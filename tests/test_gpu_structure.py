"""edge_index -> row structure, degree and normalisation: BIT-EXACT against the integer oracle
(oracle/port.py csr_oracle = stable argsort + bincount + cumsum) and torch CPU."""
import numpy as np
import pytest
import torch

from meta_gcn_b200 import ops
from meta_gcn_b200.data import synth_botnet_graph
from oracle import port
from util import assert_bitexact, check_structure, csr_numpy

pytestmark = pytest.mark.gpu
DEV = "cuda"


def build(ei_np, n, by, mode, hub_t=256):
    ei = torch.from_numpy(np.ascontiguousarray(ei_np)).long().to(DEV)
    return csr_numpy(ops.csr_build_impl(ei, n, by, mode, hub_t))


def check_against_oracle(ei_np, n, by, mode, hub_t=256):
    check_structure(build(ei_np, n, by, mode, hub_t), *port.csr_oracle(ei_np, n, by, mode), hub_t)


@pytest.mark.parametrize("n,e", [(1, 1), (5, 0), (7, 3), (100, 4095), (100, 4096), (100, 4097), (300, 8193),
                                 (1000, 50000), (70000, 200000), (300000, 100000)])
@pytest.mark.parametrize("by", [0, 1])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_csr_build_random(n, e, by, mode):
    rng = np.random.default_rng(n * 31 + e)
    ei = rng.integers(0, n, size=(2, e))
    check_against_oracle(ei, n, by, mode)


def test_csr_build_empty_graph():
    b = build(np.zeros((2, 0), np.int64), 0, 1, 0)
    assert b.rowptr.tolist() == [0] and b.hub_count[0] == 0
    b = build(np.zeros((2, 0), np.int64), 4, 1, 2)
    assert b.rowptr.tolist() == [0, 1, 2, 3, 4] and b.nbr.tolist() == [0, 1, 2, 3]
    assert b.order.tolist() == [0, 1, 2, 3]


def test_csr_build_hubs_and_duplicates():
    # star with duplicated spokes: one row of 5000 entries, stable order must keep duplicates apart
    n = 600
    spokes = np.tile(np.arange(1, 501), 10)
    ei = np.stack([spokes, np.zeros_like(spokes)])
    ei = np.concatenate([ei, ei[::-1]], axis=1)
    for by in (0, 1):
        check_against_oracle(ei, n, by, 0, hub_t=128)
        check_against_oracle(ei, n, by, 2, hub_t=128)


def test_csr_build_flags_out_of_range_indices():
    ei = np.array([[0, 1, 9], [1, 0, 2]])
    b = build(ei, 3, 1, 0)
    assert b.bad[0] == 1
    assert b.rowptr[-1] == 2  # offending edge dropped
    ei = np.array([[0, -1], [1, 0]])
    assert build(ei, 3, 0, 0).bad[0] == 1


def test_csr_build_botnet_graph_both_orders():
    g = synth_botnet_graph(seed=1, num_nodes=20000, edge_entries=220000, evil=1500)
    n = 20000
    for by in (0, 1):
        check_against_oracle(g["edge_index"], n, by, 0)
    # grouped by source, the preprocessed file is already in row order apart from the appended
    # loops (SURVEY.md §8 a12): every row is its sorted prefix segment followed by its loop
    b = build(g["edge_index"], n, 0, 0)
    e = g["edge_index"].shape[1]
    last = b.perm[b.rowptr[1:] - 1]
    assert (last == e - n + np.arange(n)).all()


def test_degree_and_norm_bitexact():
    g = synth_botnet_graph(seed=2, num_nodes=5000, edge_entries=60000, evil=300)
    n = 5000
    ei = torch.from_numpy(g["edge_index"]).to(DEV)
    rowptr = ops.csr_build_impl(ei, n, 0, 0, 256).rowptr
    deg = ops.degree_impl(rowptr)
    assert_bitexact(deg, g["x"][:, 1], "out-degree")            # data_add_degree.py:60-63
    for mode, p in ((0, -0.5), (1, -1.0)):
        dis = ops.gcn_norm_impl(deg, mode)
        ref = torch.from_numpy(g["x"][:, 1]).pow(p)             # gcn_base_models.py:128-131
        ref[ref == float("inf")] = 0
        assert_bitexact(dis, ref, f"dis mode {mode}")
    # every degree value 0..100000 (0 -> inf -> 0)
    d = torch.arange(0, 100001, dtype=torch.float32)
    for mode, p in ((0, -0.5), (1, -1.0)):
        ref = d.pow(p)
        ref[ref == float("inf")] = 0
        assert_bitexact(ops.gcn_norm_impl(d.to(DEV), mode), ref, f"all degrees mode {mode}")


def test_weighted_degree_and_edge_value_permutation():
    rng = np.random.default_rng(5)
    n, e = 400, 5000
    ei_np = rng.integers(0, n, size=(2, e))
    ew = torch.rand(e) + 0.5
    ei = torch.from_numpy(ei_np).to(DEV)
    csr = ops.csr_build_impl(ei, n, 0, 0, 256)
    wd = ops.weighted_degree_impl(csr, ew.to(DEV), 1.0)
    ref = port.scatter_rows("add", ew, torch.from_numpy(ei_np[0]), n)   # gcn_base_models.py:126
    assert_bitexact(wd, ref, "weighted degree")
    pv = ops.permute_edge_values_impl(csr, ew.to(DEV), 1.0)
    assert_bitexact(pv, ew[csr.perm.cpu().long()], "edge values in row order")
    # with appended loops (GCNConv.norm: loop weight = fill value)
    csr = ops.csr_build_impl(ei, n, 0, 2, 256)
    wd = ops.weighted_degree_impl(csr, ew.to(DEV), 2.0)
    keep = ei_np[0] != ei_np[1]
    ei_l = np.concatenate([ei_np[:, keep], np.stack([np.arange(n)] * 2)], axis=1)
    w_l = torch.cat([ew[torch.from_numpy(keep)], torch.full((n,), 2.0)])
    assert_bitexact(wd, port.scatter_rows("add", w_l, torch.from_numpy(ei_l[0]), n), "weighted degree + loops")


def test_batch_to_offsets():
    sizes = [3, 0, 5, 1, 0, 0, 7]
    batch = torch.cat([torch.full((s,), i, dtype=torch.long) for i, s in enumerate(sizes)]).to(DEV)
    off = ops.batch_to_offsets_impl(batch, len(sizes))
    assert off.cpu().tolist() == np.concatenate([[0], np.cumsum(sizes)]).tolist()


def test_edge_symmetry_fingerprint_and_structure_reuse():
    """mgcn_edge_fingerprint: symmetric edge multisets (the reference's undirected botnet data,
    data_procs/undirected.py:6-35) are recognised, any asymmetry is not; for a symmetric list the plain
    transposed structure is the forward one and the aggregation results agree with the by-source build."""
    from meta_gcn_b200 import graph as G
    g = synth_botnet_graph(seed=3, num_nodes=5000, edge_entries=40000, evil=300)
    ei = torch.from_numpy(np.ascontiguousarray(g["edge_index"])).long().to(DEV)
    assert ops.edge_symmetry_impl(ei) is True
    ei2 = ei.clone()
    ei2[1, 17] = (ei2[1, 17] + 1) % 5000            # one endpoint changed
    assert ops.edge_symmetry_impl(ei2) is False
    dup = torch.cat([ei, ei[:, :1]], 1)             # one direction duplicated: multiplicities differ
    assert ops.edge_symmetry_impl(dup) is (bool(ei[0, 0] == ei[1, 0]))
    assert ops.edge_symmetry_impl(torch.zeros(2, 0, dtype=torch.int64, device=DEV)) is True
    gs = G.GraphStructure(ei, 5000)
    # (this list is also in (src,dst) order: the plain structures are then the sort-free by-source build)
    assert gs.symmetric and gs.bwd_plain is gs.fwd_plain
    G.USE_PRESORTED = False
    try:
        gsu = G.GraphStructure(ei, 5000)
        assert gsu.symmetric and gsu.bwd_plain is gsu.fwd and gsu._bwd is None
    finally:
        G.USE_PRESORTED = True
    x = torch.randn(5000, 32, device=DEV)
    a = ops.aggregate_prescaled_impl(gs.bwd_plain, x, None, 0, None, None, 0)
    b = ops.aggregate_prescaled_impl(gs.bwd, x, None, 0, None, None, 0)
    assert gs.bwd_plain is gs.bwd                   # once built, the exact by-source structure is used
    torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-5)
    assert_bitexact(gs.out_degree().cpu().numpy(), np.diff(gs.bwd.rowptr.cpu().numpy()).astype(np.float32), "deg")
    gs2 = G.GraphStructure(ei2, 5000)
    assert not gs2.symmetric and gs2.bwd_plain is gs2.bwd


def test_int32_edge_index_builds_the_same_structures():
    """mgcn_csr_build_i32 / mgcn_edge_fingerprint_i32: an edge_index held as int32 (half the host -> device bytes)
    gives bit-identical structures, symmetry verdict and model output as the reference's int64"""
    from meta_gcn_b200 import data as D
    from meta_gcn_b200 import ops as O
    from meta_gcn_b200.gcn_meta.models import GCNModel
    g = D.synth_botnet_graph(seed=3, num_nodes=20000, edge_entries=200000, evil=1000)
    ei64 = torch.from_numpy(g["edge_index"]).to("cuda")
    ei32 = ei64.to(torch.int32)
    n = g["x"].shape[0]
    for by in (0, 1):
        for loop_mode in (0, 1, 2):
            a = O.csr_build_impl(ei64, n, by, loop_mode)
            b = O.csr_build_impl(ei32, n, by, loop_mode)
            # (hub table slots, and with them the segment tasks, are claimed in arbitrary order by every build)
            for name in ("rowptr", "nbr", "perm", "order", "hub_count", "seg_count"):
                assert torch.equal(getattr(a, name), getattr(b, name)), (by, loop_mode, name)
    assert O.edge_symmetry_impl(ei32) == O.edge_symmetry_impl(ei64) is True
    torch.manual_seed(0)
    model = GCNModel(in_channels=1, enc_sizes=[32] * 3, num_classes=2, residual_hop=1, dropout=0.0, final_type="proj",
                     deg_norm="sm", aggr="add", bias=False).to("cuda").eval()
    x = torch.from_numpy(g["x"]).to("cuda")
    with torch.no_grad():
        o64 = model(x[:, 0:1].contiguous(), ei64, deg_K=x[:, 1].contiguous())
        o32 = model(x[:, 0:1].contiguous(), ei32, deg_K=x[:, 1].contiguous())
    assert torch.equal(o64, o32)


@pytest.mark.parametrize("case", ["botnet", "sorted", "sorted_dups", "sorted_asym", "unsorted"])
@pytest.mark.parametrize("dtype", [torch.int64, torch.int32])
def test_presorted_build_equals_the_sorting_build(case, dtype):
    """mgcn_edge_layout + mgcn_csr_build_presorted: a list already in (src,dst) order (optionally + the N trailing self
    loops of data_procs/loop.py:13-17) is grouped without a sort — rowptr / nbr / perm bit-identical to the radix-sort
    build, by source always, by target when the list is symmetric"""
    from meta_gcn_b200 import data as D
    from meta_gcn_b200 import graph as G
    from meta_gcn_b200 import ops as O
    rng = np.random.default_rng(11)
    n = 5000
    if case == "botnet":
        g = D.synth_botnet_graph(seed=5, num_nodes=n, edge_entries=60000, evil=300)
        ei = g["edge_index"]
    else:
        src, dst = rng.integers(0, n, 40000), rng.integers(0, n, 40000)
        if case != "sorted_asym":
            src, dst = np.concatenate([src, dst]), np.concatenate([dst, src])     # symmetric multiset
        if case == "sorted_dups":
            src, dst = np.concatenate([src, src[:5000], dst[:5000]]), np.concatenate([dst, dst[:5000], src[:5000]])
        elif case != "unsorted":
            key = np.unique(src * n + dst)
            src, dst = key // n, key % n
        if case != "unsorted":
            o = np.lexsort((dst, src))
            src, dst = src[o], dst[o]
        ei = np.stack([src, dst])
    ei = torch.from_numpy(ei.astype(np.int64)).to("cuda").to(dtype)
    facts = O.edge_layout_impl(ei, n)
    want = {"botnet": 2, "sorted": 1, "sorted_dups": 5, "sorted_asym": 1, "unsorted": 0}[case]
    assert facts["layout"] == want, facts
    assert facts["symmetric"] == (case != "sorted_asym")
    for by in (0, 1):
        ref = O.csr_build_impl(ei, n, by, 0)
        if want and (by == 0 or facts["symmetric"]):
            fast = O.csr_build_impl(ei, n, by, 0, layout=want)
            for name in ("rowptr", "nbr", "perm", "order"):
                assert torch.equal(getattr(fast, name), getattr(ref, name)), (case, by, name)
    if want and facts["symmetric"]:
        # sorted + symmetric: the by-source rows ARE the by-target rows, entry for entry (GraphStructure.fwd_plain)
        a0, a1 = O.csr_build_impl(ei, n, 0, 0), O.csr_build_impl(ei, n, 1, 0)
        assert torch.equal(a0.rowptr, a1.rowptr) and torch.equal(a0.nbr, a1.nbr)
        gsp = G.GraphStructure(ei, n)
        assert gsp.fwd_plain is gsp.bwd and gsp._fwd is None
    # the structure cache picks the sort-free path on its own and the model result does not change
    gs = G.GraphStructure(ei, n)
    x = torch.randn(n, 32, device="cuda")
    out_fast = O.aggregate_prescaled_impl(gs.fwd_plain, x)
    assert torch.equal(out_fast, O.aggregate_prescaled_impl(gs.fwd, x))
    G.USE_PRESORTED = False
    try:
        out_ref = O.aggregate_prescaled_impl(G.GraphStructure(ei, n).fwd, x)
    finally:
        G.USE_PRESORTED = True
    assert torch.equal(out_fast, out_ref)


@pytest.mark.parametrize("dtype", [torch.int64, torch.int32])
def test_ordered_batch_is_grouped_without_a_sort(dtype):
    """a BATCH of graphs in the reference's preprocessed layout (Batch.from_data_list of sorted-unique lists with their
    loops appended, dataloader.py:11 + data_procs/loop.py:13-17): GraphBatch.structure() hands the batch boundaries to
    the structure, the per-graph order check passes, and the sort-free by-source build equals the radix-sort one"""
    from meta_gcn_b200 import data as D
    from meta_gcn_b200 import graph as G
    from meta_gcn_b200 import ops as O
    graphs = [D.synth_botnet_graph(seed=s, num_nodes=3000 + 500 * s, edge_entries=30000 + 1000 * s, evil=200) for s in range(4)]
    batch = D.GraphBatch.from_data_list(graphs)
    if dtype == torch.int32:
        batch = batch.with_int32_indices()
    batch = batch.to("cuda")
    n = batch.num_nodes
    assert O.edge_layout_impl(batch.edge_index, n)["layout"] == 0            # not ordered as ONE list ...
    gs = batch.structure()
    assert gs.facts == {"symmetric": True, "layout": 2}                       # ... but graph by graph
    assert G.structure_of(batch.edge_index, n) is gs                          # what the model classes will find
    ref0 = O.csr_build_impl(batch.edge_index, n, 0, 0)
    ref1 = O.csr_build_impl(batch.edge_index, n, 1, 0)
    for name in ("rowptr", "nbr", "perm", "order"):
        assert torch.equal(getattr(gs.bwd, name), getattr(ref0, name)), name
    assert gs.fwd_plain is gs.bwd and gs.bwd_plain is gs.bwd
    assert torch.equal(gs.fwd_plain.rowptr, ref1.rowptr) and torch.equal(gs.fwd_plain.nbr, ref1.nbr)
    for name in ("rowptr", "nbr", "perm"):                                    # the exact by-target structure still sorts
        assert torch.equal(getattr(gs.fwd, name), getattr(ref1, name)), name
    # a batch with one graph out of order falls back to the sort
    bad = [dict(g) for g in graphs]
    bad[2]["edge_index"] = np.ascontiguousarray(bad[2]["edge_index"][:, ::-1])
    bb = D.GraphBatch.from_data_list(bad).to("cuda")
    gb = bb.structure()
    assert gb.facts["layout"] == 0
    assert torch.equal(gb.bwd.nbr, O.csr_build_impl(bb.edge_index, bb.num_nodes, 0, 0).nbr)
