"""The order check (mgcn_edge_layout) and the sort-free structure build (mgcn_csr_build_presorted) against exact
references.

Every step of the botnet workload aggregates over structures built without a sort, and that build places each entry
with a closed formula that trusts the layout the order check reported.  So:
  1. the eight words of mgcn_edge_layout equal a numpy restatement of include/mgcn.h, bit for bit, and the layout /
     symmetry ops.edge_layout_impl derives from them are the ones the restatement gives;
  2. wherever GraphStructure builds without a sort, the result is bit-identical to the radix-sort build and passes the
     full structural check against the stable-argsort oracle;
  3. aggregations over GraphStructure's structures agree with an fp64 index_add_ over the edge list and are
     bit-identical to those over the sorting build; so is GCNModel on a batch of loop-free graphs.
The cases put violations on thread, block and grid-stride boundaries and at the prefix / loop junction, and cover
out-of-range ids, empty and tiny graphs, batches whose graph boundaries fall on e = 256 and e = stride, and lists of
millions of entries."""
import functools
import zlib
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from meta_gcn_b200 import _lib, ops
from meta_gcn_b200 import functional as F_mgcn
from meta_gcn_b200 import graph as G
from meta_gcn_b200.data import GraphBatch, synth_botnet_graph
from oracle import port
from util import assert_bitexact, assert_parity, check_structure, csr_numpy

gpu = pytest.mark.gpu
DEV = "cuda"
DTYPES = [torch.int64, torch.int32]
HUB_T = 16          # small, so that most cases have hub rows cut into segments
BUILD_FIELDS = ("rowptr", "nbr", "perm", "order", "hub_count", "seg_count")   # hub slots are claimed by atomics


# ------------------------------------------------------------------------------------------------
# restatement of mgcn_edge_layout (include/mgcn.h)
# ------------------------------------------------------------------------------------------------
def _mix64(z):
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xbf58476d1ce4e5b9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94d049bb133111eb)
    return z ^ (z >> np.uint64(31))


def restate_out8(ei, n, segments=None):
    """the eight uint64 words of mgcn_edge_layout for edge_index `ei` [2,E] (int32 or int64) over n nodes;
    segments = (node_off, edge_off) host lists of a batch, None for one graph.  Integer sums wrap mod 2^64."""
    s = np.asarray(ei[0]).astype(np.int64)         # int32 ids are sign-extended, as the kernel reads them
    d = np.asarray(ei[1]).astype(np.int64)
    E = s.size
    out = np.zeros(8, np.uint64)
    if E == 0:
        return out
    a, b = s.view(np.uint64), d.view(np.uint64)
    k1, k2 = np.uint64(0x9e3779b97f4a7c15), np.uint64(0xd6e8feb86659fd93)
    ab, ba = a * k1 + b, b * k1 + a
    for q, z in enumerate((ab, ba, ab ^ k2, ba ^ k2)):
        out[q] = _mix64(z).sum(dtype=np.uint64)
    e = np.arange(E, dtype=np.int64)
    if segments is None:
        n0, e0, ng, eg = (np.full(E, v, np.int64) for v in (0, 0, n, E))
    else:
        node_off, edge_off = (np.asarray(v, np.int64) for v in segments)
        g = np.searchsorted(edge_off[:-1], e, side="right") - 1         # the last graph that starts at or before e
        n0, e0 = node_off[g], edge_off[g]
        ng, eg = node_off[g + 1] - n0, edge_off[g + 1] - e0
    outside = (s < n0) | (s >= n0 + ng) | (d < n0) | (d >= n0 + ng)    # an endpoint outside its graph's node range
    ep = np.where(eg >= ng, e0 + eg - ng, -1)                           # end of the sorted prefix, -1: no such reading
    nxt = e + 1 < e0 + eg                                               # e + 1 belongs to the same graph
    s1, d1 = np.append(s[1:], 0), np.append(d[1:], 0)
    desc = nxt & ((s > s1) | ((s == s1) & (d > d1)))
    loop = n0 + e - ep
    out[4] = outside.sum() + desc.sum()
    out[5] = outside.sum() + (desc & (ep >= 0) & (e + 1 < ep)).sum()
    out[6] = (ep < 0).sum() + ((ep >= 0) & (e >= ep) & ~((s == loop) & (d == loop))).sum()
    out[7] = (nxt & (s == s1) & (d == d1)).sum()
    return out


def facts_of(w, E, n):
    """what ops.edge_layout_impl reports for the words w"""
    layout = 0
    if E > 0 and w[4] == 0:
        layout = 1
    elif E >= n > 0 and w[5] == 0 and w[6] == 0:
        layout = 2
    if layout and w[7] != 0:
        layout |= 4
    return {"symmetric": bool(w[0] == w[1] and w[2] == w[3]), "layout": layout}


def test_restatement_on_hand_made_lists():
    """the restatement itself, on lists small enough to count by hand"""
    loops = np.array([[0, 1, 2], [0, 1, 2]])
    prefix = np.array([[0, 0, 1, 2, 2], [1, 2, 0, 0, 1]])
    assert restate_out8(np.concatenate([prefix, loops], 1), 3)[4:].tolist() == [1, 0, 0, 0]
    # the prefix/loop junction is not a pair of the prefix; a descent just before it is
    swapped = np.concatenate([prefix[:, [0, 1, 2, 4, 3]], loops], 1)
    assert restate_out8(swapped, 3)[4:].tolist() == [2, 1, 0, 0]
    assert restate_out8(np.concatenate([prefix, loops[:, [0, 2, 1]]], 1), 3)[4:].tolist() == [2, 0, 2, 0]
    # E < N: no "+ loops" reading, every entry counts in [6]; repeated entries in [7]
    assert restate_out8(np.array([[0, 0, 1], [1, 1, 0]]), 5)[4:].tolist() == [0, 0, 3, 1]
    # an id outside [0, N) counts once per entry in [4] and [5]
    assert restate_out8(np.array([[0, 1, 1, 0, 1], [1, 0, 2, 0, 1]]), 2)[4:].tolist() == [2, 1, 0, 0]
    assert restate_out8(np.array([[-1, 0, 1], [0, 1, 0]]), 2)[4:].tolist() == [1, 1, 2, 0]
    # a batch: pairs across a graph boundary are not compared; an endpoint in the next graph is a violation;
    # an empty graph and a graph without entries count nothing
    batch = np.array([[0, 1, 0, 1, 4, 5], [1, 0, 0, 1, 4, 2]])
    w = restate_out8(batch, 6, ([0, 2, 2, 4, 6], [0, 4, 4, 4, 6]))
    assert w[4:].tolist() == [2, 1, 1, 0]
    assert restate_out8(batch, 6)[4:].tolist() == [1, 0, 5, 0]      # read as one graph
    # symmetric multisets: equal fingerprints, in any order; an asymmetric one: not
    sym = np.array([[0, 1, 1, 2, 2], [1, 0, 2, 1, 2]])
    assert facts_of(restate_out8(sym, 3), 5, 3)["symmetric"]
    assert facts_of(restate_out8(sym[:, ::-1], 3), 5, 3)["symmetric"]
    assert not facts_of(restate_out8(sym[:, 1:], 3), 4, 3)["symmetric"]


def test_restatement_of_a_botnet_graph():
    """the reference's preprocessed layout: sorted unique prefix + N loops -> one descent, at the junction"""
    g = synth_botnet_graph(seed=5, num_nodes=5000, edge_entries=60000)
    w = restate_out8(g["edge_index"], 5000)
    assert w[4:].tolist() == [1, 0, 0, 0]
    assert facts_of(w, g["edge_index"].shape[1], 5000) == {"symmetric": True, "layout": 2}


# ------------------------------------------------------------------------------------------------
# cases: edge lists over n nodes, with the layout they are built to have
# ------------------------------------------------------------------------------------------------
def grid_stride(E):
    """entries between two iterations of one thread of k_edge_order_check (its launch: blocks of 256 threads, one block
    per 2048 entries, at most 8 blocks an SM)"""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return min(-(-E // 2048), 8 * sms) * 256


def _sorted(src, dst):
    o = np.lexsort((dst, src))
    return np.stack([src[o], dst[o]]).astype(np.int64)


def _unique_sorted(rng, n, m, symmetric):
    """about m distinct (src, dst) entries in (src, dst) order; symmetric: with every mirror, without loops"""
    a, b = rng.integers(0, n, m), rng.integers(0, n, m)
    if symmetric:
        keep = a != b
        key = np.unique(np.concatenate([a[keep] * n + b[keep], b[keep] * n + a[keep]]))
    else:
        key = np.unique(a * n + b)
    return np.stack([key // n, key % n])


def _exact_sorted(rng, n, m):
    """exactly m distinct (src, dst) entries in (src, dst) order"""
    key = np.sort(rng.choice(n * n, size=m, replace=False))
    return np.stack([key // n, key % n]).astype(np.int64)


def _loops(n):
    return np.stack([np.arange(n), np.arange(n)]).astype(np.int64)


def _botnet(seed, n, e):
    return synth_botnet_graph(seed=seed, num_nodes=n, edge_entries=e, evil=n // 16)["edge_index"]


def _swap(ei, p):
    ei = ei.copy()
    ei[:, [p, p + 1]] = ei[:, [p + 1, p]]
    return ei


def _last_of_row(ei, stop, s):
    return int(np.nonzero(ei[0, :stop] == s)[0][-1])


SINGLE = ["sorted_sym", "sorted_asym", "sorted_dups", "botnet", "botnet_dups", "prefix_self_loops", "loops_only",
          "one_node", "fewer_entries_than_nodes", "random",
          "inv_0", "inv_255", "inv_256", "inv_stride-1", "inv_stride", "inv_prefix_end", "inv_junction", "inv_last",
          "loop_wrong", "loops_swapped", "loop_missing",
          "id_N_botnet", "id_neg_botnet", "id_N_sorted", "id_neg_sorted",
          "big", "big_inv_stride", "big_inv_prefix_end"]
BATCH = ["b_botnet", "b_loop_free", "b_empty_graphs", "b_graph_without_entries", "b_single_node",
         "b_fewer_entries", "b_fewer_entries_loop_free", "b_endpoint_in_next", "b_endpoint_in_next_loop_free",
         "b_bounds", "b_bounds_loop_free"]
CASES = SINGLE + BATCH


def _single(name):
    """(edge_index [2,E] int64, n, layout)"""
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    n = 3000
    if name == "sorted_sym":
        return _unique_sorted(rng, n, 20000, True), n, 1
    if name == "sorted_asym":
        return _unique_sorted(rng, n, 40000, False), n, 1
    if name == "sorted_dups":
        p = _unique_sorted(rng, n, 20000, True)
        k = rng.choice(p.shape[1], 4000)
        return _sorted(np.concatenate([p[0], p[0, k], p[1, k]]), np.concatenate([p[1], p[1, k], p[0, k]])), n, 5
    if name == "botnet":
        return _botnet(5, 5000, 60000), 5000, 2
    if name == "botnet_dups":       # repeated prefix entries (both directions) + the loops: layout 6
        n, ei = 5000, _botnet(6, 5000, 60000)
        p = ei[:, :-n]
        k = rng.choice(p.shape[1], 6000)
        p = _sorted(np.concatenate([p[0], p[0, k], p[1, k]]), np.concatenate([p[1], p[1, k], p[0, k]]))
        return np.concatenate([p, _loops(n)], 1), n, 6
    if name == "prefix_self_loops":  # (i, i) inside the prefix too, the last one (n-1, n-1) right before (0, 0)
        n, ei = 5000, _botnet(7, 5000, 60000)
        own = np.concatenate([[0, n - 1], rng.choice(n, 300, replace=False)])
        own = np.unique(own)
        p = _sorted(np.concatenate([ei[0, :-n], own]), np.concatenate([ei[1, :-n], own]))
        return np.concatenate([p, _loops(n)], 1), n, 2
    if name == "loops_only":        # E == N
        return _loops(n), n, 1
    if name == "one_node":
        return np.zeros((2, 1), np.int64), 1, 1
    if name == "fewer_entries_than_nodes":
        return _unique_sorted(rng, 10000, 3000, False), 10000, 1
    if name == "random":
        return rng.integers(0, n, (2, 40000)), n, 0
    if name.startswith("inv_"):     # one swapped pair of a botnet list (grid not at its cap)
        n, ei = 20000, _botnet(8, 20000, 300000)
        E = ei.shape[1]
        st = grid_stride(E)
        p = {"inv_0": 0, "inv_255": 255, "inv_256": 256, "inv_stride-1": st - 1, "inv_stride": st,
             "inv_prefix_end": E - n - 2, "inv_junction": E - n - 1, "inv_last": E - 2}[name]
        return _swap(ei, p), n, 0
    if name in ("loop_wrong", "loops_swapped", "loop_missing"):
        n, ei = 5000, _botnet(9, 5000, 60000)
        j = ei.shape[1] - n
        ei = ei.copy()
        if name == "loop_wrong":
            ei[1, j + 1234] += 1                     # (i, i+1) where (i, i) belongs
        elif name == "loops_swapped":
            ei = _swap(ei, j + 77)
        else:
            ei = np.delete(ei, j + 4321, axis=1)
        return ei, n, 0
    if name.startswith("id_"):      # one id outside [0, N) in an otherwise ordered list
        if name.endswith("botnet"):
            n, ei = 5000, _botnet(10, 5000, 60000)
            stop = ei.shape[1] - n
        else:
            ei = _unique_sorted(rng, n, 40000, False)
            stop = ei.shape[1]
        ei = ei.copy()
        if name.startswith("id_N"):
            ei[1, _last_of_row(ei, stop, 1234)] = n  # a target N at the end of a source's row
        else:
            ei[0, 0] = -1                            # a source -1 first in the list
        return ei, n, 0
    if name.startswith("big"):      # millions of entries: the grid at its cap, several strides per list
        n, ei = 150000, _botnet(11, 150000, 2_600_000)
        E = ei.shape[1]
        if name == "big":
            return ei, n, 2
        return _swap(ei, grid_stride(E) if name == "big_inv_stride" else E - n - 2), n, 0
    raise KeyError(name)


def _assemble(graphs):
    """[(local edge_index, n_g)] -> (edge_index, n, (node_off, edge_off)) as Batch.from_data_list lays them out"""
    parts, node_off, edge_off = [], [0], [0]
    for ei, ng in graphs:
        parts.append(np.asarray(ei, np.int64) + node_off[-1])
        node_off.append(node_off[-1] + ng)
        edge_off.append(edge_off[-1] + parts[-1].shape[1])
    return np.concatenate(parts, 1), node_off[-1], (node_off, edge_off)


def _batch(name):
    """(edge_index, n, segments, layout)"""
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    loop_free = name.endswith("loop_free")
    gs = [(_botnet(20 + k, 2000 + 700 * k, 20000 + 6000 * k), 2000 + 700 * k) for k in range(3)]
    if loop_free:
        gs = [(ei[:, :-ng], ng) for ei, ng in gs]
    if name in ("b_botnet", "b_loop_free"):
        return (*_assemble(gs), 1 if loop_free else 2)
    if name == "b_empty_graphs":
        empty = (np.zeros((2, 0), np.int64), 0)
        return (*_assemble([empty, gs[0], empty, empty, gs[1], empty]), 2)
    if name == "b_graph_without_entries":
        return (*_assemble([gs[0], (np.zeros((2, 0), np.int64), 50), gs[1]]), 2)
    if name == "b_single_node":
        return (*_assemble([gs[0], (np.zeros((2, 1), np.int64), 1), gs[1]]), 2)
    if name.startswith("b_fewer_entries"):
        few = (_unique_sorted(rng, 500, 200, False), 500)
        return (*_assemble([gs[0], few, gs[1]]), 1 if loop_free else 0)
    if name.startswith("b_endpoint_in_next"):
        ei, ng = gs[0]
        ei = ei.copy()
        ei[1, ei.shape[1] - (1 if loop_free else ng + 1)] = ng   # the last prefix entry points at node 0 of graph 1
        return (*_assemble([(ei, ng)] + gs[1:]), 0)
    if name.startswith("b_bounds"):   # graph boundaries at e = 256 and e = stride
        E = 400_000
        st = grid_stride(E)
        sizes = [(16, 256), (4000, st - 256), (20000, E - st)]
        out = []
        for ng, m in sizes:
            if loop_free:
                out.append((_exact_sorted(rng, ng, m), ng))
            else:
                out.append((np.concatenate([_exact_sorted(rng, ng, m - ng), _loops(ng)], 1), ng))
        ei, n, seg = _assemble(out)
        assert seg[1][1] == 256 and seg[1][2] == st
        return ei, n, seg, 1 if loop_free else 2
    raise KeyError(name)


@functools.lru_cache(maxsize=None)
def case(name):
    if name in BATCH:
        ei, n, seg, layout = _batch(name)
    else:
        (ei, n, layout), seg = _single(name), None
    ei = np.ascontiguousarray(ei, dtype=np.int64)
    in_range = bool(ei.size == 0 or (ei.min() >= 0 and ei.max() < n))
    ei.setflags(write=False)
    return SimpleNamespace(ei=ei, n=n, seg=seg, layout=layout, in_range=in_range)


def on_device(c, dtype):
    ei = torch.from_numpy(c.ei.copy()).to(dtype).to(DEV)
    segs = None if c.seg is None else tuple(torch.tensor(v, dtype=torch.int32, device=DEV) for v in c.seg)
    return ei, segs


def device_out8(ei, n, segs):
    """the raw words of mgcn_edge_layout"""
    out = torch.empty(8, dtype=torch.int64, device=ei.device)
    lib = _lib.load()
    fn = lib.mgcn_edge_layout if ei.dtype == torch.int64 else lib.mgcn_edge_layout_i32
    g = 0 if segs is None else segs[0].numel() - 1
    _lib.check(fn(ei.data_ptr(), ei.size(1), int(n), g, segs[0].data_ptr() if g else None,
                  segs[1].data_ptr() if g else None, out.data_ptr(), torch.cuda.current_stream().cuda_stream))
    return out.cpu().numpy().view(np.uint64)


# ------------------------------------------------------------------------------------------------
# 1. the order check, word for word
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["int64", "int32"])
@pytest.mark.parametrize("name", CASES)
def test_edge_layout_words_equal_the_restatement(name, dtype):
    c = case(name)
    ei, segs = on_device(c, dtype)
    host = ei.cpu().numpy()
    want = restate_out8(host, c.n, c.seg)
    assert device_out8(ei, c.n, segs).tolist() == want.tolist()
    facts = facts_of(want, host.shape[1], c.n)
    assert facts["layout"] == c.layout, (facts, c.layout)
    assert ops.edge_layout_impl(ei, c.n, segs) == facts
    if c.seg is None:       # the same list described as a batch of one graph
        one = ([0, c.n], [0, host.shape[1]])
        assert restate_out8(host, c.n, one).tolist() == want.tolist()
        assert device_out8(ei, c.n, on_device(SimpleNamespace(ei=c.ei, seg=one), dtype)[1]).tolist() == want.tolist()


# ------------------------------------------------------------------------------------------------
# 2. the sort-free build equals the sorting build
# ------------------------------------------------------------------------------------------------
def _equal_builds(got, ref, what):
    for field in BUILD_FIELDS:
        assert torch.equal(getattr(got, field), getattr(ref, field)), (what, field)
    assert torch.equal(got.bad, ref.bad), what


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["int64", "int32"])
@pytest.mark.parametrize("name", CASES)
def test_sort_free_build_equals_the_sorting_build(name, dtype):
    """for each grouping, the structure GraphStructure builds and, where the layout allows one, the sort-free build
    called directly: bit-identical to the radix-sort build, and structurally exact against the oracle.  A list with an
    id outside [0, N) must take the sorting build, which drops that entry and raises `bad`; only the integer arrays of
    such builds are compared."""
    c = case(name)
    ei, segs = on_device(c, dtype)
    facts = ops.edge_layout_impl(ei, c.n, segs)
    gs = G.GraphStructure(ei, c.n, hub_threshold=HUB_T, segments=c.seg)
    for by in (0, 1):
        ref = ops.csr_build_impl(ei, c.n, by, 0, HUB_T)
        builds = {"GraphStructure": gs.bwd if by == 0 else gs.fwd}
        layout = facts["layout"] if by == 0 or (facts["symmetric"] and c.seg is None) else 0
        if layout:
            builds["sort-free"] = ops.csr_build_impl(ei, c.n, by, 0, HUB_T, layout=layout,
                                                     segments=segs if layout & 3 == 2 else None)
        oracle = port.csr_oracle(c.ei, c.n, by, 0) if c.in_range else None
        for what, got in builds.items():
            _equal_builds(got, ref, (what, by, layout))
            if oracle is not None:
                check_structure(csr_numpy(got), *oracle, HUB_T)
        assert int(ref.bad.item()) == (0 if c.in_range else 1)


# ------------------------------------------------------------------------------------------------
# 3. through GraphStructure: aggregations and the model
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["int64", "int32"])
@pytest.mark.parametrize("name", [n for n in CASES if not n.startswith("id_")])
def test_structures_aggregate_like_the_edge_list(name, dtype, monkeypatch):
    """aggregate_prescaled over fwd_plain / bwd_plain = fp64 index_add_ over the edge list (target / source rows), and
    bit-identical to the same aggregation over the structures built with a sort"""
    c = case(name)
    assert c.in_range
    ei, _ = on_device(c, dtype)
    x = torch.randn(c.n, 32, generator=torch.Generator().manual_seed(1)).to(DEV)
    x64 = x.double().cpu()
    src, dst = (torch.from_numpy(v.copy()) for v in c.ei)
    want = {"fwd": torch.zeros(c.n, 32, dtype=torch.float64).index_add_(0, dst, x64[src]),
            "bwd": torch.zeros(c.n, 32, dtype=torch.float64).index_add_(0, src, x64[dst])}

    def aggregate():
        gs = G.GraphStructure(ei, c.n, hub_threshold=HUB_T, segments=c.seg)
        return {"fwd": ops.aggregate_prescaled_impl(gs.fwd_plain, x), "bwd": ops.aggregate_prescaled_impl(gs.bwd_plain, x)}

    got = aggregate()
    monkeypatch.setattr(G, "USE_PRESORTED", False)
    sorted_ = aggregate()
    for k in ("fwd", "bwd"):
        assert_parity(got[k], want[k], f"{name} {k}")
        assert_bitexact(got[k], sorted_[k], f"{name} {k} against the sorting build")


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["int64", "int32"])
def test_loop_free_batch_trains_like_the_sorting_build(dtype, monkeypatch):
    """a batch of graphs that are each sorted but have no appended loops (layout 1 graph by graph): GraphStructure
    builds its by-source structure as one list, and GCNModel's forward and backward are bit-identical to the run on
    structures built with a sort"""
    from meta_gcn_b200.gcn_meta.models import GCNModel
    graphs = []
    for s in range(3):
        g = synth_botnet_graph(seed=30 + s, num_nodes=3000 + 900 * s, edge_entries=40000 + 9000 * s, evil=200)
        n = g["x"].shape[0]
        graphs.append({"x": g["x"], "edge_index": g["edge_index"][:, :-n], "y": g["y"]})
    batch = GraphBatch.from_data_list(graphs)
    if dtype == torch.int32:
        batch = batch.with_int32_indices()
    batch = batch.to(DEV)
    x = torch.randn(batch.num_nodes, 1, generator=torch.Generator().manual_seed(2)).to(DEV)
    y = batch.y.long()
    cfg = dict(in_channels=1, enc_sizes=[32] * 4, num_classes=2, residual_hop=1, dropout=0.0, final_type="proj",
               deg_norm="sm", aggr="add", bias=False)

    def run():
        G.clear_structure_cache()
        gs = batch.structure()
        assert gs.facts == {"symmetric": True, "layout": 1}
        torch.manual_seed(0)
        model = GCNModel(**cfg).to(DEV)
        out = model(x, batch.edge_index)
        F_mgcn.cross_entropy(out, y).backward()
        torch.cuda.synchronize()
        return [out.detach()] + [p.grad for p in model.parameters()]

    try:
        got = run()
        monkeypatch.setattr(G, "USE_PRESORTED", False)
        ref = run()
    finally:
        G.clear_structure_cache()
    for k, (a, b) in enumerate(zip(got, ref)):
        assert_bitexact(a, b, f"output / gradient {k}")


# ------------------------------------------------------------------------------------------------
# 4. at bench scale
# ------------------------------------------------------------------------------------------------
@gpu
def test_bench_scale_batch():
    """int32 batch of full-size botnet graphs made as bench.py makes them: the words equal the restatement and the
    sort-free by-source build equals the sorting build"""
    graphs = [synth_botnet_graph(seed=s, num_nodes=143107, edge_entries=1_500_000, evil=min(10000, 143107 // 14))
              for s in range(4)]
    batch = GraphBatch.from_data_list(graphs).with_int32_indices().to(DEV)
    n, seg = batch.num_nodes, (batch.slices_x, batch.slices_e)
    ei = batch.edge_index
    segs = tuple(torch.tensor(v, dtype=torch.int32, device=DEV) for v in seg)
    host = ei.cpu().numpy()
    assert host.shape[1] > 10 * grid_stride(host.shape[1])
    want = restate_out8(host, n, seg)
    assert device_out8(ei, n, segs).tolist() == want.tolist()
    assert facts_of(want, host.shape[1], n) == {"symmetric": True, "layout": 2}
    fast = ops.csr_build_impl(ei, n, 0, 0, layout=2, segments=segs)
    _equal_builds(fast, ops.csr_build_impl(ei, n, 0, 0), "bench batch")
    check_structure(csr_numpy(fast), *port.csr_oracle(host, n, 0, 0), ops.DEFAULT_HUB_THRESHOLD)
