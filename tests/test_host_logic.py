"""Host-side logic that needs no GPU: batching contract, synthetic workloads, model mirrors'
parameter layout, CUDA-only refusal, fake-tensor tracing of the torch.library ops."""
import numpy as np
import pytest
import torch

from meta_gcn_b200 import data as D
from meta_gcn_b200 import dist as mdist
from oracle import port, use_shim
from util import assert_bitexact, golden, params_of


def test_graphbatch_matches_from_data_list_contract():
    use_shim()
    from torch_geometric.data import Batch, Data
    rng = np.random.default_rng(0)
    graphs = [D.synth_tu_graph(rng) for _ in range(5)]
    ours = D.GraphBatch.from_data_list(graphs)
    ref = Batch.from_data_list([Data(x=torch.from_numpy(g["x"]), edge_index=torch.from_numpy(g["edge_index"]),
                                     y=torch.from_numpy(g["y"])) for g in graphs])
    assert_bitexact(ours.x, ref.x, "x")
    assert_bitexact(ours.edge_index, ref.edge_index, "edge_index")
    assert_bitexact(ours.batch, ref.batch, "batch")
    assert_bitexact(ours.y, ref.y, "y")
    assert ours.slices_x == ref.__slices__["x"]
    assert ours.num_graphs == ref.num_graphs == 5
    assert (np.diff(ours.batch.numpy()) >= 0).all()


def test_botnet_generator_follows_reference_preprocessing_order():
    g = D.synth_botnet_graph(seed=3, num_nodes=3000, edge_entries=30000, evil=300)
    ei, n = g["edge_index"], 3000
    e = ei.shape[1]
    assert abs(e - 30000) <= 300
    # non-loop prefix: strictly increasing (src,dst) keys = sort-unique (undirected.py:6-16)
    key = ei[0, :e - n] * n + ei[1, :e - n]
    assert (np.diff(key) > 0).all() and (ei[0, :e - n] != ei[1, :e - n]).all()
    # loops appended at the end, in node order (loop.py:13-17)
    assert (ei[0, e - n:] == np.arange(n)).all() and (ei[1, e - n:] == np.arange(n)).all()
    # symmetric
    fwd = set(map(tuple, ei[:, :e - n].T.tolist()))
    assert all((b, a) in fwd for a, b in list(fwd)[:2000])
    # x = [1, out-degree incl. loop] (data_add_degree.py:45-65)
    assert_bitexact(g["x"][:, 1], port.out_degree(ei, n), "deg")
    assert (g["x"][:, 0] == 1).all() and g["y"].sum() == 300
    # the oracle's preprocessing reproduces the generator's ordering from the raw undirected pairs
    again = port.append_self_loops(port.to_undirected(ei[:, :e - n], n), n)
    assert_bitexact(again, ei, "ordering")
    # determinism
    g2 = D.synth_botnet_graph(seed=3, num_nodes=3000, edge_entries=30000, evil=300)
    assert_bitexact(g2["edge_index"], ei, "seeded")


def test_model_mirror_has_reference_parameter_layout():
    from meta_gcn_b200.gcn_meta.models import GCNModel
    g = golden("gcn_meta_botnet12")
    torch.manual_seed(0)
    m = GCNModel(1, [32] * 12, 2, residual_hop=1, dropout=0.0, final_type="proj", deg_norm="sm",
                 bias=False, nodemodel="additive", edge_gate=None, aggr="add", nheads=[1] * 12, att_act="lrelu")
    ref = params_of(g)
    sd = m.state_dict()
    assert set(sd) == set(ref)
    for k in sd:
        assert_bitexact(sd[k], ref[k], k)   # same seed, same initialisers, same creation order
    assert sum(p.numel() for p in m.parameters()) == 23042


@pytest.mark.parametrize("name,cls,kw", [("kernel_gcn", "GCN", {}), ("kernel_gcn_jk", "GCNWithJK", {}),
                                         ("kernel_gin0", "GIN0", {}), ("kernel_gin", "GIN", {}),
                                         ("kernel_sage", "GraphSAGE", {})])
def test_kernel_mirrors_have_reference_parameter_layout(name, cls, kw):
    import meta_gcn_b200.kernel as K
    g = golden(name)
    seed = {"kernel_gcn": 10, "kernel_gcn_jk": 11, "kernel_gin0": 12, "kernel_gin": 13, "kernel_sage": 14}[name]
    torch.manual_seed(seed)
    net = getattr(K, cls)(D.dataset_meta(3, 2), 3, 64, **kw)
    ref = params_of(g)
    sd = net.state_dict()
    assert set(sd) == set(ref)
    for k in sd:
        assert_bitexact(sd[k], ref[k], k)


def test_unsupported_reference_options_fail_loudly():
    from meta_gcn_b200.gcn_meta.models import GCNModel, scatter_
    with pytest.raises(NotImplementedError):
        GCNModel(1, [8], 2, nodemodel="hardattention")
    assert GCNModel(1, [8], 2, nodemodel="attention", nheads=2) is not None
    assert GCNModel(1, [8], 2, edge_gate="proj") is not None    # edge gates and 'max' are built (csrc/segmax.cu)
    assert GCNModel(1, [8], 2, aggr="max") is not None
    assert GCNModel(1, [8], 2, aggr="max", edge_gate="proj") is not None   # max over gated messages: primitive seam
    with pytest.raises(RuntimeError):                           # ... and, like every op, refuses CPU tensors
        scatter_("max", torch.ones(3, 2), torch.zeros(3, dtype=torch.long))


def test_ops_refuse_cpu_tensors():
    """no CPU fallback anywhere on the product path"""
    import meta_gcn_b200.ops  # noqa: F401
    from meta_gcn_b200 import functional as F_mgcn
    from meta_gcn_b200.gcn_meta.models import GCNModel
    ei = torch.tensor([[0, 1], [1, 0]])
    with pytest.raises(RuntimeError):
        torch.ops.mgcn.csr_build(ei, 2, 0, 0, 256)
    with pytest.raises(RuntimeError):
        torch.ops.mgcn.linear(torch.ones(2, 2), torch.ones(2, 2), False, None, None, 0)
    with pytest.raises(RuntimeError):
        F_mgcn.scatter_rows(torch.ones(2, 2), ei[0], 2)
    with pytest.raises(RuntimeError):
        GCNModel(1, [8], 2)(torch.ones(2, 1), ei)


def test_layer_bwd_refuses_the_removed_mma_sync_kernel():
    """ops.gcn_layer_bwd_impl runs on tcgen05 only: tensor_memory=False is refused before any tensor is looked at"""
    from meta_gcn_b200 import ops
    t, m = torch.ones(4, 32), torch.ones(32, 32)
    with pytest.raises(ValueError, match="mma.sync"):
        ops.gcn_layer_bwd_impl(t, t, t, m, m, None, None, False, False)


def test_ops_trace_with_fake_tensors():
    import meta_gcn_b200.ops  # noqa: F401
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        ei = torch.empty(2, 100, dtype=torch.int64, device="cuda")
        csr = torch.ops.mgcn.csr_build(ei, 10, 1, 2, 256)
        assert csr[0].shape == (11,) and csr[1].shape == (110,) and csr[2].dtype == torch.int32
        x = torch.empty(10, 32, device="cuda")
        y = torch.ops.mgcn.spmm(csr, 256, x, False, None, None, None, 0, None, None, 1)
        assert y.shape == (10, 32) and y.device.type == "cuda"
        w = torch.empty(32, 16, device="cuda")
        z = torch.ops.mgcn.linear(y, w, False, None, None, 0)
        assert z.shape == (10, 16)
        dw, db = torch.ops.mgcn.linear_wgrad(y, z, False, True)
        assert dw.shape == (32, 16) and db.shape == (16,)
        off = torch.ops.mgcn.batch_to_offsets(torch.empty(10, dtype=torch.int64, device="cuda"), 3)
        assert torch.ops.mgcn.segment_reduce(x, off, 1).shape == (3, 32)


def test_shard_helpers():
    covered = []
    for r in range(8):
        a, b = mdist.shard_range(25, 8, r)
        covered += list(range(a, b))
        assert 3 <= b - a <= 4
    assert covered == list(range(25))
    parts = mdist.shard_by_weight([5, 9, 1, 7, 3, 3], 3)
    assert sorted(sum(parts, [])) == list(range(6))
    loads = [sum([5, 9, 1, 7, 3, 3][i] for i in p) for p in parts]
    assert max(loads) - min(loads) <= 3


def test_numa_binding_is_a_noop_without_a_readable_topology():
    """dist.bind_to_gpu_numa_node: on a host without CUDA / sysfs topology nothing changes and None comes back"""
    import os
    from meta_gcn_b200 import dist as mdist
    before = os.sched_getaffinity(0)
    assert mdist.bind_to_gpu_numa_node(0) is None or isinstance(mdist.bind_to_gpu_numa_node(0), int)
    if not __import__("torch").cuda.is_available():
        assert os.sched_getaffinity(0) == before


def test_csr_reuse_argument_is_checked_on_the_host():
    """ops.csr_build_impl refuses CPU tensors before looking at `reuse` (no CPU fallback), and structure_of accepts the
    recycle flag"""
    import inspect
    import pytest
    import torch
    from meta_gcn_b200 import graph, ops
    assert "reuse" in inspect.signature(ops.csr_build_impl).parameters
    assert "recycle" in inspect.signature(graph.structure_of).parameters
    with pytest.raises(RuntimeError):
        ops.csr_build_impl(torch.zeros(2, 3, dtype=torch.int64), 4, 0, 0, reuse=None)
