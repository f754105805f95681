"""Edge gates (EdgeGateProj, gcn_base_models.py:322-369) on the hidden-32 tcgen05 stack: the gate kernels against fp64
restatements of include/mgcn.h, the route a gated model takes, training parity with the gated oracle
(tests/gated_oracle.py) at fp32 with an fp64 arbiter, and determinism."""
import ctypes
import math

import pytest
import torch
import torch.nn as nn

from gated_oracle import GatedOracle
from util import assert_bitexact, assert_parity

DEV = "cuda"
H = 32
BOTNET_GATE = dict(in_channels=1, enc_sizes=[32] * 12, num_classes=2, residual_hop=1, dropout=0.0,
                   final_type="proj", deg_norm="sm", aggr="add", bias=True, edge_gate="proj")


# ------------------------------------------------------------------------------------------------ kernels (GPU)
def _csr_pair(ei, n, hub_threshold=None):
    from meta_gcn_b200.graph import structure_of
    g = structure_of(ei.to(DEV), n)
    return g.fwd_plain, g.bwd_plain


def _random_graph(n, e, seed, hub=0, kind="random"):
    """edges among nodes [0, n): random (asymmetric, unordered), symmetric (both directions of each edge) or ordered
    (sorted by target, then source); one target with `hub` sources and one source with hub / 2 targets"""
    gen = torch.Generator().manual_seed(seed)
    src = torch.randint(0, n, (e,), generator=gen)
    tgt = torch.randint(0, n, (e,), generator=gen)
    if hub:
        src = torch.cat([src, torch.randint(0, n, (hub,), generator=gen)])
        tgt = torch.cat([tgt, torch.full((hub,), 7)])
        src = torch.cat([src, torch.full((hub // 2,), 11)])
        tgt = torch.cat([tgt, torch.randint(0, n, (hub // 2,), generator=gen)])
    ei = torch.stack([src, tgt])
    if kind == "symmetric":
        ei = torch.cat([ei, ei.flip(0)], 1)
    elif kind == "ordered":
        ei = ei[:, torch.argsort(ei[1] * n + ei[0], stable=True)]
    return ei


def _gate_ref(ei, ab, c):
    a, b = ab[:, 0].double(), ab[:, 1].double()
    return torch.sigmoid(a[ei[0]] + b[ei[1]] + c)


@pytest.mark.gpu
@pytest.mark.parametrize("n, e, hub, spread, kind", [
    (1000, 6000, 0, 1.0, "random"), (5003, 30000, 20000, 1.0, "random"), (777, 4000, 3000, 30.0, "random"),
    (2001, 8000, 3000, 1.0, "symmetric"), (2001, 8000, 3000, 1.0, "ordered")])
def test_gate_passes_vs_fp64(n, e, hub, spread, kind):
    """scores, gated narrow aggregation and both backward passes against fp64 on asymmetric / symmetric, unordered /
    ordered lists with 61 isolated rows at the end (N not a multiple of 128), hub rows (one above 32 segments) and gates
    saturated near 0 and 1 (|a + b + c| up to ~30)"""
    from meta_gcn_b200 import ops
    ei = _random_graph(n, e, seed=n, hub=hub, kind=kind)
    n = n + 61
    fwd, bwd = _csr_pair(ei, n)
    gen = torch.Generator().manual_seed(1)
    ab = (spread * torch.randn(n, 2, generator=gen)).to(DEV)
    c = torch.tensor([0.3]).to(DEV)
    gs = torch.randn(n, H, generator=gen).to(DEV)
    m = torch.randn(n, H, generator=gen).to(DEV)
    pre = (0.5 + torch.rand(n, generator=gen)).to(DEV)
    u, v = torch.randn(H, generator=gen).to(DEV), torch.randn(H, generator=gen).to(DEV)
    g = _gate_ref(ei, ab.cpu(), 0.3)
    dot = (gs.cpu().double()[ei[1]] * m.cpu().double()[ei[0]]).sum(1)
    dt = dot * g * (1 - g)
    db_ref = torch.zeros(n, dtype=torch.float64).index_add_(0, ei[1], dt)
    da_ref = torch.zeros(n, dtype=torch.float64).index_add_(0, ei[0], dt)
    agg = torch.zeros(n, H, dtype=torch.float64).index_add_(0, ei[0], g[:, None] * gs.cpu().double()[ei[1]])
    dxw_ref = pre.cpu().double()[:, None] * agg + da_ref[:, None] * u.cpu().double() + db_ref[:, None] * v.cpu().double()
    db = ops.gate_grad_by_target_impl(fwd, gs, m, ab, c)
    dxw, dsc = ops.gate_grad_by_source_impl(bwd, gs, m, ab, c, db, pre, u, v, pre)
    scale = dt.abs().max().item() + 1e-30
    assert (db.cpu().double() - db_ref).abs().max().item() <= 1e-4 * scale
    assert (dsc[:, 2].cpu().double() - db_ref).abs().max().item() <= 1e-4 * scale
    assert (dsc[:, 0].cpu().double() * pre.cpu().double() - da_ref).abs().max().item() <= 1e-4 * scale
    assert_parity(dxw, dxw_ref.float(), "dxw", rtol=1e-4, scale_atol=1e-4)
    # narrow gated aggregation
    x4 = torch.randn(n, 3, generator=gen).to(DEV)
    s = ops.gate_spmm_narrow_impl(fwd, x4, ab, c)
    s_ref = torch.zeros(n, 3, dtype=torch.float64).index_add_(0, ei[1], g[:, None] * x4.cpu().double()[ei[0]])
    assert_parity(s, s_ref.float(), "gate_spmm_narrow", rtol=1e-4, scale_atol=1e-5)
    # scores
    z = torch.randn(n, H, generator=gen).to(DEV)
    w = torch.randn(H, H, generator=gen).to(DEV)
    sc = ops.gate_scores_impl(z, w, u, v, pre)
    xw = (z.cpu().double() / pre.cpu().double()[:, None]) @ w.cpu().double()
    sc_ref = torch.stack([xw @ u.cpu().double(), xw @ v.cpu().double()], 1)
    assert_parity(sc, sc_ref.float(), "gate_scores", rtol=1e-4, scale_atol=1e-4)


@pytest.mark.gpu
def test_dt_of_both_passes_agree_bit_for_bit():
    """on a permutation graph each row has one in-edge and one out-edge: db of the by-target pass and da of the
    by-source pass are then the same edge's dt, and must be the same bits"""
    from meta_gcn_b200 import ops
    n = 4099
    gen = torch.Generator().manual_seed(2)
    perm = torch.randperm(n, generator=gen)
    ei = torch.stack([torch.arange(n), perm])
    fwd, bwd = _csr_pair(ei, n)
    ab = (20 * torch.randn(n, 2, generator=gen)).to(DEV)
    c = torch.tensor([-0.7]).to(DEV)
    gs, m = torch.randn(n, H, generator=gen).to(DEV), torch.randn(n, H, generator=gen).to(DEV)
    u, v = torch.randn(H).to(DEV), torch.randn(H).to(DEV)
    db = ops.gate_grad_by_target_impl(fwd, gs, m, ab, c)
    _, dsc = ops.gate_grad_by_source_impl(bwd, gs, m, ab, c, db, None, u, v, None)
    da = dsc[:, 0].cpu()
    assert torch.equal(da, db.cpu()[perm]), "dt differs between the passes"
    assert (db != 0).any()


def _layer_fwd_tc_gate(fwd, z, w, rw, rb, bias, in_scale, post, out_scale, keep, keep_scale, ab, c):
    """mgcn_gcn_layer_fwd_tc_gate called directly (ab / c may be None: NULL)"""
    from meta_gcn_b200 import _lib, ops
    n = fwd.n_rows
    z_next = torch.empty(n, H, device=DEV)
    hmask = torch.empty(n, dtype=torch.int32, device=DEV)
    lib = _lib.load()
    p = ops._ptr
    args = (ctypes.byref(fwd.struct()), p(z), z.size(0), p(w), p(rw), p(rb), p(bias), p(in_scale), p(post),
            p(out_scale), p(keep), float(keep_scale), p(ab), p(c), 1, H, p(z_next), p(hmask))
    ws, nbytes = ops._workspace(lambda w_, nb, stm: lib.mgcn_gcn_layer_fwd_tc_gate(*args, w_, nb, stm), z.device)
    _lib.check(lib.mgcn_gcn_layer_fwd_tc_gate(*args, p(ws), ctypes.byref(nbytes), ops._stream()))
    return z_next, hmask


@pytest.mark.gpu
@pytest.mark.parametrize("dropout", [False, True])
def test_gated_forward_layer_vs_fp64_and_null_gate(dropout):
    """mgcn_gcn_layer_fwd_tc_gate with gate_ab NULL is mgcn_gcn_layer_fwd_tc_ex bit for bit (keep bits, bias, degree
    factors); with varying gates (a and b drawn apart, so a swap would show) the layer matches an fp64 restatement of
    its contract on a graph with a hub above 32 segments and isolated rows"""
    from meta_gcn_b200 import ops
    n0 = 3001
    ei = _random_graph(n0, 20000, seed=4, hub=3000)
    n = n0 + 61
    fwd, _ = _csr_pair(ei, n)
    gen = torch.Generator().manual_seed(3)
    z = torch.randn(n, H, generator=gen).to(DEV)
    w, rw = torch.randn(H, H, generator=gen).to(DEV) * 0.2, torch.randn(H, H, generator=gen).to(DEV) * 0.2
    rb, b = torch.randn(H, generator=gen).to(DEV), torch.randn(H, generator=gen).to(DEV) * 0.1
    in_scale = (0.5 + torch.rand(n, generator=gen)).to(DEV)
    post = (0.5 + torch.rand(n, generator=gen)).to(DEV)
    out_scale = (0.5 + torch.rand(n, generator=gen)).to(DEV)
    keep = torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), generator=gen, dtype=torch.int64).to(torch.int32).to(DEV) \
        if dropout else None
    ks = 2.0 if dropout else 1.0
    ref_ex = ops.gcn_layer_fwd_tc_impl(fwd, z, w, rw, rb, b, in_scale, post, out_scale, 1, keep=keep, keep_scale=ks)
    null = _layer_fwd_tc_gate(fwd, z, w, rw, rb, b, in_scale, post, out_scale, keep, ks, None, None)
    assert_bitexact(null[0], ref_ex[0], "z_next, gate NULL")
    assert torch.equal(null[1], ref_ex[1])
    # varying gates: a_j in ~N(0, 3), b_i in ~N(2, 1): sigmoid(a + b + c) spans (0, 1)
    ab = torch.stack([3 * torch.randn(n, generator=gen), 2 + torch.randn(n, generator=gen)], 1).to(DEV)
    c = torch.tensor([-1.5]).to(DEV)
    zn, hm = _layer_fwd_tc_gate(fwd, z, w, rw, rb, b, in_scale, post, out_scale, keep, ks, ab, c)
    g = _gate_ref(ei, ab.cpu(), -1.5)
    zd = z.cpu().double()
    s = torch.zeros(n, H, dtype=torch.float64).index_add_(0, ei[1], g[:, None] * zd[ei[0]])
    h = torch.relu(post.cpu().double()[:, None] * (s @ w.cpu().double()) + b.cpu().double())
    if dropout:
        bits = ((keep.cpu().numpy().astype("uint32")[:, None] >> torch.arange(H).numpy().astype("uint32")) & 1)
        h = h * torch.from_numpy(bits.astype("float64")) * ks
    y = h + (zd @ rw.cpu().double().t()) / in_scale.cpu().double()[:, None] + rb.cpu().double()
    ref = torch.relu(y) * out_scale.cpu().double()[:, None]
    assert_parity(zn, ref.float(), "gated forward layer", rtol=1e-4, scale_atol=1e-5)


# ------------------------------------------------------------------------------------------------ model (GPU)
def _set_gates(model, seed=11, spread=1.0):
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if name.startswith("gcn_net.") and (name.endswith(".bias") or "edge_gate" in name):
                prm.copy_(spread * 0.1 * torch.randn(prm.shape, generator=gen))


def _parity(monkeypatch, cfg, graph, xin_of, p=0.0, use_deg=True):
    from meta_gcn_b200 import fused
    from meta_gcn_b200.gcn_meta.models import GCNModel
    from test_gpu_bench_shapes import assert_parity_arbitrated
    from test_gpu_dropout import _MaskedDropout, _pin_seed, keep_bits_ref
    g = graph()
    xin = xin_of(g)
    calls = _pin_seed(monkeypatch, 0x2)
    taken = []
    real = fused._GatedResidualGCNStack32AT.apply
    monkeypatch.setattr(fused._GatedResidualGCNStack32AT, "apply", lambda *a: taken.append(True) or real(*a))
    cfg = dict(cfg, dropout=p)
    torch.manual_seed(0)
    ref = GatedOracle(**cfg)
    _set_gates(ref)
    model = GCNModel(**cfg)
    model.load_state_dict(ref.state_dict())
    model.to(DEV).train()
    ei = torch.from_numpy(g["edge_index"])
    y = torch.from_numpy(g["y"]).long()
    deg = torch.from_numpy(g["x"])[:, 1].contiguous() if use_deg else None
    ref64 = GatedOracle(**cfg)
    ref64.load_state_dict(ref.state_dict())
    ref64 = ref64.double()
    if p:
        keep = keep_bits_ref(0x2, len(cfg["enc_sizes"]), xin.size(0), 1, p)
        ref.dropout = _MaskedDropout(keep, H, p)
        ref64.dropout = _MaskedDropout(keep, H, p)
    crit = nn.CrossEntropyLoss()
    out_r = ref(xin, ei, deg)
    loss_r = crit(out_r, y)
    loss_r.backward()
    out64 = ref64(xin.double(), ei, deg.double() if use_deg else None)
    crit(out64, y).backward()
    out = model(xin.to(DEV), ei.to(DEV), deg_K=deg.to(DEV) if use_deg else None)
    loss = crit(out, y.to(DEV))
    loss.backward()
    assert taken == [True], "the forward did not take the gated tcgen05 stack"
    assert len(calls) == (1 if p else 0)
    assert_parity_arbitrated(out, out_r, out64, "logits")
    assert abs(loss.item() - loss_r.item()) <= 1e-5 * max(1.0, abs(loss_r.item()))
    names = dict(ref.named_parameters())
    names64 = dict(ref64.named_parameters())
    n_gate = 0
    for k, prm in model.named_parameters():
        # a gate bias gradient is one scalar summed over every edge with heavy cancellation, from gates formed with
        # ex2.approx (a few ulp each): judged at 3e-5 against fp64 instead of 1e-5
        rtol = 3e-5 if k.endswith("edge_gate.bias") else 1e-5
        assert_parity_arbitrated(prm.grad, names[k].grad, names64[k].grad, "grad." + k, rtol=rtol)
        n_gate += "edge_gate" in k
    assert n_gate == 3 * len(cfg["enc_sizes"])


def _graph20k():
    from test_gpu_dropout import _graph
    return _graph()


def _botnet_input(g):
    return torch.from_numpy(g["x"][:, 0:1].copy())


@pytest.mark.gpu
@pytest.mark.parametrize("bias, p", [(True, 0.0), (False, 0.5)])
def test_gated_botnet_model_vs_oracle(monkeypatch, bias, p):
    """12 layers at hidden 32 with gates on every layer, the first aggregated before its transform"""
    _parity(monkeypatch, dict(BOTNET_GATE, bias=bias), _graph20k, _botnet_input, p)


@pytest.mark.gpu
def test_gated_rw_and_wide_input_vs_oracle(monkeypatch):
    """deg_norm 'rw' (no per-target factor), and a 32-wide input (layer 0 through the gated tcgen05 layer)"""
    _parity(monkeypatch, dict(BOTNET_GATE, enc_sizes=[32] * 4, deg_norm="rw"), _graph20k, _botnet_input, 0.5)
    _parity(monkeypatch, dict(BOTNET_GATE, in_channels=32, enc_sizes=[32] * 4), _graph20k,
            lambda g: torch.randn(g["x"].shape[0], 32, generator=torch.Generator().manual_seed(3)), 0.0)


def _sink_graph(n=5000, e=40000, n_src=4500, seed=7):
    """asymmetric graph whose last n - n_src nodes have in-edges but no out-edges: with the graph's own out-degree
    their per-source factor is 0 (sigma 1), while their gate score b still receives a gradient"""
    gen = torch.Generator().manual_seed(seed)
    ei = torch.stack([torch.randint(0, n_src, (e,), generator=gen), torch.randint(0, n, (e,), generator=gen)])
    x = torch.stack([torch.rand(n, generator=gen), torch.zeros(n)], 1)
    return {"edge_index": ei.numpy(), "x": x.numpy(), "y": torch.randint(0, 2, (n,), generator=gen).numpy()}


@pytest.mark.gpu
@pytest.mark.parametrize("deg_norm", ["rw", "sm"])
def test_gated_sink_nodes_without_degree_vector_vs_oracle(monkeypatch, deg_norm):
    """no deg_K: degree factors from the graph's out-degree, 0 on sink nodes; the first layer's lintgt gradient takes
    those rows' x W in full (the messages m = pre (.) x W are 0 there)"""
    _parity(monkeypatch, dict(BOTNET_GATE, enc_sizes=[32] * 4, deg_norm=deg_norm), _sink_graph, _botnet_input, 0.0,
            use_deg=False)


@pytest.mark.gpu
def test_gated_full_c1_graph_vs_oracle(monkeypatch):
    from meta_gcn_b200.data import synth_botnet_graph
    _parity(monkeypatch, BOTNET_GATE, lambda: synth_botnet_graph(seed=0), _botnet_input, 0.0)


def _free_gates(model, E):
    from meta_gcn_b200.gcn_meta.models.gcn_base_models import EdgeGateFree
    for layer in model.gcn_net:
        layer.gcn.node_models[0].edge_gate = EdgeGateFree(E)


def _ungate_layer1(model):
    model.gcn_net[1].gcn.node_models[0].edge_gate = None


@pytest.mark.gpu
@pytest.mark.parametrize("case, want", [
    ("sm", 4), ("rw", 4), ("no_norm", 4), ("no_bias", 4),
    ("width16", 0), ("x_requires_grad", 0), ("edge_gate_free", 0), ("mixed", 0), ("mean", 0), ("max", 0),
    ("edge_attr", 0), ("edge_weight", 0), ("degree_with_zeros", 0)])
def test_gated_routing(monkeypatch, case, want):
    """the gated stack (one by-source gate pass per layer) for sm / rw / no normalisation, with or without bias; the
    per-layer path for every excluded configuration"""
    from meta_gcn_b200 import ops
    from meta_gcn_b200.gcn_meta.models import GCNModel
    from test_gpu_dropout import _graph, _inputs
    g = _graph(seed=5, num_nodes=6000, edge_entries=50000, evil=400)
    x0, ei, deg, y = _inputs(g)
    E = ei.size(1)
    n = {"src": 0}
    real = ops.gate_grad_by_source_impl
    monkeypatch.setattr(ops, "gate_grad_by_source_impl", lambda *a: n.__setitem__("src", n["src"] + 1) or real(*a))
    cfg = dict(BOTNET_GATE, enc_sizes=[32] * 4)
    cfg.update({"rw": dict(deg_norm="rw"), "no_norm": dict(deg_norm=None), "no_bias": dict(bias=False),
                "width16": dict(enc_sizes=[16] * 4), "mean": dict(aggr="mean"), "max": dict(aggr="max"),
                "edge_attr": dict(in_edgedim=3)}.get(case, {}))
    torch.manual_seed(0)
    model = GCNModel(**cfg)
    if case == "edge_gate_free":
        _free_gates(model, E)
    if case == "mixed":
        _ungate_layer1(model)
    model = model.to(DEV).train()
    kw = {"deg_K": deg}
    if case == "edge_attr":
        kw["edge_attr_K"] = torch.rand(E, 3, device=DEV)
    if case == "edge_weight":
        kw["edge_weight_K"] = torch.rand(E, device=DEV) + 0.5
    if case == "degree_with_zeros":
        kw["deg_K"] = torch.where(torch.arange(deg.numel(), device=DEV) % 97 == 0, torch.zeros_like(deg), deg)
    x = x0.clone().requires_grad_(case == "x_requires_grad")
    nn.CrossEntropyLoss()(model(x, ei, **kw), y).backward()
    assert n["src"] == want, (case, n)
    assert all(torch.isfinite(q.grad).all() for q in model.parameters() if q.grad is not None)


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.5])
def test_gated_batch_and_graphed_adam_steps(p):
    """two runs bit-identical, a batch equal to its graphs bit for bit, three Adam steps replayed from a captured CUDA
    graph equal to the eager steps bit for bit"""
    from meta_gcn_b200 import data as D
    from meta_gcn_b200 import dist as mdist
    from meta_gcn_b200 import functional as F
    from meta_gcn_b200.gcn_meta.models import GCNModel
    from meta_gcn_b200.graphed import GraphedCall
    graphs = [D.synth_botnet_graph(seed=s, num_nodes=20000, edge_entries=220000, evil=1500) for s in (1, 2, 3)]
    batch = D.GraphBatch.from_data_list(graphs).to(DEV)
    batch.x = batch.x.contiguous()
    torch.manual_seed(3)
    model = GCNModel(**dict(BOTNET_GATE, dropout=p)).to(DEV)
    _set_gates(model, spread=3.0)
    with torch.no_grad():
        model.eval()
        whole = model(batch.x[:, 0].view(-1, 1), batch.edge_index, deg_K=batch.x[:, 1])
        assert_bitexact(whole, model(batch.x[:, 0].view(-1, 1), batch.edge_index, deg_K=batch.x[:, 1]), "rerun")
        for i, gph in enumerate(graphs):
            one = D.GraphBatch.from_data_list([gph]).to(DEV)
            part = model(one.x[:, 0].view(-1, 1), one.edge_index, deg_K=one.x[:, 1])
            assert_bitexact(whole[batch.slices_x[i]:batch.slices_x[i + 1]], part, f"graph {i} of the batch")
    model.train()
    state0 = {k: v.clone() for k, v in model.state_dict().items()}
    rng = torch.cuda.get_rng_state()
    results = []
    work = torch.cuda.Stream()
    work.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(work):
        for use_graph in (False, True):
            model.load_state_dict(state0)
            reducer = mdist.FlatGradientReducer(model.parameters())
            opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=5e-4, fused=True)

            def fwd_loss_bwd():
                reducer.zero()
                out = model(batch.x[:, 0].view(-1, 1), batch.edge_index, deg_K=batch.x[:, 1])
                loss_sum = F.cross_entropy(out, batch.y.long(), "sum")
                loss_sum.backward()
                return loss_sum
            call = GraphedCall(fwd_loss_bwd, warmup=1) if use_graph else fwd_loss_bwd
            if use_graph:
                model.load_state_dict(state0)
            torch.cuda.set_rng_state(rng)
            losses = []
            for _ in range(3):
                loss_sum = call()
                mean_loss, _ = reducer.reduce_mean(loss_sum, batch.num_nodes)
                opt.step()
                losses.append(float(mean_loss))
            results.append((losses, [q.detach().clone() for q in model.parameters()]))
    torch.cuda.current_stream().wait_stream(work)
    assert results[0][0] == results[1][0], (results[0][0], results[1][0])
    assert all(math.isfinite(x) for x in results[0][0])
    for pe, pg in zip(results[0][1], results[1][1]):
        assert torch.equal(pe, pg)
