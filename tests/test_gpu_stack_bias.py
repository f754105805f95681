"""Node-model bias on the hidden-32 tcgen05 stack (NodeModelAdditive's default bias=True, gcn_base_models.py:240):
the first-layer entry with a bias, the bias gradient of the row-local backward and the standalone masked column sum
against fp64 restatements of include/mgcn.h; the route a bias model takes; training steps against the oracle with
non-zero biases; CUDA-graph replay and batching.  Host tests are unmarked; the rest need a GPU."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn as nn

from meta_gcn_b200 import _lib, fused, ops
from meta_gcn_b200.gcn_meta.models import GCNModel
from util import assert_bitexact, assert_parity

DEV = "cuda"
H = 32
NULL, SHAPE = -1, -3
BOTNET_BIAS = dict(in_channels=1, enc_sizes=[32] * 12, num_classes=2, residual_hop=1, dropout=0.0,
                   final_type="proj", deg_norm="sm", aggr="add", bias=True)


def unpack_bits(words, n_cols=H):
    """int32 [N] mask words -> float64 0/1 [N, n_cols]"""
    u = np.asarray(words).astype(np.uint32)
    return torch.from_numpy(((u[:, None] >> np.arange(n_cols, dtype=np.uint32)[None, :]) & 1).astype(np.float64))


def masked_colsum_ref(gy, bits, scale):
    """d_bias[c] = scale * sum_i bit c of bits[i] * gy[i,c] in fp64"""
    return scale * (gy.double() * unpack_bits(bits.cpu().numpy())).sum(0)


# ------------------------------------------------------------------------------------------------ host
def test_argument_errors_without_device():
    lib = _lib.load()
    n = ctypes.c_size_t(0)
    dummy = 256                                   # 16-byte aligned, never dereferenced on these paths
    first = lambda h, **kw: lib.mgcn_gcn_first_layer_fwd_bias(  # noqa: E731
        kw.get("s"), kw.get("s"), 10, kw.get("hin", 1), kw.get("s"), kw.get("s"), None, kw.get("bias"), None, None,
        None, None, None, 1.0, 1, h, kw.get("s"), None, kw.get("s"), None)
    assert first(16) == SHAPE
    assert first(32, hin=5) == SHAPE
    assert first(32) == NULL
    bwd = lambda h, ws, nb, d_bias=None, hmask_cur=None, ptrs=None, N=100: lib.mgcn_gcn_layer_bwd_tc_ex(  # noqa: E731
        ptrs, ptrs, ptrs, None, ptrs, ptrs, None, hmask_cur, None, 2.0, N, h, None, None, ptrs, ptrs, ptrs, d_bias,
        ws, nb, None)
    assert bwd(32, None, None) == NULL                                  # no workspace size
    assert bwd(16, None, ctypes.byref(n)) == SHAPE
    assert bwd(32, None, ctypes.byref(n)) == 0
    plain = n.value
    assert bwd(32, None, ctypes.byref(n), d_bias=dummy) == 0
    assert n.value > plain                                              # the bias partials
    big = ctypes.c_size_t(n.value)
    assert bwd(32, dummy, ctypes.byref(big), d_bias=dummy, ptrs=dummy) == NULL    # d_bias without hmask_cur
    assert bwd(32, dummy, ctypes.byref(big), d_bias=dummy, ptrs=dummy, hmask_cur=dummy, N=0) == 0   # nothing to do
    colsum = lambda h, ws, nb, gy=None, bits=None, d_bias=None, N=10: lib.mgcn_mask_bits_colsum(  # noqa: E731
        gy, bits, 1.0, N, h, d_bias, ws, nb, None)
    assert colsum(32, None, None) == NULL
    assert colsum(16, None, ctypes.byref(n)) == SHAPE
    assert colsum(32, None, ctypes.byref(n), N=-1) == -2
    assert colsum(32, None, ctypes.byref(n)) == 0 and n.value >= H * 4
    big = ctypes.c_size_t(n.value)
    assert colsum(32, dummy, ctypes.byref(big), gy=dummy, bits=dummy) == NULL         # no d_bias
    assert colsum(32, dummy, ctypes.byref(big), d_bias=dummy) == NULL                 # N > 0 without gy / bits


def test_ops_refuse_cpu_and_trace_as_fakes():
    gy = torch.zeros(4, H)
    bits = torch.zeros(4, dtype=torch.int32)
    with pytest.raises(RuntimeError, match="CPU"):
        torch.ops.mgcn.mask_bits_colsum(gy, bits, 1.0)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.mask_bits_colsum_impl(gy, bits, 1.0)
    with pytest.raises(RuntimeError, match="CPU"):
        torch.ops.mgcn.gcn_first_layer_fwd_bias(torch.zeros(4, 1), torch.zeros(4, 1), torch.zeros(1, H),
                                                torch.zeros(H, 1), None, torch.zeros(H), None, None, None, 1, None)
    meta = dict(device="meta")
    assert torch.ops.mgcn.mask_bits_colsum(torch.empty(7, H, **meta), torch.empty(7, dtype=torch.int32, **meta),
                                           2.0).shape == (H,)
    outs = torch.ops.mgcn.gcn_layer_bwd_bias(*(torch.empty(7, H, **meta) for _ in range(3)),
                                             torch.empty(H, H, **meta), torch.empty(H, H, **meta), None,
                                             torch.empty(7, dtype=torch.int32, **meta), None, 2.0, False, None)
    assert [tuple(t.shape) for t in outs] == [(0,), (0,), (H, H), (H, H), (H,), (H,)]
    xn, mn, hm = torch.ops.mgcn.gcn_first_layer_fwd_bias(
        torch.empty(7, 2, **meta), torch.empty(7, 2, **meta), torch.empty(2, H, **meta), torch.empty(H, 2, **meta),
        None, torch.empty(H, **meta), None, None, None, 1, None)
    assert xn.shape == (7, H) and mn.shape == (0,) and hm.shape == (7,)


def _stack_params(widths, bias, hin=1):
    sizes = [hin] + widths
    return [((torch.zeros(a, b), torch.zeros(b)) if bias else (torch.zeros(a, b),)) + (torch.zeros(b, a), torch.zeros(b))
            for a, b in zip(sizes, sizes[1:])]


@pytest.mark.parametrize("widths,bias,hin,aggregate_first,requires_grad,want", [
    ([32] * 3, True, 1, True, False, "tc"),
    ([32] * 3, True, 32, True, False, "tc"),
    ([32] * 3, False, 1, True, False, "tc"),
    ([32] * 3, True, 8, True, False, "generic"),        # input width neither <= 4 nor 32
    ([32] * 3, True, 1, False, False, "generic"),       # a degree with zeros
    ([32] * 3, True, 1, True, True, "generic"),         # x requires grad
    ([16] * 3, True, 1, True, False, "generic"),
    ([64] * 3, True, 1, True, False, "generic"),
    ([32] * 3, False, 1, False, False, "round1"),
])
def test_routing(monkeypatch, widths, bias, hin, aggregate_first, requires_grad, want):
    """residual_gcn_stack sends a hidden-32 stack with bias to the tcgen05 stack under the conditions of the bias-free
    one; every other bias model keeps the generic stack, and bias-free models keep their routes"""
    taken = []
    for name, cls in (("tc", fused._ResidualGCNStack32AT), ("generic", fused._ResidualGCNStack),
                      ("round1", fused._ResidualGCNStack32)):
        monkeypatch.setattr(cls, "apply", lambda *a, _n=name: taken.append((_n, a)) or _n)
    x = torch.zeros(5, hin, requires_grad=requires_grad)
    got = fused.residual_gcn_stack(x, None, None, None, _stack_params(widths, bias, hin), bias,
                                   aggregate_first=aggregate_first)
    assert got == want and len(taken) == 1
    if want == "tc":
        assert taken[0][1][4] is bias                          # has_bias, then (W, [b], R, r) per layer
        assert len(taken[0][1]) == 7 + (4 if bias else 3) * len(widths)


# ------------------------------------------------------------------------------------------------ kernels
def _first_layer_inputs(n, hin, hub_threshold, seed):
    """a random graph with rows above the hub threshold, s = sum_j pre_j x_j through mgcn_spmm, and the layer's operands"""
    from meta_gcn_b200.graph import GraphStructure
    g = np.random.default_rng(seed)
    e = 6 * n
    src, dst = g.integers(0, n, e), g.integers(0, n, e)
    if n > 40:
        dst[:200] = 3                                          # hub rows (13 segments at threshold 16)
        dst[200:240] = 7
    ei = torch.from_numpy(np.stack([src, dst]).astype(np.int64))
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(n, hin, generator=gen)
    pre = torch.rand(n, generator=gen) + 0.1
    post = torch.rand(n, generator=gen) + 0.1
    w_in = torch.randn(hin, H, generator=gen)
    res_w = torch.randn(H, hin, generator=gen)
    res_b = torch.randn(H, generator=gen)
    bias = torch.randn(H, generator=gen)
    gs = GraphStructure(ei.to(DEV), n, hub_threshold=hub_threshold)
    s = ops.spmm_impl(gs.fwd, (x * pre.view(-1, 1)).to(DEV))
    agg = torch.zeros(n, hin, dtype=torch.float64).index_add_(0, ei[1], (x.double() * pre.double().view(-1, 1))[ei[0]])
    return s, agg, x, pre, post, w_in, res_w, res_b, bias


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 1003, 150001])
@pytest.mark.parametrize("hin", [1, 2, 4])
@pytest.mark.parametrize("dropout", [False, True])
def test_first_layer_bias_vs_fp64(n, hin, dropout):
    """mgcn_gcn_first_layer_fwd_bias, streaming pass: h = keep ? scale * relu(post (s W) + b) : 0,
    x' = relu(h + x R^T + r) * out_scale, mask words = (h > 0); bias = NULL is bit-identical to mgcn_gcn_first_layer_fwd_ex"""
    s, agg, x, pre, post, w_in, res_w, res_b, bias = _first_layer_inputs(n, hin, 16, seed=n + hin)
    gen = torch.Generator().manual_seed(n * 7 + hin)
    out_scale = torch.rand(n, generator=gen) + 0.1
    keep = torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), generator=gen, dtype=torch.int64).to(torch.int32) if dropout \
        else None
    scale = 2.0 if dropout else 1.0
    d = lambda t: None if t is None else t.to(DEV)   # noqa: E731
    drop = dict(keep=d(keep), keep_scale=scale) if dropout else {}
    xn, mn, hm = ops.gcn_first_layer_fwd_impl(s, d(x), d(w_in), d(res_w), d(res_b), None, None, d(post), 1,
                                              out_scale=d(out_scale), bias=d(bias), **drop)
    assert mn is None
    D = lambda t: t.double()   # noqa: E731
    pre_act = D(post).view(-1, 1) * (agg @ D(w_in)) + D(bias)
    h = torch.relu(pre_act)
    if dropout:
        h = h * unpack_bits(keep.numpy()) * scale
    y = h + D(x) @ D(res_w).t() + D(res_b)
    assert_parity(xn, torch.relu(y) * D(out_scale).view(-1, 1), "x_next")
    got = unpack_bits(hm.cpu().numpy()).bool().numpy()
    sure = np.abs(pre_act.numpy()) > 1e-5 * max(1.0, float(np.abs(pre_act.numpy()).max()))
    assert (got == (h.numpy() > 0))[sure].all()
    # bias = NULL through the new entry point == mgcn_gcn_first_layer_fwd_ex
    a = ops.gcn_first_layer_fwd_impl(s, d(x), d(w_in), d(res_w), d(res_b), None, None, d(post), 1,
                                     out_scale=d(out_scale), **drop)
    xb, hb = torch.empty(n, H, device=DEV), torch.empty(n, dtype=torch.int32, device=DEV)
    p = lambda t: None if t is None else t.data_ptr()   # noqa: E731
    args = [d(x).contiguous(), d(w_in), d(res_w), d(res_b), d(post), d(out_scale), d(keep)]
    xd, wd, rwd, rbd, postd, osd, kd = args
    _lib.check(_lib.load().mgcn_gcn_first_layer_fwd_bias(
        p(s), p(xd), n, hin, p(wd), p(rwd), p(rbd), None, None, None, p(postd), p(osd), p(kd), scale, 1, H, p(xb), None,
        p(hb), ops._stream()))
    assert_bitexact(xb, a[0], "x_next, bias NULL")
    assert_bitexact(hb, a[2], "mask, bias NULL")
    # run-to-run identical
    xn2, _, hm2 = ops.gcn_first_layer_fwd_impl(s, d(x), d(w_in), d(res_w), d(res_b), None, None, d(post), 1,
                                               out_scale=d(out_scale), bias=d(bias), **drop)
    assert_bitexact(xn, xn2, "run-to-run")
    assert_bitexact(hm, hm2, "run-to-run mask")


@pytest.mark.gpu
@pytest.mark.parametrize("n,hin", [(1003, 1), (37, 4)])
def test_first_layer_bias_tile_kernel_vs_fp64(n, hin):
    """with a following transform (w_next) the same entry runs the tile kernel: m' = pre (x' W') too"""
    s, agg, x, pre, post, w_in, res_w, res_b, bias = _first_layer_inputs(n, hin, 16, seed=n)
    w_next = torch.randn(H, H, generator=torch.Generator().manual_seed(1)) / H ** 0.5
    d = lambda t: t.to(DEV)   # noqa: E731
    xn, mn, hm = ops.gcn_first_layer_fwd_impl(s, d(x), d(w_in), d(res_w), d(res_b), d(w_next), d(pre), d(post), 1,
                                              bias=d(bias))
    D = lambda t: t.double()   # noqa: E731
    h = torch.relu(D(post).view(-1, 1) * (agg @ D(w_in)) + D(bias))
    x_ref = torch.relu(h + D(x) @ D(res_w).t() + D(res_b))
    assert_parity(xn, x_ref, "x_next")
    assert_parity(mn, D(pre).view(-1, 1) * (x_ref @ D(w_next)), "m_next")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [150, 1000, 9541, 300001])     # 3 tiles; 16; 150 (> one per SM, odd); 4688
@pytest.mark.parametrize("scale", [1.0, 2.0])
def test_layer_bwd_tc_ex_bias_gradient(n, scale):
    """mgcn_gcn_layer_bwd_tc_ex: d_bias = scale * colsum(gy * bits(hmask_cur)) within fp32 rounding of fp64 and the same
    from run to run; every other output bit-identical to mgcn_gcn_layer_bwd_tc on the same inputs"""
    gen = torch.Generator().manual_seed(n + 5)
    dxw, gy, x = (torch.randn(n, H, generator=gen) for _ in range(3))
    w = torch.randn(H, H, generator=gen) / H ** 0.5
    res_w = torch.randn(H, H, generator=gen) / H ** 0.5
    post = torch.rand(n, generator=gen)
    post[::5] = 0.0                                   # post does not enter d_bias
    sigma = torch.rand(n, generator=gen) + 0.1
    bits_prev, bits_cur = (torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), generator=gen, dtype=torch.int64).to(torch.int32)
                           for _ in range(2))
    d = lambda t: t.to(DEV)   # noqa: E731
    args = (d(dxw), d(gy), d(x * sigma.view(-1, 1)), d(w), d(res_w), d(bits_prev))
    for want_prev in (True, False):
        got = ops.gcn_layer_bwd_bias_impl(*args, d(bits_cur), d(post), scale, want_prev, x_scale=d(sigma))
        base = ops.gcn_layer_bwd_impl(*args, d(post), want_prev, True, x_scale=d(sigma))
        for a, b, name in zip(got[:5], base, ("gy_prev", "gs_prev", "dW", "dR", "dr")):
            if b is None:
                assert a is None
            else:
                assert_bitexact(a, b, name + " vs mgcn_gcn_layer_bwd_tc")
        assert_parity(got[5], masked_colsum_ref(gy, bits_cur, scale), "d_bias")
        again = ops.gcn_layer_bwd_bias_impl(*args, d(bits_cur), d(post), scale, want_prev, x_scale=d(sigma))
        assert_bitexact(got[5], again[5], "run-to-run d_bias")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 31, 1003, 300001])
@pytest.mark.parametrize("scale", [1.0, 2.0, 1.0 / 0.9])
def test_mask_bits_colsum_vs_fp64(n, scale):
    gen = torch.Generator().manual_seed(n + 9)
    gy = torch.randn(n, H, generator=gen)
    bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), generator=gen, dtype=torch.int64).to(torch.int32)
    got = ops.mask_bits_colsum_impl(gy.to(DEV), bits.to(DEV), scale)
    if n == 0:
        assert_bitexact(got, torch.zeros(H), "empty")
        return
    assert_parity(got, masked_colsum_ref(gy, bits, scale), "d_bias")
    assert_bitexact(got, ops.mask_bits_colsum_impl(gy.to(DEV), bits.to(DEV), scale), "run-to-run")
    assert_bitexact(got, torch.ops.mgcn.mask_bits_colsum(gy.to(DEV), bits.to(DEV), scale), "torch.ops.mgcn")


# ------------------------------------------------------------------------------------------------ model
def _set_biases(model, seed=11):
    """the reference initialises node-model biases to zeros, which would leave the forward untested"""
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if name.startswith("gcn_net.") and name.endswith(".bias"):
                prm.copy_(0.1 * torch.randn(prm.shape, generator=gen))


@pytest.mark.gpu
def test_bias_model_takes_the_tcgen05_stack(monkeypatch):
    """a bias=True hidden-32 GCNModel runs k_gcn_fwd_tc for every layer after the first; 16- and 64-wide ones the
    generic stack"""
    from test_gpu_dropout import _graph, _inputs
    g = _graph(seed=5, num_nodes=6000, edge_entries=50000, evil=400)
    x0, ei, deg, y = _inputs(g)
    calls = {"tc": 0, "generic": 0}
    real_tc, real_generic = ops.gcn_layer_fwd_tc_impl, fused._ResidualGCNStack.apply

    def spy_tc(*a, **k):
        calls["tc"] += 1
        return real_tc(*a, **k)

    def spy_generic(*a, **k):
        calls["generic"] += 1
        return real_generic(*a, **k)
    monkeypatch.setattr(ops, "gcn_layer_fwd_tc_impl", spy_tc)
    monkeypatch.setattr(fused._ResidualGCNStack, "apply", spy_generic)
    for width, want in ((32, {"tc": 3, "generic": 0}), (16, {"tc": 0, "generic": 1}), (64, {"tc": 0, "generic": 1})):
        calls.update(tc=0, generic=0)
        torch.manual_seed(0)
        model = GCNModel(**dict(BOTNET_BIAS, enc_sizes=[width] * 4)).to(DEV).train()
        loss = nn.CrossEntropyLoss()(model(x0, ei, deg_K=deg), y)
        loss.backward()
        assert calls == want, (width, calls)
        assert all(torch.isfinite(p.grad).all() for p in model.parameters())


def _parity_vs_oracle(monkeypatch, cfg, graph, xin_of, p, mask_seed, arbitrated):
    """logits, loss and every parameter gradient (bias gradients included) against the fp32 oracle with the same biases
    and dropout masks; arbitrated: entries that miss rtol 1e-5 are judged against fp64 (tests/test_gpu_bench_shapes.py)"""
    from oracle import port
    from test_gpu_bench_shapes import assert_parity_arbitrated
    from test_gpu_dropout import _MaskedDropout, _pin_seed, keep_bits_ref
    cfg = dict(cfg, dropout=p)
    g = graph()
    xin = xin_of(g)
    calls = _pin_seed(monkeypatch, mask_seed)
    taken = []
    real = fused._ResidualGCNStack32AT.apply
    monkeypatch.setattr(fused._ResidualGCNStack32AT, "apply", lambda *a: taken.append(1) or real(*a))
    torch.manual_seed(0)
    ref = port.OracleGCNModel(**cfg)
    _set_biases(ref)
    model = GCNModel(**cfg)
    model.load_state_dict(ref.state_dict())
    model.to(DEV).train()
    x = torch.from_numpy(g["x"])
    ei = torch.from_numpy(g["edge_index"])
    y = torch.from_numpy(g["y"]).long()
    deg = x[:, 1].contiguous()
    N, L = x.size(0), len(cfg["enc_sizes"])
    crit = nn.CrossEntropyLoss()
    ref64 = port.OracleGCNModel(**cfg)
    ref64.load_state_dict(ref.state_dict())
    ref64 = ref64.double()
    if p:
        keep = keep_bits_ref(mask_seed, L, N, 1, p)
        ref.dropout = _MaskedDropout(keep, H, p)
        ref64.dropout = _MaskedDropout(keep, H, p)
    out_r = ref(xin, ei, deg)
    loss_r = crit(out_r, y)
    loss_r.backward()
    out64 = ref64(xin.double(), ei, deg.double())
    crit(out64, y).backward()
    out = model(xin.to(DEV), ei.to(DEV), deg_K=deg.to(DEV))
    loss = crit(out, y.to(DEV))
    loss.backward()
    assert taken == [1], "the forward did not take the tcgen05 stack"
    assert len(calls) == (1 if p else 0)
    check = (lambda a, r32, r64, what: assert_parity_arbitrated(a, r32, r64, what)) if arbitrated else \
        (lambda a, r32, r64, what: assert_parity(a, r32, what))
    check(out, out_r, out64, "logits")
    assert abs(loss.item() - loss_r.item()) <= 1e-5 * max(1.0, abs(loss_r.item())), (loss.item(), loss_r.item())
    names = []
    for (k, prm), (_, pr), (_, p64) in zip(model.named_parameters(), ref.named_parameters(), ref64.named_parameters()):
        check(prm.grad, pr.grad, p64.grad, "grad." + k)
        names.append(k)
    assert sum(k.endswith("node_models.0.bias") for k in names) == L
    assert_parity(out, out64.detach(), "logits vs fp64")


def _botnet_input(g):
    return torch.from_numpy(g["x"][:, 0:1].copy())


def _graph20k():
    from test_gpu_dropout import _graph
    return _graph()


def _c1():
    from meta_gcn_b200.data import synth_botnet_graph
    return synth_botnet_graph(seed=0)


def _wide(g):
    return torch.randn(g["x"].shape[0], 32, generator=torch.Generator().manual_seed(3))


MASK_SEED = 0x2


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.5])
def test_botnet_model_with_bias_vs_oracle(monkeypatch, p):
    """the 12-layer botnet model with bias=True on the 20k-node hub graph: first layer through the streaming pass with
    its bias and the standalone column sum, then k_gcn_fwd_tc and mgcn_gcn_layer_bwd_tc_ex"""
    _parity_vs_oracle(monkeypatch, BOTNET_BIAS, _graph20k, _botnet_input, p, MASK_SEED, arbitrated=True)


@pytest.mark.gpu
def test_rw_normalisation_with_bias_vs_oracle(monkeypatch):
    """deg_norm='rw': no per-target factor"""
    _parity_vs_oracle(monkeypatch, dict(BOTNET_BIAS, enc_sizes=[32] * 4, deg_norm="rw"), _graph20k, _botnet_input, 0.5,
                      MASK_SEED, arbitrated=True)


@pytest.mark.gpu
def test_wide_input_with_bias_vs_oracle(monkeypatch):
    """a 32-wide input: every layer through k_gcn_fwd_tc and mgcn_gcn_layer_bwd_tc_ex, layer 0 included"""
    _parity_vs_oracle(monkeypatch, dict(BOTNET_BIAS, in_channels=32, enc_sizes=[32] * 4), _graph20k, _wide, 0.5,
                      MASK_SEED, arbitrated=True)


@pytest.mark.gpu
def test_full_c1_graph_with_bias_vs_oracle(monkeypatch):
    """the full C1 graph, fp64 arbitrating the entries where the fp32 oracle itself is ~1e-5 away"""
    _parity_vs_oracle(monkeypatch, BOTNET_BIAS, _c1, _botnet_input, 0.0, MASK_SEED, arbitrated=True)


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.5])
def test_batch_equals_per_graph_and_graphed_adam_steps_equal_eager(p):
    """a batch of graphs equals the per-graph results bit for bit; three Adam steps replayed from one captured CUDA
    graph equal the eager steps bit for bit (after the first step the biases are non-zero)"""
    from meta_gcn_b200 import data as D
    from meta_gcn_b200 import dist as mdist
    from meta_gcn_b200 import functional as F
    from meta_gcn_b200.graphed import GraphedCall
    graphs = [D.synth_botnet_graph(seed=s, num_nodes=20000, edge_entries=220000, evil=1500) for s in (1, 2, 3)]
    batch = D.GraphBatch.from_data_list(graphs).to(DEV)
    batch.x = batch.x.contiguous()
    torch.manual_seed(3)
    model = GCNModel(**dict(BOTNET_BIAS, dropout=p)).to(DEV)
    with torch.no_grad():
        model.eval()
        whole = model(batch.x[:, 0].view(-1, 1), batch.edge_index, deg_K=batch.x[:, 1])
        for i, gph in enumerate(graphs):
            one = D.GraphBatch.from_data_list([gph]).to(DEV)
            part = model(one.x[:, 0].view(-1, 1), one.edge_index, deg_K=one.x[:, 1])
            assert_bitexact(whole[batch.slices_x[i]:batch.slices_x[i + 1]], part, f"graph {i} of the batch")
    model.train()
    state0 = {k: v.clone() for k, v in model.state_dict().items()}
    rng = torch.cuda.get_rng_state()             # the same dropout seeds in the eager and the replayed steps
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
            losses, biases = [], []
            for _ in range(3):
                loss_sum = call()
                mean_loss, _ = reducer.reduce_mean(loss_sum, batch.num_nodes)
                opt.step()
                losses.append(float(mean_loss))
                biases.append(float(model.gcn_net[1].gcn.node_models[0].bias.abs().max()))
            results.append((losses, [q.detach().clone() for q in model.parameters()], biases))
    torch.cuda.current_stream().wait_stream(work)
    assert results[0][0] == results[1][0], (results[0][0], results[1][0])
    for pe, pg in zip(results[0][1], results[1][1]):
        assert torch.equal(pe, pg)
    assert all(b > 0 for b in results[0][2])               # non-zero biases from the first update on
