"""Fused residual-GCN layer kernels (csrc/gcn_layer.cu) against an fp64 dense restatement of
gcn_model.py:89-106 / gcn_base_models.py:199-243 on the same seeded inputs: forward outputs, mask
words, and every backward product; ragged shapes (N not a multiple of the 16-row tile), empty rows,
hub rows (longer than the hub threshold) and isolated nodes included."""
import numpy as np
import pytest
import torch

from meta_gcn_b200 import ops
from meta_gcn_b200.graph import GraphStructure
from util import assert_bitexact, assert_parity

pytestmark = pytest.mark.gpu
DEV = "cuda"
H = 32


def rand_graph(n, e, seed, hubs=2):
    g = np.random.default_rng(seed)
    src = g.integers(0, n, e)
    dst = g.integers(0, n, e)
    # a few hub targets / hub sources, and nodes n-3.. left isolated
    for k in range(hubs):
        dst[g.integers(0, e, 300)] = k
        src[g.integers(0, e, 200)] = k + 5
    keep = (src < n - 3) & (dst < n - 3)
    ei = np.stack([src[keep], dst[keep]]).astype(np.int64)
    return torch.from_numpy(ei)


def dense_adj(ei, n):
    """A[i, j] = number of edges j -> i (row = target), fp64"""
    a = torch.zeros(n, n, dtype=torch.float64)
    a.index_put_((ei[1], ei[0]), torch.ones(ei.size(1), dtype=torch.float64), accumulate=True)
    return a


@pytest.mark.parametrize("n,e,act_out,with_next,resid_mode", [
    (1000, 9000, 1, True, False),
    (1003, 12000, 0, False, False),
    (517, 3000, 1, True, True),
    (16, 40, 1, True, False),
    (5, 0, 1, True, False),
])
def test_layer_fwd(n, e, act_out, with_next, resid_mode):
    ei = rand_graph(n, e, seed=n) if e else torch.zeros(2, 0, dtype=torch.int64)
    gen = torch.Generator().manual_seed(n + 1)
    m = torch.randn(n, H, generator=gen)
    x = torch.randn(n, H, generator=gen)
    res_w = torch.randn(H, H, generator=gen) / H ** 0.5
    res_b = torch.randn(H, generator=gen)
    w_next = torch.randn(H, H, generator=gen) / H ** 0.5
    pre = torch.rand(n, generator=gen) + 0.1
    post = torch.rand(n, generator=gen) + 0.1
    gs = GraphStructure(ei.to(DEV), n, hub_threshold=64)
    d = lambda t: t.to(DEV)
    resid = (x.double() @ res_w.double().t() + res_b.double()).float()
    xn, mn, hm = ops.gcn_layer_fwd_impl(
        gs.fwd, d(m), None if resid_mode else d(x), d(resid) if resid_mode else None, d(res_w), d(res_b),
        d(w_next) if with_next else None, None, d(pre), d(post), act_out)
    a = dense_adj(ei, n)
    h = torch.relu(post.double().view(-1, 1) * (a @ m.double()))
    y = h + (resid.double() if resid_mode else x.double() @ res_w.double().t() + res_b.double())
    x_ref = torch.relu(y) if act_out else y
    assert_parity(xn, x_ref, "x_next")
    if with_next:
        assert_parity(mn, pre.double().view(-1, 1) * (x_ref @ w_next.double()), "m_next")
    else:
        assert mn is None
    # mask words: bit c = h[:, c] > 0; compare where h is not within rounding of 0
    bits = hm.cpu().numpy().astype(np.uint32)
    got = ((bits[:, None] >> np.arange(H, dtype=np.uint32)[None, :]) & 1).astype(bool)
    hn = h.numpy()
    sure = np.abs(hn) > 1e-6 * max(1.0, np.abs(hn).max())
    assert (got[sure] == (hn[sure] > 0)).all()
    assert not got[hn == 0].any()


def test_layer_fwd_is_deterministic_and_order_exact():
    """row sums run in edge_index order: with unit factors and no dense part the h bits equal a
    sequential fp32 scatter_add (the reference's CPU order) for rows within the hub threshold"""
    n, e = 800, 6000
    ei = rand_graph(n, e, seed=3, hubs=0)
    gen = torch.Generator().manual_seed(0)
    m = torch.randn(n, H, generator=gen)
    zeros = torch.zeros(n, H)
    gs = GraphStructure(ei.to(DEV), n, hub_threshold=1 << 20)
    outs = []
    for _ in range(2):
        xn, _, _ = ops.gcn_layer_fwd_impl(gs.fwd, m.to(DEV), None, zeros.to(DEV), None, None, None, None,
                                          None, None, 0)
        outs.append(xn.cpu())
    assert_bitexact(outs[0], outs[1], "run-to-run")
    ref = torch.zeros(n, H).scatter_add_(0, ei[1].view(-1, 1).expand(-1, H), m[ei[0]])
    assert_bitexact(outs[0], torch.relu(ref), "edge-order sum")


@pytest.mark.parametrize("n,want_prev", [(1000, True), (1003, True), (131, False), (7, True), (40000, True), (300001, True), (151617, False)])
def test_layer_bwd(n, want_prev):
    gen = torch.Generator().manual_seed(n)
    dxw = torch.randn(n, H, generator=gen)
    gy = torch.randn(n, H, generator=gen)
    x = torch.randn(n, H, generator=gen)
    w = torch.randn(H, H, generator=gen) / H ** 0.5
    res_w = torch.randn(H, H, generator=gen) / H ** 0.5
    post = torch.rand(n, generator=gen) + 0.1
    bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), generator=gen, dtype=torch.int64).to(torch.int32)
    d = lambda t: t.to(DEV)
    gyp, gsp, dw, drw, drb = ops.gcn_layer_bwd_impl(d(dxw), d(gy), d(x), d(w), d(res_w), d(bits), d(post),
                                                    want_prev)
    D = lambda t: t.double()
    assert_parity(dw, D(x).t() @ D(dxw), "dW")
    assert_parity(drw, D(gy).t() @ D(x), "dR")
    assert_parity(drb, D(gy).sum(0), "dr")
    if not want_prev:
        assert gyp is None and gsp is None
        return
    G = D(dxw) @ D(w).t() + D(gy) @ D(res_w)
    gy_ref = G * (x > 0)
    assert_parity(gyp, gy_ref, "gy_prev")
    b = ((bits.numpy().astype(np.uint32)[:, None] >> np.arange(H, dtype=np.uint32)[None, :]) & 1).astype(np.float64)
    assert_parity(gsp, D(post).view(-1, 1) * gy_ref * torch.from_numpy(b), "gs_prev")
    gs2 = ops.mask_bits_scale_impl(d(gy), d(bits), d(post))
    assert_bitexact(gs2, post.view(-1, 1) * torch.where(torch.from_numpy(b > 0), gy, torch.zeros(())), "mask_bits_scale")


@pytest.mark.parametrize("n", [1000, 1003, 9])
def test_layer_fwd_row_local_mode(n):
    """csr None: m is the finished pre-activation of every row (first layer aggregated before its transform)"""
    gen = torch.Generator().manual_seed(n + 5)
    z = torch.randn(n, H, generator=gen)
    resid = torch.randn(n, H, generator=gen)
    w_next = torch.randn(H, H, generator=gen) / H ** 0.5
    pre = torch.rand(n, generator=gen) + 0.1
    d = lambda t: t.to(DEV)
    xn, mn, hm = ops.gcn_layer_fwd_impl(None, d(z), None, d(resid), None, None, d(w_next), None, d(pre), None, 1)
    h = torch.relu(z.double())
    x_ref = torch.relu(h + resid.double())
    assert_parity(xn, x_ref, "x_next")
    assert_parity(mn, pre.double().view(-1, 1) * (x_ref @ w_next.double()), "m_next")
    bits = hm.cpu().numpy().astype(np.uint32)
    got = ((bits[:, None] >> np.arange(H, dtype=np.uint32)[None, :]) & 1).astype(bool)
    assert (got == (z.numpy() > 0)).all()


@pytest.mark.parametrize("n,hin,act_out,with_next", [(1000, 1, 1, True), (1003, 2, 0, False), (37, 4, 1, True), (150001, 1, 1, True),
                                                     (1001, 1, 1, None)])
def test_first_layer_fwd_narrow_input(n, hin, act_out, with_next):
    """mgcn_gcn_first_layer_fwd: h = relu(post (s W)), y = h + x R^T + r, x' = act(y), m' = pre (x' W') from the
    two [N, H_in] operands (gcn_base_models.py:199-243 + gcn_model.py:96-105 for layer 0), fp64 restatement"""
    gen = torch.Generator().manual_seed(n + hin)
    s = torch.randn(n, hin, generator=gen)
    x = torch.randn(n, hin, generator=gen)
    w_in = torch.randn(hin, H, generator=gen)
    res_w = torch.randn(H, hin, generator=gen)
    res_b = torch.randn(H, generator=gen)
    w_next = torch.randn(H, H, generator=gen) / H ** 0.5
    pre = torch.rand(n, generator=gen) + 0.1
    post = torch.rand(n, generator=gen) + 0.1
    d = lambda t: t.to(DEV)
    out_scale = torch.rand(n, generator=gen) + 0.1 if with_next is None else None   # the scaled-rows output format
    xn, mn, hm = ops.gcn_first_layer_fwd_impl(d(s), d(x), d(w_in), d(res_w), d(res_b), d(w_next) if with_next else None,
                                              d(pre), d(post), act_out,
                                              out_scale=None if out_scale is None else d(out_scale))
    D = lambda t: t.double()
    z = D(post).view(-1, 1) * (D(s) @ D(w_in))
    y = torch.relu(z) + D(x) @ D(res_w).t() + D(res_b)
    x_ref = torch.relu(y) if act_out else y
    if out_scale is not None:
        x_ref = x_ref * D(out_scale).view(-1, 1)
    assert_parity(xn, x_ref, "x_next")
    if with_next:
        assert_parity(mn, D(pre).view(-1, 1) * (x_ref @ D(w_next)), "m_next")
    else:
        assert mn is None
    bits = hm.cpu().numpy().astype(np.uint32)
    got = ((bits[:, None] >> np.arange(H, dtype=np.uint32)[None, :]) & 1).astype(bool)
    zf = (post.view(-1, 1) * (s @ w_in)).numpy()
    sure = np.abs(z.numpy()) > 1e-5          # sign of z is unambiguous away from zero
    assert (got == (zf > 0))[sure].all()


def test_giant_hub_rows_cta_wide_reduce():
    """rows with more than 32 hub segments (k_hub_reduce's CTA-wide path) next to ordinary hubs: the hidden-32
    aggregation equals the edge-order scatter_add within fp32 rounding and is run-to-run identical"""
    n = 4000
    g = np.random.default_rng(7)
    src = g.integers(0, n, 30000)
    dst = g.integers(0, n, 30000)
    dst[:9000] = 11           # 141 segments at threshold 64
    dst[9000:12500] = 12      # 55 segments
    dst[12500:13000] = 13     # 8 segments: warp path
    ei = torch.from_numpy(np.stack([src, dst]).astype(np.int64))
    x = torch.randn(n, H, generator=torch.Generator().manual_seed(3))
    gs = GraphStructure(ei.to(DEV), n, hub_threshold=64)
    outs = [ops.aggregate_prescaled_impl(gs.fwd, x.to(DEV), None, 0, None, None, 0).cpu() for _ in range(2)]
    assert_bitexact(outs[0], outs[1], "run-to-run")
    ref = torch.zeros(n, H, dtype=torch.float64).index_add_(0, ei[1], x.double()[ei[0]])
    assert_parity(outs[0], ref, "aggregation with giant hubs")


def _giant_hub_graph(n=4000):
    g = np.random.default_rng(7)
    src = g.integers(0, n, 30000)
    dst = g.integers(0, n, 30000)
    dst[:9000] = 11           # 141 segments at threshold 64
    dst[9000:12500] = 12      # 55 segments
    dst[12500:13000] = 13     # 8 segments
    return torch.from_numpy(np.stack([src, dst]).astype(np.int64))


@pytest.mark.parametrize("n,e,act_out,scaled,with_bias", [
    (1000, 9000, 1, True, False),
    (1003, 12000, 0, True, True),
    (517, 3000, 1, False, False),
    (128, 700, 1, True, False),
    (16, 40, 1, True, True),
    (5, 0, 1, True, False),
    (40000, 400000, 1, True, False),
    (4000, -1, 1, True, False),      # giant hubs (141 / 55 / 8 segments)
    (300001, 1500000, 1, True, False),
])
def test_layer_fwd_tc_aggregate_then_transform(n, e, act_out, scaled, with_bias):
    """mgcn_gcn_layer_fwd_tc against an fp64 dense / sparse restatement of gcn_model.py:89-106 +
    gcn_base_models.py:199-243 with the stored format z = sigma (.) x: outputs (scaled by out_scale), mask words;
    ragged tile counts, empty rows, isolated nodes, hub rows, several tiles per CTA."""
    if e == -1:
        ei = _giant_hub_graph(n)
    else:
        ei = rand_graph(n, e, seed=n) if e else torch.zeros(2, 0, dtype=torch.int64)
    gen = torch.Generator().manual_seed(n + 11)
    x = torch.randn(n, H, generator=gen)
    w = torch.randn(H, H, generator=gen) / H ** 0.5
    res_w = torch.randn(H, H, generator=gen) / H ** 0.5
    res_b = torch.randn(H, generator=gen)
    bias = torch.randn(H, generator=gen) if with_bias else None
    sigma = torch.rand(n, generator=gen) + 0.1 if scaled else None
    post = torch.rand(n, generator=gen) + 0.1
    outs = torch.rand(n, generator=gen) + 0.1 if scaled else None
    z = x * sigma.view(-1, 1) if scaled else x
    gs = GraphStructure(ei.to(DEV), n, hub_threshold=64)
    d = lambda t: None if t is None else t.to(DEV)
    zn, hm = ops.gcn_layer_fwd_tc_impl(gs.fwd, d(z), d(w), d(res_w), d(res_b), d(bias), d(sigma), d(post), d(outs),
                                       act_out)
    D = lambda t: t.double()
    agg = torch.zeros(n, H, dtype=torch.float64).index_add_(0, ei[1], D(z)[ei[0]])
    s = D(post).view(-1, 1) * agg
    pre_act = s @ D(w) + (D(bias) if with_bias else 0.0)
    h = torch.relu(pre_act)
    xin = D(z) / D(sigma).view(-1, 1) if scaled else D(z)
    y = h + xin @ D(res_w).t() + D(res_b)
    x_ref = torch.relu(y) if act_out else y
    if scaled:
        x_ref = x_ref * D(outs).view(-1, 1)
    assert_parity(zn, x_ref, "z_next")
    bits = hm.cpu().numpy().astype(np.uint32)
    got = ((bits[:, None] >> np.arange(H, dtype=np.uint32)[None, :]) & 1).astype(bool)
    hn = pre_act.numpy()
    sure = np.abs(hn) > 1e-5 * max(1.0, np.abs(hn).max())
    assert (got[sure] == (hn[sure] > 0)).all()
    # run-to-run identical (fixed summation orders, no atomics on data)
    zn2, hm2 = ops.gcn_layer_fwd_tc_impl(gs.fwd, d(z), d(w), d(res_w), d(res_b), d(bias), d(sigma), d(post), d(outs),
                                         act_out)
    assert_bitexact(zn, zn2, "run-to-run")
    assert_bitexact(hm, hm2, "run-to-run mask")


@pytest.mark.parametrize("n", [1000, 40000])
def test_layer_bwd_tc_scaled_input(n):
    """x_scale: the x operand of the tcgen05 backward is stored as sigma (.) x"""
    gen = torch.Generator().manual_seed(n)
    dxw, gy, x = (torch.randn(n, H, generator=gen) for _ in range(3))
    w = torch.randn(H, H, generator=gen) / H ** 0.5
    res_w = torch.randn(H, H, generator=gen) / H ** 0.5
    post = torch.rand(n, generator=gen) + 0.1
    sigma = torch.rand(n, generator=gen) + 0.1
    bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), generator=gen, dtype=torch.int64).to(torch.int32)
    d = lambda t: t.to(DEV)
    gyp, gsp, dw, drw, drb = ops.gcn_layer_bwd_impl(d(dxw), d(gy), d(x * sigma.view(-1, 1)), d(w), d(res_w), d(bits),
                                                    d(post), True, True, x_scale=d(sigma))
    D = lambda t: t.double()
    assert_parity(dw, D(x).t() @ D(dxw), "dW")
    assert_parity(drw, D(gy).t() @ D(x), "dR")
    assert_parity(drb, D(gy).sum(0), "dr")
    G = D(dxw) @ D(w).t() + D(gy) @ D(res_w)
    assert_parity(gyp, G * (x > 0), "gy_prev")


@pytest.mark.parametrize("n,e,scaled,want_prev", [
    (1000, 9000, True, True),
    (1003, 12000, True, True),
    (517, 3000, False, True),
    (131, 700, True, False),
    (16, 40, True, True),
    (5, 0, True, True),
    (40000, 400000, True, True),
    (4000, -1, True, True),          # giant hubs (141 / 55 / 8 segments)
    (300001, 1500000, True, True),
    (151617, 700000, True, False),
])
def test_layer_bwd_two_launch(n, e, scaled, want_prev):
    """the layer backward of the hidden-32 stack as it runs there, mgcn_aggregate_prescaled over the by-source structure
    followed by mgcn_gcn_layer_bwd_tc, against an fp64 restatement of the autograd of gcn_model.py:89-106 /
    gcn_base_models.py:199-243 in the stored format z = sigma (.) x: ragged tile counts, rows without entries, hub rows,
    several tiles per CTA."""
    if e == -1:
        ei = _giant_hub_graph(n)
    else:
        ei = rand_graph(n, e, seed=n) if e else torch.zeros(2, 0, dtype=torch.int64)
    gen = torch.Generator().manual_seed(n + 23)
    gs_in = torch.randn(n, H, generator=gen)
    gy = torch.randn(n, H, generator=gen)
    x = torch.randn(n, H, generator=gen)
    w = torch.randn(H, H, generator=gen) / H ** 0.5
    res_w = torch.randn(H, H, generator=gen) / H ** 0.5
    post = torch.rand(n, generator=gen) + 0.1
    pre = torch.rand(n, generator=gen) + 0.1 if scaled else None
    sigma = torch.rand(n, generator=gen) + 0.1 if scaled else None
    bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), generator=gen, dtype=torch.int64).to(torch.int32)
    z = x * sigma.view(-1, 1) if scaled else x
    struct = GraphStructure(ei.to(DEV), n, hub_threshold=64)
    d = lambda t: None if t is None else t.to(DEV)

    def backward():
        dxw = ops.aggregate_prescaled_impl(struct.bwd, d(gs_in), d(pre), 0, None, None, 0)
        return ops.gcn_layer_bwd_impl(dxw, d(gy), d(z), d(w), d(res_w), d(bits), d(post), want_prev, x_scale=d(sigma))

    gyp, gsp, dw, drw, drb = backward()
    D = lambda t: t.double()
    # dxw_j = pre_j * sum over edges j -> i of gs_i
    dxw = torch.zeros(n, H, dtype=torch.float64).index_add_(0, ei[0], D(gs_in)[ei[1]])
    if scaled:
        dxw = dxw * D(pre).view(-1, 1)
    xin = D(z) / D(sigma).view(-1, 1) if scaled else D(z)
    assert_parity(dw, xin.t() @ dxw, "dW")
    assert_parity(drw, D(gy).t() @ xin, "dR")
    assert_parity(drb, D(gy).sum(0), "dr")
    if not want_prev:
        assert gyp is None and gsp is None
        return
    G = dxw @ D(w).t() + D(gy) @ D(res_w)
    gy_ref = G * (x > 0)
    assert_parity(gyp, gy_ref, "gy_prev")
    b = ((bits.numpy().astype(np.uint32)[:, None] >> np.arange(H, dtype=np.uint32)[None, :]) & 1).astype(np.float64)
    assert_parity(gsp, D(post).view(-1, 1) * gy_ref * torch.from_numpy(b), "gs_prev")
    # run-to-run identical (fixed summation orders, no atomics on data)
    again = backward()
    for got, ref, name in zip((gyp, gsp, dw, drw, drb), again, ("gy_prev", "gs_prev", "dW", "dR", "dr")):
        assert_bitexact(got, ref, "run-to-run " + name)
