"""The 'max' aggregation (k_segment_max, k_segment_max_bwd, k_scatter_max_bwd) and the per-edge dot product
(k_edge_dot) against exact references, at sizes where the grid-stride loops take several passes, with hub rows,
empty rows, duplicate edges, self loops and exact ties, and on both sides of torch_scatter's fill value.

The max kernels are checked bit for bit: the maximum of fp32 values and the first position attaining it are exact,
and the layer-seam backward adds, per source, the routed gradients in edge order — what an unbuffered np.add.at in
edge order does.  The dot products are checked against fp64 with a per-edge bound."""
import numpy as np
import pytest
import torch

from meta_gcn_b200 import functional as F_mgcn
from meta_gcn_b200 import ops
from meta_gcn_b200.data import synth_botnet_graph
from meta_gcn_b200.gcn_meta.models import GCNModel
from meta_gcn_b200.graph import GraphStructure
from oracle import port
from util import assert_bitexact, assert_parity

pytestmark = pytest.mark.gpu
DEV = "cuda"
FLT_MAX = float(np.finfo(np.float32).max)
F32 = np.float32
# the max kernels cap their grid at 148 * 16 blocks of 256 threads: one pass covers this many (row, column) pairs
ONE_PASS = 148 * 16 * 256


# ------------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------------
def first_max_ref(vals, rows, n, fill=None):
    """torch_scatter's scatter_max over vals [E,H] fp32 (edge order) grouped by rows [E] into n rows ->
    (out [n,H] fp32, arg [n,H] int64): arg = the edge id of the first entry attaining the row's maximum, out =
    vals[arg] (so a tie between -0 and +0 keeps the winning entry's bits); (0, -1) where nothing wins (an empty row,
    or with ``fill`` every entry <= fill)."""
    vals = np.asarray(vals, dtype=F32)
    if vals.ndim == 1:
        vals = vals[:, None]
    rows = np.asarray(rows, dtype=np.int64)
    E, H = vals.shape
    out = np.zeros((n, H), dtype=F32)
    arg = np.full((n, H), -1, dtype=np.int64)
    if E == 0:
        return out, arg
    order = np.argsort(rows, kind="stable")
    sr, sv = rows[order], vals[order]
    starts = np.flatnonzero(np.r_[True, sr[1:] != sr[:-1]])
    group = np.cumsum(np.r_[True, sr[1:] != sr[:-1]]) - 1
    ok = np.ones_like(sv, dtype=bool) if fill is None else sv > F32(fill)
    masked = np.where(ok, sv, F32(-np.inf))
    m = np.maximum.reduceat(masked, starts, axis=0)
    hit = ok & (sv == m[group])
    pos = np.arange(E, dtype=np.int64)[:, None]
    first = np.minimum.reduceat(np.where(hit, pos, E), starts, axis=0)
    won = first < E
    edge = np.where(won, order[np.minimum(first, E - 1)], -1)
    tgt = sr[starts]
    arg[tgt] = edge
    out[tgt] = np.where(won, np.take_along_axis(vals, np.maximum(edge, 0), axis=0), F32(0))
    return out, arg


def scatter_max_grad_ref(arg, g, n_src):
    """primitive-seam backward: dsrc [n_src,H] = 0, dsrc[arg[i,c], c] = g[i,c] where arg >= 0"""
    g = np.asarray(g, dtype=F32).reshape(arg.shape)
    d = np.zeros((n_src, arg.shape[1]), dtype=F32)
    i, c = np.nonzero(arg >= 0)
    d[arg[i, c], c] = g[i, c]
    return d


def layer_max_grad_ref(arg, g, src, ev, n):
    """layer-seam backward in fp32: dx[src_e, c] += g[i,c] * ev[e] for every (i,c) won by edge e, added per source
    in edge order from 0 (np.add.at is unbuffered and sequential)"""
    i, c = np.nonzero(arg >= 0)
    e = arg[i, c]
    v = np.asarray(g, dtype=F32)[i, c]
    if ev is not None:
        v = v * np.asarray(ev, dtype=F32)[e]
    o = np.argsort(e, kind="stable")
    dx = np.zeros((n, arg.shape[1]), dtype=F32)
    np.add.at(dx, (np.asarray(src)[e[o]], c[o]), v[o])
    return dx


def edge_dot_ref(ei, a, b):
    """fp64 <a[col_e], b[row_e]> and sum_k |a[col_e,k] b[row_e,k]| per edge (chunked over the edges)"""
    r, c = np.asarray(ei[0]), np.asarray(ei[1])
    E, H = r.shape[0], a.shape[1]
    dot, mag = np.zeros(E), np.zeros(E)
    step = max(1, (1 << 22) // H)
    for s in range(0, E, step):
        p = a[c[s:s + step]].astype(np.float64) * b[r[s:s + step]].astype(np.float64)
        dot[s:s + step] = p.sum(1)
        mag[s:s + step] = np.abs(p).sum(1)
    return dot, mag


def check_edge_dot(actual, dot, mag, s, H, slack, what):
    """|actual - s*dot| <= (H + slack) 2^-24 |s| sum|a_k b_k| per edge: the fp32 error of an H-term dot product and of
    the scale multiplications, judged edge by edge (a cancelling edge is not measured against the largest one)"""
    a = actual.detach().cpu().numpy().astype(np.float64)
    ref = s * dot
    bound = (H + slack) * 2.0 ** -24 * np.abs(s) * mag
    bad = np.abs(a - ref) > bound
    assert not bad.any(), (f"{what}: {int(bad.sum())}/{a.size} edges outside the per-edge bound, worst excess "
                           f"{np.max(np.abs(a - ref) - bound):.3e}")


# ------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------
_GRAPHS = {}


def hub_graph(n, hub_in=50_000, hub_out=0, seed=0):
    """edge_index int64 [2,E] on n nodes, in shuffled (unsorted) order: one target with hub_in in-edges, optionally
    one source with hub_out out-edges, a dozen rows above the hub threshold, ~2 random edges per node, self loops,
    repeated edges, and a tenth of the nodes isolated.  Returns (edge_index, hub_target, hub_source)."""
    key = (n, hub_in, hub_out, seed)
    if key not in _GRAPHS:
        rng = np.random.default_rng(seed)
        active = rng.permutation(n)[: n - n // 10]
        ht, hs = int(active[0]), int(active[1])
        src = [rng.choice(active, hub_in), np.full(hub_out, hs)]
        dst = [np.full(hub_in, ht), rng.choice(active, hub_out)]
        for t in active[2:14]:
            k = int(rng.integers(65, 400))
            src.append(rng.choice(active, k))
            dst.append(np.full(k, t))
        src.append(rng.choice(active, 2 * n))
        dst.append(rng.choice(active, 2 * n))
        loops = rng.choice(active, min(200, len(active)), replace=False)
        src.append(loops)
        dst.append(loops)
        s, d = np.concatenate(src), np.concatenate(dst)
        dup = rng.choice(len(s), len(s) // 20)
        s, d = np.concatenate([s, s[dup]]), np.concatenate([d, d[dup]])
        perm = rng.permutation(len(s))
        _GRAPHS[key] = (np.stack([s[perm], d[perm]]).astype(np.int64), ht, hs)
    return _GRAPHS[key]


def node_values(kind, n, H, rng):
    if kind == "normal":
        return rng.standard_normal((n, H)).astype(F32)
    if kind == "ties":
        return rng.integers(-2, 3, (n, H)).astype(F32)
    assert kind == "const"                        # one feature that is the same on every node (botnet x = ones)
    x = rng.standard_normal((n, H)).astype(F32)
    x[:, 0] = 1.0
    return x


def edge_values(kind, ei, n, rng):
    if kind is None:
        return None
    if kind == "norm":                            # degree normalisation: positive, many equal values
        deg = np.bincount(ei[0], minlength=n).astype(F32)
        dis = np.where(deg > 0, np.maximum(deg, 1) ** F32(-0.5), F32(0)).astype(F32)
        return (dis[ei[0]] * dis[ei[1]]).astype(F32)
    assert kind == "mixed"                        # both signs and zeros: x * 0 gives +0 and -0, which tie
    return rng.choice(np.array([-1.5, -1.0, -0.5, 0.0, 0.0, 0.5, 1.0, 2.0], dtype=F32), ei.shape[1])


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


# ------------------------------------------------------------------------------------------------
# 1. layer seam forward
# ------------------------------------------------------------------------------------------------
# (H, n): n*H below and above one grid pass
LAYER_SHAPES = [(1, 200_003), (3, 200_003), (4, 200_003), (16, 20_000), (32, 20_000), (33, 60_000), (64, 8_000),
                (128, 8_000), (257, 3_001)]


def test_layer_shapes_cover_one_and_several_grid_passes():
    sizes = [H * n for H, n in LAYER_SHAPES]
    assert min(sizes) < ONE_PASS < max(sizes) and sum(s > 3 * ONE_PASS for s in sizes) >= 1


@pytest.mark.parametrize("values", ["normal", "ties", "const"])
@pytest.mark.parametrize("H,n", LAYER_SHAPES)
def test_segment_max_layer_seam_forward_bitexact(H, n, values):
    ei, ht, _ = hub_graph(n)
    rng = np.random.default_rng(H * 7 + len(values))
    x = node_values(values, n, H, rng)
    gs = GraphStructure(dev(ei), n)
    assert int(gs.fwd.rowptr[ht + 1] - gs.fwd.rowptr[ht]) >= 50_000
    for ev_kind in (None, "norm", "mixed"):
        ev = edge_values(ev_kind, ei, n, rng)
        vals = x[ei[0]] if ev is None else x[ei[0]] * ev[:, None]
        out_r, arg_r = first_max_ref(vals, ei[1], n)
        ev_fwd = None if ev is None else gs.edge_values(dev(ev))[0]
        out, arg = ops.segment_max_impl(gs.fwd, dev(x), False, ev_fwd)
        assert_bitexact(out, out_r, f"out H={H} n={n} {values} edge_val={ev_kind}")
        assert_bitexact(arg, arg_r.astype(np.int32), f"arg H={H} n={n} {values} edge_val={ev_kind}")


# ------------------------------------------------------------------------------------------------
# 2. primitive seam: forward through the three public entry points, backward bit-exact
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("E,H,dim_size", [(1_000_003, 1, 1_300_000), (400_009, 3, 250_000), (150_001, 8, 90_000),
                                          (5_000, 5, 7_000)])
def test_scatter_max_primitive_seam_bitexact(E, H, dim_size):
    from meta_gcn_b200.compat.torch_scatter import scatter_max
    from meta_gcn_b200.gcn_meta.models import scatter_
    rng = np.random.default_rng(E)
    top = dim_size - 17                           # the last rows receive nothing
    index = rng.integers(0, top, E)
    index[rng.choice(E, min(50_000, E // 3), replace=False)] = top // 2        # a hub row
    src = rng.standard_normal((E, H)).astype(F32)
    src[:, ::2] = rng.integers(-2, 3, (E, (H + 1) // 2))                        # tie-heavy columns
    out_r, arg_r = first_max_ref(src, index, dim_size, fill=-1e38)
    squeeze = H == 1                              # the 1-D form of the call
    s = dev(src[:, 0] if squeeze else src).requires_grad_(True)
    idx = dev(index)
    out, arg = F_mgcn.scatter_rows_max(s, idx, dim_size)
    shape = (dim_size,) if squeeze else (dim_size, H)
    assert_bitexact(out, out_r.reshape(shape), "scatter_rows_max out")
    assert_bitexact(arg, arg_r.reshape(shape), "scatter_rows_max arg")
    g = rng.standard_normal((dim_size, H)).astype(F32)
    out.backward(dev(g.reshape(shape)))
    assert_bitexact(s.grad, scatter_max_grad_ref(arg_r, g, E).reshape(s.shape), "scatter_max backward")
    with torch.no_grad():
        assert_bitexact(scatter_("max", s, idx, dim_size=dim_size), out_r.reshape(shape), "scatter_('max')")
        o2, a2 = scatter_max(s, idx, 0, None, dim_size)
    assert_bitexact(a2, arg_r.reshape(shape), "compat scatter_max arg")
    assert_bitexact(o2, np.where(arg_r >= 0, out_r, -FLT_MAX).astype(F32).reshape(shape), "compat scatter_max out")


def test_duplicate_edges_route_the_gradient_to_the_first_copy():
    """(0 -> 1) three times, (2 -> 1) once: node 1's maximum comes from node 0, and only the first copy of the
    repeated edge receives its gradient, at both seams"""
    ei = dev(np.array([[2, 0, 0, 3, 0], [1, 1, 1, 0, 1]], dtype=np.int64))
    x = dev(np.array([[5.0], [0.0], [1.0], [2.0]], dtype=F32)).requires_grad_(True)
    out = F_mgcn.aggregate_max(x, GraphStructure(ei, 4))
    out.backward(dev(np.array([[7.0], [3.0], [11.0], [13.0]], dtype=F32)))
    assert out[:, 0].tolist() == [2.0, 5.0, 0.0, 0.0]
    assert x.grad[:, 0].tolist() == [3.0, 0.0, 0.0, 7.0]
    msg = x.detach()[ei[0]].clone().requires_grad_(True)
    out, arg = F_mgcn.scatter_rows_max(msg, ei[1], 4)
    assert arg[:, 0].tolist() == [3, 1, -1, -1]
    out.backward(torch.ones_like(out))
    assert msg.grad[:, 0].tolist() == [0.0, 1.0, 0.0, 1.0, 0.0]


# ------------------------------------------------------------------------------------------------
# 3. layer seam backward
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("values,ev_kind", [("normal", None), ("ties", "mixed"), ("const", "norm")])
@pytest.mark.parametrize("H,n", [(1, 200_003), (33, 60_000), (128, 8_000)])
def test_aggregate_max_backward_bitexact(H, n, values, ev_kind):
    ei, _, hs = hub_graph(n, hub_out=50_000, seed=1)
    rng = np.random.default_rng(H + n)
    x = node_values(values, n, H, rng)
    x[hs] += 2.0                                  # the source hub wins often
    ev = edge_values(ev_kind, ei, n, rng)
    gs = GraphStructure(dev(ei), n)
    assert int(gs.bwd.rowptr[hs + 1] - gs.bwd.rowptr[hs]) >= 50_000
    vals = x[ei[0]] if ev is None else x[ei[0]] * ev[:, None]
    out_r, arg_r = first_max_ref(vals, ei[1], n, fill=-1e38)
    g = rng.standard_normal((n, H)).astype(F32)
    dx_r = layer_max_grad_ref(arg_r, g, ei[0], ev, n)
    grads = []
    for _ in range(2):
        xt = dev(x).requires_grad_(True)
        out = F_mgcn.aggregate_max(xt, gs, None if ev is None else dev(ev))
        out.backward(dev(g))
        grads.append(xt.grad)
    assert_bitexact(out, out_r, "aggregate_max out")
    assert_bitexact(grads[0], dx_r, "aggregate_max dx")
    assert_bitexact(grads[1], grads[0], "aggregate_max dx, run to run")


# ------------------------------------------------------------------------------------------------
# 4. torch_scatter's fill value: an entry <= fill never wins
# ------------------------------------------------------------------------------------------------
def _fill_rows():
    """(src [E,2] fp32, index [E], dim_size): rows on both sides of the fills -1e38, -1e16, -1e9 and -FLT_MAX,
    column 1 holding each row's entries in reverse"""
    inf = float("inf")
    rows = [[-2e38, -2e38, -3e38], [-FLT_MAX, -FLT_MAX], [-inf, -inf, -inf], [-1e38, -1e38],
            [-2e38, -1e38, -FLT_MAX, -inf], [-2e38, -9.9e37, -1e38, -9.9e37], [1.5, -0.0, 0.0, 1.5],
            [],                                                                 # empty
            [-1e16, -1e16], [-2e16, -5e15, -1e16, -5e15], [-1e9, -1e9], [-3e9, -1e9, -2e8, -2e8],
            [-FLT_MAX, -5e37], [-0.0, 0.0], [0.0, -0.0, -inf]]
    v0, v1, idx = [], [], []
    for r, vs in enumerate(rows):
        v0 += vs
        v1 += vs[::-1]
        idx += [r] * len(vs)
    # interleave the rows in edge order, keeping each row's entries in the order listed
    index = np.asarray(idx, dtype=np.int64)[np.random.default_rng(5).permutation(len(idx))]
    src = np.empty((len(idx), 2), dtype=F32)
    src[np.argsort(index, kind="stable")] = np.stack([np.asarray(v0, dtype=F32), np.asarray(v1, dtype=F32)], 1)
    return src, index, len(rows) + 3


def test_fill_rows_cover_both_sides_of_each_fill():
    src, index, n = _fill_rows()
    rmax = np.full(n, -np.inf, dtype=F32)
    np.maximum.at(rmax, index, src[:, 0])
    rmax = rmax[np.bincount(index, minlength=n) > 0]
    for f in (-1e38, -1e16, -1e9, -FLT_MAX):
        f = F32(f)
        assert (rmax < f).any() and (rmax > f).any() and (src == f).any(), f


def test_scatter_max_fill_matches_reference():
    """common.py's scatter_('max') (fill -1e38, untouched entries 0) at the layer seam and the primitive seam: values
    against the oracle's scatter_rows, argmax and gradient against the first-maximum rule of segment_max_first"""
    from meta_gcn_b200.gcn_meta.models import scatter_
    src, index, n = _fill_rows()
    E = src.shape[0]
    s_cpu, i_cpu = torch.from_numpy(src), torch.from_numpy(index)
    out_r = port.scatter_rows("max", s_cpu, i_cpu, n)
    _, arg_r = port.segment_max_first(s_cpu, i_cpu, n)
    w = np.random.default_rng(1).standard_normal((n, 2)).astype(F32)
    grad_r = scatter_max_grad_ref(arg_r, w, E)

    s = dev(src).requires_grad_(True)
    out = scatter_("max", s, dev(index), dim_size=n)
    assert_bitexact(out, out_r, "scatter_('max') out")
    out.backward(dev(w))
    assert_bitexact(s.grad, grad_r, "scatter_('max') gradient")
    assert_bitexact(F_mgcn.scatter_rows_max(s.detach(), dev(index), n)[1], arg_r, "scatter_rows_max arg")

    # layer seam: node e's feature row is src[e], edge e runs e -> index[e]
    N = max(E, n)
    x = np.zeros((N, 2), dtype=F32)
    x[:E] = src
    xt = dev(x).requires_grad_(True)
    gs = GraphStructure(dev(np.stack([np.arange(E), index])), N)
    out = F_mgcn.aggregate_max(xt, gs)
    assert_bitexact(out[:n], out_r, "aggregate_max out")
    assert_bitexact(out[n:], np.zeros((N - n, 2), dtype=F32), "aggregate_max empty rows")
    wN = np.zeros((N, 2), dtype=F32)
    wN[:n] = w
    out.backward(dev(wN))
    dx_r = np.zeros((N, 2), dtype=F32)
    dx_r[:E] = grad_r
    assert_bitexact(xt.grad, dx_r, "aggregate_max gradient")


@pytest.mark.parametrize("fill", [-1e16, None])
def test_compat_scatter_max_fill_matches_torch_scatter(fill):
    """compat torch_scatter.scatter_max (softmax passes -1e16; the default is the dtype's lowest value) against the
    oracle's torch_scatter 1.x: out = max(fill, entries), argmax -1 where no entry exceeds the fill, gradient to the
    argmax only"""
    from meta_gcn_b200.compat.torch_scatter import scatter_max
    from oracle.shim import torch_scatter as ts_ref
    src, index, n = _fill_rows()
    w = np.random.default_rng(2).standard_normal((n, 2)).astype(F32)
    s_cpu = torch.from_numpy(src).requires_grad_(True)
    o_r, a_r = ts_ref.scatter_max(s_cpu, torch.from_numpy(index), 0, None, n, fill)
    (o_r * torch.from_numpy(w)).sum().backward()
    s = dev(src).requires_grad_(True)
    o, a = scatter_max(s, dev(index), 0, None, n, fill)
    assert_bitexact(o, o_r, f"scatter_max out, fill {fill}")
    assert_bitexact(a, a_r, f"scatter_max arg, fill {fill}")
    o.backward(dev(w))
    assert_bitexact(s.grad, s_cpu.grad, f"scatter_max gradient, fill {fill}")


def test_pyg_scatter_max_fill_matches_reference():
    """compat torch_geometric.utils.scatter_('max'): torch_scatter's scatter_max from -1e9, entries still at the fill
    set to 0 (PyG 1.3)"""
    from meta_gcn_b200.compat.torch_geometric.utils import scatter_ as pyg_scatter_
    from oracle.shim import torch_scatter as ts_ref
    src, index, n = _fill_rows()
    w = np.random.default_rng(3).standard_normal((n, 2)).astype(F32)
    s_cpu = torch.from_numpy(src).requires_grad_(True)
    o_r = ts_ref.scatter_max(s_cpu, torch.from_numpy(index), 0, None, n, -1e9)[0]
    o_r = torch.where(o_r == F32(-1e9), torch.zeros_like(o_r), o_r)
    (o_r * torch.from_numpy(w)).sum().backward()
    s = dev(src).requires_grad_(True)
    o = pyg_scatter_("max", s, dev(index), n)
    assert_bitexact(o, o_r, "PyG scatter_('max') out")
    o.backward(dev(w))
    assert_bitexact(s.grad, s_cpu.grad, "PyG scatter_('max') gradient")


# ------------------------------------------------------------------------------------------------
# 5. per-edge dot product
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("E", [0, 1, 7, 33, 75_777, 1_000_003])
@pytest.mark.parametrize("H", [1, 2, 7, 8, 9, 16, 33, 64, 100, 256])
def test_edge_dot_against_fp64(H, E):
    rng = np.random.default_rng(H * 1000 + E)
    N = 100_003 if E > 100_000 else 5_003
    ei = rng.integers(0, N, (2, E))
    a = rng.standard_normal((N, H)).astype(F32)
    b = rng.standard_normal((N, H)).astype(F32)
    ss = rng.standard_normal(N).astype(F32)
    st = rng.standard_normal(N).astype(F32)
    dot, mag = edge_dot_ref(ei, a, b)
    ta, tb, tss, tst = dev(a), dev(b), dev(ss), dev(st)
    ei64 = dev(ei)
    ei32 = ei64.to(torch.int32)
    for name, s_src, s_tgt in [("none", None, None), ("src", tss, None), ("tgt", None, tst), ("both", tss, tst)]:
        out = ops.edge_dot_impl(ei64, ta, tb, s_src, s_tgt)
        assert out.shape == (E,)
        s = np.ones(E)
        if s_src is not None:
            s = s * ss[ei[0]].astype(np.float64)
        if s_tgt is not None:
            s = s * st[ei[1]].astype(np.float64)
        check_edge_dot(out, dot, mag, s, H, 5, f"edge_dot H={H} E={E} scales={name}")
        assert_bitexact(ops.edge_dot_impl(ei32, ta, tb, s_src, s_tgt), out.cpu(), f"edge_dot int32 H={H} E={E}")


def test_edge_dot_rejects_other_index_types():
    a = torch.ones(4, 3, device=DEV)
    for bad in (torch.zeros(2, 5, dtype=torch.int16, device=DEV), torch.zeros(2, 5, device=DEV),
                torch.zeros(3, 5, dtype=torch.int64, device=DEV)):
        with pytest.raises(TypeError):
            ops.edge_dot_impl(bad, a, a)


# ------------------------------------------------------------------------------------------------
# 6. gradient w.r.t. a per-edge weight (the edge-gate path) through F.aggregate
# ------------------------------------------------------------------------------------------------
def _aggregate_ref(ei, n, x, ew, s_nbr, s_row, reduce, bias, mask, w):
    """torch fp64 CPU autograd of the explicit message form: x[row] * w_e * s_nbr[row] * s_row[col] index_added into
    col (mean: divided by the in-degree clamped to 1), + bias, ReLU with the given mask"""
    row, col = torch.from_numpy(ei[0]), torch.from_numpy(ei[1])
    x64 = torch.from_numpy(x).double().requires_grad_(True)
    ew64 = torch.from_numpy(ew).double().requires_grad_(True)
    b64 = None if bias is None else torch.from_numpy(bias).double().requires_grad_(True)
    f = ew64
    if s_nbr is not None:
        f = f * torch.from_numpy(s_nbr).double()[row]
    if s_row is not None:
        f = f * torch.from_numpy(s_row).double()[col]
    agg = torch.zeros(n, x.shape[1], dtype=torch.float64).index_add(0, col, x64[row] * f[:, None])
    if reduce == "mean":
        agg = agg / torch.bincount(col, minlength=n).clamp(min=1).double()[:, None]
    if b64 is not None:
        agg = agg + b64
    pre = agg.detach().clone()
    out = agg if mask is None else agg * torch.from_numpy(mask).double()
    (out * torch.from_numpy(w).double()).sum().backward()
    return out.detach(), pre, x64.grad, ew64.grad, None if b64 is None else b64.grad


@pytest.mark.parametrize("relu_bias", [False, True])
@pytest.mark.parametrize("scales", ["none", "nbr", "both"])
@pytest.mark.parametrize("reduce", ["add", "mean"])
def test_aggregate_edge_weight_gradient_against_fp64(reduce, scales, relu_bias):
    n, H = 50_000, 16
    ei, _, _ = hub_graph(n, hub_out=50_000, seed=2)
    rng = np.random.default_rng(len(reduce) + len(scales) + relu_bias)
    x = rng.standard_normal((n, H)).astype(F32)
    ew = rng.uniform(0.1, 2.0, ei.shape[1]).astype(F32)
    s_nbr = rng.uniform(0.2, 1.5, n).astype(F32) if scales != "none" else None
    s_row = rng.uniform(0.2, 1.5, n).astype(F32) if scales == "both" else None
    bias = rng.standard_normal(H).astype(F32) if relu_bias else None
    w = rng.standard_normal((n, H)).astype(F32)
    res = {}
    for dt in (torch.int64, torch.int32):
        gs = GraphStructure(dev(ei).to(dt), n)
        xt, ewt = dev(x).requires_grad_(True), dev(ew).requires_grad_(True)
        bt = None if bias is None else dev(bias).requires_grad_(True)
        out = F_mgcn.aggregate(xt, gs, None if s_nbr is None else dev(s_nbr), None if s_row is None else dev(s_row),
                               ewt, reduce, bt, None, "relu" if relu_bias else None)
        out.backward(dev(w))
        res[dt] = (out.detach(), xt.grad, ewt.grad, None if bt is None else bt.grad)
    for k, what in enumerate(("out", "dx", "d_edge_weight", "d_bias")):
        if res[torch.int64][k] is not None:
            assert_bitexact(res[torch.int32][k], res[torch.int64][k].cpu(), f"{what}: int32 vs int64 edge_index")
    out, dx, dew, db = res[torch.int64]
    mask = (out > 0).cpu().numpy().astype(F32) if relu_bias else None
    o_r, pre, dx_r, dew_r, db_r = _aggregate_ref(ei, n, x, ew, s_nbr, s_row, reduce, bias, mask, w)
    if mask is not None:                          # the ReLU decided on the fp32 side only where fp64 is near zero
        tol = 1e-5 * float(pre.abs().max())
        assert (pre[torch.from_numpy(mask) == 0] <= tol).all() and (pre[torch.from_numpy(mask) == 1] >= -tol).all()
    assert_parity(out, o_r, "aggregate out")
    assert_parity(dx, dx_r, "aggregate dx")
    if db is not None:
        assert_parity(db, db_r, "aggregate d_bias")
    # d w_e = s_nbr[row] s_row[col] <gg[col], x[row]>, gg = the upstream gradient (ReLU-masked, / in-degree for mean)
    gg = w.astype(np.float64) * (1.0 if mask is None else mask)
    if reduce == "mean":
        gg = gg / np.maximum(np.bincount(ei[1], minlength=n), 1)[:, None]
    dot, mag = edge_dot_ref(ei, gg, x)
    s = np.ones(ei.shape[1])
    if s_nbr is not None:
        s = s * s_nbr[ei[0]]
    if s_row is not None:
        s = s * s_row[ei[1]]
    np.testing.assert_allclose(dot * s, dew_r.numpy(), rtol=1e-9, atol=1e-10)
    check_edge_dot(dew, dot, mag, s, H, 8, "aggregate d_edge_weight")


# ------------------------------------------------------------------------------------------------
# 7. attention: compat softmax over groups, then an aggregation weighted by it
# ------------------------------------------------------------------------------------------------
def test_softmax_then_weighted_aggregate_against_fp64():
    from meta_gcn_b200.gcn_meta.models.common import softmax
    n, H = 20_000, 8
    ei, ht, _ = hub_graph(n, seed=3)
    E = ei.shape[1]
    cnt = np.bincount(ei[1], minlength=n)
    assert cnt[ht] >= 50_000 and (cnt == 1).sum() > 1000
    rng = np.random.default_rng(7)
    logits = (3 * rng.standard_normal(E)).astype(F32)
    x = rng.standard_normal((n, H)).astype(F32)
    w = rng.standard_normal((n, H)).astype(F32)

    col = dev(ei[1])
    st, xt = dev(logits).requires_grad_(True), dev(x).requires_grad_(True)
    alpha = softmax(st, col, n)
    out = F_mgcn.aggregate(xt, GraphStructure(dev(ei), n), None, None, alpha, "add")
    out.backward(dev(w))

    row_c, col_c = torch.from_numpy(ei[0]), torch.from_numpy(ei[1])
    s64 = torch.from_numpy(logits).double().requires_grad_(True)
    x64 = torch.from_numpy(x).double().requires_grad_(True)
    m = torch.full((n,), -1e16, dtype=torch.float64).scatter_reduce(0, col_c, s64.detach(), "amax")
    e = (s64 - m[col_c]).exp()
    a64 = e / (torch.zeros(n, dtype=torch.float64).index_add(0, col_c, e)[col_c] + 1e-16)
    o64 = torch.zeros(n, H, dtype=torch.float64).index_add(0, col_c, x64[row_c] * a64[:, None])
    (o64 * torch.from_numpy(w).double()).sum().backward()
    assert_parity(alpha, a64.detach(), "softmax")
    assert_parity(out, o64.detach(), "attention out")
    assert_parity(st.grad, s64.grad, "d logits")
    assert_parity(xt.grad, x64.grad, "dx")


# ------------------------------------------------------------------------------------------------
# 8. models
# ------------------------------------------------------------------------------------------------
class _FirstMax(torch.autograd.Function):
    """the oracle's scatter_('max') with torch_scatter's gradient rule (the first maximal entry receives it)"""

    @staticmethod
    def forward(ctx, src, index, dim_size):
        out, arg = first_max_ref(src.detach().numpy(), index.numpy(), dim_size, fill=-1e38)
        ctx.arg, ctx.n_src = arg, src.size(0)
        return torch.from_numpy(out).reshape((dim_size,) + tuple(src.shape[1:]))

    @staticmethod
    def backward(ctx, g):
        d = scatter_max_grad_ref(ctx.arg, g.contiguous().numpy(), ctx.n_src)
        return torch.from_numpy(d), None, None


@pytest.fixture(scope="module")
def botnet20k():
    g = synth_botnet_graph(seed=2, num_nodes=20_000, edge_entries=200_000, evil=500)
    deg = g["x"][:, 1]
    # five features, many nodes sharing the same row (equal degree): their messages tie exactly
    x = np.stack([np.ones_like(deg), deg, np.log1p(deg), deg % 3, np.zeros_like(deg)], 1).astype(F32)
    return x, g["edge_index"], deg.astype(F32), g["y"].astype(np.int64)


MODEL = dict(in_channels=5, enc_sizes=[16, 16, 16], num_classes=2, residual_hop=1, dropout=0.0, final_type="proj",
             aggr="max", bias=True)


@pytest.mark.parametrize("deg_norm", ["sm", "rw"])
def test_gcn_model_max_against_oracle(botnet20k, deg_norm, monkeypatch):
    x, ei, deg, y = botnet20k
    orig = port.scatter_rows

    def scatter_rows(name, src, index, dim_size):
        return _FirstMax.apply(src, index, dim_size) if name == "max" else orig(name, src, index, dim_size)

    monkeypatch.setattr(port, "scatter_rows", scatter_rows)
    cfg = dict(MODEL, deg_norm=deg_norm)
    torch.manual_seed(4)
    ref = port.OracleGCNModel(**cfg)
    xr, eir, degr, yr = (torch.from_numpy(v) for v in (x, ei, deg, y))
    out_r = ref(xr, eir, degr)
    torch.nn.CrossEntropyLoss()(out_r, yr).backward()

    model = GCNModel(**cfg)
    model.load_state_dict(ref.state_dict())
    model.to(DEV).train()
    out = model(dev(x), dev(ei), deg_K=dev(deg))
    torch.nn.CrossEntropyLoss()(out, dev(y)).backward()
    assert_parity(out, out_r.detach(), f"max/{deg_norm} logits")
    ref_grads = dict(ref.named_parameters())
    for k, p in model.named_parameters():
        assert_parity(p.grad, ref_grads[k].grad, f"max/{deg_norm} grad.{k}")


@pytest.mark.parametrize("aggr", ["add", "max"])
def test_gcn_model_edge_gate_int32_int64_and_run_to_run_bitwise(botnet20k, aggr):
    x, ei, deg, y = botnet20k
    torch.manual_seed(5)
    model = GCNModel(**dict(MODEL, aggr=aggr, deg_norm="sm", edge_gate="proj")).to(DEV).train()
    xt, dt, yt = dev(x), dev(deg), dev(y)
    ei64 = dev(ei)
    runs = []
    for e in (ei64, ei64.to(torch.int32), ei64):
        model.zero_grad(set_to_none=True)
        out = model(xt, e, deg_K=dt)
        torch.nn.CrossEntropyLoss()(out, yt).backward()
        runs.append([out.detach()] + [p.grad.clone() for _, p in model.named_parameters()])
    names = ["out"] + [k for k, _ in model.named_parameters()]
    for k, name in enumerate(names):
        assert_bitexact(runs[1][k], runs[0][k].cpu(), f"gate/{aggr} {name}: int32 vs int64 edge_index")
        assert_bitexact(runs[2][k], runs[0][k].cpu(), f"gate/{aggr} {name}: run to run")
