"""torch.library custom ops (namespace ``mgcn``) over the C-ABI of libmgcn.so.

Every op takes/returns torch CUDA tensors and forwards raw device pointers, sizes and the current
CUDA stream to the library; PyTorch only provides memory and streams.  CUDA-only: a CPU tensor
raises, there is no fallback (the CPU restatement lives in oracle/ and is test infrastructure).

Raw ops (no autograd) are registered as ``torch.ops.mgcn.*`` with fake (meta) implementations;
the differentiable wrappers used by the model classes are in ``meta_gcn_b200.functional``.
"""
import ctypes
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import MgcnCsr

DEFAULT_HUB_THRESHOLD = 64
WIDE_WIDTHS = (64, 128, 192, 256)   # output widths served by the tcgen05 transform


def _ptr(t):
    return None if t is None else t.data_ptr()


# torch.cuda.current_stream() costs ~15 us of Python per call (device-index resolution, is_available, a Stream object);
# a step of the small-graph nets makes 33 such calls.  The raw handle comes straight from the C extension.
_RAW_STREAM = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_RAW_DEVICE = getattr(torch._C, "_cuda_getDevice", None)


def _stream():
    if _RAW_STREAM is not None and _RAW_DEVICE is not None:
        return _RAW_STREAM(_RAW_DEVICE())
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("mgcn ops run on CUDA tensors only (no CPU fallback)")


def _f32c(t, name):
    if t is None:
        return None
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    return t.contiguous()


CSR_FIELDS = ("rowptr", "nbr", "perm", "order", "hub_rows", "hub_seg0", "hub_count", "seg_row",
              "seg_beg", "seg_count", "tasks", "nbr_w")


class Csr:
    """Device buffers of one mgcn_csr_t (include/mgcn.h) plus the ctypes view handed to the library."""

    __slots__ = CSR_FIELDS + ("bad", "hub_threshold", "_struct")

    def __init__(self, tensors, hub_threshold, bad=None):
        for name, t in zip(CSR_FIELDS, tensors):
            setattr(self, name, t)
        self.bad = bad
        self.hub_threshold = int(hub_threshold)
        self._struct = None

    def tensors(self):
        return [getattr(self, n) for n in CSR_FIELDS]

    @property
    def n_rows(self):
        return self.rowptr.numel() - 1

    def struct(self):
        if self._struct is None:
            s = MgcnCsr()
            s.n_rows = self.rowptr.numel() - 1
            s.nnz_cap = self.nbr.numel()
            s.hub_cap = self.hub_rows.numel()
            s.seg_cap = self.seg_row.numel()
            s.hub_threshold = self.hub_threshold
            for name in CSR_FIELDS:
                t = getattr(self, name)
                setattr(s, name, t.data_ptr() if t is not None and t.numel() else None)
            self._struct = s
        return self._struct


def _as_csr(csr, hub_threshold=None):
    if isinstance(csr, Csr):
        return csr
    return Csr(list(csr), hub_threshold)


# ------------------------------------------------------------------------------------------------
# implementations (plain functions; also what meta_gcn_b200.functional calls directly)
# ------------------------------------------------------------------------------------------------
def csr_build_impl(edge_index, N, by, loop_mode, hub_threshold=DEFAULT_HUB_THRESHOLD, layout=0, segments=None,
                   reuse=None):
    """layout != 0 (from edge_layout_impl; loop_mode 0 only): the list is already in (src,dst) order — no sort.
    segments = (node_off, edge_off) int32 device tensors [G+1] for a batch of graphs (by = 0 only).
    reuse: a Csr whose buffers may be overwritten (same sizes, device and hub threshold, else ignored): the new
    structure then lives at the same addresses and nothing is allocated for it."""
    _need_cuda(edge_index)
    if edge_index.dtype not in (torch.int64, torch.int32) or edge_index.dim() != 2 or edge_index.size(0) != 2:
        raise TypeError("edge_index must be int64 (the reference's dtype) or int32, shape [2,E]")
    ei = edge_index.contiguous()
    E = ei.size(1)
    N = int(N)
    dev = ei.device
    lib = _lib.load()
    if layout:
        if int(loop_mode) != 0:
            raise ValueError("a presorted build keeps the edges as given (loop_mode 0)")
        build = lib.mgcn_csr_build_presorted if ei.dtype == torch.int64 else lib.mgcn_csr_build_presorted_i32
        g_ = 0 if segments is None else segments[0].numel() - 1
        mode_arg = (int(layout), g_, _ptr(segments[0]) if g_ else None, _ptr(segments[1]) if g_ else None)
    else:
        build = lib.mgcn_csr_build if ei.dtype == torch.int64 else lib.mgcn_csr_build_i32
        mode_arg = (int(loop_mode),)
    caps = [ctypes.c_int64(0) for _ in range(3)]
    _lib.check(lib.mgcn_csr_capacities(E, N, int(loop_mode), int(hub_threshold),
                                       *[ctypes.byref(c) for c in caps]))
    nnz_cap, hub_cap, seg_cap = (c.value for c in caps)
    i32 = dict(dtype=torch.int32, device=dev)
    sizes = dict(rowptr=N + 1, nbr=nnz_cap, perm=nnz_cap, order=N, hub_rows=hub_cap, hub_seg0=hub_cap,
                 hub_count=1, seg_row=seg_cap, seg_beg=seg_cap, seg_count=1, tasks=4 * (N + seg_cap),
                 nbr_w=nnz_cap)
    csr = None
    if reuse is not None and reuse.hub_threshold == int(hub_threshold) and reuse.bad is not None:
        old = reuse.tensors()
        if all(t is not None and t.device == dev and t.numel() == sizes[n] for n, t in zip(CSR_FIELDS, old)):
            csr = Csr(old, hub_threshold, reuse.bad)
    if csr is None:
        csr = Csr([torch.empty(sizes[n], **i32) for n in CSR_FIELDS], hub_threshold,
                  torch.empty(1, **i32))
    nbytes = ctypes.c_size_t(0)
    st = csr.struct()
    _lib.check(build(_ptr(ei), E, N, int(by), *mode_arg, ctypes.byref(st),
                     _ptr(csr.bad), None, ctypes.byref(nbytes), None))
    ws = torch.empty(max(nbytes.value, 1), dtype=torch.uint8, device=dev)
    _lib.check(build(_ptr(ei), E, N, int(by), *mode_arg, ctypes.byref(st),
                     _ptr(csr.bad), _ptr(ws), ctypes.byref(nbytes), _stream()))
    return csr


def preprocess_edges_impl(edge_index, N, undirected=True, add_loops=True):
    """mgcn_preprocess_edges: returns (edge_index_out int64 [2, count], deg f32 [N], perm int32 [count]);
    one host sync to read the number of kept edges (as torch.unique does)."""
    _need_cuda(edge_index)
    if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.size(0) != 2:
        raise TypeError("edge_index must be int64 [2,E]")
    ei = edge_index.contiguous()
    E, N = ei.size(1), int(N)
    dev = ei.device
    cap = (2 * E if undirected else E) + (N if add_loops else 0)
    out = torch.empty(2, max(cap, 1), dtype=torch.int64, device=dev)
    perm = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    deg = torch.empty(N, dtype=torch.float32, device=dev)
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    bad = torch.zeros(1, dtype=torch.int32, device=dev)
    lib = _lib.load()
    args = (_ptr(ei), E, N, int(bool(undirected)), int(bool(add_loops)), out.size(1), _ptr(out), _ptr(perm),
            _ptr(deg), _ptr(count), _ptr(bad))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_preprocess_edges(*args, w_, nb, stm), dev)
    _lib.check(lib.mgcn_preprocess_edges(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    n_out, is_bad = int(count.item()), int(bad.item())
    if is_bad:
        raise IndexError("edge_index contains node ids outside [0, num_nodes)")
    return out[:, :n_out], deg, perm[:n_out]


def degree_impl(rowptr):
    _need_cuda(rowptr)
    N = rowptr.numel() - 1
    deg = torch.empty(N, dtype=torch.float32, device=rowptr.device)
    _lib.check(_lib.load().mgcn_degree_from_rowptr(_ptr(rowptr), N, _ptr(deg), _stream()))
    return deg


def weighted_degree_impl(csr, edge_weight, loop_weight):
    _need_cuda(csr.rowptr, edge_weight)
    ew = _f32c(edge_weight, "edge_weight")
    deg = torch.empty(csr.n_rows, dtype=torch.float32, device=csr.rowptr.device)
    _lib.check(_lib.load().mgcn_weighted_degree(ctypes.byref(csr.struct()), _ptr(ew), ew.numel(),
                                                float(loop_weight), _ptr(deg), _stream()))
    return deg


def binary_confusion_impl(target, logits=None, pred=None):
    """device int64[5] = {TP, FP, TN, FN, correct} (mgcn_binary_confusion); no host synchronisation"""
    if (logits is None) == (pred is None):
        raise ValueError("exactly one of logits / pred")
    src = logits if logits is not None else pred
    _need_cuda(src, target)
    if target.dtype != torch.int64:
        raise TypeError("target must be int64 (batch.y.long())")
    target = target.contiguous()
    if logits is not None:
        logits = _f32c(logits, "logits")
        N, C = logits.shape
    else:
        if pred.dtype != torch.int64:
            raise TypeError("pred must be int64")
        pred = pred.contiguous()
        N, C = pred.numel(), 2
    if target.numel() != N:
        raise ValueError("pred / logits and target differ in length")
    out = torch.empty(5, dtype=torch.int64, device=src.device)
    _lib.check(_lib.load().mgcn_binary_confusion(_ptr(logits) if logits is not None else None,
                                                 _ptr(pred) if pred is not None else None, N, C,
                                                 _ptr(target), _ptr(out), _stream()))
    return out


def edge_symmetry_impl(edge_index):
    """True iff the directed edge multiset equals its transpose (mgcn_edge_fingerprint).  Reads four words
    back from the device: one host synchronisation per edge_index."""
    _need_cuda(edge_index)
    if edge_index.dtype not in (torch.int64, torch.int32) or edge_index.dim() != 2 or edge_index.size(0) != 2:
        raise TypeError("edge_index must be int64 or int32, shape [2, E]")
    ei = edge_index.contiguous()
    out = torch.empty(4, dtype=torch.int64, device=ei.device)
    lib = _lib.load()
    fn = lib.mgcn_edge_fingerprint if ei.dtype == torch.int64 else lib.mgcn_edge_fingerprint_i32
    _lib.check(fn(_ptr(ei), ei.size(1), _ptr(out), _stream()))
    f = out.tolist()
    return f[0] == f[1] and f[2] == f[3]


def edge_layout_impl(edge_index, N, segments=None):
    """One pass pair + ONE host read per edge_index (mgcn_edge_layout): {'symmetric': the directed multiset equals its
    transpose, 'layout': 0 unsorted | 1 sorted by (src,dst) | 2 sorted prefix + N trailing self loops (+4: repeated
    entries)} — what decides whether the structures need a sort and whether the by-source one is needed at all."""
    _need_cuda(edge_index)
    if edge_index.dtype not in (torch.int64, torch.int32) or edge_index.dim() != 2 or edge_index.size(0) != 2:
        raise TypeError("edge_index must be int64 or int32, shape [2, E]")
    ei = edge_index.contiguous()
    out = torch.empty(8, dtype=torch.int64, device=ei.device)
    lib = _lib.load()
    fn = lib.mgcn_edge_layout if ei.dtype == torch.int64 else lib.mgcn_edge_layout_i32
    g_ = 0 if segments is None else segments[0].numel() - 1
    _lib.check(fn(_ptr(ei), ei.size(1), int(N), g_, _ptr(segments[0]) if g_ else None,
                  _ptr(segments[1]) if g_ else None, _ptr(out), _stream()))
    f = out.tolist()
    E = ei.size(1)
    layout = 0
    if E > 0 and f[4] == 0:
        layout = 1
    elif E >= N > 0 and f[5] == 0 and f[6] == 0:
        layout = 2
    if layout and f[7] != 0:
        layout |= 4
    return {"symmetric": f[0] == f[1] and f[2] == f[3], "layout": layout}


def gcn_norm_impl(deg, mode):
    _need_cuda(deg)
    d = _f32c(deg, "deg")
    dis = torch.empty_like(d)
    _lib.check(_lib.load().mgcn_gcn_norm(_ptr(d), d.numel(), int(mode), _ptr(dis), _stream()))
    return dis


def permute_edge_values_impl(csr, vals, loop_value):
    _need_cuda(csr.rowptr, vals)
    v = _f32c(vals, "vals")
    out = torch.empty(csr.nbr.numel(), dtype=torch.float32, device=csr.rowptr.device)
    _lib.check(_lib.load().mgcn_permute_edge_values(ctypes.byref(csr.struct()), _ptr(v), v.numel(),
                                                    float(loop_value), _ptr(out), _stream()))
    return out


def _workspace(fn, dev):
    """two-phase workspace protocol: fn(ws_ptr, byref(nbytes)) -> rc"""
    nbytes = ctypes.c_size_t(0)
    _lib.check(fn(None, ctypes.byref(nbytes), None))
    ws = torch.empty(max(nbytes.value, 1), dtype=torch.uint8, device=dev)
    return ws, nbytes


def spmm_impl(csr, x, gather_perm=False, edge_val=None, nbr_scale=None, row_scale=None, reduce=0,
              bias=None, residual=None, act=0):
    _need_cuda(csr.rowptr, x, edge_val, nbr_scale, row_scale, bias, residual)
    if x.dim() != 2:
        raise ValueError("x must be [n_in, H]")
    x = _f32c(x, "x")
    edge_val = _f32c(edge_val, "edge_val")
    nbr_scale = _f32c(nbr_scale, "nbr_scale")
    row_scale = _f32c(row_scale, "row_scale")
    bias = _f32c(bias, "bias")
    residual = _f32c(residual, "residual")
    n_rows = csr.n_rows
    H = x.size(1)
    if edge_val is not None and edge_val.numel() != csr.nbr.numel():
        raise ValueError("edge_val must be in row order with nnz_cap entries")
    if row_scale is not None and row_scale.numel() != n_rows:
        raise ValueError("row_scale must have one entry per row")
    if residual is not None and tuple(residual.shape) != (n_rows, H):
        raise ValueError("residual must be [n_rows, H]")
    if bias is not None and bias.numel() != H:
        raise ValueError("bias must have H entries")
    out = torch.empty(n_rows, H, dtype=torch.float32, device=x.device)
    lib = _lib.load()
    st = ctypes.byref(csr.struct())
    args = (st, _ptr(x), x.size(0), H, int(bool(gather_perm)), _ptr(edge_val), _ptr(nbr_scale),
            _ptr(row_scale), int(reduce), _ptr(bias), _ptr(residual), int(act), _ptr(out))
    ws, nbytes = _workspace(lambda w, nb, stm: lib.mgcn_spmm(*args, w, nb, stm), x.device)
    _lib.check(lib.mgcn_spmm(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return out


def edge_dot_impl(edge_index, a, b, scale_src=None, scale_tgt=None):
    """out[e] = scale_src[row_e] * scale_tgt[col_e] * <a[col_e], b[row_e]>   (mgcn_edge_dot / _i32)"""
    _need_cuda(edge_index, a, b, scale_src, scale_tgt)
    if edge_index.dtype not in (torch.int64, torch.int32) or edge_index.dim() != 2 or edge_index.size(0) != 2:
        raise TypeError("edge_index must be int64 or int32, shape [2, E]")
    a = _f32c(a, "a")
    b = _f32c(b, "b")
    scale_src = _f32c(scale_src, "scale_src")
    scale_tgt = _f32c(scale_tgt, "scale_tgt")
    ei = edge_index.contiguous()
    E = ei.size(1)
    out = torch.empty(E, dtype=torch.float32, device=a.device)
    lib = _lib.load()
    fn = lib.mgcn_edge_dot if ei.dtype == torch.int64 else lib.mgcn_edge_dot_i32
    _lib.check(fn(_ptr(ei), E, _ptr(a), _ptr(b), a.size(1), _ptr(scale_src), _ptr(scale_tgt), _ptr(out), _stream()))
    return out


def segment_max_impl(csr, x, gather_perm=False, edge_val=None, fill=None):
    """(out [n_rows,H], arg int32 [n_rows,H]) of mgcn_segment_max, or of mgcn_segment_max_ex with a fill value
    (torch_scatter's rule: only an entry strictly greater than fill can win; no winner -> 0 / -1)"""
    _need_cuda(csr.rowptr, x, edge_val)
    x = _f32c(x, "x")
    edge_val = _f32c(edge_val, "edge_val")
    if edge_val is not None and edge_val.numel() != csr.nbr.numel():
        raise ValueError("edge_val must be in row order with nnz_cap entries")
    H = x.size(1)
    out = torch.empty(csr.n_rows, H, dtype=torch.float32, device=x.device)
    arg = torch.empty(csr.n_rows, H, dtype=torch.int32, device=x.device)
    lib = _lib.load()
    head = (ctypes.byref(csr.struct()), _ptr(x), x.size(0), H, int(bool(gather_perm)), _ptr(edge_val))
    if fill is None:
        _lib.check(lib.mgcn_segment_max(*head, _ptr(out), _ptr(arg), _stream()))
    else:
        _lib.check(lib.mgcn_segment_max_ex(*head, float(fill), _ptr(out), _ptr(arg), _stream()))
    return out, arg


def segment_max_bwd_impl(csr_t, grad, arg, edge_val=None):
    """layer seam: gradient w.r.t. the gathered operand, by the structure grouped by source"""
    _need_cuda(csr_t.rowptr, grad, arg, edge_val)
    grad = _f32c(grad, "grad")
    edge_val = _f32c(edge_val, "edge_val")
    H = grad.size(1)
    dx = torch.empty(csr_t.n_rows, H, dtype=torch.float32, device=grad.device)
    _lib.check(_lib.load().mgcn_segment_max_bwd(ctypes.byref(csr_t.struct()), _ptr(grad), _ptr(arg.contiguous()),
                                                _ptr(edge_val), H, _ptr(dx), _stream()))
    return dx


def scatter_max_bwd_impl(arg, grad, n_src):
    """primitive seam: gradient w.r.t. src [n_src,H]"""
    _need_cuda(arg, grad)
    grad = _f32c(grad, "grad")
    N, H = grad.shape
    dsrc = torch.empty(n_src, H, dtype=torch.float32, device=grad.device)
    _lib.check(_lib.load().mgcn_scatter_max_bwd(_ptr(arg.contiguous()), _ptr(grad), N, H, n_src, _ptr(dsrc), _stream()))
    return dsrc


def aggregate_prescaled_impl(csr, x, post_scale=None, reduce=0, bias=None, residual=None, act=0):
    """out_i = act(post_scale[i] * sum_k x[nbr_k] (/len) + bias + residual_i) for x that already
    carries the per-source factor; H in {16, 32, 64, 128}."""
    _need_cuda(csr.rowptr, x, post_scale, bias, residual)
    x = _f32c(x, "x")
    post_scale = _f32c(post_scale, "post_scale")
    bias = _f32c(bias, "bias")
    residual = _f32c(residual, "residual")
    n_rows, H = csr.n_rows, x.size(1)
    out = torch.empty(n_rows, H, dtype=torch.float32, device=x.device)
    lib = _lib.load()
    args = (ctypes.byref(csr.struct()), _ptr(x), x.size(0), H, _ptr(post_scale), int(reduce),
            _ptr(bias), _ptr(residual), int(act), _ptr(out))
    ws, nbytes = _workspace(lambda w, nb, stm: lib.mgcn_aggregate_prescaled(*args, w, nb, stm), x.device)
    _lib.check(lib.mgcn_aggregate_prescaled(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return out


def linear_impl(x, w, w_out_in, bias=None, add=None, act=0, xmask=None, row_scale=None):
    """y = row_scale * act((x * (xmask > 0)) @ W + bias + add); w is [Hi,Ho] (weight_node) or, if
    w_out_in, [Ho,Hi] (nn.Linear)."""
    _need_cuda(x, w, bias, add, xmask, row_scale)
    x = _f32c(x, "x")
    w = _f32c(w, "w")
    bias = _f32c(bias, "bias")
    add = _f32c(add, "add")
    xmask = _f32c(xmask, "xmask")
    row_scale = _f32c(row_scale, "row_scale")
    N, Hi = x.shape
    if w_out_in:
        Ho, Hi_w = w.shape
        sk, sc = 1, Hi
    else:
        Hi_w, Ho = w.shape
        sk, sc = Ho, 1
    if Hi_w != Hi:
        raise ValueError(f"width mismatch: x has {Hi}, weight expects {Hi_w}")
    if xmask is not None and xmask.shape != x.shape:
        raise ValueError("xmask must have the shape of x")
    y = torch.empty(N, Ho, dtype=torch.float32, device=x.device)
    if xmask is None and Ho in WIDE_WIDTHS and Hi >= 32 and Hi % 4 == 0 and N > 0:
        # wide output: tcgen05 / TMEM tile GEMM (csrc/linear_wide.cu)
        lib = _lib.load()
        args = (_ptr(x), N, Hi, _ptr(w), sk, sc, Ho, _ptr(bias), _ptr(add), int(act), _ptr(row_scale), _ptr(y))
        ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_linear_wide(*args, w_, nb, stm), x.device)
        _lib.check(lib.mgcn_linear_wide(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
        return y
    _lib.check(_lib.load().mgcn_linear_ex(_ptr(x), _ptr(xmask), N, Hi, _ptr(w), sk, sc, Ho, _ptr(bias),
                                          _ptr(add), int(act), _ptr(row_scale), _ptr(y), _stream()))
    return y


def linear_wgrad_impl(x, g, w_out_in, want_bias, gmask=None):
    _need_cuda(x, g, gmask)
    x = _f32c(x, "x")
    g = _f32c(g, "g")
    gmask = _f32c(gmask, "gmask")
    N, Hi = x.shape
    Ho = g.size(1)
    dev = x.device
    if w_out_in:
        dw = torch.empty(Ho, Hi, dtype=torch.float32, device=dev)
        sk, sc = 1, Hi
    else:
        dw = torch.empty(Hi, Ho, dtype=torch.float32, device=dev)
        sk, sc = Ho, 1
    db = torch.empty(Ho if want_bias else 0, dtype=torch.float32, device=dev)
    lib = _lib.load()
    args = (_ptr(x), N, Hi, _ptr(g), _ptr(gmask), Ho, _ptr(dw), sk, sc, _ptr(db) if want_bias else None)
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_linear_wgrad_ex(*args, w_, nb, stm), dev)
    _lib.check(lib.mgcn_linear_wgrad_ex(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return dw, db


def masked_scale_impl(g, m1=None, m2=None, row_scale=None):
    """out = row_scale[:,None] * g * (m1 > 0) * (m2 > 0)"""
    _need_cuda(g, m1, m2, row_scale)
    g = _f32c(g, "g")
    m1 = _f32c(m1, "m1")
    m2 = _f32c(m2, "m2")
    row_scale = _f32c(row_scale, "row_scale")
    out = torch.empty_like(g)
    _lib.check(_lib.load().mgcn_masked_scale(_ptr(g), _ptr(m1), _ptr(m2), _ptr(row_scale), g.size(0),
                                             g.size(1), _ptr(out), _stream()))
    return out


def gcn_layer_fwd_impl(csr, m, x, resid, res_w, res_b, w_next, bias, pre, post, act_out):
    """one fused forward layer at hidden 32 (mgcn_gcn_layer_fwd): returns (x_next, m_next | None,
    hmask int32[N]).  csr None = row-local mode (m is the finished pre-activation)."""
    _need_cuda(m, x, resid, res_w, res_b, w_next, bias, pre, post)
    m = _f32c(m, "m")
    x = _f32c(x, "x")
    resid = _f32c(resid, "resid")
    res_w = _f32c(res_w, "res_w")
    res_b = _f32c(res_b, "res_b")
    w_next = _f32c(w_next, "w_next")
    bias = _f32c(bias, "bias")
    pre = _f32c(pre, "pre")
    post = _f32c(post, "post")
    n_rows, H = (csr.n_rows if csr is not None else m.size(0)), m.size(1)
    dev = m.device
    x_next = torch.empty(n_rows, H, dtype=torch.float32, device=dev)
    m_next = torch.empty(n_rows, H, dtype=torch.float32, device=dev) if w_next is not None else None
    hmask = torch.empty(n_rows, dtype=torch.int32, device=dev)
    lib = _lib.load()
    args = (ctypes.byref(csr.struct()) if csr is not None else None, _ptr(m), m.size(0), _ptr(x), _ptr(resid),
            _ptr(res_w), _ptr(res_b), _ptr(w_next), _ptr(bias), _ptr(pre), _ptr(post), int(act_out), H,
            _ptr(x_next), _ptr(m_next), _ptr(hmask))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_gcn_layer_fwd(*args, w_, nb, stm), dev)
    _lib.check(lib.mgcn_gcn_layer_fwd(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return x_next, m_next, hmask


def gcn_first_layer_fwd_impl(s, x, w_in, res_w, res_b, w_next, pre, post, act_out, out_scale=None, keep=None,
                             keep_scale=1.0, bias=None):
    """first layer with a narrow input (mgcn_gcn_first_layer_fwd_ex): s = aggregated input [N,Hin], x = layer input
    [N,Hin]; returns (x_next [N,32], m_next | None, hmask int32[N]); out_scale [N]: x_next rows leave scaled;
    keep int32 [N] (w_next None only): dropout keep bits of the layer, kept entries of h multiplied by keep_scale;
    bias [32]: the node-model bias, h = relu(post (s W) + bias) (mgcn_gcn_first_layer_fwd_bias)"""
    _need_cuda(s, x, w_in, res_w, res_b, w_next, pre, post, out_scale, keep, bias)
    bias = _f32c(bias, "bias")
    out_scale = _f32c(out_scale, "out_scale")
    s = _f32c(s, "s")
    x = _f32c(x, "x")
    w_in = _f32c(w_in, "w_in")
    res_w = _f32c(res_w, "res_w")
    res_b = _f32c(res_b, "res_b")
    w_next = _f32c(w_next, "w_next")
    pre = _f32c(pre, "pre")
    post = _f32c(post, "post")
    N, Hin = x.shape
    H = w_in.size(1)
    if s.shape != x.shape or w_in.size(0) != Hin or tuple(res_w.shape) != (H, Hin):
        raise ValueError("shape mismatch in gcn_first_layer_fwd")
    dev = x.device
    x_next = torch.empty(N, H, dtype=torch.float32, device=dev)
    m_next = torch.empty(N, H, dtype=torch.float32, device=dev) if w_next is not None else None
    hmask = torch.empty(N, dtype=torch.int32, device=dev)
    keep = _keep_rows(keep, N, 1)
    lib = _lib.load()
    if bias is not None:
        if bias.numel() != H:
            raise ValueError(f"bias must have {H} entries, got {bias.numel()}")
        _lib.check(lib.mgcn_gcn_first_layer_fwd_bias(
            _ptr(s), _ptr(x), N, Hin, _ptr(w_in), _ptr(res_w), _ptr(res_b), _ptr(bias), _ptr(w_next), _ptr(pre),
            _ptr(post), _ptr(out_scale), _ptr(keep), float(keep_scale), int(act_out), H, _ptr(x_next), _ptr(m_next),
            _ptr(hmask), _stream()))
        return x_next, m_next, hmask
    _lib.check(lib.mgcn_gcn_first_layer_fwd_ex(
        _ptr(s), _ptr(x), N, Hin, _ptr(w_in), _ptr(res_w), _ptr(res_b), _ptr(w_next), _ptr(pre), _ptr(post),
        _ptr(out_scale), _ptr(keep), float(keep_scale), int(act_out), H, _ptr(x_next), _ptr(m_next), _ptr(hmask),
        _stream()))
    return x_next, m_next, hmask


def _keep_rows(keep, N, W):
    """keep bits of one layer as a contiguous int32 [N, W] (or [N] for W = 1)"""
    if keep is None:
        return None
    if keep.dtype != torch.int32 or keep.numel() != N * W:
        raise ValueError(f"keep must be int32 with {N} x {W} words, got {keep.dtype} {tuple(keep.shape)}")
    return keep.contiguous()


# forward layer of the hidden-32 stack: A operands through tensor memory (csrc/gcn_fwd_tm.cu) or as shared-memory
# images (csrc/gcn_fwd_tc.cu); both pass the same parity tests
FWD_TMEM_OPERANDS = False


def gcn_layer_fwd_tc_impl(csr, z, w, res_w, res_b, bias, in_scale, post, out_scale, act_out, tmem_operands=None,
                          keep=None, keep_scale=1.0, gate_ab=None, gate_c=None):
    """one aggregate-then-transform forward layer at hidden 32 on tcgen05 (mgcn_gcn_layer_fwd_tc_ex): z = in_scale (.) x
    [N,32]; returns (z_next = out_scale (.) x_next [N,32], hmask int32[N]).  keep int32 [N]: dropout keep bits of the
    layer (kept entries of h multiplied by keep_scale, dropped ones cleared in hmask too).  gate_ab [N,2] (from
    gate_scores_impl) and gate_c [1]: every gathered row weighted by its edge gate (mgcn_gcn_layer_fwd_tc_gate)"""
    _need_cuda(z, w, res_w, res_b, bias, in_scale, post, out_scale, keep, gate_ab, gate_c)
    tmem = FWD_TMEM_OPERANDS if tmem_operands is None else tmem_operands
    if (keep is not None or gate_ab is not None) and tmem:
        raise ValueError("dropout keep bits and edge gates need the shared-memory operand forward "
                         "(mgcn_gcn_layer_fwd_tc_gate), not the TMEM-operand kernel")
    z = _f32c(z, "z")
    w = _f32c(w, "w")
    res_w = _f32c(res_w, "res_w")
    res_b = _f32c(res_b, "res_b")
    bias = _f32c(bias, "bias")
    in_scale = _f32c(in_scale, "in_scale")
    post = _f32c(post, "post")
    out_scale = _f32c(out_scale, "out_scale")
    n_rows, H = csr.n_rows, z.size(1)
    if tuple(w.shape) != (H, H) or tuple(res_w.shape) != (H, H):
        raise ValueError("gcn_layer_fwd_tc needs square [32,32] weights")
    dev = z.device
    z_next = torch.empty(n_rows, H, dtype=torch.float32, device=dev)
    hmask = torch.empty(n_rows, dtype=torch.int32, device=dev)
    lib = _lib.load()
    lead = (ctypes.byref(csr.struct()), _ptr(z), z.size(0), _ptr(w), _ptr(res_w), _ptr(res_b), _ptr(bias),
            _ptr(in_scale), _ptr(post), _ptr(out_scale))
    tail = (int(act_out), H, _ptr(z_next), _ptr(hmask))
    if tmem:
        fn, args = lib.mgcn_gcn_layer_fwd_tm, lead + tail
    elif gate_ab is not None:
        keep = _keep_rows(keep, n_rows, 1)
        gate_ab, gate_c = _gate_operands(gate_ab, gate_c, z.size(0))
        fn, args = lib.mgcn_gcn_layer_fwd_tc_gate, lead + (_ptr(keep), float(keep_scale), _ptr(gate_ab),
                                                          _ptr(gate_c)) + tail
    else:
        keep = _keep_rows(keep, n_rows, 1)
        fn, args = lib.mgcn_gcn_layer_fwd_tc_ex, lead + (_ptr(keep), float(keep_scale)) + tail
    ws, nbytes = _workspace(lambda w_, nb, stm: fn(*args, w_, nb, stm), dev)
    _lib.check(fn(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return z_next, hmask


def _gate_operands(ab, c, n):
    ab = _f32c(ab, "gate_ab")
    c = _f32c(c, "gate_c")
    if tuple(ab.shape) != (n, 2):
        raise ValueError(f"gate_ab must be [{n}, 2], got {tuple(ab.shape)}")
    if c is not None and c.numel() != 1:
        raise ValueError("gate_c must have one entry")
    return ab, c


def gate_scores_impl(x, w, u, v, in_scale=None):
    """per-node gate scores (mgcn_gate_scores): [N,2] = ((x w) . u, (x w) . v) / in_scale for x [N,H<=32] (x = the
    stored z = in_scale (.) x of the stack), w [H,32], u / v with 32 entries"""
    _need_cuda(x, w, u, v, in_scale)
    x = _f32c(x, "x")
    w = _f32c(w, "w")
    u = _f32c(u, "u")
    v = _f32c(v, "v")
    in_scale = _f32c(in_scale, "in_scale")
    N, H = x.shape
    if tuple(w.shape) != (H, 32) or u.numel() != 32 or v.numel() != 32:
        raise ValueError("gate_scores needs w [H,32] and u, v with 32 entries")
    ab = torch.empty(N, 2, dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().mgcn_gate_scores(_ptr(x), N, H, _ptr(in_scale), _ptr(w), _ptr(u), _ptr(v), _ptr(ab),
                                            _stream()))
    return ab


def gate_spmm_narrow_impl(csr, x, ab, c):
    """out_i = sum_{j -> i} gate_ij x_j for x [n_in, H<=4] (mgcn_gate_spmm_narrow)"""
    _need_cuda(csr.rowptr, x, ab, c)
    x = _f32c(x, "x")
    ab, c = _gate_operands(ab, c, x.size(0))
    out = torch.empty(csr.n_rows, x.size(1), dtype=torch.float32, device=x.device)
    _lib.check(_lib.load().mgcn_gate_spmm_narrow(ctypes.byref(csr.struct()), _ptr(x), x.size(0), x.size(1), _ptr(ab),
                                                 _ptr(c), _ptr(out), _stream()))
    return out


def gate_grad_by_target_impl(csr, gs, m, ab, c):
    """db [N]: db_i = sum_{j -> i} <gs_i, m_j> g_ij (1 - g_ij) over the forward structure (mgcn_gate_grad_by_target)"""
    _need_cuda(csr.rowptr, gs, m, ab, c)
    gs = _f32c(gs, "gs")
    m = _f32c(m, "m")
    ab, c = _gate_operands(ab, c, m.size(0))
    db = torch.empty(csr.n_rows, dtype=torch.float32, device=gs.device)
    lib = _lib.load()
    args = (ctypes.byref(csr.struct()), _ptr(gs), _ptr(m), _ptr(ab), _ptr(c), _ptr(db))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_gate_grad_by_target(*args, w_, nb, stm), gs.device)
    _lib.check(lib.mgcn_gate_grad_by_target(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return db


def gate_grad_by_source_impl(csr_t, gs, m, ab, c, db, pre, u, v, sigma):
    """(dxw [N,32], dsc [N,3]) of mgcn_gate_grad_by_source: dxw_j = pre_j sum_i g_ij gs_i + da_j u + db_j v and
    dsc_j = (da_j / sigma_j, db_j / sigma_j, db_j)"""
    _need_cuda(csr_t.rowptr, gs, m, ab, c, db, pre, u, v, sigma)
    gs = _f32c(gs, "gs")
    m = _f32c(m, "m")
    ab, c = _gate_operands(ab, c, m.size(0))
    db = _f32c(db, "db")
    pre = _f32c(pre, "pre")
    u = _f32c(u, "u")
    v = _f32c(v, "v")
    sigma = _f32c(sigma, "sigma")
    n = csr_t.n_rows
    dxw = torch.empty(n, 32, dtype=torch.float32, device=gs.device)
    dsc = torch.empty(n, 3, dtype=torch.float32, device=gs.device)
    lib = _lib.load()
    args = (ctypes.byref(csr_t.struct()), _ptr(gs), _ptr(m), _ptr(ab), _ptr(c), _ptr(db), _ptr(pre), _ptr(u), _ptr(v),
            _ptr(sigma), _ptr(dxw), _ptr(dsc))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_gate_grad_by_source(*args, w_, nb, stm), gs.device)
    _lib.check(lib.mgcn_gate_grad_by_source(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return dxw, dsc


def gcn_layer_bwd_impl(dxw, gy, x, w, res_w, hmask_prev, post, want_prev=True, tensor_memory=False, x_scale=None):
    """row-local backward of one layer at hidden 32 (mgcn_gcn_layer_bwd): returns
    (gy_prev | None, gs_prev | None, dw, d_res_w, d_res_b).  x_scale [N] (tensor_memory only): x holds x_scale (.) x"""
    _need_cuda(dxw, gy, x, w, res_w, hmask_prev, post, x_scale)
    if x_scale is not None and not tensor_memory:
        raise ValueError("x_scale needs the tcgen05 backward")
    x_scale = _f32c(x_scale, "x_scale")
    dxw = _f32c(dxw, "dxw")
    gy = _f32c(gy, "gy")
    x = _f32c(x, "x")
    w = _f32c(w, "w")
    res_w = _f32c(res_w, "res_w")
    post = _f32c(post, "post")
    N, H = x.shape
    dev = x.device
    gy_prev = torch.empty_like(x) if want_prev else None
    gs_prev = torch.empty_like(x) if want_prev else None
    dw = torch.empty(H, H, dtype=torch.float32, device=dev)
    drw = torch.empty(H, H, dtype=torch.float32, device=dev)
    drb = torch.empty(H, dtype=torch.float32, device=dev)
    lib = _lib.load()
    args = (_ptr(dxw), _ptr(gy), _ptr(x), *((_ptr(x_scale),) if tensor_memory else ()), _ptr(w), _ptr(res_w),
            _ptr(hmask_prev) if want_prev else None,
            _ptr(post), N, H, _ptr(gy_prev), _ptr(gs_prev), _ptr(dw), _ptr(drw), _ptr(drb))
    fn = lib.mgcn_gcn_layer_bwd_tc if tensor_memory else lib.mgcn_gcn_layer_bwd
    ws, nbytes = _workspace(lambda w_, nb, stm: fn(*args, w_, nb, stm), dev)
    _lib.check(fn(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return gy_prev, gs_prev, dw, drw, drb


def gcn_layer_bwd_bias_impl(dxw, gy, x, w, res_w, hmask_prev, hmask_cur, post, bias_scale=1.0, want_prev=True,
                            x_scale=None):
    """gcn_layer_bwd_impl on tcgen05 plus the node-model bias gradient (mgcn_gcn_layer_bwd_tc_ex): returns
    (gy_prev | None, gs_prev | None, dw, d_res_w, d_res_b, d_bias) with
    d_bias[c] = bias_scale * sum_i bit c of hmask_cur[i] * gy[i,c]   (hmask_cur: this layer's mask words)"""
    _need_cuda(dxw, gy, x, w, res_w, hmask_prev, hmask_cur, post, x_scale)
    if hmask_cur is None:
        raise ValueError("the bias gradient needs this layer's mask words (hmask_cur)")
    x_scale = _f32c(x_scale, "x_scale")
    dxw = _f32c(dxw, "dxw")
    gy = _f32c(gy, "gy")
    x = _f32c(x, "x")
    w = _f32c(w, "w")
    res_w = _f32c(res_w, "res_w")
    post = _f32c(post, "post")
    hmask_cur = _keep_rows(hmask_cur, x.size(0), 1)
    N, H = x.shape
    dev = x.device
    gy_prev = torch.empty_like(x) if want_prev else None
    gs_prev = torch.empty_like(x) if want_prev else None
    dw = torch.empty(H, H, dtype=torch.float32, device=dev)
    drw = torch.empty(H, H, dtype=torch.float32, device=dev)
    drb = torch.empty(H, dtype=torch.float32, device=dev)
    db = torch.empty(H, dtype=torch.float32, device=dev)
    lib = _lib.load()
    args = (_ptr(dxw), _ptr(gy), _ptr(x), _ptr(x_scale), _ptr(w), _ptr(res_w), _ptr(hmask_prev) if want_prev else None,
            _ptr(hmask_cur), _ptr(post), float(bias_scale), N, H, _ptr(gy_prev), _ptr(gs_prev), _ptr(dw), _ptr(drw),
            _ptr(drb), _ptr(db))
    fn = lib.mgcn_gcn_layer_bwd_tc_ex
    ws, nbytes = _workspace(lambda w_, nb, stm: fn(*args, w_, nb, stm), dev)
    _lib.check(fn(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return gy_prev, gs_prev, dw, drw, drb, db


def mask_bits_colsum_impl(gy, bits, scale=1.0):
    """d_bias[c] = scale * sum_i bit c of bits[i] * gy[i,c]   (H = 32; fixed order, mgcn_mask_bits_colsum)"""
    _need_cuda(gy, bits)
    gy = _f32c(gy, "gy")
    bits = _keep_rows(bits, gy.size(0), 1)
    d_bias = torch.empty(gy.size(1), dtype=torch.float32, device=gy.device)
    lib = _lib.load()
    args = (_ptr(gy), _ptr(bits), float(scale), gy.size(0), gy.size(1), _ptr(d_bias))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_mask_bits_colsum(*args, w_, nb, stm), gy.device)
    _lib.check(lib.mgcn_mask_bits_colsum(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return d_bias


def gcn_layer_bwd_fused_impl(csr_t, gs, gy, z, w, res_w, hmask_prev, post, row_scale=None, x_scale=None, want_prev=True):
    """the whole backward of one hidden-32 layer in one launch (mgcn_gcn_layer_bwd_fused): transposed aggregation of gs
    over the by-source structure csr_t (scaled by row_scale) + the row-local products with x = z / x_scale; returns
    (gy_prev | None, gs_prev | None, dw, d_res_w, d_res_b)"""
    _need_cuda(gs, gy, z, w, res_w, hmask_prev, post, row_scale, x_scale)
    gs = _f32c(gs, "gs")
    gy = _f32c(gy, "gy")
    z = _f32c(z, "z")
    w = _f32c(w, "w")
    res_w = _f32c(res_w, "res_w")
    post = _f32c(post, "post")
    row_scale = _f32c(row_scale, "row_scale")
    x_scale = _f32c(x_scale, "x_scale")
    N, H = z.shape
    if csr_t.n_rows != N or gs.size(0) != N or gy.size(0) != N:
        raise ValueError("gcn_layer_bwd_fused needs a square structure and [N,32] operands")
    dev = z.device
    gy_prev = torch.empty_like(z) if want_prev else None
    gs_prev = torch.empty_like(z) if want_prev else None
    dw = torch.empty(H, H, dtype=torch.float32, device=dev)
    drw = torch.empty(H, H, dtype=torch.float32, device=dev)
    drb = torch.empty(H, dtype=torch.float32, device=dev)
    lib = _lib.load()
    args = (ctypes.byref(csr_t.struct()), _ptr(gs), _ptr(gy), _ptr(z), _ptr(x_scale), _ptr(row_scale), _ptr(w),
            _ptr(res_w), _ptr(hmask_prev) if want_prev else None, _ptr(post), H, _ptr(gy_prev), _ptr(gs_prev),
            _ptr(dw), _ptr(drw), _ptr(drb))
    fn = lib.mgcn_gcn_layer_bwd_fused
    ws, nbytes = _workspace(lambda w_, nb, stm: fn(*args, w_, nb, stm), dev)
    _lib.check(fn(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return gy_prev, gs_prev, dw, drw, drb


def mask_bits_scale_impl(gy, bits, post):
    """gs = post[:,None] * gy * bit(bits, column)   (H = 32)"""
    _need_cuda(gy, bits, post)
    gy = _f32c(gy, "gy")
    post = _f32c(post, "post")
    out = torch.empty_like(gy)
    _lib.check(_lib.load().mgcn_mask_bits_scale(_ptr(gy), _ptr(bits), _ptr(post), gy.size(0), gy.size(1),
                                                _ptr(out), _stream()))
    return out


def dropout_keep_bits_impl(seed, L, N, W, p):
    """dropout keep masks of L layers as bits (mgcn_dropout_keep_bits): int32 [L, N, W], bit b of word w = column
    32 w + b kept; a pure function of (seed[0], layer, row, column) — include/mgcn.h states the generator exactly"""
    _need_cuda(seed)
    if seed.dtype != torch.int64 or seed.numel() != 1:
        raise TypeError("seed must be one int64 on the device")
    keep = torch.empty(L, N, W, dtype=torch.int32, device=seed.device)
    _lib.check(_lib.load().mgcn_dropout_keep_bits(_ptr(seed.contiguous()), int(L), int(N), int(W), float(p),
                                                  _ptr(keep), _stream()))
    return keep


def dropout_apply_impl(h, keep, scale):
    """h[n,c] = keep bit ? h[n,c] * scale : 0 IN PLACE (mgcn_dropout_apply); keep int32 [N, W] (one layer's bits)"""
    _need_cuda(h, keep)
    if h.dtype != torch.float32 or not h.is_contiguous():
        raise TypeError("h must be a contiguous float32 tensor (updated in place)")
    N, H = h.shape
    W = keep.size(-1) if keep.dim() > 1 else 1
    keep = _keep_rows(keep, N, W)
    _lib.check(_lib.load().mgcn_dropout_apply(_ptr(h), _ptr(keep), N, H, W, float(scale), _stream()))
    return h


def cross_entropy_fwd_impl(logits, target, mean):
    _need_cuda(logits, target)
    logits = _f32c(logits, "logits")
    if target.dtype != torch.int64:
        raise TypeError("target must be int64 (batch.y.long())")
    target = target.contiguous()
    N, C = logits.shape
    loss = torch.empty(1, dtype=torch.float32, device=logits.device)
    bad = torch.empty(1, dtype=torch.int32, device=logits.device)
    lib = _lib.load()
    args = (_ptr(logits), _ptr(target), N, C, int(bool(mean)), _ptr(loss), _ptr(bad))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_cross_entropy_fwd(*args, w_, nb, stm), logits.device)
    _lib.check(lib.mgcn_cross_entropy_fwd(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return loss, bad


def cross_entropy_bwd_impl(logits, target, mean, upstream):
    _need_cuda(logits, target, upstream)
    logits = _f32c(logits, "logits")
    N, C = logits.shape
    up = None if upstream is None else _f32c(upstream, "upstream").reshape(-1)
    out = torch.empty_like(logits)
    _lib.check(_lib.load().mgcn_cross_entropy_bwd(_ptr(logits), _ptr(target.contiguous()), N, C,
                                                  int(bool(mean)), _ptr(up), _ptr(out), _stream()))
    return out


def relu_backward_impl(g, y):
    _need_cuda(g, y)
    g = _f32c(g, "g")
    y = _f32c(y, "y")
    out = torch.empty_like(g)
    _lib.check(_lib.load().mgcn_relu_backward(_ptr(g), _ptr(y), g.numel(), _ptr(out), _stream()))
    return out


def batch_to_offsets_impl(batch, G):
    _need_cuda(batch)
    if batch.dtype != torch.int64:
        raise TypeError("batch must be int64")
    b = batch.contiguous()
    off = torch.empty(int(G) + 1, dtype=torch.int32, device=b.device)
    _lib.check(_lib.load().mgcn_batch_to_offsets(_ptr(b), b.numel(), int(G), _ptr(off), _stream()))
    return off


def segment_reduce_impl(x, offsets, mode):
    _need_cuda(x, offsets)
    x = _f32c(x, "x")
    G = offsets.numel() - 1
    out = torch.empty(G, x.size(1), dtype=torch.float32, device=x.device)
    lib = _lib.load()
    args = (_ptr(x), x.size(1), _ptr(offsets), G, x.size(0), int(mode), _ptr(out))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_segment_reduce(*args, w_, nb, stm), x.device)
    _lib.check(lib.mgcn_segment_reduce(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return out


def segment_broadcast_impl(gout, offsets, N, mode):
    _need_cuda(gout, offsets)
    gout = _f32c(gout, "gout")
    G = offsets.numel() - 1
    dx = torch.empty(int(N), gout.size(1), dtype=torch.float32, device=gout.device)
    _lib.check(_lib.load().mgcn_segment_broadcast(_ptr(gout), gout.size(1), _ptr(offsets), G, int(N),
                                                  int(mode), _ptr(dx), _stream()))
    return dx


def head_cross_entropy_fwd_impl(x, w, b, target, mean, want_counts=False):
    """mgcn_head_cross_entropy_fwd: returns (logits [N,C], loss [1], counts int64[5] | None, bad int32[1])"""
    _need_cuda(x, w, b, target)
    x = _f32c(x, "x")
    w = _f32c(w, "w")
    b = _f32c(b, "b")
    if target.dtype != torch.int64:
        raise TypeError("target must be int64 (batch.y.long())")
    target = target.contiguous()
    N, H = x.shape
    C = w.size(0)
    dev = x.device
    logits = torch.empty(N, C, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    counts = torch.empty(5, dtype=torch.int64, device=dev) if want_counts else None
    bad = torch.empty(1, dtype=torch.int32, device=dev)
    lib = _lib.load()
    args = (_ptr(x), N, H, _ptr(w), _ptr(b), C, _ptr(target), int(bool(mean)), _ptr(logits), _ptr(loss), _ptr(counts),
            _ptr(bad))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_head_cross_entropy_fwd(*args, w_, nb, stm), dev)
    _lib.check(lib.mgcn_head_cross_entropy_fwd(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return logits, loss, counts, bad


def head_cross_entropy_bwd_impl(x, logits, w, target, mean, upstream, want_dx=True):
    """mgcn_head_cross_entropy_bwd: returns (dx | None, dw [C,H], db [C])"""
    _need_cuda(x, logits, w, target, upstream)
    N, H = x.shape
    C = w.size(0)
    dev = x.device
    dx = torch.empty_like(x) if want_dx else None
    dw = torch.empty(C, H, dtype=torch.float32, device=dev)
    db = torch.empty(C, dtype=torch.float32, device=dev)
    lib = _lib.load()
    args = (_ptr(x), _ptr(logits), N, H, _ptr(w), C, _ptr(target), int(bool(mean)), _ptr(upstream), _ptr(dx), _ptr(dw),
            _ptr(db))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_head_cross_entropy_bwd(*args, w_, nb, stm), dev)
    _lib.check(lib.mgcn_head_cross_entropy_bwd(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return dx, dw, db


def batchnorm_fwd_impl(x, gamma, beta, running_mean, running_var, training, momentum, eps):
    """mgcn_batchnorm_fwd: returns (y, mean [H], rstd [H]); running statistics are updated in place when training"""
    _need_cuda(x, gamma, beta, running_mean, running_var)
    x = _f32c(x, "x")
    gamma = _f32c(gamma, "gamma")
    beta = _f32c(beta, "beta")
    N, H = x.shape
    dev = x.device
    y = torch.empty_like(x)
    mean = torch.empty(H, dtype=torch.float32, device=dev)
    rstd = torch.empty(H, dtype=torch.float32, device=dev)
    lib = _lib.load()
    args = (_ptr(x), N, H, _ptr(gamma), _ptr(beta), float(eps), float(momentum), int(bool(training)),
            _ptr(running_mean), _ptr(running_var), _ptr(mean), _ptr(rstd), _ptr(y))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_batchnorm_fwd(*args, w_, nb, stm), dev)
    _lib.check(lib.mgcn_batchnorm_fwd(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return y, mean, rstd


def batchnorm_bwd_impl(x, g, gamma, mean, rstd, training, want_dx=True):
    """mgcn_batchnorm_bwd: returns (dx | None, dgamma [H], dbeta [H])"""
    _need_cuda(x, g, gamma, mean, rstd)
    x = _f32c(x, "x")
    g = _f32c(g, "g")
    gamma = _f32c(gamma, "gamma")
    N, H = x.shape
    dev = x.device
    dx = torch.empty_like(x) if want_dx else None
    dgamma = torch.empty(H, dtype=torch.float32, device=dev)
    dbeta = torch.empty(H, dtype=torch.float32, device=dev)
    lib = _lib.load()
    args = (_ptr(x), _ptr(g), N, H, _ptr(gamma), _ptr(mean), _ptr(rstd), int(bool(training)), _ptr(dx),
            _ptr(dgamma), _ptr(dbeta))
    ws, nbytes = _workspace(lambda w_, nb, stm: lib.mgcn_batchnorm_bwd(*args, w_, nb, stm), dev)
    _lib.check(lib.mgcn_batchnorm_bwd(*args, _ptr(ws), ctypes.byref(nbytes), _stream()))
    return dx, dgamma, dbeta


# ------------------------------------------------------------------------------------------------
# torch.library registration
# ------------------------------------------------------------------------------------------------
_LIBDEF = torch.library.Library("mgcn", "DEF")
# `csr` is the list of the int32 tensors of a row structure, in CSR_FIELDS order
_LIBDEF.define("csr_build(Tensor edge_index, int N, int by, int loop_mode, int hub_threshold) -> Tensor[]")
_LIBDEF.define("degree(Tensor rowptr) -> Tensor")
_LIBDEF.define("weighted_degree(Tensor[] csr, Tensor edge_weight, float loop_weight) -> Tensor")
_LIBDEF.define("gcn_norm(Tensor deg, int mode) -> Tensor")
_LIBDEF.define("permute_edge_values(Tensor[] csr, Tensor vals, float loop_value) -> Tensor")
_LIBDEF.define("spmm(Tensor[] csr, int hub_threshold, Tensor x, bool gather_perm, Tensor? edge_val, "
               "Tensor? nbr_scale, Tensor? row_scale, int reduce, Tensor? bias, Tensor? residual, "
               "int act) -> Tensor")
_LIBDEF.define("aggregate_prescaled(Tensor[] csr, int hub_threshold, Tensor x, Tensor? post_scale, "
               "int reduce, Tensor? bias, Tensor? residual, int act) -> Tensor")
_LIBDEF.define("linear(Tensor x, Tensor w, bool w_out_in, Tensor? bias, Tensor? add, int act, "
               "Tensor? xmask=None, Tensor? row_scale=None) -> Tensor")
_LIBDEF.define("linear_wgrad(Tensor x, Tensor g, bool w_out_in, bool want_bias, Tensor? gmask=None) -> "
               "(Tensor, Tensor)")
_LIBDEF.define("masked_scale(Tensor g, Tensor? m1, Tensor? m2, Tensor? row_scale) -> Tensor")
_LIBDEF.define("relu_backward(Tensor g, Tensor y) -> Tensor")
_LIBDEF.define("cross_entropy_fwd(Tensor logits, Tensor target, bool mean) -> (Tensor, Tensor)")
_LIBDEF.define("cross_entropy_bwd(Tensor logits, Tensor target, bool mean, Tensor? upstream) -> Tensor")
_LIBDEF.define("batch_to_offsets(Tensor batch, int G) -> Tensor")
_LIBDEF.define("segment_reduce(Tensor x, Tensor offsets, int mode) -> Tensor")
_LIBDEF.define("segment_broadcast(Tensor gout, Tensor offsets, int N, int mode) -> Tensor")


def _op_csr_build(edge_index, N, by, loop_mode, hub_threshold):
    return csr_build_impl(edge_index, N, by, loop_mode, hub_threshold).tensors()


def _op_weighted_degree(csr, edge_weight, loop_weight):
    return weighted_degree_impl(_as_csr(csr, DEFAULT_HUB_THRESHOLD), edge_weight, loop_weight)


def _op_permute_edge_values(csr, vals, loop_value):
    return permute_edge_values_impl(_as_csr(csr, DEFAULT_HUB_THRESHOLD), vals, loop_value)


def _op_spmm(csr, hub_threshold, x, gather_perm, edge_val, nbr_scale, row_scale, reduce, bias,
             residual, act):
    return spmm_impl(_as_csr(csr, hub_threshold), x, gather_perm, edge_val, nbr_scale, row_scale,
                     reduce, bias, residual, act)


def _op_aggregate_prescaled(csr, hub_threshold, x, post_scale, reduce, bias, residual, act):
    return aggregate_prescaled_impl(_as_csr(csr, hub_threshold), x, post_scale, reduce, bias,
                                    residual, act)


_IMPLS = {
    "csr_build": _op_csr_build,
    "degree": degree_impl,
    "weighted_degree": _op_weighted_degree,
    "gcn_norm": gcn_norm_impl,
    "permute_edge_values": _op_permute_edge_values,
    "spmm": _op_spmm,
    "aggregate_prescaled": _op_aggregate_prescaled,
    "linear": linear_impl,
    "linear_wgrad": linear_wgrad_impl,
    "masked_scale": masked_scale_impl,
    "relu_backward": relu_backward_impl,
    "cross_entropy_fwd": cross_entropy_fwd_impl,
    "cross_entropy_bwd": cross_entropy_bwd_impl,
    "batch_to_offsets": batch_to_offsets_impl,
    "segment_reduce": segment_reduce_impl,
    "segment_broadcast": segment_broadcast_impl,
}
for _name, _fn in _IMPLS.items():
    _LIBDEF.impl(_name, _fn, "CUDA")


def _cpu_refusal(name):
    def _raise(*args, **kwargs):
        raise RuntimeError(f"mgcn::{name} has no CPU implementation (CUDA sm_100a only)")
    return _raise


for _name in _IMPLS:
    _LIBDEF.impl(_name, _cpu_refusal(_name), "CPU")


# fake (meta) implementations so the ops trace under FakeTensor / torch.export
@torch.library.register_fake("mgcn::csr_build")
def _(edge_index, N, by, loop_mode, hub_threshold):
    E = edge_index.size(1)
    cap = E + (N if loop_mode == 2 else 0)
    hub_cap = cap // max(hub_threshold, 1) + 1
    seg_cap = cap // max(hub_threshold, 1) + hub_cap + 1
    i32 = dict(dtype=torch.int32, device=edge_index.device)
    sizes = (N + 1, cap, cap, N, hub_cap, hub_cap, 1, seg_cap, seg_cap, 1, 4 * (N + seg_cap), cap)
    return [torch.empty(n, **i32) for n in sizes]


@torch.library.register_fake("mgcn::degree")
def _(rowptr):
    return torch.empty(rowptr.numel() - 1, dtype=torch.float32, device=rowptr.device)


@torch.library.register_fake("mgcn::weighted_degree")
def _(csr, edge_weight, loop_weight):
    return torch.empty(csr[0].numel() - 1, dtype=torch.float32, device=csr[0].device)


@torch.library.register_fake("mgcn::gcn_norm")
def _(deg, mode):
    return torch.empty_like(deg)


@torch.library.register_fake("mgcn::permute_edge_values")
def _(csr, vals, loop_value):
    return torch.empty(csr[1].numel(), dtype=torch.float32, device=csr[0].device)


@torch.library.register_fake("mgcn::spmm")
def _(csr, hub_threshold, x, gather_perm, edge_val, nbr_scale, row_scale, reduce, bias, residual, act):
    return torch.empty(csr[0].numel() - 1, x.size(1), dtype=torch.float32, device=x.device)


@torch.library.register_fake("mgcn::aggregate_prescaled")
def _(csr, hub_threshold, x, post_scale, reduce, bias, residual, act):
    return torch.empty(csr[0].numel() - 1, x.size(1), dtype=torch.float32, device=x.device)


@torch.library.register_fake("mgcn::masked_scale")
def _(g, m1, m2, row_scale):
    return torch.empty_like(g)


@torch.library.register_fake("mgcn::linear")
def _(x, w, w_out_in, bias, add, act, xmask=None, row_scale=None):
    Ho = w.size(0) if w_out_in else w.size(1)
    return torch.empty(x.size(0), Ho, dtype=torch.float32, device=x.device)


@torch.library.register_fake("mgcn::linear_wgrad")
def _(x, g, w_out_in, want_bias, gmask=None):
    Hi, Ho = x.size(1), g.size(1)
    shape = (Ho, Hi) if w_out_in else (Hi, Ho)
    return (torch.empty(shape, dtype=torch.float32, device=x.device),
            torch.empty(Ho if want_bias else 0, dtype=torch.float32, device=x.device))


@torch.library.register_fake("mgcn::cross_entropy_fwd")
def _(logits, target, mean):
    return (torch.empty(1, dtype=torch.float32, device=logits.device),
            torch.empty(1, dtype=torch.int32, device=logits.device))


@torch.library.register_fake("mgcn::cross_entropy_bwd")
def _(logits, target, mean, upstream):
    return torch.empty_like(logits)


@torch.library.register_fake("mgcn::relu_backward")
def _(g, y):
    return torch.empty_like(g)


@torch.library.register_fake("mgcn::batch_to_offsets")
def _(batch, G):
    return torch.empty(G + 1, dtype=torch.int32, device=batch.device)


@torch.library.register_fake("mgcn::segment_reduce")
def _(x, offsets, mode):
    return torch.empty(offsets.numel() - 1, x.size(1), dtype=torch.float32, device=x.device)


@torch.library.register_fake("mgcn::segment_broadcast")
def _(gout, offsets, N, mode):
    return torch.empty(N, gout.size(1), dtype=torch.float32, device=gout.device)



# ------------------------------------------------------------------------------------------------
# second group: the fused layer launches, the wide transform, 'max' aggregation, edge gates, preprocessing and
# metrics as torch.ops.mgcn.* too (SURVEY.md §8b: the op table is the library's Python surface), plus
# register_autograd for the differentiable core (propagate, linear, segment_reduce) so that
# torch.ops.mgcn.propagate / linear / segment_reduce carry gradients without the wrappers of functional.py
# ------------------------------------------------------------------------------------------------
_LIBDEF.define("gcn_layer_fwd_tc(Tensor[] csr, int hub_threshold, Tensor z, Tensor w, Tensor res_w, Tensor? res_b, "
               "Tensor? bias, Tensor? in_scale, Tensor? post, Tensor? out_scale, int act_out) -> (Tensor, Tensor)")
_LIBDEF.define("gcn_first_layer_fwd(Tensor s, Tensor x, Tensor w_in, Tensor res_w, Tensor? res_b, Tensor? w_next, "
               "Tensor? pre, Tensor? post, int act_out, Tensor? out_scale) -> (Tensor, Tensor, Tensor)")
_LIBDEF.define("gcn_layer_bwd(Tensor dxw, Tensor gy, Tensor x, Tensor w, Tensor res_w, Tensor? hmask_prev, Tensor? post, "
               "bool want_prev, bool tensor_memory, Tensor? x_scale) -> (Tensor, Tensor, Tensor, Tensor, Tensor)")
_LIBDEF.define("mask_bits_scale(Tensor gy, Tensor bits, Tensor? post) -> Tensor")
_LIBDEF.define("gcn_first_layer_fwd_bias(Tensor s, Tensor x, Tensor w_in, Tensor res_w, Tensor? res_b, Tensor bias, "
               "Tensor? w_next, Tensor? pre, Tensor? post, int act_out, Tensor? out_scale) -> (Tensor, Tensor, Tensor)")
_LIBDEF.define("gcn_layer_bwd_bias(Tensor dxw, Tensor gy, Tensor x, Tensor w, Tensor res_w, Tensor? hmask_prev, "
               "Tensor hmask_cur, Tensor? post, float bias_scale, bool want_prev, Tensor? x_scale) "
               "-> (Tensor, Tensor, Tensor, Tensor, Tensor, Tensor)")
_LIBDEF.define("mask_bits_colsum(Tensor gy, Tensor bits, float scale) -> Tensor")
_LIBDEF.define("gate_scores(Tensor x, Tensor w, Tensor u, Tensor v, Tensor? in_scale) -> Tensor")
_LIBDEF.define("gcn_layer_fwd_tc_gate(Tensor[] csr, int hub_threshold, Tensor z, Tensor w, Tensor res_w, Tensor? res_b, "
               "Tensor? bias, Tensor? in_scale, Tensor? post, Tensor? out_scale, int act_out, Tensor? keep, "
               "float keep_scale, Tensor gate_ab, Tensor? gate_c) -> (Tensor, Tensor)")
_LIBDEF.define("gate_spmm_narrow(Tensor[] csr, int hub_threshold, Tensor x, Tensor ab, Tensor? c) -> Tensor")
_LIBDEF.define("gate_grad_by_target(Tensor[] csr, int hub_threshold, Tensor gs, Tensor m, Tensor ab, Tensor? c) "
               "-> Tensor")
_LIBDEF.define("gate_grad_by_source(Tensor[] csr_t, int hub_threshold, Tensor gs, Tensor m, Tensor ab, Tensor? c, "
               "Tensor db, Tensor? pre, Tensor u, Tensor v, Tensor? sigma) -> (Tensor, Tensor)")
_LIBDEF.define("dropout_keep_bits(Tensor seed, int L, int N, int W, float p) -> Tensor")
_LIBDEF.define("segment_max(Tensor[] csr, int hub_threshold, Tensor x, bool gather_perm, Tensor? edge_val) -> (Tensor, Tensor)")
_LIBDEF.define("segment_max_bwd(Tensor[] csr_t, int hub_threshold, Tensor grad, Tensor arg, Tensor? edge_val) -> Tensor")
_LIBDEF.define("scatter_max_bwd(Tensor arg, Tensor grad, int n_src) -> Tensor")
_LIBDEF.define("edge_dot(Tensor edge_index, Tensor a, Tensor b, Tensor? scale_src, Tensor? scale_tgt) -> Tensor")
_LIBDEF.define("binary_confusion(Tensor target, Tensor? logits, Tensor? pred) -> Tensor")
_LIBDEF.define("preprocess_edges(Tensor edge_index, int N, bool undirected, bool add_loops) -> (Tensor, Tensor, Tensor)")
_LIBDEF.define("edge_fingerprint(Tensor edge_index) -> Tensor")
_LIBDEF.define("propagate(Tensor[] csr, Tensor[] csr_t, int hub_threshold, Tensor x, Tensor? nbr_scale, "
               "Tensor? row_scale, int act) -> Tensor")


def _none_to_empty(t, like):
    return t if t is not None else torch.empty(0, dtype=torch.float32, device=like.device)


def _op_layer_fwd_tc(csr, hub_threshold, z, w, res_w, res_b, bias, in_scale, post, out_scale, act_out):
    return gcn_layer_fwd_tc_impl(_as_csr(csr, hub_threshold), z, w, res_w, res_b, bias, in_scale, post, out_scale,
                                 act_out)


def _op_first_layer_fwd(s, x, w_in, res_w, res_b, w_next, pre, post, act_out, out_scale):
    xn, mn, hm = gcn_first_layer_fwd_impl(s, x, w_in, res_w, res_b, w_next, pre, post, act_out, out_scale)
    return xn, _none_to_empty(mn, xn), hm


def _op_layer_bwd(dxw, gy, x, w, res_w, hmask_prev, post, want_prev, tensor_memory, x_scale):
    gyp, gsp, dw, drw, drb = gcn_layer_bwd_impl(dxw, gy, x, w, res_w, hmask_prev, post, want_prev, tensor_memory,
                                                x_scale)
    return _none_to_empty(gyp, dw), _none_to_empty(gsp, dw), dw, drw, drb


def _op_first_layer_fwd_bias(s, x, w_in, res_w, res_b, bias, w_next, pre, post, act_out, out_scale):
    xn, mn, hm = gcn_first_layer_fwd_impl(s, x, w_in, res_w, res_b, w_next, pre, post, act_out, out_scale, bias=bias)
    return xn, _none_to_empty(mn, xn), hm


def _op_layer_bwd_bias(dxw, gy, x, w, res_w, hmask_prev, hmask_cur, post, bias_scale, want_prev, x_scale):
    gyp, gsp, dw, drw, drb, db = gcn_layer_bwd_bias_impl(dxw, gy, x, w, res_w, hmask_prev, hmask_cur, post, bias_scale,
                                                         want_prev, x_scale)
    return _none_to_empty(gyp, dw), _none_to_empty(gsp, dw), dw, drw, drb, db


def _op_edge_fingerprint(edge_index):
    _need_cuda(edge_index)
    ei = edge_index.contiguous()
    out = torch.empty(4, dtype=torch.int64, device=ei.device)
    lib = _lib.load()
    fn = lib.mgcn_edge_fingerprint if ei.dtype == torch.int64 else lib.mgcn_edge_fingerprint_i32
    _lib.check(fn(_ptr(ei), ei.size(1), _ptr(out), _stream()))
    return out


def _op_propagate(csr, csr_t, hub_threshold, x, nbr_scale, row_scale, act):
    return spmm_impl(_as_csr(csr, hub_threshold), x, False, None, nbr_scale, row_scale, 0, None, None, act)


def _op_layer_fwd_tc_gate(csr, hub_threshold, z, w, res_w, res_b, bias, in_scale, post, out_scale, act_out, keep,
                          keep_scale, gate_ab, gate_c):
    return gcn_layer_fwd_tc_impl(_as_csr(csr, hub_threshold), z, w, res_w, res_b, bias, in_scale, post, out_scale,
                                 act_out, tmem_operands=False, keep=keep, keep_scale=keep_scale, gate_ab=gate_ab,
                                 gate_c=gate_c)


_IMPLS2 = {
    "gate_scores": gate_scores_impl,
    "gcn_layer_fwd_tc_gate": _op_layer_fwd_tc_gate,
    "gate_spmm_narrow": lambda csr, ht, x, ab, c: gate_spmm_narrow_impl(_as_csr(csr, ht), x, ab, c),
    "gate_grad_by_target": lambda csr, ht, gs, m, ab, c: gate_grad_by_target_impl(_as_csr(csr, ht), gs, m, ab, c),
    "gate_grad_by_source": lambda csr_t, ht, gs, m, ab, c, db, pre, u, v, sigma: gate_grad_by_source_impl(
        _as_csr(csr_t, ht), gs, m, ab, c, db, pre, u, v, sigma),
    "gcn_layer_fwd_tc": _op_layer_fwd_tc,
    "gcn_first_layer_fwd": _op_first_layer_fwd,
    "gcn_layer_bwd": _op_layer_bwd,
    "mask_bits_scale": mask_bits_scale_impl,
    "gcn_first_layer_fwd_bias": _op_first_layer_fwd_bias,
    "gcn_layer_bwd_bias": _op_layer_bwd_bias,
    "mask_bits_colsum": mask_bits_colsum_impl,
    "dropout_keep_bits": dropout_keep_bits_impl,
    "segment_max": lambda csr, ht, x, gp, ev: segment_max_impl(_as_csr(csr, ht), x, gp, ev),
    "segment_max_bwd": lambda csr_t, ht, grad, arg, ev: segment_max_bwd_impl(_as_csr(csr_t, ht), grad, arg, ev),
    "scatter_max_bwd": scatter_max_bwd_impl,
    "edge_dot": edge_dot_impl,
    "binary_confusion": binary_confusion_impl,
    "preprocess_edges": preprocess_edges_impl,
    "edge_fingerprint": _op_edge_fingerprint,
    "propagate": _op_propagate,
}
for _name, _fn in _IMPLS2.items():
    _LIBDEF.impl(_name, _fn, "CUDA")
    _LIBDEF.impl(_name, _cpu_refusal(_name), "CPU")
_IMPLS.update(_IMPLS2)


def _rows_of(csr):
    return csr[0].numel() - 1


@torch.library.register_fake("mgcn::gcn_layer_fwd_tc")
def _(csr, hub_threshold, z, w, res_w, res_b, bias, in_scale, post, out_scale, act_out):
    n = _rows_of(csr)
    return (torch.empty(n, z.size(1), dtype=torch.float32, device=z.device),
            torch.empty(n, dtype=torch.int32, device=z.device))


@torch.library.register_fake("mgcn::gcn_first_layer_fwd")
def _(s, x, w_in, res_w, res_b, w_next, pre, post, act_out, out_scale):
    n, h = x.size(0), w_in.size(1)
    return (torch.empty(n, h, dtype=torch.float32, device=x.device),
            torch.empty((n, h) if w_next is not None else (0,), dtype=torch.float32, device=x.device),
            torch.empty(n, dtype=torch.int32, device=x.device))


@torch.library.register_fake("mgcn::gcn_layer_bwd")
def _(dxw, gy, x, w, res_w, hmask_prev, post, want_prev, tensor_memory, x_scale):
    h = x.size(1)
    prev = torch.empty_like(x) if want_prev else torch.empty(0, dtype=torch.float32, device=x.device)
    f = dict(dtype=torch.float32, device=x.device)
    return prev, torch.empty_like(prev), torch.empty(h, h, **f), torch.empty(h, h, **f), torch.empty(h, **f)


@torch.library.register_fake("mgcn::mask_bits_scale")
def _(gy, bits, post):
    return torch.empty_like(gy)


@torch.library.register_fake("mgcn::gcn_first_layer_fwd_bias")
def _(s, x, w_in, res_w, res_b, bias, w_next, pre, post, act_out, out_scale):
    n, h = x.size(0), w_in.size(1)
    return (torch.empty(n, h, dtype=torch.float32, device=x.device),
            torch.empty((n, h) if w_next is not None else (0,), dtype=torch.float32, device=x.device),
            torch.empty(n, dtype=torch.int32, device=x.device))


@torch.library.register_fake("mgcn::gcn_layer_bwd_bias")
def _(dxw, gy, x, w, res_w, hmask_prev, hmask_cur, post, bias_scale, want_prev, x_scale):
    h = x.size(1)
    prev = torch.empty_like(x) if want_prev else torch.empty(0, dtype=torch.float32, device=x.device)
    f = dict(dtype=torch.float32, device=x.device)
    return (prev, torch.empty_like(prev), torch.empty(h, h, **f), torch.empty(h, h, **f), torch.empty(h, **f),
            torch.empty(h, **f))


@torch.library.register_fake("mgcn::mask_bits_colsum")
def _(gy, bits, scale):
    return torch.empty(gy.size(1), dtype=torch.float32, device=gy.device)


@torch.library.register_fake("mgcn::gate_scores")
def _(x, w, u, v, in_scale):
    return torch.empty(x.size(0), 2, dtype=torch.float32, device=x.device)


@torch.library.register_fake("mgcn::gcn_layer_fwd_tc_gate")
def _(csr, hub_threshold, z, w, res_w, res_b, bias, in_scale, post, out_scale, act_out, keep, keep_scale, gate_ab,
      gate_c):
    n = _rows_of(csr)
    return (torch.empty(n, z.size(1), dtype=torch.float32, device=z.device),
            torch.empty(n, dtype=torch.int32, device=z.device))


@torch.library.register_fake("mgcn::gate_spmm_narrow")
def _(csr, hub_threshold, x, ab, c):
    return torch.empty(_rows_of(csr), x.size(1), dtype=torch.float32, device=x.device)


@torch.library.register_fake("mgcn::gate_grad_by_target")
def _(csr, hub_threshold, gs, m, ab, c):
    return torch.empty(_rows_of(csr), dtype=torch.float32, device=gs.device)


@torch.library.register_fake("mgcn::gate_grad_by_source")
def _(csr_t, hub_threshold, gs, m, ab, c, db, pre, u, v, sigma):
    n = _rows_of(csr_t)
    return (torch.empty(n, 32, dtype=torch.float32, device=gs.device),
            torch.empty(n, 3, dtype=torch.float32, device=gs.device))


@torch.library.register_fake("mgcn::dropout_keep_bits")
def _(seed, L, N, W, p):
    return torch.empty(L, N, W, dtype=torch.int32, device=seed.device)


@torch.library.register_fake("mgcn::segment_max")
def _(csr, hub_threshold, x, gather_perm, edge_val):
    n = _rows_of(csr)
    return (torch.empty(n, x.size(1), dtype=torch.float32, device=x.device),
            torch.empty(n, x.size(1), dtype=torch.int32, device=x.device))


@torch.library.register_fake("mgcn::segment_max_bwd")
def _(csr_t, hub_threshold, grad, arg, edge_val):
    return torch.empty(_rows_of(csr_t), grad.size(1), dtype=torch.float32, device=grad.device)


@torch.library.register_fake("mgcn::scatter_max_bwd")
def _(arg, grad, n_src):
    return torch.empty(n_src, grad.size(1), dtype=torch.float32, device=grad.device)


@torch.library.register_fake("mgcn::edge_dot")
def _(edge_index, a, b, scale_src, scale_tgt):
    return torch.empty(edge_index.size(1), dtype=torch.float32, device=a.device)


@torch.library.register_fake("mgcn::binary_confusion")
def _(target, logits, pred):
    return torch.empty(5, dtype=torch.int64, device=target.device)


@torch.library.register_fake("mgcn::edge_fingerprint")
def _(edge_index):
    return torch.empty(4, dtype=torch.int64, device=edge_index.device)


@torch.library.register_fake("mgcn::propagate")
def _(csr, csr_t, hub_threshold, x, nbr_scale, row_scale, act):
    return torch.empty(_rows_of(csr), x.size(1), dtype=torch.float32, device=x.device)


# ---- autograd formulas (deterministic: the transposed aggregation is the same row-owned kernel on csr_t) ----
def _propagate_setup(ctx, inputs, output):
    csr, csr_t, hub_threshold, x, nbr_scale, row_scale, act = inputs
    ctx.csr_t, ctx.hub_threshold, ctx.act, ctx.n_csr = csr_t, hub_threshold, act, len(csr)
    ctx.save_for_backward(output if act else None, nbr_scale, row_scale)


def _propagate_backward(ctx, g):
    out, nbr_scale, row_scale = ctx.saved_tensors
    g = g.contiguous()
    if ctx.act:
        g = torch.ops.mgcn.relu_backward(g, out)
    # transpose: rows = sources; the per-target factor is gathered, the per-source factor scales the row
    dx = torch.ops.mgcn.spmm(ctx.csr_t, ctx.hub_threshold, g, False, None, row_scale, nbr_scale, 0, None, None, 0)
    # gradients mirror the input structure: one entry per tensor of the two structure lists
    return [None] * ctx.n_csr, [None] * len(ctx.csr_t), None, dx, None, None, None


torch.library.register_autograd("mgcn::propagate", _propagate_backward, setup_context=_propagate_setup)


def _linear_setup(ctx, inputs, output):
    x, w, w_out_in, bias, add, act, xmask, row_scale = inputs
    if xmask is not None or row_scale is not None:
        raise RuntimeError("mgcn::linear is differentiable without xmask / row_scale only")
    ctx.cfg = (w_out_in, act, bias is not None, add is not None)
    ctx.save_for_backward(x, w, output if act else None)


def _linear_backward(ctx, g):
    x, w, y = ctx.saved_tensors
    w_out_in, act, has_bias, has_add = ctx.cfg
    g = g.contiguous()
    if act:
        g = torch.ops.mgcn.relu_backward(g, y)
    dx = torch.ops.mgcn.linear(g, w, not w_out_in, None, None, 0) if ctx.needs_input_grad[0] else None
    dw = db = None
    if ctx.needs_input_grad[1] or (has_bias and ctx.needs_input_grad[3]):
        dw, db_ = torch.ops.mgcn.linear_wgrad(x, g, w_out_in, has_bias)
        db = db_ if has_bias else None
    return dx, dw, None, db, (g if has_add else None), None, None, None


torch.library.register_autograd("mgcn::linear", _linear_backward, setup_context=_linear_setup)


def _segred_setup(ctx, inputs, output):
    x, offsets, mode = inputs
    ctx.n, ctx.mode = x.size(0), mode
    ctx.save_for_backward(offsets)


def _segred_backward(ctx, g):
    (offsets,) = ctx.saved_tensors
    return torch.ops.mgcn.segment_broadcast(g.contiguous(), offsets, ctx.n, ctx.mode), None, None


torch.library.register_autograd("mgcn::segment_reduce", _segred_backward, setup_context=_segred_setup)

OP_NAMES = tuple(_IMPLS)
