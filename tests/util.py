"""Shared helpers of the parity tests."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# north_star tolerance for fp32 features and gradients
RTOL = 1e-5


def golden(name):
    with np.load(os.path.join(GOLDEN, name + ".npz")) as z:
        return {k: z[k] for k in z.files}


def params_of(g, prefix="param."):
    return {k[len(prefix):]: torch.from_numpy(v.copy()) for k, v in g.items() if k.startswith(prefix)}


def to_np(t):
    if isinstance(t, torch.Tensor):
        return t.detach().cpu().numpy()
    return np.asarray(t)


def assert_parity(actual, expected, what="", rtol=RTOL, scale_atol=RTOL):
    """fp32 parity: |a-e| <= rtol*|e| + scale_atol*max|e| elementwise, and normwise relative error
    <= rtol.  (A pure relative bound is meaningless for entries that cancel to ~0; the absolute
    term is tied to the tensor's own scale, not a free constant.)"""
    a = to_np(actual).astype(np.float64)
    e = to_np(expected).astype(np.float64)
    assert a.shape == e.shape, f"{what}: shape {a.shape} vs {e.shape}"
    if e.size == 0:
        return
    assert np.isfinite(a).all(), f"{what}: non-finite values"
    scale = np.abs(e).max()
    err = np.abs(a - e)
    bound = rtol * np.abs(e) + scale_atol * scale
    bad = err > bound
    nrm = np.linalg.norm(e.ravel())
    rel = np.linalg.norm((a - e).ravel()) / nrm if nrm > 0 else np.linalg.norm(a.ravel())
    assert not bad.any(), (f"{what}: {int(bad.sum())}/{e.size} entries outside tolerance, "
                           f"max err {err.max():.3e} (scale {scale:.3e}), normwise rel {rel:.3e}")
    assert rel <= max(rtol, 1e-12), f"{what}: normwise relative error {rel:.3e} > {rtol}"


def assert_bitexact(actual, expected, what=""):
    a, e = to_np(actual), to_np(expected)
    assert a.shape == e.shape, f"{what}: shape {a.shape} vs {e.shape}"
    assert a.dtype == e.dtype or a.dtype.kind == e.dtype.kind, f"{what}: dtype {a.dtype} vs {e.dtype}"
    if a.dtype.kind == "f":
        same = a.view(np.uint32 if a.dtype == np.float32 else np.uint64) == \
            e.astype(a.dtype).view(np.uint32 if a.dtype == np.float32 else np.uint64)
    else:
        same = a == e
    assert same.all(), f"{what}: {int((~same).sum())}/{a.size} entries differ bitwise"


def csr_numpy(csr):
    """the device buffers of an ops.Csr as host arrays: one attribute per ops.CSR_FIELDS entry, plus `bad`"""
    from types import SimpleNamespace
    from meta_gcn_b200 import ops
    torch.cuda.synchronize()
    b = SimpleNamespace(**{name: getattr(csr, name).cpu().numpy() for name in ops.CSR_FIELDS})
    b.bad = csr.bad.cpu().numpy()
    return b


def check_structure(b, o_rowptr, o_nbr, o_perm, hub_t):
    """Everything include/mgcn.h promises of a built structure `b` (csr_numpy), against the stable grouping
    o_rowptr / o_nbr / o_perm of the same list (oracle.port.csr_oracle): rows, entries and edge ids bit for bit,
    perm = -1 past the kept entries, the hub table and its segments, the work order, the task descriptors and nbr_w."""
    n = len(o_rowptr) - 1
    assert b.bad[0] == 0
    assert_bitexact(b.rowptr, o_rowptr, "rowptr")
    nnz = int(o_rowptr[-1])
    assert_bitexact(b.nbr[:nnz], o_nbr, "nbr")
    assert_bitexact(b.perm[:nnz], o_perm, "perm")
    assert (b.perm[nnz:] == -1).all()
    rowptr = o_rowptr.astype(np.int64)
    deg = np.diff(rowptr)
    # hubs and their segments: every hub once, segments contiguous, covering the row in order
    want_hubs = np.nonzero(deg > hub_t)[0]
    nh = int(b.hub_count[0])
    assert nh == len(want_hubs)
    hub_rows = b.hub_rows[:nh].astype(np.int64)
    assert np.sort(hub_rows).tolist() == want_hubs.tolist()
    nseg = -(-deg[hub_rows] // hub_t)
    total_segs = int(nseg.sum())
    q = np.arange(total_segs) - np.repeat(np.cumsum(nseg) - nseg, nseg)      # segment number inside its hub
    at = np.repeat(b.hub_seg0[:nh].astype(np.int64), nseg) + q
    assert (b.seg_row[at] == np.repeat(hub_rows, nseg)).all()
    assert (b.seg_beg[at] == np.repeat(rowptr[hub_rows], nseg) + q * hub_t).all()
    assert int(b.seg_count[0]) == total_segs
    # work order: a permutation of the rows, sorted by (row // 16384, min(len, 1023)), stable
    assert sorted(b.order.tolist()) == list(range(n))
    key = (b.order.astype(np.int64) >> 14) * 1024 + np.minimum(deg[b.order], 1023)
    assert (np.diff(key) >= 0).all()
    same = np.diff(key) == 0
    assert (np.diff(b.order)[same] > 0).all()
    # work descriptors {row, beg, end, partial_slot}: n + total_segs tasks sorted (stably, by task id)
    # by (window, length; segments behind the rows of their window); positions contiguous in nbr_w
    t = b.tasks.reshape(-1, 4).astype(np.int64)
    nt = n + total_segs
    tid_len = np.concatenate([np.minimum(deg, 1023), np.full(total_segs, 1024)]).astype(np.int64)
    tid_win = np.concatenate([np.arange(n) >> 14, b.seg_row[:total_segs] >> 14]).astype(np.int64)
    want = np.argsort(tid_win * 2048 + tid_len, kind="stable")
    row, beg, end, slot = t[:nt].T
    assert (beg == np.concatenate([[0], end[:-1]])).all()
    assert (end[-1] if nt else 0) == nnz
    is_row = want < n
    rid = want[is_row]
    hub = deg[rid] > hub_t
    assert (slot[is_row] == 0).all()
    assert (row[is_row][hub] == -1).all() and (end[is_row][hub] == beg[is_row][hub]).all()
    assert (row[is_row][~hub] == rid[~hub]).all()
    assert ((end - beg)[is_row][~hub] == deg[rid[~hub]]).all()
    qs = want[~is_row] - n
    s_row = row[~is_row]
    assert (slot[~is_row] == qs + 1).all() and (s_row == b.seg_row[qs]).all()
    sb = b.seg_beg[qs].astype(np.int64)
    se = np.minimum(sb + hub_t, rowptr[s_row + 1])
    assert ((end - beg)[~is_row] == se - sb).all()
    # the entries of task p are those of its row (or segment) in row order: nbr_w[beg + i] = nbr[first + i]
    first = np.zeros(nt, np.int64)
    first[is_row] = rowptr[rid]
    first[~is_row] = sb
    src = np.repeat(first - beg, end - beg) + np.arange(nnz)
    assert (b.nbr_w[:nnz] == o_nbr[src]).all()
    pad = t[nt:]
    assert (pad[:, 0] == -1).all() and (pad[:, 1] == nnz).all() and (pad[:, 2] == nnz).all()
