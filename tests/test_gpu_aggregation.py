"""The generic sum aggregation — mgcn_spmm (csrc/spmm.cu) and mgcn_aggregate_prescaled (csrc/agg_pipelined.cu, with
k_agg_flat / k_agg_flat_hub_finish of csrc/gcn_layer.cu at H = 32) — bit for bit against a restatement of the contract
of include/mgcn.h that uses no libmgcn structure.

restate_aggregate groups the entries with a stable torch.sort of the row endpoint, forms w = nbr_scale * edge_val *
row_scale (each product rounded to fp32, left to right), sums msg = x * w in row order from 0 (hub rows: per segment of
hub_threshold entries), combines the segment sums of a hub in the order the kernel documents and applies the epilogue
in kernel order (post scale, / max(len, 1), + bias, + residual, ReLU).  It is vectorised by position inside a segment,
so the same code runs on the CPU at small sizes and on the GPU at the configs[4] sweep shapes; elementwise fp32 torch
ops round once and never contract, so both give the same bits.

Which k_spmm instantiation (LPR = lanes per row, VEC4 = float4 columns) each width of the matrix reaches:
    H    16-byte aligned x         x at a 4-byte offset (scalar loads)
    1    LPR 1                     LPR 1
    2    LPR 2                     LPR 2
    3    LPR 4                     LPR 4
    4    LPR 1  VEC4               LPR 4
    5    LPR 8                     LPR 8
    8    LPR 2  VEC4               LPR 8
    12   LPR 4  VEC4               LPR 16
    16   LPR 4  VEC4               LPR 16
    17   LPR 32                    LPR 32
    32   LPR 8  VEC4               LPR 32
    33   LPR 32 (2 column passes)  same
    48   LPR 16 VEC4               LPR 32 (2 passes)
    64   LPR 16 VEC4               LPR 32 (2 passes)
    100  LPR 32 VEC4               LPR 32 (4 passes)
    128  LPR 32 VEC4               LPR 32 (4 passes)
    132  LPR 32 VEC4 (2 passes)    LPR 32 (5 passes)
    256  LPR 32 VEC4 (2 passes)    LPR 32 (8 passes)
    512  LPR 32 VEC4 (4 passes)    LPR 32 (16 passes)
each with kExact (any per-entry factor) and kPlain (none), and with the segment pass + k_spmm_hub_combine when the
graph has hub rows.
"""
import time

import numpy as np
import pytest
import torch

from meta_gcn_b200 import data as D
from meta_gcn_b200 import functional as F_mgcn
from meta_gcn_b200 import ops
from meta_gcn_b200.graph import GraphStructure, clear_structure_cache
from oracle import port
from util import assert_bitexact, assert_parity, check_structure, csr_numpy

DEV = "cuda"
gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------------------------
# the restatement
# ------------------------------------------------------------------------------------------------------------------
class Grouping:
    """Entries of an edge list grouped by one endpoint with a stable sort (each row keeps edge_index order), with the
    loop handling of mgcn_csr_build: loop_mode 1 drops self loops, 2 drops them and appends one loop per node at the
    END of the list (perm = E + i)."""

    def __init__(self, edge_index, n, by=1, loop_mode=0, device=None):
        ei = edge_index.to(device) if device is not None else edge_index
        dev = ei.device
        E = ei.size(1)
        src, dst = ei[0].long(), ei[1].long()
        pos = torch.arange(E, device=dev)
        if loop_mode in (1, 2):
            keep = src != dst
            src, dst, pos = src[keep], dst[keep], pos[keep]
        if loop_mode == 2:
            loop = torch.arange(n, device=dev)
            src, dst, pos = torch.cat([src, loop]), torch.cat([dst, loop]), torch.cat([pos, E + loop])
        key, other = (dst, src) if by == 1 else (src, dst)
        order = torch.sort(key, stable=True).indices
        self.n, self.E = n, E
        self.rows, self.nbr, self.perm = key[order], other[order], pos[order]
        self.cnt = torch.bincount(key, minlength=n)
        self.rowptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        self.rowptr[1:] = torch.cumsum(self.cnt, 0)


def _positional_sum(src_rows, beg, length, weight=None, idx=None):
    """sum_{p < length[r]} src[idx[beg[r] + p]] (* weight[beg[r] + p]) for every r, one rounded add per entry in
    position order, starting from +0 — vectorised by position: the r are sorted by length, so the rows still
    active at position p are a prefix"""
    R = beg.numel()
    acc = torch.zeros(R, src_rows.size(1), dtype=torch.float32, device=src_rows.device)
    if R == 0:
        return acc
    order = torch.sort(length, descending=True, stable=True).indices
    b, ln = beg[order], length[order]
    maxlen = int(ln[0].item())
    if maxlen > 0:
        hist = torch.bincount(ln, minlength=maxlen + 1).cpu().numpy()
        active = R - np.cumsum(hist)[:maxlen]           # active[p] = number of r with length > p
        for p in range(maxlen):
            c = int(active[p])
            e = b[:c] + p
            v = src_rows[idx[e]] if idx is not None else src_rows[e]
            if weight is not None:
                v = v * weight[e].unsqueeze(1)
            acc[:c].add_(v)
    out = torch.empty_like(acc)
    out[order] = acc
    return out


def _run_lengths(ns, combine):
    if combine == "ltr":
        return torch.ones_like(ns)
    if combine == "runs8":
        return (ns + 7) // 8
    assert combine == "runs"
    return torch.where(ns <= 32, (ns + 7) // 8, (ns + 63) // 64)


def restate_aggregate(edge_index, n, x, *, by=1, loop_mode=0, loop_value=1.0, gather_perm=False, edge_weight=None,
                      nbr_scale=None, row_scale=None, post_scale=None, reduce=0, bias=None, residual=None, act=0,
                      hub_threshold=64, combine="ltr", grouping=None, col_block=None):
    """out [n, H] of the aggregation contract of include/mgcn.h, on x's device.

    combine: how the segment sums p_0 .. p_{ns-1} of a hub row are added —
      "ltr"   ((p_0 + p_1) + p_2) + ...                        k_spmm_hub_combine, k_agg_hub_combine
      "runs"  runs of per = ceil(ns/8) (ns <= 32) or ceil(ns/64) (ns > 32) segments, each run summed from 0 left to
              right, the run sums then added left to right       k_agg_flat_hub_finish, k_hub_reduce
      "runs8" the same with per = ceil(ns/8) for every ns         the tcgen05 layer kernels"""
    dev = x.device
    g = grouping if grouping is not None else Grouping(edge_index, n, by, loop_mode, dev)
    w = None
    if nbr_scale is not None:
        w = nbr_scale[g.nbr]
    if edge_weight is not None:
        ev = torch.full((g.perm.numel(),), float(loop_value), dtype=torch.float32, device=dev)
        real = g.perm < g.E
        ev[real] = edge_weight[g.perm[real]]
        w = ev if w is None else w * ev
    if row_scale is not None:
        rs = row_scale[g.rows]
        w = rs if w is None else w * rs
    gidx = g.perm if gather_perm else g.nbr
    t = int(hub_threshold)
    cnt = g.cnt
    hub = cnt > t
    nseg = torch.where(hub, (cnt + t - 1) // t, torch.ones_like(cnt))
    S = int(nseg.sum().item())
    seg_row = torch.repeat_interleave(torch.arange(n, device=dev), nseg)
    first = torch.cumsum(nseg, 0) - nseg
    q = torch.arange(S, device=dev) - first[seg_row]
    seg_beg = g.rowptr[seg_row] + q * t
    seg_len = torch.where(hub[seg_row], torch.clamp(cnt[seg_row] - q * t, max=t), cnt[seg_row])
    hub_ids = torch.nonzero(hub).flatten()
    ns = nseg[hub_ids]
    per = _run_lengths(ns, combine)
    nrun = (ns + per - 1) // per
    n_runs = int(nrun.sum().item())
    run_hub = torch.repeat_interleave(torch.arange(hub_ids.numel(), device=dev), nrun)
    run_first = torch.cumsum(nrun, 0) - nrun
    gq = torch.arange(n_runs, device=dev) - run_first[run_hub]
    run_beg = first[hub_ids][run_hub] + gq * per[run_hub]
    run_len = torch.minimum(per[run_hub], ns[run_hub] - gq * per[run_hub])
    H = x.size(1)
    out = torch.empty(n, H, dtype=torch.float32, device=dev)
    if col_block is None:
        col_block = max(1, min(H, (1 << 28) // max(S, 1)))
    for c0 in range(0, H, col_block):
        c1 = min(H, c0 + col_block)
        xc = x[:, c0:c1].contiguous()
        part = _positional_sum(xc, seg_beg, seg_len, w, gidx)
        res = part[first]                                   # rows within the threshold: their one segment
        if hub_ids.numel():
            runs = _positional_sum(part, run_beg, run_len)
            # run sums of each hub added left to right: vectorised by run number over the hubs sorted by run count
            ho = torch.sort(nrun, descending=True, stable=True).indices
            tot = runs[run_first[ho]].clone()
            nr = nrun[ho]
            hist = torch.bincount(nr).cpu().numpy()
            active = hub_ids.numel() - np.cumsum(hist)
            for gi in range(1, int(nr[0].item())):
                c = int(active[gi])
                tot[:c].add_(runs[run_first[ho[:c]] + gi])
            res[hub_ids[ho]] = tot
        if post_scale is not None:
            res = res * post_scale.unsqueeze(1)
        if reduce == 1:
            res = res / torch.clamp(cnt, min=1).to(torch.float32).unsqueeze(1)
        if bias is not None:
            res = res + bias[c0:c1]
        if residual is not None:
            res = res + residual[:, c0:c1]
        if act == 1:
            res = torch.where(res < 0, torch.zeros_like(res), res)
        out[:, c0:c1] = res
    return out


def assert_same_bits(actual, expected, what=""):
    """bitwise equality, compared on the device (the configs[4] outputs are gigabytes)"""
    assert actual.shape == expected.shape, f"{what}: shape {tuple(actual.shape)} vs {tuple(expected.shape)}"
    diff = actual.contiguous().view(torch.int32) != expected.contiguous().view(torch.int32)
    bad = int(diff.sum().item())
    if bad:
        rows = torch.nonzero(diff.any(1)).flatten()
        assert False, (f"{what}: {bad}/{actual.numel()} entries differ bitwise in {rows.numel()} rows "
                       f"(first rows {rows[:8].tolist()})")


def giants_per_cta(csr, sms, giant_segs=32):
    """The most giant hubs (more than giant_segs segments) one CTA of k_agg_flat_hub_finish / k_hub_reduce meets:
    CTA b owns the hub table slots k with (k mod 8W) // 8 == b, W = min(ceil(hub_cap / 8), 8 * sms)."""
    nh = min(int(csr.hub_count.item()), csr.hub_rows.numel())
    if nh == 0:
        return 0
    rows = csr.hub_rows[:nh].long()
    ns = (csr.rowptr[rows + 1] - csr.rowptr[rows] + csr.hub_threshold - 1) // csr.hub_threshold
    blocks = min(-(-csr.hub_rows.numel() // 8), 8 * sms)
    k = torch.nonzero(ns > giant_segs).flatten()
    if k.numel() == 0:
        return 0
    return int(torch.bincount((k % (8 * blocks)) // 8).max().item())


# ------------------------------------------------------------------------------------------------------------------
# the restatement itself
# ------------------------------------------------------------------------------------------------------------------
def planted_graph(seed, t, n=700):
    """~700 nodes: targets 0..9 receive 0, 1, t-1, t, t+1, 2t, 2t+1, 8t+1, 33t+1, 150t entries, sources 10..19 send
    as many, 30 self loops, 3000 random edges among the first n-50 nodes (the last 50 are isolated); shuffled"""
    rng = np.random.default_rng(seed)
    lengths = [0, 1, t - 1, t, t + 1, 2 * t, 2 * t + 1, 8 * t + 1, 33 * t + 1, 150 * t]
    live = n - 50
    parts = []
    for i, L in enumerate(lengths):
        parts.append(np.stack([rng.integers(0, live, L), np.full(L, i)]))
        parts.append(np.stack([np.full(L, 10 + i), rng.integers(0, live, L)]))
    loops = rng.integers(0, live, 30)
    parts.append(np.stack([loops, loops]))
    parts.append(rng.integers(20, live, size=(2, 3000)))
    ei = np.concatenate(parts, axis=1)
    return torch.from_numpy(ei[:, rng.permutation(ei.shape[1])].astype(np.int64))


def test_restatement_matches_fp64_index_add_on_cpu():
    """no GPU needed: the restatement (every combine order, with hubs, loops and all factors) within fp32 rounding of
    an fp64 index_add_ of the same messages"""
    t = 8
    ei = planted_graph(1, t, n=300)
    n = 300
    gen = torch.Generator().manual_seed(0)
    x = torch.randn(n, 5, generator=gen)
    ew = torch.rand(ei.size(1), generator=gen) + 0.5
    ns, rs = torch.rand(n, generator=gen) + 0.5, torch.rand(n, generator=gen) + 0.5
    bias, res = torch.randn(5, generator=gen), torch.randn(n, 5, generator=gen)
    for loop_mode in (0, 2):
        src, dst = ei[0], ei[1]
        w64 = ew.double()
        if loop_mode == 2:
            keep = src != dst
            src, dst, w64 = src[keep], dst[keep], w64[keep]
            src, dst = torch.cat([src, torch.arange(n)]), torch.cat([dst, torch.arange(n)])
            w64 = torch.cat([w64, torch.full((n,), 2.5, dtype=torch.float64)])
        w64 = ns.double()[src] * w64 * rs.double()[dst]
        ref = torch.zeros(n, 5, dtype=torch.float64).index_add_(0, dst, x.double()[src] * w64.unsqueeze(1))
        deg = torch.bincount(dst, minlength=n).clamp(min=1).double().unsqueeze(1)
        ref = torch.relu(ref / deg + bias.double() + res.double())
        for combine in ("ltr", "runs", "runs8"):
            got = restate_aggregate(ei, n, x, loop_mode=loop_mode, loop_value=2.5, edge_weight=ew, nbr_scale=ns,
                                    row_scale=rs, reduce=1, bias=bias, residual=res, act=1, hub_threshold=t,
                                    combine=combine)
            assert_parity(got, ref, f"restatement loop_mode={loop_mode} {combine}")
    # rows within the threshold: exactly the reference's CPU scatter_add (index_select -> mul -> scatter_add)
    plain = restate_aggregate(ei, n, x, hub_threshold=1 << 30)
    assert_bitexact(plain, port.scatter_rows("add", x[ei[0]], ei[1], n), "no hubs == scatter_add")
    # the combine orders really differ on hubs of more than 8 segments (so the tests below can tell them apart)
    a = restate_aggregate(ei, n, x, hub_threshold=t, combine="ltr")
    b = restate_aggregate(ei, n, x, hub_threshold=t, combine="runs")
    assert not torch.equal(a, b)


@gpu
def test_restatement_cpu_equals_cuda_bitwise():
    t = 16
    ei = planted_graph(2, t)
    n = 700
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(n, 33, generator=gen)
    ew = torch.rand(ei.size(1), generator=gen) + 0.5
    ns, rs, post = (torch.rand(n, generator=gen) + 0.5 for _ in range(3))
    bias, res = torch.randn(33, generator=gen), torch.randn(n, 33, generator=gen)
    for combine in ("ltr", "runs"):
        kw = dict(loop_mode=2, loop_value=2.5, edge_weight=ew, nbr_scale=ns, row_scale=rs, post_scale=post, reduce=1,
                  bias=bias, residual=res, act=1, hub_threshold=t, combine=combine)
        cpu = restate_aggregate(ei, n, x, **kw)
        cuda = restate_aggregate(ei.to(DEV), n, x.to(DEV), **{k: (v.to(DEV) if torch.is_tensor(v) else v)
                                                              for k, v in kw.items()})
        assert_bitexact(cuda, cpu, f"restatement CUDA == CPU ({combine})")


# ------------------------------------------------------------------------------------------------------------------
# mgcn_spmm: the specialisation matrix
# ------------------------------------------------------------------------------------------------------------------
SPMM_H = [1, 2, 3, 4, 5, 8, 12, 16, 17, 32, 33, 48, 64, 100, 128, 132, 256, 512]
HUB_T = [16, 64, 1 << 30]
MODES = ["none", "nbr_scale", "edge_val", "row_scale", "all"]


def _x_at(n, H, offset_floats, gen):
    """x [n, H] as a contiguous view starting offset_floats floats into its storage"""
    store = torch.randn(n * H + offset_floats, generator=gen).to(DEV)
    return store[offset_floats:].view(n, H)


@gpu
@pytest.mark.parametrize("hub_t", HUB_T)
@pytest.mark.parametrize("H", SPMM_H)
def test_spmm_specialisations_bitexact(H, hub_t):
    """every row of mgcn_spmm == the restatement bit for bit, over a pairwise cover of x layout x weight mode x reduce
    x epilogue x loop mode (loop_value 2.5); two runs identical"""
    hi, ti = SPMM_H.index(H), HUB_T.index(hub_t)
    t_plant = hub_t if hub_t < (1 << 30) else 16        # no hubs: rows up to 2400 entries, all summed by one group
    n = 700
    ei = planted_graph(100 + hi, t_plant, n).to(DEV)
    gen = torch.Generator().manual_seed(1000 * hi + ti)
    ew = (torch.rand(ei.size(1), generator=gen) + 0.5).to(DEV)
    nbr_s, row_s = ((torch.rand(n, generator=gen) + 0.5).to(DEV) for _ in range(2))
    bias, res = torch.randn(H, generator=gen).to(DEV), torch.randn(n, H, generator=gen).to(DEV)
    structs = {}
    for i, mode in enumerate(MODES):
        offset = (i + ti + hi) % 2                      # 0: aligned (VEC4 if H % 4 == 0), 1: 4-byte offset (scalar)
        reduce = (i + ti) % 2
        epi = (i // 2 + ti + hi) % 2
        loop_mode = (i + ti + hi) % 3
        if loop_mode not in structs:
            structs[loop_mode] = GraphStructure(ei, n, loop_mode, hub_threshold=hub_t)
        gs = structs[loop_mode]
        x = _x_at(n, H, offset, gen)
        assert (x.data_ptr() % 16 == 0) == (offset == 0)
        ns = nbr_s if mode in ("nbr_scale", "all") else None
        ew_m = ew if mode in ("edge_val", "all") else None
        rs = row_s if mode in ("row_scale", "all") else None
        ev = gs.edge_values(ew_m, 2.5)[0] if ew_m is not None else None
        kw = dict(reduce=reduce, bias=bias if epi else None, residual=res if epi else None, act=epi)
        what = f"H={H} t={hub_t} {mode} offset={offset} reduce={reduce} epi={epi} loops={loop_mode}"
        out = ops.spmm_impl(gs.fwd, x, False, ev, ns, rs, **kw)
        ref = restate_aggregate(ei, n, x, loop_mode=loop_mode, loop_value=2.5, edge_weight=ew_m, nbr_scale=ns,
                                row_scale=rs, hub_threshold=hub_t, combine="ltr", **kw)
        assert_same_bits(out, ref, what)
        assert_same_bits(ops.spmm_impl(gs.fwd, x, False, ev, ns, rs, **kw), out, what + " run 2")


@gpu
@pytest.mark.parametrize("reduce", ["add", "mean"])
@pytest.mark.parametrize("H", [1, 3, 4, 16, 32, 33, 128])
def test_scatter_rows_with_hub_index_bitexact(H, reduce):
    """scatter_(name, src, index) — the gather_perm path — with an index whose values repeat thousands of times (every
    one of them a hub row of the default threshold), plus rows of 0..64 entries and empty rows"""
    rng = np.random.default_rng(H)
    dim = 300
    idx = np.concatenate([np.full(5000, 7), np.full(3000, 42), rng.integers(0, 4, 6000), np.full(64, 100),
                          np.full(65, 101), rng.integers(150, 250, 2000)])
    idx = torch.from_numpy(idx[rng.permutation(idx.size)].astype(np.int64)).to(DEV)
    src = torch.randn(idx.numel(), H, device=DEV)
    out = F_mgcn.scatter_rows(src, idx, dim, reduce)
    ref = restate_aggregate(torch.stack([idx, idx]), dim, src, gather_perm=True, reduce=int(reduce == "mean"),
                            hub_threshold=ops.DEFAULT_HUB_THRESHOLD, combine="ltr")
    assert_same_bits(out, ref, f"scatter_{reduce} H={H}")
    assert_same_bits(F_mgcn.scatter_rows(src, idx, dim, reduce), out, "run 2")


@gpu
def test_spmm_empty_edge_list():
    n = 40
    for H in (3, 32):
        x = torch.randn(n, H, device=DEV)
        res, bias = torch.randn(n, H, device=DEV), torch.randn(H, device=DEV)
        ei = torch.zeros(2, 0, dtype=torch.long, device=DEV)
        ns = torch.rand(n, device=DEV) + 0.5
        for loop_mode in (0, 2):
            for nbr_scale in (None, ns):
                gs = GraphStructure(ei, n, loop_mode)
                out = ops.spmm_impl(gs.fwd, x, False, None, nbr_scale, None, 1, bias, res, 1)
                ref = restate_aggregate(ei, n, x, loop_mode=loop_mode, nbr_scale=nbr_scale, reduce=1, bias=bias,
                                        residual=res, act=1)
                assert_same_bits(out, ref, f"empty edge list H={H} loop_mode={loop_mode}")


# ------------------------------------------------------------------------------------------------------------------
# mgcn_aggregate_prescaled
# ------------------------------------------------------------------------------------------------------------------
EPILOGUES = {"none": (False, 0), "relu": (False, 1), "bias_res_relu": (True, 1)}


@gpu
@pytest.mark.parametrize("epi", sorted(EPILOGUES))
@pytest.mark.parametrize("reduce", [0, 1])
@pytest.mark.parametrize("post", [False, True])
@pytest.mark.parametrize("H", [16, 32, 64, 128])
def test_prescaled_bitexact_in_documented_order(H, post, reduce, epi):
    """k_agg_plain + k_agg_hub_combine (left to right) and, at H = 32 without mean / bias / residual on a 32-byte
    aligned x, k_agg_flat + k_agg_flat_hub_finish (8 / 64 runs); at H = 32 also x at a 16-byte offset, which takes
    k_agg_plain<8> whatever the epilogue"""
    n = 700
    with_br, act = EPILOGUES[epi]
    layouts = [0, 4] if H == 32 else [0]
    for t in (16, 64):
        ei = planted_graph(7 + t + H, t, n).to(DEV)
        gs = GraphStructure(ei, n, hub_threshold=t)
        gen = torch.Generator().manual_seed(H + t)
        ps = (torch.rand(n, generator=gen) + 0.5).to(DEV) if post else None
        bias = torch.randn(H, generator=gen).to(DEV) if with_br else None
        res = torch.randn(n, H, generator=gen).to(DEV) if with_br else None
        for off in layouts:
            x = _x_at(n, H, off, gen)
            flat = H == 32 and reduce == 0 and not with_br and x.data_ptr() % 32 == 0
            assert flat == (H == 32 and reduce == 0 and not with_br and off == 0)
            out = ops.aggregate_prescaled_impl(gs.fwd, x, ps, reduce, bias, res, act)
            ref = restate_aggregate(ei, n, x, post_scale=ps, reduce=reduce, bias=bias, residual=res, act=act,
                                    hub_threshold=t, combine="runs" if flat else "ltr")
            what = f"H={H} t={t} post={post} reduce={reduce} {epi} offset={4 * off}B ({'flat' if flat else 'plain'})"
            assert_same_bits(out, ref, what)
            assert_same_bits(ops.aggregate_prescaled_impl(gs.fwd, x, ps, reduce, bias, res, act), out, what + " run 2")


@gpu
def test_prescaled_argument_checks():
    n = 100
    ei = planted_graph(3, 16, n).to(DEV)
    gs = GraphStructure(ei, n, hub_threshold=16)
    x4 = _x_at(n, 32, 1, torch.Generator().manual_seed(0))
    with pytest.raises(RuntimeError, match=r"\(-4\)"):          # MGCN_ERR_ALIGN
        ops.aggregate_prescaled_impl(gs.fwd, x4)
    with pytest.raises(RuntimeError, match=r"\(-3\)"):          # MGCN_ERR_SHAPE
        ops.aggregate_prescaled_impl(gs.fwd, torch.randn(n, 48, device=DEV))


# ------------------------------------------------------------------------------------------------------------------
# autograd
# ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("reduce", ["add", "mean"])
@pytest.mark.parametrize("H", [1, 4, 17, 32, 64, 132])
def test_aggregate_autograd_dx_bitexact_and_edge_weight_grad(H, reduce):
    """dx of functional.aggregate is the aggregation over the by-source list with the factors swapped (and g / in_degree
    for the mean): bit-exact against the restatement; the edge-weight gradient against fp64"""
    n, t = 700, 16
    ei = planted_graph(50 + H, t, n).to(DEV)
    gs = GraphStructure(ei, n, hub_threshold=t)
    gen = torch.Generator().manual_seed(H)
    x = torch.randn(n, H, generator=gen).to(DEV).requires_grad_(True)
    ew = (torch.rand(ei.size(1), generator=gen) + 0.5).to(DEV).requires_grad_(True)
    ns, rs = ((torch.rand(n, generator=gen) + 0.5).to(DEV) for _ in range(2))
    up = torch.randn(n, H, generator=gen).to(DEV)
    out = F_mgcn.aggregate(x, gs, ns, rs, ew, reduce)
    out.backward(up)
    ref = restate_aggregate(ei, n, x.detach(), edge_weight=ew.detach(), nbr_scale=ns, row_scale=rs,
                            reduce=int(reduce == "mean"), hub_threshold=t)
    assert_same_bits(out.detach(), ref, f"forward H={H} {reduce}")
    gg = up
    if reduce == "mean":
        gg = up / torch.bincount(ei[1], minlength=n).clamp(min=1).to(torch.float32).unsqueeze(1)
    ref_dx = restate_aggregate(ei, n, gg, by=0, edge_weight=ew.detach(), nbr_scale=rs, row_scale=ns, hub_threshold=t)
    assert_same_bits(x.grad, ref_dx, f"dx H={H} {reduce}")
    src, dst = ei[0], ei[1]
    d64 = (ns.double()[src] * rs.double()[dst] * (gg.double()[dst] * x.detach().double()[src]).sum(1))
    assert_parity(ew.grad, d64, f"d edge_weight H={H} {reduce}")


# ------------------------------------------------------------------------------------------------------------------
# giant hubs: more than 32 of them in one CTA of k_agg_flat_hub_finish / k_hub_reduce
# ------------------------------------------------------------------------------------------------------------------
@gpu
def test_giant_hubs_beyond_one_list_get_the_64_run_order():
    """60 000 rows of 66 entries at hub_threshold 2 (33 segments each: 'giants'): the hub table has more than 32
    giants for every CTA of the hub kernels, whatever the order of the table.  Every giant is combined in 64 runs —
    k_agg_flat_hub_finish (mgcn_aggregate_prescaled, H = 32) and k_hub_reduce (mgcn_gcn_layer_fwd: its output equals
    the row-local mode of the same launch fed with the restated sums) — and the results do not depend on the order of
    the hub table"""
    t, G, L = 2, 60_000, 66
    n = G + 1000
    rng = np.random.default_rng(9)
    ei = np.concatenate([np.stack([rng.integers(0, n, G * L), np.repeat(np.arange(G), L)]),
                         np.stack([rng.integers(0, n, 1000), np.arange(G, n)])], axis=1)
    ei = torch.from_numpy(ei[:, rng.permutation(ei.shape[1])].astype(np.int64)).to(DEV)
    gs = GraphStructure(ei, n, hub_threshold=t)
    csr = gs.fwd
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    most = giants_per_cta(csr, sms)
    print(f"giants per CTA (most): {most} on {sms} SMs")
    assert most > 32
    gen = torch.Generator().manual_seed(3)
    m = torch.randn(n, 32, generator=gen).to(DEV)
    x = torch.randn(n, 32, generator=gen).to(DEV)
    res_w = (torch.randn(32, 32, generator=gen) / 6).to(DEV)
    res_b = torch.randn(32, generator=gen).to(DEV)
    post = (torch.rand(n, generator=gen) + 0.5).to(DEV)
    grouping = Grouping(ei, n, 1)
    want = restate_aggregate(ei, n, m, post_scale=post, act=1, hub_threshold=t, combine="runs", grouping=grouping)
    s = restate_aggregate(ei, n, m, hub_threshold=t, combine="runs", grouping=grouping)
    local = ops.gcn_layer_fwd_impl(None, s, x, None, res_w, res_b, None, None, None, None, 1)
    results = []
    for flip in (False, True):
        if flip:      # the same structure with its hub table in reverse order
            nh = int(csr.hub_count.item())
            csr.hub_rows[:nh] = csr.hub_rows[:nh].flip(0).clone()
            csr.hub_seg0[:nh] = csr.hub_seg0[:nh].flip(0).clone()
            assert giants_per_cta(csr, sms) > 32
        agg = ops.aggregate_prescaled_impl(csr, m, post, 0, None, None, 1)
        assert_same_bits(agg, want, f"k_agg_flat_hub_finish, hub table reversed={flip}")
        x_next, _, hmask = ops.gcn_layer_fwd_impl(csr, m, x, None, res_w, res_b, None, None, None, None, 1)
        assert_same_bits(x_next, local[0], f"k_hub_reduce (mgcn_gcn_layer_fwd), hub table reversed={flip}")
        assert torch.equal(hmask, local[2])
        results.append(x_next)
    assert_same_bits(results[1], results[0], "hub table order")


# ------------------------------------------------------------------------------------------------------------------
# configs[4] at its own shapes: N = 1 M, power-law sources, average degree 2..128
# ------------------------------------------------------------------------------------------------------------------
C4_N = 1_000_000
C4_DEG = [2, 8, 32, 128]


class C4:
    def __init__(self, d):
        t0 = time.perf_counter()
        self.d = d
        self.ei_h = torch.from_numpy(D.synth_powerlaw_graph(5, C4_N, C4_N * d))     # exactly as config4 builds it
        self.ei = self.ei_h.to(DEV)
        clear_structure_cache()
        self.gs = GraphStructure(self.ei, C4_N)
        self.gs.fwd
        self.gs.bwd
        self.norm = torch.rand(self.ei.size(1), generator=torch.Generator().manual_seed(d)).to(DEV)
        self.ev_fwd, self.ev_bwd = self.gs.edge_values(self.norm)
        self.grouping = {1: Grouping(self.ei, C4_N, 1), 0: Grouping(self.ei, C4_N, 0)}
        self.sms = torch.cuda.get_device_properties(0).multi_processor_count
        torch.cuda.synchronize()
        print(f"configs[4] graph d={d}: E={self.ei.size(1)}, built in {time.perf_counter() - t0:.1f} s; giants per CTA "
              f"(most) by target {giants_per_cta(self.gs.fwd, self.sms)}, by source {giants_per_cta(self.gs.bwd, self.sms)}")

    def csr(self, by):
        return self.gs.fwd if by == 1 else self.gs.bwd

    def x(self, H):
        return torch.randn(C4_N, H, generator=torch.Generator(device=DEV).manual_seed(H), device=DEV)


@pytest.fixture(scope="module", params=C4_DEG, ids=lambda d: f"deg{d}")
def c4(request):
    g = C4(request.param)
    yield g
    del g
    clear_structure_cache()
    torch.cuda.empty_cache()


@gpu
def test_c4_structures_equal_stable_sort_grouping(c4):
    for by in (1, 0):
        grp = c4.grouping[by]
        csr = c4.csr(by)
        nnz = grp.nbr.numel()
        assert torch.equal(csr.rowptr.long(), grp.rowptr), f"rowptr by={by}"
        assert torch.equal(csr.nbr[:nnz].long(), grp.nbr), f"nbr by={by}"
        assert torch.equal(csr.perm[:nnz].long(), grp.perm), f"perm by={by}"
        if c4.d <= 32:     # everything else include/mgcn.h promises (hub table, work order, tasks), on the host
            o_rowptr, o_nbr, o_perm = port.csr_oracle(c4.ei_h.numpy(), C4_N, by)
            check_structure(csr_numpy(csr), o_rowptr, o_nbr, o_perm, csr.hub_threshold)


@gpu
@pytest.mark.parametrize("weighted", [False, True], ids=["plain", "edge_val"])
@pytest.mark.parametrize("H", [16, 32, 64, 128, 256, 512])
def test_c4_spmm_forward_bitexact(c4, H, weighted):
    x = c4.x(H)
    ev = c4.ev_fwd if weighted else None
    out = ops.spmm_impl(c4.gs.fwd, x, False, ev)
    ref = restate_aggregate(c4.ei, C4_N, x, edge_weight=c4.norm if weighted else None, grouping=c4.grouping[1])
    assert_same_bits(out, ref, f"configs[4] d={c4.d} H={H} forward {'edge_val' if weighted else 'plain'}")
    del ref
    assert_same_bits(ops.spmm_impl(c4.gs.fwd, x, False, ev), out, "run 2")


@gpu
@pytest.mark.parametrize("weighted", [False, True], ids=["plain", "edge_val"])
@pytest.mark.parametrize("H", [32, 256])
def test_c4_spmm_transposed_bitexact(c4, H, weighted):
    """the by-source structure: power-law rows up to ~1.7 M entries (tens of thousands of segments)"""
    x = c4.x(H)
    ev = c4.ev_bwd if weighted else None
    out = ops.spmm_impl(c4.gs.bwd, x, False, ev)
    ref = restate_aggregate(c4.ei, C4_N, x, by=0, edge_weight=c4.norm if weighted else None, grouping=c4.grouping[0])
    assert_same_bits(out, ref, f"configs[4] d={c4.d} H={H} transposed {'edge_val' if weighted else 'plain'}")
    del ref
    assert_same_bits(ops.spmm_impl(c4.gs.bwd, x, False, ev), out, "run 2")


@gpu
@pytest.mark.parametrize("by", [1, 0], ids=["by_target", "by_source"])
@pytest.mark.parametrize("H", [16, 32, 64, 128])
def test_c4_prescaled_bitexact(c4, H, by):
    x = c4.x(H)
    assert x.data_ptr() % 32 == 0
    out = ops.aggregate_prescaled_impl(c4.csr(by), x)
    ref = restate_aggregate(c4.ei, C4_N, x, by=by, grouping=c4.grouping[by], combine="runs" if H == 32 else "ltr")
    assert_same_bits(out, ref, f"configs[4] d={c4.d} H={H} prescaled by={by}")
    del ref
    assert_same_bits(ops.aggregate_prescaled_impl(c4.csr(by), x), out, "run 2")


# ------------------------------------------------------------------------------------------------------------------
# configs[2] at its own shape: kernel/ nets, 3 layers, hidden 64, a batch of 128 TU-shaped graphs
# ------------------------------------------------------------------------------------------------------------------
def _no_dropout(fn):
    import torch.nn.functional as F
    real = F.dropout
    F.dropout = lambda x, p=0.5, training=True, inplace=False: x
    try:
        return fn()
    finally:
        F.dropout = real


class _Data:
    pass


def _arbitrated(actual, ref32, ref64, what, rtol=1e-5):
    """rtol against the fp32 oracle; where an entry misses it, the CUDA value must be no farther from fp64 than twice
    the fp32 oracle's worst distance, and the normwise error against fp64 within max(rtol, twice the oracle's)"""
    a = actual.detach().cpu().double().numpy()
    e32, e64 = ref32.detach().double().numpy(), ref64.detach().double().numpy()
    assert np.isfinite(a).all(), what
    bound = rtol * np.abs(e32) + rtol * np.abs(e64).max()
    miss = np.abs(a - e32) > bound
    if miss.any():
        ours, theirs = np.abs(a - e64)[miss], np.abs(e32 - e64)
        worse = ours > np.maximum(2.0 * theirs.max(), bound[miss])
        assert not worse.any(), f"{what}: {int(worse.sum())} entries farther from fp64 than the fp32 oracle"
    nrm = max(np.linalg.norm(e64.ravel()), 1e-300)
    rel = np.linalg.norm((a - e64).ravel()) / nrm
    rel32 = np.linalg.norm((e32 - e64).ravel()) / nrm
    assert rel <= max(rtol, 2.0 * rel32), f"{what}: normwise error vs fp64 {rel:.3e} (fp32 oracle {rel32:.3e})"


@gpu
@pytest.mark.parametrize("name,kind", [("GCN", "gcn"), ("GIN0", "gin0"), ("GIN", "gin"), ("GraphSAGE", "sage")])
def test_c2_tu_batch_vs_fp64_oracle(name, kind):
    import meta_gcn_b200.kernel as K
    from oracle.kernel_nets import OracleGraphNet
    host = D.synth_tu_batch(seed=0, num_graphs=128)
    tb = host.to(DEV)
    y = host.y.view(-1).long()
    torch.manual_seed(0)
    ref = OracleGraphNet(kind, 3, 2, 3, 64, dropout=False).train()
    d = _Data()
    d.x, d.edge_index, d.batch = host.x, host.edge_index, host.batch
    out_r = ref(d)
    torch.nn.functional.nll_loss(out_r, y).backward()
    ref64 = OracleGraphNet(kind, 3, 2, 3, 64, dropout=False)
    ref64.load_state_dict(ref.state_dict())
    ref64 = ref64.double().train()
    d64 = _Data()
    d64.x, d64.edge_index, d64.batch = host.x.double(), host.edge_index, host.batch
    out64 = ref64(d64)
    torch.nn.functional.nll_loss(out64, y).backward()
    net = getattr(K, name)(D.dataset_meta(3, 2), 3, 64)
    net.load_state_dict(ref.state_dict(), strict=True)
    net.to(DEV).train()

    def step():
        clear_structure_cache()          # as config2: a new mini-batch every step, structure build included
        net.zero_grad(set_to_none=True)
        out = net(tb)
        torch.nn.functional.nll_loss(out, y.to(DEV)).backward()
        return out
    out = _no_dropout(step)
    grads64 = dict(ref64.named_parameters())
    grads32 = dict(ref.named_parameters())
    if not kind.startswith("gin"):
        _arbitrated(out, out_r, out64, f"{name} log-probabilities")
        for k, p in net.named_parameters():
            _arbitrated(p.grad, grads32[k].grad, grads64[k].grad, f"{name} grad.{k}")
        return
    # GIN: BatchNorm1d batch statistics; the bar is "no farther from fp64 than the fp32 oracle's own run, or 1e-5"
    # (the rule of test_gpu_models.py::test_kernel_nets_match_reference_golden)
    assert_parity(out, out64, f"{name} log-probabilities vs fp64")
    for k, p in net.named_parameters():
        r64 = grads64[k].grad.numpy()
        nrm = max(np.linalg.norm(r64), 1e-30)
        ours = np.linalg.norm(p.grad.cpu().double().numpy() - r64) / nrm
        theirs = np.linalg.norm(grads32[k].grad.double().numpy() - r64) / nrm
        assert ours <= max(1e-5, 2.0 * theirs), f"{name}.grad.{k}: ours {ours:.2e} vs fp32 oracle {theirs:.2e}"
