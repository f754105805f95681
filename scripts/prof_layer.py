"""Runs the three per-layer kernels of the botnet step alone at the C2 shape (for ncu / CUDA-event timing).
    python scripts/prof_layer.py [--graphs 25] [--reps 5]"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap = argparse.ArgumentParser()
ap.add_argument("--graphs", type=int, default=25)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--hub", type=int, default=64)
ap.add_argument("--only", default="")
args = ap.parse_args()

from bench import make_graphs, b_agg  # noqa: E402

graphs = make_graphs(list(range(args.graphs)), 143107, 1_500_000)
import torch  # noqa: E402
from meta_gcn_b200 import ops  # noqa: E402
from meta_gcn_b200.data import GraphBatch  # noqa: E402
from meta_gcn_b200.graph import GraphStructure  # noqa: E402

dev = torch.device("cuda")
b = GraphBatch.from_data_list(graphs).to(dev)
n, e = b.num_nodes, b.num_edges
H = 32
gs = GraphStructure(b.edge_index, n, hub_threshold=args.hub)
gs.fwd, gs.bwd
dis = ops.gcn_norm_impl(b.x[:, 1].contiguous(), 0)
m = torch.randn(n, H, device=dev)
x = torch.randn(n, H, device=dev)
gy = torch.randn(n, H, device=dev)
w = torch.randn(H, H, device=dev) / H ** 0.5
r = torch.randn(H, H, device=dev) / H ** 0.5
rb = torch.randn(H, device=dev)
bits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), device=dev, dtype=torch.int64).to(torch.int32)


def timeit(name, fn, byts):
    if args.only and not any(o in name for o in args.only.split("|")):
        return
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / args.reps
    print(f"{name:34s} {ms:8.3f} ms  {byts / ms / 1e6:8.1f} GB/s (bytes model {byts / 1e6:.0f} MB)")


nh = 4 * n * H
print(f"N={n} E={e} hubs={int(gs.fwd.hub_count)} segs={int(gs.fwd.seg_count)}")
timeit("layer_fwd (gather+2 products)", lambda: ops.gcn_layer_fwd_impl(gs.fwd, m, x, None, r, rb, w, None, dis, dis, 1),
       4 * e + 8 * n + 4 * nh)
if hasattr(ops, "gcn_layer_fwd_tc_impl"):
    timeit("layer_fwd_tc (aggregate-then-transform)",
           lambda: ops.gcn_layer_fwd_tc_impl(gs.fwd, x, w, r, rb, None, dis, dis, dis, 1), b_agg(n, e, H))
timeit("layer_fwd last (no next)", lambda: ops.gcn_layer_fwd_impl(gs.fwd, m, x, None, r, rb, None, None, dis, dis, 0),
       4 * e + 8 * n + 3 * nh)
x1 = torch.ones(n, 1, device=dev)
timeit("first layer: spmm H=1 (pre-scaled)", lambda: ops.spmm_impl(gs.fwd, x1, nbr_scale=dis), 4 * e + 16 * n)
timeit("first layer: spmm H=1 (plain, as the stack calls it)", lambda: ops.spmm_impl(gs.fwd, x1), 4 * e + 16 * n)
timeit("first layer: row-local fwd", lambda: ops.gcn_layer_fwd_impl(None, m, None, x, None, None, w, None, dis, None, 1), 4 * nh)
timeit("agg_plain bwd structure", lambda: ops.aggregate_prescaled_impl(gs.bwd, gy, dis, 0, None, None, 0),
       b_agg(n, e, H))
timeit("agg_plain fwd structure", lambda: ops.aggregate_prescaled_impl(gs.fwd, gy, dis, 0, None, None, 1),
       b_agg(n, e, H))
timeit("layer_bwd (row-local, tcgen05)", lambda: ops.gcn_layer_bwd_impl(m, gy, x, w, r, bits, dis, True), 5 * nh + 8 * n)
timeit("mask_bits_scale", lambda: ops.mask_bits_scale_impl(gy, bits, dis), 2 * nh + 8 * n)
timeit("torch copy", lambda: m.copy_(x), 2 * nh)
# the step's first and last stages (H_in = 1 first layer, output layer + loss)
hw = torch.randn(2, H, device=dev) / H ** 0.5
hb = torch.zeros(2, device=dev)
tgt = torch.randint(0, 2, (n,), device=dev)
timeit("head fwd (Linear 32->2 + CE)", lambda: ops.head_cross_entropy_fwd_impl(x, hw, hb, tgt, False), nh + 16 * n)
logits_ = ops.head_cross_entropy_fwd_impl(x, hw, hb, tgt, False)[0]
one = torch.ones(1, device=dev)
timeit("head bwd", lambda: ops.head_cross_entropy_bwd_impl(x, logits_, hw, tgt, False, one), 2 * nh + 16 * n)
s1 = torch.randn(n, 1, device=dev)
w0 = torch.randn(1, H, device=dev)
r0 = torch.randn(H, 1, device=dev)
timeit("first layer fwd (narrow input)", lambda: ops.gcn_first_layer_fwd_impl(s1, x1, w0, r0, rb, None, None, dis, 1, out_scale=dis),
       nh + 20 * n)
timeit("wgrad narrow (x0^T gy)", lambda: ops.linear_wgrad_impl(x1, gy, True, True), nh + 4 * n)
