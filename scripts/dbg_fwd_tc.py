"""Diagnostic cases for mgcn_gcn_layer_fwd_tc (csrc/gcn_fwd_tc.cu): isolates the operand-image / descriptor
conventions from the gather and the epilogue.  python scripts/dbg_fwd_tc.py"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from meta_gcn_b200 import ops
from meta_gcn_b200.graph import GraphStructure

dev = "cuda"
H = 32
torch.manual_seed(0)


def run(name, n, ei, x, w, r, rb, post=None, sigma=None, outs=None, act=0):
    gs = GraphStructure(ei.to(dev), n, hub_threshold=64)
    d = lambda t: None if t is None else t.to(dev)
    zn, hm = ops.gcn_layer_fwd_tc_impl(gs.fwd, d(x), d(w), d(r), d(rb), None, d(sigma), d(post), d(outs), act)
    torch.cuda.synchronize()
    D = lambda t: t.double()
    agg = torch.zeros(n, H, dtype=torch.float64).index_add_(0, ei[1], D(x)[ei[0]])
    if post is not None:
        agg = agg * D(post).view(-1, 1)
    h = torch.relu(agg @ D(w))
    xin = D(x) / D(sigma).view(-1, 1) if sigma is not None else D(x)
    y = h + xin @ D(r).t() + D(rb)
    if act:
        y = torch.relu(y)
    if outs is not None:
        y = y * D(outs).view(-1, 1)
    got = zn.cpu().double()
    err = (got - y).abs()
    rel = err.max().item() / max(y.abs().max().item(), 1e-30)
    print(f"{name:44s} n={n:7d} E={ei.size(1):8d}  max err {err.max().item():.3e}  rel {rel:.3e}  nan {int(torch.isnan(got).sum())}")
    if rel > 1e-5:
        bad = (err > 1e-4 * y.abs().max()).nonzero()
        print("   first bad entries (row, col):", bad[:8].tolist())
        rows = sorted(set(bad[:, 0].tolist()))[:4]
        for rr in rows:
            print("   row", rr, "got", got[rr, :8].tolist(), "ref", y[rr, :8].tolist())
    return rel


eye = torch.eye(H)
zero = torch.zeros(H, H)
zb = torch.zeros(H)
for n in (128, 200, 1000, 200000):
    x = torch.randn(n, H)
    noe = torch.zeros(2, 0, dtype=torch.int64)
    run("no edges, R = I  (row-local product only)", n, noe, x, zero, eye, zb)
    run("no edges, R random", n, noe, x, zero, torch.randn(H, H) / 6, torch.randn(H))
    loops = torch.arange(n).repeat(2, 1)
    run("self loops, W = I, R = 0 (gather -> s image)", n, loops, x.abs(), eye, zero, zb)
    run("self loops, W random, R = 0", n, loops, x, torch.randn(H, H) / 6, zero, zb)
    g = np.random.default_rng(n)
    ei = torch.from_numpy(np.stack([g.integers(0, n, 8 * n), g.integers(0, n, 8 * n)]).astype(np.int64))
    run("random graph, W = I, R = 0", n, ei, x.abs(), eye, zero, zb)
    run("random graph, full layer", n, ei, x, torch.randn(H, H) / 6, torch.randn(H, H) / 6, torch.randn(H),
        post=torch.rand(n) + 0.1, sigma=torch.rand(n) + 0.1, outs=torch.rand(n) + 0.1, act=1)
