"""Why the dropout parity cases of tests/test_gpu_dropout.py use the mask seeds they do.  A ReLU whose exact input lies
within rounding of zero has a derivative decided by the order of the fp32 sums: the stack and the fp32 oracle may land
on different sides, and that single element moves many gradients past 1e-5 of their norm (the same effect that picked
the seed of __graft_entry__.smoke(), scripts/relu_boundary_check.py).  Dropout at p = 0.5 doubles the kept entries and
draws new masks per seed, so each (case, mask seed) is a new input.  For each mask seed this prints the smallest
|pre-activation| of both ReLUs of every layer relative to its layer's scale (fp64 restatement with the same masks), and
the worst normwise error of the parameter gradients of the stack and of the fp32 oracle, each against the fp64 oracle.
    python scripts/dropout_boundary_check.py --case botnet --p 0.5 --mask-seeds 1,2,3      (needs a GPU)"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np
import torch

import test_gpu_dropout as T
from meta_gcn_b200 import fused
from meta_gcn_b200.gcn_meta.models import GCNModel
from oracle import port


def margins(cfg, sd, x_in, ei, deg, keep, p):
    """smallest |u| (inner ReLU, kept entries) and |y| (outer ReLU) over all layers, relative to the layer's max"""
    L, H = len(cfg["enc_sizes"]), cfg["enc_sizes"][0]
    masks = T.unpack(keep, H).double()
    scale = float(np.float32(1.0 / (1.0 - p)))
    n = x_in.shape[0]
    dis = deg.double().pow(-0.5 if cfg["deg_norm"] == "sm" else -1.0)
    dis[torch.isinf(dis)] = 0
    w_e = (dis[ei[0]] * dis[ei[1]] if cfg["deg_norm"] == "sm" else dis[ei[0]]).view(-1, 1)
    xc, worst = x_in.double(), (np.inf, np.inf)
    for l in range(L):
        xw = xc @ sd[f"gcn_net.{l}.gcn.node_models.0.weight_node"].double()
        u = torch.zeros(n, H, dtype=torch.float64).index_add_(0, ei[1], xw[ei[0]] * w_e)
        kept = masks[l] > 0
        mu = (u.abs()[kept].min() / u.abs().max()).item()
        yv = torch.relu(u) * masks[l] * scale + xc @ sd[f"residuals.{l}.weight"].double().t() + \
            sd[f"residuals.{l}.bias"].double()
        my = (yv.abs().min() / yv.abs().max()).item() if l < L - 1 else np.inf
        worst = (min(worst[0], mu), min(worst[1], my))
        xc = torch.relu(yv) if l < L - 1 else yv
    return worst


def grad_errors(cfg, sd, x_in, ei, deg, y, keep, p, mask_seed):
    H = cfg["enc_sizes"][0]
    dev = "cuda"
    fused.dropout_seed = lambda device: torch.tensor([mask_seed], dtype=torch.int64, device=device)
    model = GCNModel(**cfg)
    model.load_state_dict(sd)
    model.to(dev).train()
    torch.nn.CrossEntropyLoss()(model(x_in.to(dev), ei.to(dev), deg_K=deg.to(dev)), y.to(dev)).backward()
    refs = []
    for dt in (torch.float32, torch.float64):
        r = port.OracleGCNModel(**cfg)
        r.load_state_dict(sd)
        r = r.to(dt)
        r.dropout = T._MaskedDropout(keep, H, p)
        torch.nn.CrossEntropyLoss()(r(x_in.to(dt), ei, deg.to(dt)), y).backward()
        refs.append(r)
    worst = [0.0, 0.0]
    for (k, pm), (_, p32), (_, p64) in zip(model.named_parameters(), refs[0].named_parameters(),
                                          refs[1].named_parameters()):
        e = p64.grad.numpy()
        nrm = max(np.linalg.norm(e), 1e-300)
        worst[0] = max(worst[0], np.linalg.norm(pm.grad.cpu().double().numpy() - e) / nrm)
        worst[1] = max(worst[1], np.linalg.norm(p32.grad.double().numpy() - e) / nrm)
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", default="botnet", choices=sorted(T.CASES))
    ap.add_argument("--p", type=float, default=0.5)
    ap.add_argument("--mask-seeds", default=str(T.SEED))
    a = ap.parse_args()
    cfg, g, x_in = T.case_inputs(a.case, a.p)
    x = torch.from_numpy(g["x"])
    ei = torch.from_numpy(g["edge_index"])
    y = torch.from_numpy(g["y"]).long()
    deg = x[:, 1].contiguous()
    torch.manual_seed(0)
    sd = port.OracleGCNModel(**cfg).state_dict()
    L, H = len(cfg["enc_sizes"]), cfg["enc_sizes"][0]
    for s in (int(v, 0) for v in a.mask_seeds.split(",")):
        keep = T.keep_bits_ref(s, L, x.shape[0], (H + 31) // 32, a.p)
        mu, my = margins(cfg, sd, x_in, ei, deg, keep, a.p)
        ours, theirs = grad_errors(cfg, sd, x_in, ei, deg, y, keep, a.p, s)
        print(f"case {a.case} p {a.p} mask seed {s:#x}: min |u|/scale {mu:.1e}, min |y|/scale {my:.1e}; "
              f"worst gradient error vs fp64: stack {ours:.1e}, fp32 oracle {theirs:.1e}", flush=True)


if __name__ == "__main__":
    main()
