"""gather_bf16 mode of the hidden-32 stack against fp32 — an experiment that is NOT part of libmgcn.so: it runs on a
tree with scripts/experiments/bf16_gather.patch applied (the mode, its contract in include/mgcn.h and its tests),
after `python -m meta_gcn_b200.build`:

    git apply scripts/experiments/bf16_gather.patch
    python scripts/experiments/bench_bf16_gather.py [--reps 20] [--rounds 3] [--out profiles/bf16_gather_bench.log]

Writes one JSON object per measurement (and the card's name and power limit, read in the same run):
  step     C1 (one botnet graph) and C2 (bench.py's configs[1], 25 graphs): forward + mean cross entropy + backward,
           median of --reps single steps timed with CUDA events, eager and replayed from one captured CUDA graph; fp32
           and bf16 alternate for --rounds rounds, so the spread of the per-round medians of one mode is the run-to-run
           spread of the same call
  launch   C2: CUDA-event times of one forward-layer launch (mgcn_gcn_layer_fwd_tc_ex against _bf16, both its
           launches) and one transposed aggregation (mgcn_aggregate_prescaled against _bf16), median of 50, for the
           library as built (MGCN_GATHER_U_BF16 = 4) and for a variant compiled with MGCN_GATHER_U_BF16 = 8 into a
           temporary directory
  adam     C1: 50 Adam steps (lr 1e-3) from the same seed in both modes, the loss of every step (recorded, not judged)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

CFG = dict(in_channels=1, enc_sizes=[32] * 12, num_classes=2, residual_hop=1, final_type="proj", deg_norm="sm",
           aggr="add", bias=False, dropout=0.0)


def _batch(graphs):
    import torch
    from meta_gcn_b200.data import GraphBatch
    b = GraphBatch.from_data_list(graphs).to(torch.device("cuda"))
    return b, b.x[:, 0].reshape(-1, 1).contiguous(), b.x[:, 1].contiguous(), b.y.long()


def steps(name, graphs, reps, rounds):
    import torch
    from bench_dropout import median_ms
    from meta_gcn_b200 import functional as F
    from meta_gcn_b200.gcn_meta.models import GCNModel
    from meta_gcn_b200.graph import clear_structure_cache
    from meta_gcn_b200.graphed import GraphedCall
    clear_structure_cache()
    b, x0, deg, y = _batch(graphs)
    torch.manual_seed(0)
    model = GCNModel(**CFG).to("cuda").train()

    def step():
        model.zero_grad(set_to_none=True)
        loss = F.cross_entropy(model(x0, b.edge_index, deg_K=deg), y, "mean")
        loss.backward()
        return loss

    modes = {"fp32": torch.float32, "bf16": torch.bfloat16}
    graphed = {}
    for label, dt in modes.items():
        model.gather_dtype = dt
        graphed[label] = GraphedCall(step)
    res = {k: {"eager": [], "graph": []} for k in modes}
    for _ in range(rounds):
        for label, dt in modes.items():
            model.gather_dtype = dt
            res[label]["eager"].append(median_ms(step, reps))
            res[label]["graph"].append(median_ms(graphed[label], reps))
    row = {"what": "step", "config": name, "graphs": len(graphs), "n": b.num_nodes, "e": b.num_edges,
           "reps": reps, "rounds": rounds}
    for label in modes:
        for kind in ("eager", "graph"):
            v = res[label][kind]
            row[f"{label}_{kind}_ms"] = statistics.median(v)
            row[f"{label}_{kind}_spread_ms"] = max(v) - min(v)
            row[f"{label}_{kind}_rounds_ms"] = v
    for kind in ("eager", "graph"):
        row[f"bf16_over_fp32_{kind}"] = row[f"bf16_{kind}_ms"] / row[f"fp32_{kind}_ms"]
    del graphed
    clear_structure_cache()
    return row


def launches(graphs, tag):
    """one forward layer and one transposed aggregation of layer 5's shape at C2, both modes"""
    import torch
    from bench_dropout import median_ms
    from meta_gcn_b200 import ops
    b, _, deg, _ = _batch(graphs)
    gs = b.structure()
    n = b.num_nodes
    g = torch.Generator(device="cuda").manual_seed(0)
    dis = ops.gcn_norm_impl(deg, 0)
    z = torch.randn(n, 32, device="cuda", generator=g) * dis.view(-1, 1)
    zb = z.to(torch.bfloat16)
    w, rw = (torch.randn(32, 32, device="cuda", generator=g) / 32 ** 0.5 for _ in range(2))
    rb = torch.randn(32, device="cuda", generator=g)
    gsd = torch.randn(n, 32, device="cuda", generator=g)
    gsb = gsd.to(torch.bfloat16)
    fwd, bwd = gs.fwd_plain, gs.bwd_plain
    cases = {
        "fwd_layer_fp32": lambda: ops.gcn_layer_fwd_tc_impl(fwd, z, w, rw, rb, None, dis, dis, dis, 1,
                                                            tmem_operands=False),
        "fwd_layer_bf16": lambda: ops.gcn_layer_fwd_tc_bf16_impl(fwd, z, zb, w, rw, rb, None, dis, dis, dis, 1),
        "transposed_agg_fp32": lambda: ops.aggregate_prescaled_impl(bwd, gsd, dis, 0, None, None, 0),
        "transposed_agg_bf16": lambda: ops.aggregate_prescaled_bf16_impl(bwd, gsb, dis),
    }
    row = {"what": "launch", "config": "C2", "n": n, "e": b.num_edges, "MGCN_GATHER_U_BF16": tag}
    for rnd in range(2):
        for k, fn in cases.items():
            row.setdefault(k + "_ms", []).append(median_ms(fn, 50))
    return row


def adam(graphs, n_steps=50):
    import torch
    from meta_gcn_b200 import functional as F
    from meta_gcn_b200.gcn_meta.models import GCNModel
    b, x0, deg, y = _batch(graphs)
    row = {"what": "adam", "config": "C1", "steps": n_steps, "lr": 1e-3}
    for label, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        torch.manual_seed(0)
        model = GCNModel(**CFG, gather_dtype=dt).to("cuda").train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        losses = []
        for _ in range(n_steps):
            opt.zero_grad(set_to_none=True)
            loss = F.cross_entropy(model(x0, b.edge_index, deg_K=deg), y, "mean")
            loss.backward()
            opt.step()
            losses.append(loss.item())
        row[f"{label}_loss"] = losses
    return row


def _variant_lib(tmp):
    """libmgcn.so with MGCN_GATHER_U_BF16 = 8, built into tmp"""
    from meta_gcn_b200 import build
    objs, procs = [], []
    for src in build.sources():
        obj = os.path.join(tmp, os.path.basename(src)[:-3] + ".o")
        cmd = [build._nvcc(), *build.NVCC_FLAGS, "-DMGCN_GATHER_U_BF16=8", "-I", os.path.join(ROOT, "include"),
               "-I", build.CSRC, "-c", src, "-o", obj]
        procs.append(subprocess.Popen(cmd))
        objs.append(obj)
    if any(p.wait() != 0 for p in procs):
        raise RuntimeError("variant build failed")
    lib = os.path.join(tmp, "libmgcn_u8.so")
    subprocess.run([build._nvcc(), "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-Xcompiler", "-fPIC", "-o", lib, *objs], check=True)
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bf16_gather_bench.log"))
    ap.add_argument("--launches-only", action="store_true", help=argparse.SUPPRESS)   # the U = 8 child process
    a = ap.parse_args()
    from meta_gcn_b200 import _lib
    if "mgcn_aggregate_prescaled_bf16" not in _lib.SIGNATURES:
        sys.exit("the gather_bf16 mode is not in this tree: git apply scripts/experiments/bf16_gather.patch, then build")
    import bench
    from meta_gcn_b200.data import synth_botnet_graph
    c2 = bench.make_graphs(list(range(25)), 143107, 1_500_000)    # configs[1] of bench.py, before CUDA starts
    if a.launches_only:
        print(json.dumps(launches(c2, os.environ.get("MGCN_GATHER_U_BF16_TAG", "?"))), flush=True)
        return
    import torch
    from bench_dropout import gpu_info
    torch.cuda.set_stream(torch.cuda.Stream(torch.device("cuda")))
    c1 = [synth_botnet_graph(seed=0)]
    rows = [dict(what="device", **gpu_info())]
    rows.append(steps("C1", c1, a.reps, a.rounds))
    rows.append(steps("C2", c2, a.reps, a.rounds))
    rows.append(launches(c2, "4"))
    with tempfile.TemporaryDirectory() as tmp:
        env = dict(os.environ, MGCN_LIB=_variant_lib(tmp), MGCN_GATHER_U_BF16_TAG="8")
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--launches-only"], env=env,
                             capture_output=True, text=True, check=True).stdout
        rows.append(json.loads(out.strip().splitlines()[-1]))
    rows.append(adam(c1))
    with open(a.out, "w") as fh:
        fh.write("# scripts/experiments/bench_bf16_gather.py with scripts/experiments/bf16_gather.patch applied; "
                 "step = forward + loss + backward, median ms (DESIGN §3.8)\n")
        for r in rows:
            fh.write(json.dumps(r) + "\n")
            print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
