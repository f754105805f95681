"""Training step of the botnet model with edge gates (edge_gate='proj', EdgeGateProj) on every layer: on the hidden-32
tcgen05 stack, against the same model without gates on that stack and against the gated model on the per-layer path
(forced here with the model's private _no_stack switch), at p = 0 and p = 0.5, on the configs[1] batch of bench.py
(C2: 25 graphs) and on one graph (C1).  All three with the node-model bias (the default).

    python scripts/bench_gate.py [--reps 20] [--rounds 5] [--only c1,c2]      one JSON object per (config, p)
    python scripts/bench_gate.py --kernels                                  per-launch kernel times at C2

Step = forward + mean cross entropy + backward (gradients dropped, not zeroed), timed with CUDA events, eager and
replayed from one captured CUDA graph.  The three variants are built once and then timed in alternation, `rounds` times:
each round gives one median over `reps` steps per variant; the line reports the median of the rounds and their spread
(min, max).  libmgcn launches are counted over one eager step."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p_ in (ROOT, os.path.join(ROOT, "scripts")):
    if p_ not in sys.path:
        sys.path.insert(0, p_)

from bench_dropout import gpu_info, median_ms  # noqa: E402

CFG = dict(in_channels=1, enc_sizes=[32] * 12, num_classes=2, residual_hop=1, final_type="proj", deg_norm="sm",
           aggr="add")
VARIANTS = (("ungated_tc_stack", None, True), ("gated_tc_stack", "proj", True), ("gated_per_layer", "proj", False))


def measure(name, graphs, p, reps, rounds):
    import torch
    from meta_gcn_b200 import _lib, fused, functional as F
    from meta_gcn_b200.data import GraphBatch
    from meta_gcn_b200.gcn_meta.models import GCNModel
    from meta_gcn_b200.graph import clear_structure_cache
    from meta_gcn_b200.graphed import GraphedCall
    dev = torch.device("cuda")
    clear_structure_cache()
    b = GraphBatch.from_data_list(graphs).to(dev)
    x0, deg, y = b.x[:, 0].reshape(-1, 1).contiguous(), b.x[:, 1].contiguous(), b.y.long()
    b.structure().fwd_plain
    row = {"config": name, "p": p, "graphs": len(graphs), "n": b.num_nodes, "e": b.num_edges, **gpu_info(),
           "reps": reps, "rounds": rounds}
    runs = {}
    for label, gate, tc in VARIANTS:
        torch.manual_seed(0)
        model = GCNModel(**CFG, bias=True, edge_gate=gate, dropout=p).to(dev).train()
        with torch.no_grad():           # non-zero biases, as after the first optimiser step
            for k, prm in model.named_parameters():
                if k.startswith("gcn_net.") and k.endswith(".bias"):
                    prm.normal_(0.0, 0.1)
        taken = []
        real = fused.residual_gcn_stack

        def step(model=model, taken=taken, real=real, tc=tc):
            def spy(*a, **k):
                out = real(*a, **k)
                taken.append(out is not None)
                return out
            fused.residual_gcn_stack = spy
            try:
                model.zero_grad(set_to_none=True)
                loss = F.cross_entropy(model(x0, b.edge_index, deg_K=deg, _no_stack=not tc), y, "mean")
                loss.backward()
            finally:
                fused.residual_gcn_stack = real
            return loss

        step()
        torch.cuda.synchronize()
        assert any(taken) == tc, f"{label}: the tcgen05 stack was {'not ' if tc else ''}taken"
        c0 = _lib.launch_count()
        step()
        torch.cuda.synchronize()
        row[label] = {"libmgcn_launches": _lib.launch_count() - c0, "ms_eager_rounds": [], "ms_cuda_graph_rounds": []}
        try:
            graphed = GraphedCall(step)
        except RuntimeError as err:   # a path that synchronises with the host cannot be captured
            graphed, row[label]["cuda_graph_error"] = None, str(err)[:200]
        runs[label] = (step, graphed)
    for _ in range(rounds):
        for label, _, _ in VARIANTS:
            step, graphed = runs[label]
            if graphed is not None:
                row[label]["ms_cuda_graph_rounds"].append(median_ms(graphed, reps))
            row[label]["ms_eager_rounds"].append(median_ms(step, reps))
    for label, _, _ in VARIANTS:
        r = row[label]
        for kind in ("ms_cuda_graph", "ms_eager"):
            v = r[kind + "_rounds"]
            if v:
                r[kind] = statistics.median(v)
                r[kind + "_spread"] = [min(v), max(v)]
    for kind in ("ms_cuda_graph", "ms_eager"):
        base = row["ungated_tc_stack"][kind]
        row["gated_tc_over_ungated_" + kind] = row["gated_tc_stack"][kind] / base
        if kind in row["gated_per_layer"]:
            row["gated_per_layer_over_gated_tc_" + kind] = row["gated_per_layer"][kind] / row["gated_tc_stack"][kind]
    del runs
    torch.cuda.empty_cache()
    clear_structure_cache()
    return row


def kernel_times(name, graphs, steps):
    """per-launch CUDA time of every kernel of an eager step, ungated and gated stack (torch.profiler, a run of its own:
    tracing slows the host, so the step times above are taken without it)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from meta_gcn_b200 import functional as F
    from meta_gcn_b200.data import GraphBatch
    from meta_gcn_b200.gcn_meta.models import GCNModel
    from meta_gcn_b200.graph import clear_structure_cache
    dev = torch.device("cuda")
    clear_structure_cache()
    b = GraphBatch.from_data_list(graphs).to(dev)
    x0, deg, y = b.x[:, 0].reshape(-1, 1).contiguous(), b.x[:, 1].contiguous(), b.y.long()
    row = {"config": name, "p": 0.0, "steps": steps, "unit": "ms per launch (count per step)", **gpu_info()}
    for label, gate in (("ungated_tc_stack", None), ("gated_tc_stack", "proj")):
        torch.manual_seed(0)
        model = GCNModel(**CFG, bias=True, edge_gate=gate, dropout=0.0).to(dev).train()

        def step():
            model.zero_grad(set_to_none=True)
            F.cross_entropy(model(x0, b.edge_index, deg_K=deg), y, "mean").backward()
        step()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                step()
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            if ev.device_type.name != "CUDA" or ev.count == 0:
                continue
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            if t <= 0:
                continue
            key = ev.key if len(ev.key) <= 90 else ev.key[:90]
            per[key] = [round(t / ev.count / 1000.0, 4), ev.count // steps]
        row[label] = dict(sorted(per.items(), key=lambda kv: -kv[1][0] * kv[1][1]))
    clear_structure_cache()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--only", default="c1,c2")
    ap.add_argument("--kernels", action="store_true", help="per-launch kernel times at C2 (profiler) instead")
    a = ap.parse_args()
    if a.kernels:
        import bench
        c2 = bench.make_graphs(list(range(25)), 143107, 1_500_000)
        print(json.dumps(kernel_times("C2", c2, 3)), flush=True)
        return
    import bench
    from meta_gcn_b200.data import synth_botnet_graph
    want = a.only.split(",")
    # configs[1] as bench.py builds it (seeds 0..24, generated before CUDA is initialised)
    c2 = bench.make_graphs(list(range(25)), 143107, 1_500_000) if "c2" in want else None
    import torch
    torch.cuda.set_stream(torch.cuda.Stream(torch.device("cuda")))
    for p in (0.0, 0.5):
        if "c1" in want:
            print(json.dumps(measure("C1", [synth_botnet_graph(seed=0)], p, a.reps, a.rounds)), flush=True)
        if c2 is not None:
            print(json.dumps(measure("C2", c2, p, max(5, a.reps // 2), a.rounds)), flush=True)


if __name__ == "__main__":
    main()
