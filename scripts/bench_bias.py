"""Training step of the botnet model with the node-model bias (bias=True, the default of GCNLayer / NodeModelAdditive)
on the hidden-32 tcgen05 stack, against the same model without bias on that stack and against bias=True on the generic
stack (fused._ResidualGCNStack, forced here for the comparison only by turning fused.FORWARD_AGGREGATE_FIRST off), at
p = 0 and p = 0.5, on the configs[1] batch of bench.py (C2: 25 graphs) and on one graph (C1).

    python scripts/bench_bias.py [--reps 20] [--rounds 5] [--only c1,c2]      one JSON object per (config, p)

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
VARIANTS = (("nobias_tc_stack", False, True), ("bias_tc_stack", True, True), ("bias_generic_stack", True, False))


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
    for label, bias, tc in VARIANTS:
        torch.manual_seed(0)
        model = GCNModel(**CFG, bias=bias, dropout=p).to(dev).train()
        if bias:
            with torch.no_grad():           # non-zero biases, as after the first optimiser step
                for k, prm in model.named_parameters():
                    if k.startswith("gcn_net.") and k.endswith(".bias"):
                        prm.normal_(0.0, 0.1)
        taken = []
        real = fused._ResidualGCNStack32AT.apply

        def step(model=model, taken=taken, real=real, tc=tc):
            fused.FORWARD_AGGREGATE_FIRST = tc
            fused._ResidualGCNStack32AT.apply = lambda *a: taken.append(1) or real(*a)
            try:
                model.zero_grad(set_to_none=True)
                loss = F.cross_entropy(model(x0, b.edge_index, deg_K=deg), y, "mean")
                loss.backward()
            finally:
                fused.FORWARD_AGGREGATE_FIRST = True
                fused._ResidualGCNStack32AT.apply = real
            return loss

        step()
        torch.cuda.synchronize()
        assert bool(taken) == tc, f"{label}: the tcgen05 stack was {'not ' if tc else ''}taken"
        c0 = _lib.launch_count()
        step()
        torch.cuda.synchronize()
        row[label] = {"libmgcn_launches": _lib.launch_count() - c0, "ms_eager_rounds": [], "ms_cuda_graph_rounds": []}
        runs[label] = (step, GraphedCall(step))
    for _ in range(rounds):
        for label, _, _ in VARIANTS:
            step, graphed = runs[label]
            row[label]["ms_cuda_graph_rounds"].append(median_ms(graphed, reps))
            row[label]["ms_eager_rounds"].append(median_ms(step, reps))
    for label, _, _ in VARIANTS:
        r = row[label]
        for kind in ("ms_cuda_graph", "ms_eager"):
            v = r[kind + "_rounds"]
            r[kind] = statistics.median(v)
            r[kind + "_spread"] = [min(v), max(v)]
    for kind in ("ms_cuda_graph", "ms_eager"):
        base = row["nobias_tc_stack"][kind]
        row["bias_tc_over_nobias_" + kind] = row["bias_tc_stack"][kind] / base
        row["bias_generic_over_bias_tc_" + kind] = row["bias_generic_stack"][kind] / row["bias_tc_stack"][kind]
    del runs
    torch.cuda.empty_cache()
    clear_structure_cache()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--only", default="c1,c2")
    a = ap.parse_args()
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
