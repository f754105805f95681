"""Training step of the botnet model with dropout (gcn_model.py:42, the reference's default p = 0.5): the fused stack at
p = 0 and p = 0.5 against the per-layer composition at p = 0.5 (`_no_stack=True`: what any p > 0 ran before the stack
took dropout), on the configs[1] batch of bench.py (C2: 25 graphs) and on one graph (C1).

    python scripts/bench_dropout.py [--reps 20] [--only c1,c2]      one JSON object per configuration

Step = forward + mean cross entropy + backward (gradients dropped, not zeroed, as in scripts/bench_configs.py), median
over single steps timed with CUDA events, eager and replayed from one captured CUDA graph; k_dropout_keep_bits (the
masks of all 12 layers in one launch) timed alone the same way; libmgcn launches counted over one eager step."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CFG = dict(in_channels=1, enc_sizes=[32] * 12, num_classes=2, residual_hop=1, final_type="proj", deg_norm="sm",
           aggr="add", bias=False)
VARIANTS = (("stack_p0", 0.0, False), ("stack_p0.5", 0.5, False), ("per_layer_p0.5", 0.5, True))


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        lim, clk = (v.strip() for v in out.strip().split(","))
        info.update(power_limit_w=float(lim), sm_max_mhz=float(clk))
    except (OSError, ValueError, subprocess.TimeoutExpired):
        info.update(power_limit_w=None, sm_max_mhz=None)
    return info


def median_ms(fn, reps, warm=3):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for e0, e1 in evs:
        e0.record()
        fn()
        e1.record()
    torch.cuda.synchronize()
    return statistics.median(e0.elapsed_time(e1) for e0, e1 in evs)


def measure(name, graphs, reps):
    import torch
    from meta_gcn_b200 import _lib, functional as F, ops
    from meta_gcn_b200.data import GraphBatch
    from meta_gcn_b200.gcn_meta.models import GCNModel
    from meta_gcn_b200.graph import clear_structure_cache
    from meta_gcn_b200.graphed import GraphedCall
    dev = torch.device("cuda")
    clear_structure_cache()
    b = GraphBatch.from_data_list(graphs).to(dev)
    x0, deg, y = b.x[:, 0].reshape(-1, 1).contiguous(), b.x[:, 1].contiguous(), b.y.long()
    b.structure().fwd_plain
    row = {"config": name, "graphs": len(graphs), "n": b.num_nodes, "e": b.num_edges, **gpu_info()}
    for label, p, per_layer in VARIANTS:
        torch.manual_seed(0)
        model = GCNModel(**CFG, dropout=p).to(dev).train()
        kw = {"_no_stack": True} if per_layer else {}

        def step():
            model.zero_grad(set_to_none=True)
            loss = F.cross_entropy(model(x0, b.edge_index, deg_K=deg, **kw), y, "mean")
            loss.backward()
            return loss

        ms_eager = median_ms(step, reps)
        c0 = _lib.launch_count()
        step()
        torch.cuda.synchronize()
        launches = _lib.launch_count() - c0
        try:
            graphed = GraphedCall(step)
            ms_graph = median_ms(graphed, reps)
            del graphed
        except Exception as exc:      # report a refused capture instead of a number
            ms_graph = f"capture failed: {exc!r}"
        row[label] = {"ms_eager": ms_eager, "ms_cuda_graph": ms_graph, "libmgcn_launches": launches}
        del model
        torch.cuda.empty_cache()
    seed = torch.zeros(1, dtype=torch.int64, device=dev)
    row["k_dropout_keep_bits_ms"] = median_ms(
        lambda: ops.dropout_keep_bits_impl(seed, 12, b.num_nodes, 1, 0.5), max(reps, 20))
    row["keep_words"] = 12 * b.num_nodes
    p0, p5 = row["stack_p0"]["ms_cuda_graph"], row["stack_p0.5"]["ms_cuda_graph"]
    if isinstance(p0, float) and isinstance(p5, float):
        row["stack_p0.5_over_p0_graphed"] = p5 / p0
    clear_structure_cache()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--only", default="c1,c2")
    a = ap.parse_args()
    import bench
    from meta_gcn_b200.data import synth_botnet_graph
    want = a.only.split(",")
    # configs[1] as bench.py builds it (seeds 0..24, generated before CUDA is initialised)
    c2 = bench.make_graphs(list(range(25)), 143107, 1_500_000) if "c2" in want else None
    import torch
    torch.cuda.set_stream(torch.cuda.Stream(torch.device("cuda")))
    if "c1" in want:
        print(json.dumps(measure("C1", [synth_botnet_graph(seed=0)], a.reps)), flush=True)
    if c2 is not None:
        print(json.dumps(measure("C2", c2, max(5, a.reps // 2))), flush=True)


if __name__ == "__main__":
    main()
