"""bench.py — GCN fwd+bwd throughput on botnet-shaped graph batches (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = forward + cross-entropy + backward (+ gradient all-reduce for N>1) + Adam step of the
12-layer residual GCN (hidden 32) over one batch of `--graphs` synthetic botnet graphs per GPU
(143k nodes / 1.5M edge entries each).  Graphs are sharded by batch (weak scaling: every GPU owns
its own batch, gradients are summed and divided by the global node count).

Printed JSON (rank 0): metric = GCN fwd+bwd GEdges/s = sum_graphs(E) * L * 2 / t_step, whole job.
  value     device-resident inputs and structures, CUDA events, max over ranks
  e2e       through the public model API from pinned HOST buffers: H2D of x/edge_index/y, structure
            build, step, D2H of the loss, every step
  roofline  dominant kernel (row-owned aggregation, forward form) timed alone with CUDA events
  cpu_baseline / --impl reference: the oracle port of the reference's CPU path on the host cores
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

LAYERS = 12
HIDDEN = 32
# dram__bytes_read.sum + dram__bytes_write.sum per launch at the default workload, from the ncu --set full captures
# summarised under profiles/ (None until captured for the current kernel)
TRAFFIC = {
    "fwd": 1_238_066_944,    # profiles/r2_ncu_k_gcn_fwd_tc.csv: k_gcn_fwd_tc<0> 770.9 MB read + 448.1 MB written, <1> 19.0 MB
    "agg": 1_208_880_128,    # profiles/r1b_ncu_k_agg_flat.csv: 767.7 MB read + 441.1 MB written
    "bwd": 2_262_567_000,    # profiles/r1b_ncu_k_layer_bwd_tc.csv: 1402.5 MB read + 860.0 MB written
}
CFG = dict(in_channels=1, enc_sizes=[HIDDEN] * LAYERS, num_classes=2, non_linear="relu",
           non_linear_layer_wise="relu", residual_hop=1, dropout=0.0, final_type="proj",
           pred_on="node", nodemodel="additive", deg_norm="sm", edge_gate=None, aggr="add", bias=False)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--graphs", type=int, default=25, help="botnet graphs per GPU (configs[1]: 25)")
    ap.add_argument("--nodes", type=int, default=143107)
    ap.add_argument("--edges", type=int, default=1_500_000)
    ap.add_argument("--no-cuda-graph", action="store_true")
    ap.add_argument("--config", type=int, default=1, choices=[0, 1, 2, 3, 4],
                    help="BASELINE.json configs[k]; 1 (default) is the contract line, the others print one JSON line "
                         "with their own results and cpu_baseline (scripts/bench_configs.py)")
    ap.add_argument("--e2e-steps", type=int, default=20)   # the first copy of a loop cannot be overlapped
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--strong-graphs", default="24,25",
                    help="global batch sizes of the strong-scaling measurement (configs[1]: 25 graphs sharded over "
                         "the GPUs by edge count; 24 divides evenly); empty = skip")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of the device-resident measurement, write what its last step computed "
                         "(mean loss, logits, parameter gradients, updated parameters) as DIR/<name>.npy, rank 0's "
                         "shard, at most 64 MB (beyond that a fixed, seeded sample of the logits rows)")
    args = ap.parse_args()
    if args.dump_outputs and (args.config != 1 or args.impl != "ours"):
        ap.error("--dump-outputs needs --config 1 --impl ours")
    return args


def _gen(args):
    from meta_gcn_b200.data import synth_botnet_graph
    seed, nodes, edges = args
    return synth_botnet_graph(seed=seed, num_nodes=nodes, edge_entries=edges,
                              evil=min(10000, nodes // 14))


def make_graphs(seeds, nodes, edges):
    """seeded numpy generation, fanned out over host cores (before CUDA is initialised)"""
    import multiprocessing as mp
    jobs = [(s, nodes, edges) for s in seeds]
    workers = max(1, min(len(jobs), (os.cpu_count() or 2) // 2, 16))
    if workers == 1:
        return [_gen(j) for j in jobs]
    with mp.get_context("fork").Pool(workers) as pool:
        return pool.map(_gen, jobs)


def b_agg(n, e, h):
    """algorithmic bytes of one aggregation pass (SURVEY.md §8d)"""
    return 4 * e + 4 * (n + 1) + 4 * n + 8 * n * h


def b_step(n, e, h, layers):
    return layers * (2 * b_agg(n, e, h) + 4 * n * h)


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, loss, logits, model):
    """--dump-outputs: the step's mean loss, its logits, every parameter's gradient and the parameters after the
    optimiser step, each as out_dir/<name>.npy in float32.  The logits take what the others leave of DUMP_BYTES; a
    larger batch keeps a sample of rows drawn with a fixed seed (same rows for the same shape), listed in
    logits_rows.npy."""
    import numpy as np
    arrays = {"loss": loss}
    for name, p in model.named_parameters():
        arrays[f"grad.{name}"] = p.grad
        arrays[f"param.{name}"] = p
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    logits = logits.detach().float().cpu().numpy()
    header = 128        # bytes of an .npy header
    room = DUMP_BYTES - sum(a.nbytes + header for a in arrays.values()) - 2 * header
    if logits.nbytes > room:
        row_bytes = logits.itemsize * logits.shape[1]
        rows = np.random.default_rng(0).choice(logits.shape[0], room // (row_bytes + 8), replace=False)
        rows.sort()
        arrays["logits_rows"] = rows.astype(np.float64)
        logits = logits[rows]
    arrays["logits"] = logits
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(len(r) >= 7 and r[3 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's CPU path
# ------------------------------------------------------------------------------------------------
def cpu_step_time(graph, steps, warmup):
    import torch
    from oracle import port
    torch.manual_seed(0)
    model = port.OracleGCNModel(**{k: v for k, v in CFG.items() if k not in ("nodemodel", "edge_gate")})
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=5e-4)
    x = torch.from_numpy(graph["x"])
    ei = torch.from_numpy(graph["edge_index"])
    y = torch.from_numpy(graph["y"]).long()
    crit = torch.nn.CrossEntropyLoss()
    times = []
    state0 = {k: v.clone() for k, v in model.state_dict().items()}
    loss0 = None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad()
        out = model(x[:, 0].view(-1, 1), ei, x[:, 1])      # train_botnet.py:286
        loss = crit(out, y)
        if loss0 is None:
            loss0 = float(loss.detach())
        loss.backward()
        opt.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return times, float(loss.detach()), loss0, state0


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; /root/reference is pure Python over
    un-vendored torch_scatter/PyG and does not exist on the GPU box), all host threads, one graph of
    the workload per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    g = make_graphs([0], args.nodes, args.edges)[0]
    e = g["edge_index"].shape[1]
    times, loss, _, _ = cpu_step_time(g, args.steps, args.warmup)
    t = sum(times) / len(times)
    gedges = e * LAYERS * 2 / t / 1e9
    sample = (f"1 of the {args.graphs} graphs of a batch per step (N={g['x'].shape[0]}, E={e}), "
              f"fwd+loss+bwd+Adam, oracle port of src/gcn_meta on torch CPU fp32")
    line = {
        "impl": "reference", "metric": "GCN fwd+bwd GEdges/s", "value": gedges, "unit": "GEdges/s",
        "graphs_per_s": 1.0 / t, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args, args.gpus), graphs_in_step=1,
                       note="the CPU arm steps ONE of the batch's graphs per step (bounded sample) and is normalised "
                            "to edges/s; the GPU arm steps all graphs_per_gpu graphs"),
        "cpu_baseline": {"value": gedges, "unit": "GEdges/s", "cores": torch.get_num_threads(),
                         "kind": "port", "sample": sample},
        "e2e": {"value": gedges, "unit": "GEdges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(args, world):
    return {"workload": f"configs[1]: 12-layer residual GCN (hidden 32, sm norm, final proj) fwd+bwd on "
                        f"batches of {args.graphs} synthetic botnet graphs per GPU "
                        f"({args.nodes} nodes, ~{args.edges} edge entries each)",
            "graphs_per_gpu": args.graphs, "global_batch_graphs": args.graphs * world,
            "layers": LAYERS, "hidden": HIDDEN, "parallelism": f"graph-sharded dp{world}",
            "l2": "inputs larger than L2 (per-layer activations 458 MB vs 126 MB L2); no flush needed"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    seeds = [rank * args.graphs + i for i in range(args.graphs)]
    # strong scaling (configs[1] as written: ONE global batch of 25 graphs sharded over the GPUs; 24 divides evenly):
    # graph i of the global batch goes to rank i % world — the greedy balance by edge count (dist.shard_by_weight) of
    # graphs whose nominal sizes are equal
    strong_sizes = [int(v) for v in args.strong_graphs.split(",") if v.strip()]
    strong_seeds = sorted({i for g_ in strong_sizes for i in range(g_) if i % world == rank})
    all_seeds = sorted(set(seeds) | set(strong_seeds))
    by_seed = dict(zip(all_seeds, make_graphs(all_seeds, args.nodes, args.edges)))   # before CUDA init (fork-safe)
    graphs = [by_seed[s_] for s_ in seeds]

    import torch
    import torch.distributed as dist
    from meta_gcn_b200 import _lib, dist as mdist, ops
    from meta_gcn_b200 import functional as F_mgcn
    from meta_gcn_b200.data import GraphBatch
    from meta_gcn_b200.gcn_meta.models import GCNModel
    from meta_gcn_b200.graph import clear_structure_cache, structure_of

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # several ranks on one host: each keeps its pinned batch buffers on its GPU's NUMA node (first touch after binding)
    numa_node = mdist.bind_to_gpu_numa_node(local) if world > 1 else None
    mdist.init_from_env("nccl")
    # the whole run, eager warm-up included, on one non-default stream: autograd's AccumulateGrad nodes remember the
    # stream they were created on, and the CUDA-graph capture of the step must not touch the legacy default stream
    torch.cuda.set_stream(torch.cuda.Stream(dev))

    host = GraphBatch.from_data_list(graphs).pin_memory()
    n_nodes, n_edges = host.num_nodes, host.num_edges
    torch.manual_seed(0)
    model = GCNModel(**CFG).to(dev)
    reducer = mdist.FlatGradientReducer(model.parameters())
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=5e-4, fused=True)
    def crit_sum(out, target):   # nn.CrossEntropyLoss(reduction="sum") as deterministic kernels
        return F_mgcn.cross_entropy(out, target, "sum")

    # logits of the latest forward, for --dump-outputs (under a CUDA graph: its output buffer, rewritten by each replay)
    latest = {}

    # model.forward_loss = model(...) + CrossEntropyLoss(reduction="sum") (train_botnet.py:286-287) with the output
    # layer and the loss in one launch (csrc/head.cu); same values as the two separate calls (tests/test_gpu_head.py)
    def step(batch_dev):
        reducer.zero()
        loss_sum, latest["logits"] = model.forward_loss(batch_dev.x[:, 0].view(-1, 1), batch_dev.edge_index,
                                                        batch_dev.y.long(), deg_K=batch_dev.x[:, 1], reduction="sum")
        loss_sum.backward()
        mean_loss, _ = reducer.reduce_mean(loss_sum, batch_dev.num_nodes)
        opt.step()
        return mean_loss

    def fwd_loss_bwd(batch_dev):
        reducer.zero()
        loss_sum, latest["logits"] = model.forward_loss(batch_dev.x[:, 0].view(-1, 1), batch_dev.edge_index,
                                                        batch_dev.y.long(), deg_K=batch_dev.x[:, 1], reduction="sum")
        loss_sum.backward()
        return loss_sum

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def measure_resident(batch, steps, dump_dir=None):
        """structures built once outside the timed region; forward + loss + backward of the fixed-shape batch replayed
        as ONE CUDA graph (meta_gcn_b200/graphed.py), all-reduce and Adam eager; --no-cuda-graph times the eager
        step.  Returns (ms per step as max over ranks, libmgcn launches in the timed region, graphed?, last loss).
        With dump_dir, rank 0 writes what the last timed step computed there (dump_outputs)."""
        batch.structure()      # registers the batch boundaries with the structure cache (ordered batches: no sort)
        structure_of(batch.edge_index, batch.num_nodes).fwd_plain
        structure_of(batch.edge_index, batch.num_nodes).bwd_plain
        for _ in range(args.warmup):
            step(batch)
        use_graph = not args.no_cuda_graph
        graph_launches = 0
        resident_step = step
        if use_graph:
            from meta_gcn_b200.graphed import GraphedCall
            try:
                c0 = _lib.launch_count()
                graphed = GraphedCall(lambda: fwd_loss_bwd(batch), warmup=1)
                graph_launches = (_lib.launch_count() - c0) // 2      # one warm-up call + the captured call

                def resident_step(_b):
                    loss_sum = graphed()
                    mean_loss, _ = reducer.reduce_mean(loss_sum, batch.num_nodes)
                    opt.step()
                    return mean_loss
                for _ in range(2):
                    resident_step(batch)
            except Exception as exc:   # capture refused: report it and time the eager step instead
                print(f"[bench] CUDA-graph capture failed, timing the eager step: {exc!r}", file=sys.stderr)
                use_graph = False
                resident_step = step
                torch.cuda.synchronize()
        barrier()
        launches0 = _lib.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            loss = resident_step(batch)
        ev1.record()
        barrier()
        ms_ = max_over_ranks(ev0.elapsed_time(ev1)) / steps
        # kernels of libmgcn.so inside the timed region: host-side launches + those replayed from the graph
        n_launch = (_lib.launch_count() - launches0) + (graph_launches * steps if use_graph else 0)
        if dump_dir and rank == 0:
            dump_outputs(dump_dir, loss, latest["logits"], model)
        return ms_, n_launch, use_graph, float(loss.item())

    # ---- device-resident arm (weak scaling: every rank its own batch of --graphs graphs) ----
    batch = host.to(dev)
    batch.x = batch.x.contiguous()
    sampler = ClockSampler(local)
    batch.structure().fwd_plain
    if rank == 0:
        sampler.start()
    ms, launches, use_graph, final_loss = measure_resident(batch, args.steps, args.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None

    # ---- strong scaling: one GLOBAL batch of G graphs sharded over the ranks ----
    strong = []
    for g_total in strong_sizes:
        mine = [by_seed[i] for i in range(g_total) if i % world == rank]
        clear_structure_cache()
        sb = GraphBatch.from_data_list(mine).to(dev)
        sb.x = sb.x.contiguous()
        s_ms, _, s_graph, _ = measure_resident(sb, args.steps)
        e_mine = torch.tensor([float(sb.num_edges)], device=dev)
        if world > 1:
            dist.all_reduce(e_mine)
        strong.append({"global_batch_graphs": g_total, "graphs_on_rank0": len(mine), "ms_per_step": s_ms,
                       "graphs_per_s": g_total / (s_ms / 1e3),
                       "gedges_per_s": float(e_mine.item()) * LAYERS * 2 / (s_ms / 1e3) / 1e9, "cuda_graph": s_graph})
        del sb
    clear_structure_cache()

    # ---- dominant kernel alone: the fused forward layer (aggregation + dense tail) and the plain
    # aggregation of the backward, over this rank's batch, CUDA events on the launching stream ----
    gs = structure_of(batch.edge_index, n_nodes)
    dis = ops.gcn_norm_impl(batch.x[:, 1].contiguous(), 0)
    feat = torch.randn(n_nodes, HIDDEN, device=dev)
    xin = torch.randn(n_nodes, HIDDEN, device=dev)
    w_a = torch.randn(HIDDEN, HIDDEN, device=dev) / HIDDEN ** 0.5
    w_b = torch.randn(HIDDEN, HIDDEN, device=dev) / HIDDEN ** 0.5
    r_b = torch.zeros(HIDDEN, device=dev)

    def time_kernel(fn, reps=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(reps):
            fn()
        k1.record()
        torch.cuda.synchronize()
        return k0.elapsed_time(k1) / reps

    # the three per-layer launches of the hidden-32 stack (meta_gcn_b200/fused.py), each alone over this rank's batch
    fwd_ms = time_kernel(lambda: ops.gcn_layer_fwd_tc_impl(gs.fwd_plain, xin, w_a, w_b, r_b, None, dis, dis, dis, 1))
    agg_ms = time_kernel(lambda: ops.aggregate_prescaled_impl(gs.bwd_plain, feat, dis, 0, None, None, 0))
    hbits = torch.randint(-2 ** 31, 2 ** 31 - 1, (n_nodes,), device=dev, dtype=torch.int64).to(torch.int32)
    gyv = torch.randn(n_nodes, HIDDEN, device=dev)
    bwd_ms = time_kernel(lambda: ops.gcn_layer_bwd_impl(feat, gyv, xin, w_a, w_b, hbits, dis, True, True, x_scale=dis))
    del feat, xin, gyv, hbits

    # ---- end to end from pinned host buffers through the public API ----
    e2e_ms = None
    if args.e2e_steps > 0:
        # Every step: H2D of that step's x / edge_index / y from pinned host memory, structure build from
        # the raw int64 edge_index, forward + loss + backward (+ all-reduce) + Adam, D2H read of the loss.
        # The copy of step k+1 is issued on a second stream while step k computes (a prefetching loader,
        # src/gcn_meta/data/dataloader.py:6-30 has num_workers for the same purpose); all K copies lie
        # inside the timed region.
        # (meta_gcn_b200.data.DeviceLoader: two preallocated device slots per field, no allocation per step)
        import itertools
        from meta_gcn_b200.data import DeviceLoader

        from meta_gcn_b200.graph import all_positive
        from meta_gcn_b200.graphed import GraphedSlots

        def time_e2e(host_b):
            loader = DeviceLoader((), dev, fields=("x", "edge_index", "y"))
            # forward + loss + backward of a loader slot replayed as a CUDA graph: the slot's tensors and its (recycled)
            # structure buffers keep their addresses, so the graph captured the first time a slot is seen serves every
            # later batch of the same shape in it.  Per batch, eagerly: the structure build (order / symmetry test with
            # its host read, grouping kernels) and the check that decides the stack's code path.
            slots = GraphedSlots(fwd_loss_bwd, warmup=1)

            def e2e_step(b):
                gs = b.structure(recycle=True)
                gs.fwd_plain, gs.bwd_plain
                if args.no_cuda_graph:
                    return step(b)
                path = all_positive(b.x[:, 1])
                loss_sum = slots(b, extra_key=(path,))
                mean_loss, _ = reducer.reduce_mean(loss_sum, b.num_nodes)
                opt.step()
                return mean_loss

            def e2e_loop(k):
                out = []
                loader.batches = itertools.repeat(host_b, k)
                for b in loader:
                    out.append(float(e2e_step(b).item()))      # D2H read of the step's result
                return out

            e2e_loop(max(3, args.warmup))      # both loader slots, their structures and the allocator in steady state
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            e2e_loop(args.e2e_steps)
            e1.record()
            barrier()
            return max_over_ranks(e0.elapsed_time(e1)) / args.e2e_steps, loader.bytes_per_batch(host_b)

        # headline: edge_index held as int32 on the host (converted once, outside the timed region — a dataset-load
        # step; every structure entry point takes either dtype); also timed with the reference's int64 indices
        host32 = host.with_int32_indices().pin_memory()
        e2e_ms, e2e_h2d = time_e2e(host32)
        e2e64_ms, e2e64_h2d = time_e2e(host)
        del host32
        clear_structure_cache()

    if rank != 0:
        if world > 1:
            dist.barrier()
        return

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peaks = json.load(fh)
    except OSError:
        pass
    peak_bw = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"

    edges_global = n_edges * world     # every rank holds the same shape
    t = ms / 1e3
    gedges = edges_global * LAYERS * 2 / t / 1e9
    agg_bytes = b_agg(n_nodes, n_edges, HIDDEN)
    nh4 = 4 * n_nodes * HIDDEN
    step_bytes = b_step(n_nodes, n_edges, HIDDEN, LAYERS)

    def kernel_entry(name, alg_bytes, own_bytes, ms_, traffic):
        """SURVEY §8d: achieved = ALGORITHMIC bytes / time; kernel_bytes = the bytes this design's kernel has to move
        (its own operand arrays, each once); traffic = DRAM bytes ncu measured"""
        gbs = alg_bytes / (ms_ / 1e3) / 1e9
        return {"kernel": name, "algorithmic_bytes_per_launch": int(alg_bytes), "ms_per_launch": ms_,
                "achieved": gbs, "frac": gbs / peak_bw, "kernel_bytes": int(own_bytes),
                "traffic": traffic, "traffic_over_algorithmic": (traffic / alg_bytes) if traffic else None}

    k_fwd = kernel_entry("k_gcn_fwd_tc<0> + <1>: forward layer, aggregate-then-transform — row-owned gather of the "
                         "stored activations, both dense products on tcgen05 (TMEM accumulators), ReLUs / residual / "
                         "mask word in the epilogue, bulk row stores; one [N,32] array read, one written",
                         agg_bytes, agg_bytes + 28 * n_nodes, fwd_ms, TRAFFIC["fwd"])
    k_fwd["gather_l2_to_sm_gbs"] = n_edges * HIDDEN * 4 / (fwd_ms / 1e3) / 1e9
    k_agg = kernel_entry("k_agg_flat (+k_hub_reduce, k_agg_flat_hubs): transposed aggregation of the backward",
                         agg_bytes, agg_bytes + 16 * n_nodes, agg_ms, TRAFFIC["agg"])
    k_agg["gather_l2_to_sm_gbs"] = n_edges * HIDDEN * 4 / (agg_ms / 1e3) / 1e9
    k_bwd = kernel_entry("k_layer_bwd_tc: row-local backward (4 products, both ReLU masks) on tcgen05.mma / TMEM, "
                         "warp-specialised; §8d charges a layer's backward B_agg + 4NH in total, of which this launch "
                         "owns the 4NH re-read of the saved layer input",
                         nh4, 5 * nh4 + 8 * n_nodes, bwd_ms, TRAFFIC["bwd"])
    per_layer_ms = fwd_ms + agg_ms + bwd_ms
    line = {
        "metric": "GCN fwd+bwd GEdges/s", "value": gedges, "unit": "GEdges/s",
        "graphs_per_s": args.graphs * world / t,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": dict(workload_config(args, world), cuda_graph=bool(use_graph)),
        "loss": final_loss,
        "strong_scaling": {"scaling": "strong", "partition": "graph i of the global batch -> rank i % n_gpus",
                           "runs": strong},
        "clocks": clocks,
        "gpu_launches": int(launches),
        # dominant kernel = largest share of the step (the forward layer launch: 11 of them per step)
        "roofline": dict({"bound": "hbm", "peak": peak_bw, "unit": "GB/s", "peak_source": peak_src}, **k_fwd,
                         second_kernel=k_agg, third_kernel=k_bwd,
                         layer={"what": "one hidden layer forward + backward = the three launches above",
                                "ms": per_layer_ms,
                                "algorithmic_bytes": int(2 * agg_bytes + nh4),
                                "frac": (2 * agg_bytes + nh4) / (per_layer_ms / 1e3) / 1e9 / peak_bw,
                                "traffic": sum(TRAFFIC.values()),
                                "traffic_over_algorithmic": sum(TRAFFIC.values()) / (2 * agg_bytes + nh4)},
                         step_algorithmic_bytes=int(step_bytes),
                         step_frac=step_bytes / t / 1e9 / peak_bw,
                         step_frac_of_nominal_8TBs=step_bytes / t / 1e9 / 8000.0),
    }
    if e2e_ms is not None:
        line["e2e"] = {"value": edges_global * LAYERS * 2 / (e2e_ms / 1e3) / 1e9, "unit": "GEdges/s",
                       "graphs_per_s": args.graphs * world / (e2e_ms / 1e3), "ms_per_step": e2e_ms,
                       "h2d_bytes_per_step": int(e2e_h2d), "d2h_bytes_per_step": 4,
                       "index_dtype": "int32 on the host (converted once at dataset load)",
                       "numa_node_of_rank0": numa_node,
                       "int64_indices": {"value": edges_global * LAYERS * 2 / (e2e64_ms / 1e3) / 1e9,
                                         "graphs_per_s": args.graphs * world / (e2e64_ms / 1e3),
                                         "ms_per_step": e2e64_ms, "h2d_bytes_per_step": int(e2e64_h2d),
                                         "note": "the reference's edge_index dtype, copied as is"}}
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        times, _, cpu_loss0, state0 = cpu_step_time(graphs[0], args.cpu_steps, 1)
        tc = min(times)
        # same graph, same initial weights: the CUDA path's loss must equal the CPU arm's first loss
        chk = GCNModel(**CFG)
        chk.load_state_dict(state0)
        chk.to(dev)
        one = GraphBatch.from_data_list([graphs[0]]).to(dev)
        with torch.no_grad():
            o_ = chk(one.x[:, 0].contiguous().view(-1, 1), one.edge_index, deg_K=one.x[:, 1].contiguous())
            gpu_loss0 = float(F_mgcn.cross_entropy(o_, one.y.long(), "mean").item())
        if abs(gpu_loss0 - cpu_loss0) > 1e-5 * max(1.0, abs(cpu_loss0)):
            raise RuntimeError(f"loss mismatch between the CUDA path ({gpu_loss0}) and the CPU arm ({cpu_loss0})")
        line["loss_check"] = {"graph": 0, "gpu": gpu_loss0, "cpu": cpu_loss0, "abs_diff": abs(gpu_loss0 - cpu_loss0),
                              "tolerance": "1e-5 relative (asserted)"}
        e1g = graphs[0]["edge_index"].shape[1]
        line["cpu_baseline"] = {
            "value": e1g * LAYERS * 2 / tc / 1e9, "unit": "GEdges/s", "graphs_per_s": 1.0 / tc,
            "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"1 of the {args.graphs} graphs (N={graphs[0]['x'].shape[0]}, E={e1g}), best of "
                      f"{args.cpu_steps} steps after 1 warm-up, oracle port on torch CPU fp32"}
    emit(line)
    if world > 1:
        dist.barrier()


def run_secondary(args):
    """--config 0 / 2 / 3 / 4: the other BASELINE.json configurations, one GPU, with the reference's CPU path beside
    each (bounded samples; see scripts/bench_configs.py)"""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import bench_configs
    rows = bench_configs.CONFIGS[args.config](not args.no_cpu_baseline)
    emit({"metric": "see results", "config": {"workload": f"BASELINE.json configs[{args.config}]"}, "n_gpus": 1,
          "data": "synthetic", "dtype": "f32", "results": rows})


_JSON_OUT = None


def emit(line):
    """the ONE JSON line goes to the real stdout; everything else this process (or NCCL, which prints its
    version banner on fd 1 when NCCL_DEBUG is set) writes to fd 1 is diverted to stderr"""
    os.write(_JSON_OUT if _JSON_OUT is not None else 1, (json.dumps(line) + "\n").encode())


def main():
    global _JSON_OUT
    args = parse()
    sys.stdout.flush()
    _JSON_OUT = os.dup(1)
    os.dup2(2, 1)
    if args.config != 1:
        run_secondary(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
