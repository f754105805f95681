"""Parity at the shapes bench.py runs (BASELINE.json configs 0/1/3), not only at golden-vector sizes:

  (i)   the full C1 graph (143 107 nodes / 1.5 M edge entries, hubs of degree ~10^4): 12-layer residual GCN
        forward + loss + backward against the fp32 oracle port, fp64 oracle as arbiter (train_botnet.py:286-293);
  (ii)  a C2-shaped batch of full-size graphs: batched == per-graph results bit for bit, and the step bench.py times
        (CUDA-graph replay + FlatGradientReducer + fused Adam) == the eager step after 3 updates;
  (iii) kernel/graph_sage.py at hidden 256 on a 50k-node power-law graph: the model-level path through the tcgen05
        wide transform / weight gradient against the oracle net;
  (iv)  2 ranks over NCCL (skipped with fewer than 2 GPUs): graph-sharded gradients == single-GPU batched gradients
        (mean over ALL nodes of the global batch, train_botnet.py:225,287).
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import meta_gcn_b200.kernel as K
from meta_gcn_b200 import data as D
from meta_gcn_b200 import dist as mdist
from meta_gcn_b200 import functional as F_mgcn
from meta_gcn_b200.gcn_meta.models import GCNModel
from oracle import port
from oracle.kernel_nets import OracleGraphNet
from util import assert_bitexact, assert_parity

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BOTNET = dict(in_channels=1, enc_sizes=[32] * 12, num_classes=2, residual_hop=1, dropout=0.0,
              final_type="proj", deg_norm="sm", aggr="add", bias=False)


def assert_parity_arbitrated(actual, ref32, ref64, what, rtol=1e-5):
    """rtol 1e-5 against the fp32 reference result; where an entry misses it, the fp64 result arbitrates: the CUDA
    value must be within twice the fp32 reference's own WORST distance from fp64 on this tensor (sums of 10^4..10^5
    terms in another order: the fp32 reference itself sits at ~1e-5 of the tensor's scale there) — and the normwise
    error against fp64 stays within max(rtol, twice the fp32 reference's)."""
    a = actual.detach().cpu().double().numpy()
    e32 = ref32.detach().double().numpy()
    e64 = ref64.detach().double().numpy()
    assert np.isfinite(a).all(), what
    scale = np.abs(e64).max()
    bound = rtol * np.abs(e32) + rtol * scale
    miss = np.abs(a - e32) > bound
    if miss.any():
        ours, theirs = np.abs(a - e64)[miss], np.abs(e32 - e64)
        worse = ours > np.maximum(2.0 * theirs.max(), bound[miss])
        assert not worse.any(), (f"{what}: {int(worse.sum())} entries outside rtol {rtol} of the fp32 reference and "
                                 f"farther from fp64 than it (max {ours.max():.3e} vs {theirs.max():.3e})")
    nrm = max(np.linalg.norm(e64.ravel()), 1e-300)
    rel = np.linalg.norm((a - e64).ravel()) / nrm
    rel32 = np.linalg.norm((e32 - e64).ravel()) / nrm
    assert rel <= max(rtol, 2.0 * rel32), f"{what}: normwise error vs fp64 {rel:.3e} (fp32 reference {rel32:.3e})"
    return rel, rel32


def test_c1_full_graph_12_layers_vs_oracle():
    g = D.synth_botnet_graph(seed=0)
    x = torch.from_numpy(g["x"])
    ei = torch.from_numpy(g["edge_index"])
    y = torch.from_numpy(g["y"]).long()
    assert x.shape[0] == 143107 and abs(ei.shape[1] - 1_500_000) < 15_000
    torch.manual_seed(0)
    ref = port.OracleGCNModel(**BOTNET)
    crit = torch.nn.CrossEntropyLoss()
    out_r = ref(x[:, 0:1], ei, x[:, 1])
    loss_r = crit(out_r, y)
    loss_r.backward()
    ref64 = port.OracleGCNModel(**BOTNET)
    ref64.load_state_dict(ref.state_dict())
    ref64 = ref64.double()
    out64 = ref64(x[:, 0:1].double(), ei, x[:, 1].double())
    loss64 = crit(out64, y)
    loss64.backward()

    model = GCNModel(**BOTNET)
    model.load_state_dict(ref.state_dict())
    model.to(DEV)
    xd = x.to(DEV)
    out = model(xd[:, 0].view(-1, 1), ei.to(DEV), deg_K=xd[:, 1])       # train_botnet.py:286
    loss = crit(out, y.to(DEV))
    loss.backward()
    worst = assert_parity_arbitrated(out, out_r, out64, "C1 logits")
    assert abs(loss.item() - loss_r.item()) <= 1e-5 * max(1.0, abs(loss_r.item())), (loss.item(), loss_r.item())
    for (k, p), (_, pr), (_, p64) in zip(model.named_parameters(), ref.named_parameters(), ref64.named_parameters()):
        r = assert_parity_arbitrated(p.grad, pr.grad, p64.grad, "C1 grad." + k)
        worst = max(worst, r)
    print(f"C1 worst normwise error vs fp64 (ours, fp32 oracle): {worst}")


def _bench_like_step(model, batch, reducer, opt, graphed=None):
    def fwd_loss_bwd():
        reducer.zero()
        out = model(batch.x[:, 0].view(-1, 1), batch.edge_index, deg_K=batch.x[:, 1])
        loss_sum = F_mgcn.cross_entropy(out, batch.y.long(), "sum")
        loss_sum.backward()
        return loss_sum
    return fwd_loss_bwd


def test_c2_batch_equals_per_graph_and_graphed_adam_step_equals_eager():
    graphs = [D.synth_botnet_graph(seed=s) for s in (0, 7, 24)]
    batch = D.GraphBatch.from_data_list(graphs).to(DEV)
    batch.x = batch.x.contiguous()
    torch.manual_seed(3)
    model = GCNModel(**BOTNET).to(DEV)
    with torch.no_grad():
        whole = model(batch.x[:, 0].view(-1, 1), batch.edge_index, deg_K=batch.x[:, 1])
        for i, gph in enumerate(graphs):
            one = D.GraphBatch.from_data_list([gph]).to(DEV)
            part = model(one.x[:, 0].view(-1, 1), one.edge_index, deg_K=one.x[:, 1])
            assert_bitexact(whole[batch.slices_x[i]:batch.slices_x[i + 1]], part, f"graph {i} of the batch")
    # the step bench.py times: graph replay of fwd + loss + bwd, flat-buffer reduce, fused Adam — against eager;
    # everything under one non-default stream, as bench.py runs it (see GraphedCall)
    from meta_gcn_b200.graphed import GraphedCall
    state0 = {k: v.clone() for k, v in model.state_dict().items()}
    results = []
    work = torch.cuda.Stream()
    work.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(work):
        for use_graph in (False, True):
            model.load_state_dict(state0)
            reducer = mdist.FlatGradientReducer(model.parameters())
            opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=5e-4, fused=True)
            fn = _bench_like_step(model, batch, reducer, opt)
            call = GraphedCall(fn, warmup=1) if use_graph else fn
            if use_graph:                       # the warm-up call of the capture must not count as an update
                model.load_state_dict(state0)
            losses = []
            for _ in range(3):
                loss_sum = call()
                mean_loss, _ = reducer.reduce_mean(loss_sum, batch.num_nodes)
                opt.step()
                losses.append(float(mean_loss))
            results.append((losses, [p.detach().clone() for p in model.parameters()]))
    torch.cuda.current_stream().wait_stream(work)
    assert results[0][0] == results[1][0], (results[0][0], results[1][0])
    for pe, pg in zip(results[0][1], results[1][1]):
        assert torch.equal(pe, pg)
    assert results[0][0][2] < results[0][0][0]          # three Adam updates lowered the loss


def test_sage_hidden_256_model_level_vs_oracle():
    """kernel/graph_sage.py:7-33 at hidden 256 (the C4 width, 47 classes) on a 50k-node power-law graph: crosses
    k_linear_wide / k_wgrad_wide (tcgen05) from the model API; log-probabilities and every gradient"""
    n, e, f_in, classes = 50_000, 600_000, 100, 47
    ei = torch.from_numpy(D.synth_powerlaw_graph(5, n, e, alpha=0.8))
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(n, f_in, generator=gen)
    batch = torch.zeros(n, dtype=torch.int64)
    y = torch.randint(0, classes, (1,), generator=gen)
    torch.manual_seed(2)
    ref = OracleGraphNet("sage", f_in, classes, 3, 256, dropout=False)

    class Data:
        pass
    dr = Data()
    dr.x, dr.edge_index, dr.batch = x, ei, batch
    out_r = ref(dr)
    loss_r = torch.nn.functional.nll_loss(out_r, y)
    loss_r.backward()
    ref64 = OracleGraphNet("sage", f_in, classes, 3, 256, dropout=False)
    ref64.load_state_dict(ref.state_dict())
    ref64 = ref64.double()
    d64 = Data()
    d64.x, d64.edge_index, d64.batch = x.double(), ei, batch
    out64 = ref64(d64)
    loss64 = torch.nn.functional.nll_loss(out64, y)
    loss64.backward()

    class DatasetStub:
        num_features, num_classes = f_in, classes
    model = K.GraphSAGE(DatasetStub(), 3, 256)
    model.load_state_dict(ref.state_dict())
    model.to(DEV).eval()            # eval: dropout off (oracle built without it); BatchNorm-free net
    dd = Data()
    dd.x, dd.edge_index, dd.batch = x.to(DEV), ei.to(DEV), batch.to(DEV)
    out = model(dd)
    loss = torch.nn.functional.nll_loss(out, y.to(DEV))
    loss.backward()
    assert_parity_arbitrated(out, out_r, out64, "SAGE-256 log-probabilities")
    for (k, p), (_, pr), (_, p64) in zip(model.named_parameters(), ref.named_parameters(), ref64.named_parameters()):
        assert_parity_arbitrated(p.grad, pr.grad, p64.grad, "SAGE-256 grad." + k)


_TWO_RANK = r"""
import os, sys
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
from meta_gcn_b200 import data as D, dist as mdist, functional as F
from meta_gcn_b200.gcn_meta.models import GCNModel
rank, local, world = mdist.init_from_env("nccl")
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
cfg = {cfg!r}
graphs = [D.synth_botnet_graph(seed=s, num_nodes=20000 + 1000 * s, edge_entries=200000, evil=1500) for s in range(5)]
torch.manual_seed(0)
model = GCNModel(**cfg).to(dev)
def grads_of(items):
    b = D.GraphBatch.from_data_list(items).to(dev)
    red = mdist.FlatGradientReducer(model.parameters())
    red.zero()
    out = model(b.x[:, 0].contiguous().view(-1, 1), b.edge_index, deg_K=b.x[:, 1].contiguous())
    loss_sum = F.cross_entropy(out, b.y.long(), "sum")
    loss_sum.backward()
    return red, loss_sum, b.num_nodes
parts = mdist.shard_by_weight([g["edge_index"].shape[1] for g in graphs], world)
red, ls, cnt = grads_of([graphs[i] for i in parts[rank]])
mean_loss, total = red.reduce_mean(ls, cnt)
sharded = red.grads.clone()
single, ls1, cnt1 = grads_of(graphs)
m1, t1 = single.flat[single.numel] , None
single.flat[:single.numel].div_(float(cnt1))
ref = single.grads
err = ((sharded - ref).double().norm() / ref.double().norm()).item()
lerr = abs(float(mean_loss) - float(ls1) / cnt1)
if rank == 0:
    print("RESULT", err, lerr, int(total.item()), cnt1)
assert int(total.item()) == cnt1
assert err < 1e-5 and lerr < 1e-5, (err, lerr)
dist.barrier()
dist.destroy_process_group()
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_sharded_gradients_equal_single_gpu(tmp_path):
    script = tmp_path / "two_rank.py"
    script.write_text(_TWO_RANK.format(root=ROOT, cfg=BOTNET))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert "RESULT" in res.stdout
