"""The output layer and the cross entropy against fp64 on the CPU: the fused head (csrc/head.cu) at every template
instantiation and on both sides of its grid cap, the unfused output layer (csrc/dense_narrow.cu) and the loss kernels
(csrc/loss.cu) on both sides of theirs, confidently classified rows, labels outside [0, C), empty batches and the
bench step's batch.  Every output is also checked for run-to-run bit equality."""
import numpy as np
import pytest
import torch

from meta_gcn_b200 import functional as F
from meta_gcn_b200 import ops
from util import assert_bitexact, assert_parity

pytestmark = pytest.mark.gpu
DEV = "cuda"
UPSTREAM = 1.7


def assert_loss(actual, expected, what="loss"):
    """a scalar loss within 1e-5 of the fp64 value, relative, with no absolute floor"""
    a = float(actual)
    assert abs(a - expected) <= 1e-5 * abs(expected), f"{what}: {a!r} vs {expected!r}"


def ce64(z, y, reduction, upstream=UPSTREAM):
    """fp64 cross entropy of the logits z and its gradient d(upstream * loss) / dz"""
    z = torch.as_tensor(z).detach().cpu().double().requires_grad_(True)
    loss = torch.nn.functional.cross_entropy(z, y.cpu(), reduction=reduction)
    (loss * upstream).backward()
    return loss.item(), z.grad


def counters_np(logits, y):
    """{TP, FP, TN, FN, correct} over the first maximal class of each row, rows with a label outside [0, C) skipped"""
    z, y = logits.detach().cpu().numpy(), y.cpu().numpy()
    ok = (y >= 0) & (y < z.shape[1])
    p, y = z.argmax(1)[ok], y[ok]
    return np.array([((p == 1) & (y == 1)).sum(), ((p == 1) & (y == 0)).sum(), ((p == 0) & (y == 0)).sum(),
                     ((p == 0) & (y == 1)).sum(), (p == y).sum()], np.int64)


def head_linear(h, c, bias, gen):
    lin = torch.nn.Linear(h, c, bias=bias)
    with torch.no_grad():
        lin.weight.copy_(torch.randn(c, h, generator=gen) / h ** 0.5)
        if bias:
            lin.bias.copy_(torch.randn(c, generator=gen))
    return lin.to(DEV)


def run_head(x, lin, y, reduction, want_dx):
    """F.head_cross_entropy forward and backward with a device upstream gradient"""
    xd = x.to(DEV).requires_grad_(want_dx)
    lin.zero_grad(set_to_none=True)
    loss, logits, counts = F.head_cross_entropy(xd, lin, y, reduction, confusion=True)
    assert not logits.requires_grad and not counts.requires_grad     # the loss alone carries the gradient
    (loss * torch.tensor(UPSTREAM, device=DEV)).backward()
    return dict(loss=loss.detach(), logits=logits, counts=counts, dx=xd.grad, dw=lin.weight.grad,
                db=None if lin.bias is None else lin.bias.grad)


def assert_same_bits(a, b):
    for k in a:
        if a[k] is not None:
            assert_bitexact(b[k], a[k], f"{k} run-to-run")


def head_grads64(z, x, w, y, reduction, upstream=UPSTREAM):
    """fp64 loss, dlogits, dx, dw and db of the head over the given logits"""
    loss, dl = ce64(z, y, reduction, upstream)
    x64 = x.double()
    return loss, dl, dl @ w.detach().cpu().double(), dl.t() @ x64, dl.sum(0)


# ------------------------------------------------------------------------------------------------
# 1. the fused head: every <L, CM> instantiation, odd and even trip counts of the two-row loop, both sides of the
#    888-block cap (2048 rows a block below it), blocks without rows above it
# ------------------------------------------------------------------------------------------------
HC = [(h, c) for h in (16, 32, 64, 128) for c in (1, 2, 3, 8)] + [(32, c) for c in (4, 5, 6, 7)]
HEAD_CASES = []
for _i, (_h, _c) in enumerate(HC):
    for _j, _n in enumerate((1, 2, 33, 2049)):
        _k = _i + _j     # the options rotate so that every instantiation meets each of them
        HEAD_CASES.append((_n, _h, _c, ("mean", "sum")[_k % 2], _k % 3 != 1, _k % 4 != 2))
HEAD_CASES += [(1_818_624, 32, 2, "sum", True, True), (1_818_625, 32, 2, "mean", False, True),
               (1_818_625, 16, 3, "sum", True, False),
               (2_841_601, 32, 2, "sum", True, True)]   # H = 32: blocks 880-887 own no rows


@pytest.mark.parametrize("n,h,c,reduction,bias,want_dx", HEAD_CASES,
                         ids=[f"n{n}-h{h}-c{c}-{r}{'' if b else '-nobias'}{'' if d else '-nodx'}"
                              for n, h, c, r, b, d in HEAD_CASES])
def test_head_cross_entropy_matches_separate_steps(n, h, c, reduction, bias, want_dx):
    gen = torch.Generator().manual_seed(n + h + c)
    x = torch.randn(n, h, generator=gen)
    x[::5] = 0       # rows whose logits are the bias: ties, where the first maximal class wins
    lin = head_linear(h, c, bias, gen)
    if bias and c > 1:
        with torch.no_grad():
            lin.bias[1] = lin.bias[0] = lin.bias.max()
    y = torch.randint(0, c, (n,), generator=gen)
    yd = y.to(DEV)
    got = run_head(x, lin, yd, reduction, want_dx)
    w, b = lin.weight.detach().cpu().double(), None if lin.bias is None else lin.bias.detach().cpu().double()
    z64 = x.double() @ w.t() + (b if b is not None else 0)
    loss, _, dx, dw, db = head_grads64(z64, x, lin.weight, y, reduction)
    assert_parity(got["logits"], z64, "logits")
    assert_loss(got["loss"], loss)
    if want_dx:
        assert_parity(got["dx"], dx, "dx")
    else:
        assert got["dx"] is None
    assert_parity(got["dw"], dw, "dw")
    if bias:
        assert_parity(got["db"], db, "db")
    assert_bitexact(got["counts"], counters_np(got["logits"], y), "counters")
    assert_same_bits(got, run_head(x, lin, yd, reduction, want_dx))


# ------------------------------------------------------------------------------------------------
# 2. confidently classified rows: every row labelled with its argmax, margins 8-14, offsets up to +-50.  The loss and
#    the gradients are checked against fp64 over the kernel's own logits, so fp32 rounding in x w^T does not enter.
# ------------------------------------------------------------------------------------------------
def confident_logits(n, c, gen):
    z = torch.randn(n, c, generator=gen, dtype=torch.float64)
    y = torch.randint(0, c, (n,), generator=gen)
    margin = 8 + 6 * torch.rand(n, generator=gen, dtype=torch.float64)
    z[torch.arange(n), y] = z.max(1).values + margin
    return z + (100 * torch.rand(n, 1, generator=gen, dtype=torch.float64) - 50), y


@pytest.mark.parametrize("h,c", [(32, 2), (16, 3), (64, 8)])
@pytest.mark.parametrize("reduction", ["sum", "mean"])
def test_head_confident_rows(h, c, reduction):
    n = 200_003
    gen = torch.Generator().manual_seed(7 * h + c)
    z, y = confident_logits(n, c, gen)
    lin = head_linear(h, c, True, gen)
    # x with x w^T + b = z: a random x moved by the least-squares correction
    w, b = lin.weight.detach().cpu().double(), lin.bias.detach().cpu().double()
    x = torch.randn(n, h, generator=gen, dtype=torch.float64)
    x = (x + (z - b - x @ w.t()) @ torch.linalg.pinv(w.t())).float()
    yd = y.to(DEV)
    got = run_head(x, lin, yd, reduction, True)
    logits = got["logits"].cpu()
    assert (logits.argmax(1) == y).all()
    assert_parity(logits, x.double() @ w.t() + b, "logits")
    loss, _, dx, dw, db = head_grads64(logits, x, lin.weight, y, reduction)
    assert_loss(got["loss"], loss)
    assert_parity(got["dx"], dx, "dx")
    assert_parity(got["dw"], dw, "dw")
    assert_parity(got["db"], db, "db")
    assert_bitexact(got["counts"], counters_np(logits, y), "counters")
    assert_same_bits(got, run_head(x, lin, yd, reduction, True))


@pytest.mark.parametrize("c", [2, 3, 9])
@pytest.mark.parametrize("reduction", ["sum", "mean"])
def test_cross_entropy_confident_rows(c, reduction):
    n = 200_003
    z, y = confident_logits(n, c, torch.Generator().manual_seed(11 * c))
    z = z.float()
    loss64, dl64 = ce64(z, y, reduction)
    runs = []
    for _ in range(2):
        zd = z.to(DEV).requires_grad_(True)
        loss = F.cross_entropy(zd, y.to(DEV), reduction)
        (loss * torch.tensor(UPSTREAM, device=DEV)).backward()
        runs.append((loss.detach(), zd.grad))
    assert_loss(runs[0][0], loss64)
    assert_parity(runs[0][1], dl64, "dlogits")
    assert_bitexact(runs[1][0], runs[0][0], "loss run-to-run")
    assert_bitexact(runs[1][1], runs[0][1], "dlogits run-to-run")


# ------------------------------------------------------------------------------------------------
# 3. a label outside [0, C) in a large batch: the loss is NaN, the ops-level flag is set, the gradient is NaN on that
#    row (and, through it, in dw and db) and correct on every other row; the counters skip the row
# ------------------------------------------------------------------------------------------------
BAD_ROW = 77_777


@pytest.mark.parametrize("label", ["C", -1, -100, 2 ** 40])
@pytest.mark.parametrize("c", [2, 5])
@pytest.mark.parametrize("path", ["fused", "unfused"])
def test_label_outside_the_classes(path, c, label):
    n, h = 100_003, 32
    gen = torch.Generator().manual_seed(c)
    x = torch.randn(n, h, generator=gen)
    lin = head_linear(h, c, True, gen)
    y = torch.randint(0, c, (n,), generator=gen)
    y_ok = y.clone()
    y[BAD_ROW] = c if label == "C" else label
    yd = y.to(DEV)
    others = torch.ones(n, dtype=torch.bool)
    others[BAD_ROW] = False
    with torch.no_grad():
        logits = F.linear(x.to(DEV), lin.weight, lin.bias, weight_layout="out_in")
    for reduction in ("sum", "mean"):
        if path == "fused":
            _, _, counts, bad = ops.head_cross_entropy_fwd_impl(x.to(DEV), lin.weight, lin.bias, yd, reduction == "mean",
                                                                True)
            got = run_head(x, lin, yd, reduction, True)
            assert torch.isnan(got["loss"]).item()
            assert_bitexact(got["counts"], counts, "counters")
            assert_bitexact(counts, ops.binary_confusion_impl(yd, logits=got["logits"]), "counters of both paths")
            assert_bitexact(counts, counters_np(got["logits"], y), "counters")
            dx = got["dx"].cpu()
            assert torch.isnan(dx[BAD_ROW]).all()
            _, _, dx64, _, _ = head_grads64(got["logits"], x, lin.weight, y_ok, reduction)
            assert_parity(dx[others], dx64[others], "dx of the other rows")
            assert torch.isnan(got["dw"]).all() and torch.isnan(got["db"]).all()
            assert_same_bits(got, run_head(x, lin, yd, reduction, True))
        else:
            loss_, bad = ops.cross_entropy_fwd_impl(logits, yd, reduction == "mean")
            zd = logits.clone().requires_grad_(True)
            loss = F.cross_entropy(zd, yd, reduction)
            (loss * torch.tensor(UPSTREAM, device=DEV)).backward()
            assert torch.isnan(loss).item() and torch.isnan(loss_).item()
            dl = zd.grad.cpu()
            assert torch.isnan(dl[BAD_ROW]).all()
            _, dl64 = ce64(logits, y_ok, reduction)
            assert_parity(dl[others], dl64[others], "dlogits of the other rows")
            assert_bitexact(ops.binary_confusion_impl(yd, logits=logits), counters_np(logits, y), "counters")
        assert int(bad.item()) == 1
    # the flag stays clear without such a label
    assert int(ops.cross_entropy_fwd_impl(logits, y_ok.to(DEV), True)[1].item()) == 0
    assert int(ops.head_cross_entropy_fwd_impl(x.to(DEV), lin.weight, lin.bias, y_ok.to(DEV), True)[3].item()) == 0


# ------------------------------------------------------------------------------------------------
# 4. no rows: torch's values (the mean is NaN, the sum 0, parameter gradients 0)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("reduction", ["sum", "mean"])
@pytest.mark.parametrize("path", ["fused", "unfused"])
def test_empty_batch(path, reduction):
    h, c = 32, 2
    lin = head_linear(h, c, True, torch.Generator().manual_seed(0))
    ref = torch.nn.Linear(h, c).double()
    ref.load_state_dict({k: v.detach().cpu().double() for k, v in lin.state_dict().items()})
    x64 = torch.zeros(0, h, dtype=torch.float64, requires_grad=True)
    want = torch.nn.functional.cross_entropy(ref(x64), torch.zeros(0, dtype=torch.long), reduction=reduction)
    (want * UPSTREAM).backward()
    y = torch.zeros(0, dtype=torch.int64, device=DEV)
    if path == "fused":
        got = run_head(torch.zeros(0, h), lin, y, reduction, True)
        loss = got["loss"]
        assert got["dx"].shape == (0, h) and got["counts"].tolist() == [0] * 5
        assert (ref.weight.grad == 0).all() and (got["dw"] == 0).all()
        assert (ref.bias.grad == 0).all() and (got["db"] == 0).all()
    else:
        zd = torch.zeros(0, c, device=DEV, requires_grad=True)
        loss = F.cross_entropy(zd, y, reduction)
        (loss * UPSTREAM).backward()
        assert zd.grad.shape == (0, c)
    if reduction == "mean":
        assert torch.isnan(want).item() and torch.isnan(loss).item()
    else:
        assert want.item() == 0 and loss.item() == 0


# ------------------------------------------------------------------------------------------------
# 5. the bench step's output layer: forward_loss(reduction="sum", confusion=True) on the int32 batch of 25 full-size
#    botnet graphs (3,577,675 rows), against fp64 from the model's hidden output
# ------------------------------------------------------------------------------------------------
def test_bench_batch_forward_loss():
    from bench import CFG
    from meta_gcn_b200 import data as D
    from meta_gcn_b200.gcn_meta.models import GCNModel
    graphs = [D.synth_botnet_graph(seed=s, num_nodes=143107, edge_entries=1_500_000, evil=min(10000, 143107 // 14))
              for s in range(25)]
    batch = D.GraphBatch.from_data_list(graphs).with_int32_indices().to(DEV)
    assert batch.num_nodes == 3_577_675
    x0, deg, y = batch.x[:, 0].view(-1, 1), batch.x[:, 1], batch.y.long()
    torch.manual_seed(0)
    model = GCNModel(**CFG).to(DEV)

    def run():
        model.zero_grad(set_to_none=True)
        loss, logits, counts = model.forward_loss(x0, batch.edge_index, y, deg_K=deg, reduction="sum", confusion=True)
        loss.backward()
        hid = model(x0, batch.edge_index, deg_K=deg, _hidden=True).detach()
        hd = hid.clone().requires_grad_(True)     # the same head over the same hidden output, for dx
        loss2, _ = F.head_cross_entropy(hd, model.final, y, "sum")
        assert_bitexact(loss2.detach(), loss.detach(), "head over the hidden output")
        dx, = torch.autograd.grad(loss2, hd)
        return dict(loss=loss.detach(), logits=logits, counts=counts, hid=hid, dx=dx,
                    dw=model.final.weight.grad.clone(), db=model.final.bias.grad.clone())

    got = run()
    hid = got["hid"].cpu()
    w, b = model.final.weight.detach().cpu().double(), model.final.bias.detach().cpu().double()
    z64 = hid.double() @ w.t() + b
    assert_parity(got["logits"], z64, "logits")
    loss, _, dx, dw, db = head_grads64(z64, hid, model.final.weight, y, "sum", upstream=1.0)
    assert_loss(got["loss"], loss)
    assert_parity(got["dx"], dx, "dx")
    assert_parity(got["dw"], dw, "dw")
    assert_parity(got["db"], db, "db")
    assert_bitexact(got["counts"], counters_np(got["logits"], y), "counters")
    assert_same_bits(got, run())


# ------------------------------------------------------------------------------------------------
# 6. the unfused output layer GCNModel.forward runs, with its autograd: k_linear_small_out<L> forward,
#    k_wgrad_narrow (the gradient is the narrow operand) and k_linear_small_in_fixed for dx, below and above the grid
#    caps (1184 blocks of 256 / L rows; 592 blocks of 64 rows)
# ------------------------------------------------------------------------------------------------
SMALL_OUT_CAP = {16: 75_776, 32: 37_888, 64: 18_944, 128: 9_472}


@pytest.mark.parametrize("n", ["below", "above", "above_wgrad"])
@pytest.mark.parametrize("c", [1, 2, 3, 4])
@pytest.mark.parametrize("h", [16, 32, 64, 128])
def test_output_layer_autograd(h, c, n):
    n = {"below": SMALL_OUT_CAP[h] - 1, "above": 2 * SMALL_OUT_CAP[h] + 3, "above_wgrad": 37_889}[n]
    gen = torch.Generator().manual_seed(h * c + n)
    x = torch.randn(n, h, generator=gen)
    w = torch.randn(c, h, generator=gen) / h ** 0.5
    b = torch.randn(c, generator=gen)
    gy = torch.randn(n, c, generator=gen)
    x64 = x.double()
    y64 = x64 @ w.double().t() + b.double()

    def run():
        xd, wd, bd = (t.to(DEV).requires_grad_(True) for t in (x, w, b))
        out = F.linear(xd, wd, bd, weight_layout="out_in")
        out.backward(gy.to(DEV))
        return dict(y=out.detach(), dx=xd.grad, dw=wd.grad, db=bd.grad)

    got = run()
    assert_parity(got["y"], y64, "y")
    assert_parity(got["dx"], gy.double() @ w.double(), "dx")
    assert_parity(got["dw"], gy.double().t() @ x64, "dw")
    assert_parity(got["db"], gy.double().sum(0), "db")
    assert_same_bits(got, run())


# the first layer's routes, Hi <= 4 -> Ho: k_linear_small_in_fixed (256 % (Ho / 4) == 0) or k_linear_small_in
# (Ho = 12) with masks, row scale, add and ReLU, and k_wgrad_narrow with the input as the narrow operand
@pytest.mark.parametrize("n", [4097, 110_001])
@pytest.mark.parametrize("ho", [12, 16, 32, 64, 128])
@pytest.mark.parametrize("hi", [1, 2, 3, 4])
def test_narrow_input_layer(hi, ho, n):
    gen = torch.Generator().manual_seed(hi * ho + n)
    x = torch.randn(n, hi, generator=gen)
    xmask = (torch.rand(n, hi, generator=gen) > 0.3).float()
    w = torch.randn(hi, ho, generator=gen)
    b = torch.randn(ho, generator=gen)
    add = torch.randn(n, ho, generator=gen)
    rs = torch.rand(n, generator=gen) + 0.5
    g = torch.randn(n, ho, generator=gen)
    gmask = (torch.rand(n, ho, generator=gen) > 0.5).float() - 0.25 * (torch.rand(n, ho, generator=gen) > 0.5).float()
    pre = (x.double() * (xmask > 0)) @ w.double() + b.double() + add.double()
    y64 = rs.double()[:, None] * pre.clamp(min=0)
    gm = g.double() * (gmask > 0)

    def run():
        d = [t.to(DEV) for t in (x, w, b, add, xmask, rs, g, gmask)]
        y = ops.linear_impl(d[0], d[1], False, d[2], d[3], 1, xmask=d[4], row_scale=d[5])
        dw, db = ops.linear_wgrad_impl(d[0], d[6], False, True, gmask=d[7])
        return dict(y=y, dw=dw, db=db)

    got = run()
    assert_parity(got["y"], y64, "y")
    assert_parity(got["dw"], x.double().t() @ gm, "dw")
    assert_parity(got["db"], gm.sum(0), "db")
    assert_same_bits(got, run())


# ------------------------------------------------------------------------------------------------
# 7. the loss kernels alone, above both grid caps (forward 1184 blocks of 2048 rows, backward 2368 of 256), and
#    forward_loss on the configurations the fused head does not take
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,c,reduction", [(2_424_833, 1, "sum"), (2_424_833, 2, "mean"), (2_424_833, 9, "sum"),
                                           (606_209, 100, "mean"), (3001, 4096, "sum"), (606_207, 2, "sum")])
def test_cross_entropy_kernels(n, c, reduction):
    gen = torch.Generator().manual_seed(n + c)
    z = 3 * torch.randn(n, c, generator=gen)
    y = torch.randint(0, c, (n,), generator=gen)
    loss64, dl64 = ce64(z, y, reduction)
    zd, yd = z.to(DEV), y.to(DEV)

    def run():
        loss, bad = ops.cross_entropy_fwd_impl(zd, yd, reduction == "mean")
        dl = ops.cross_entropy_bwd_impl(zd, yd, reduction == "mean", torch.tensor([UPSTREAM], device=DEV))
        assert int(bad.item()) == 0
        return dict(loss=loss, dl=dl)

    got = run()
    assert_loss(got["loss"], loss64)
    assert_parity(got["dl"], dl64, "dlogits")
    assert_same_bits(got, run())


@pytest.mark.parametrize("hidden,classes", [(32, 9), (48, 2)])
def test_forward_loss_fallback(hidden, classes):
    """forward_loss on a head the fused kernel does not take (C > 8, H not in {16, 32, 64, 128}) = forward + the
    cross entropy of its logits in fp64, with the counters of its logits"""
    from meta_gcn_b200 import data as D
    from meta_gcn_b200.gcn_meta.models import GCNModel
    cfg = dict(in_channels=1, enc_sizes=[hidden] * 3, num_classes=classes, residual_hop=1, dropout=0.0,
               final_type="proj", deg_norm="sm", aggr="add", bias=False)
    g = D.synth_botnet_graph(seed=3, num_nodes=6000, edge_entries=60000, evil=400)
    b = D.GraphBatch.from_data_list([g]).to(DEV)
    x0, deg = b.x[:, 0:1].contiguous(), b.x[:, 1].contiguous()
    y = torch.randint(0, classes, (b.num_nodes,), generator=torch.Generator().manual_seed(hidden)).to(DEV)
    torch.manual_seed(0)
    model = GCNModel(**cfg).to(DEV)
    with torch.no_grad():
        out = model(x0, b.edge_index, deg_K=deg)
    for reduction in ("sum", "mean"):
        loss, logits, counts = model.forward_loss(x0, b.edge_index, y, deg_K=deg, reduction=reduction, confusion=True)
        assert_parity(logits, out, "logits")
        assert_loss(loss.detach(), ce64(logits, y, reduction)[0])
        assert_bitexact(counts, counters_np(logits.detach(), y), "counters")


def test_forward_loss_equals_forward_plus_loss():
    """GCNModel.forward_loss == GCNModel.forward + CrossEntropyLoss (train_botnet.py:286-287), values and gradients"""
    from meta_gcn_b200 import data as D
    from meta_gcn_b200.gcn_meta.models import GCNModel
    cfg = dict(in_channels=1, enc_sizes=[32] * 4, num_classes=2, residual_hop=1, dropout=0.0, final_type="proj",
               deg_norm="sm", aggr="add", bias=False)
    g = D.synth_botnet_graph(seed=2, num_nodes=5000, edge_entries=50000, evil=300)
    b = D.GraphBatch.from_data_list([g]).to(DEV)
    x0, deg, y = b.x[:, 0:1].contiguous(), b.x[:, 1].contiguous(), b.y.long()
    torch.manual_seed(0)
    model = GCNModel(**cfg).to(DEV)
    out = model(x0, b.edge_index, deg_K=deg)
    loss_a = torch.nn.CrossEntropyLoss()(out, y)
    loss_a.backward()
    grads_a = [p.grad.clone() for p in model.parameters()]
    model.zero_grad()
    loss_b, logits, counts = model.forward_loss(x0, b.edge_index, y, deg_K=deg, confusion=True)
    loss_b.backward()
    assert_parity(logits, out, "logits")
    assert abs(loss_a.item() - loss_b.item()) <= 1e-6
    for ga, p in zip(grads_a, model.parameters()):
        assert_parity(p.grad, ga, "grad")
    assert int(counts[4]) == int((out.argmax(1) == y).sum())
