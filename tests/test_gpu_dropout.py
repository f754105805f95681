"""Dropout on the fused residual stack (gcn_model.py:92, the reference's default p = 0.5): the keep-mask generator
(csrc/philox.cuh, csrc/dropout.cu) against a numpy restatement of its contract (include/mgcn.h), its statistics, and
training steps of the stack against the oracle with the same masks.  Host tests are unmarked; the rest need a GPU."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn as nn

from meta_gcn_b200 import _lib, fused, ops
from meta_gcn_b200.gcn_meta.models import GCNModel
from oracle import port
from util import assert_bitexact, assert_parity

DEV = "cuda"
BOTNET = dict(in_channels=1, enc_sizes=[32] * 12, num_classes=2, residual_hop=1, dropout=0.5,
              final_type="proj", deg_norm="sm", aggr="add", bias=False)
SEED = -0x1234_5678_9ABC_DEF1          # both key halves non-zero, the high bit set

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c, k):
    """Philox4x32-10 on uint64 arrays holding 32-bit words: c = (c0, c1, c2, c3), k = (k0, k1)"""
    c0, c1, c2, c3 = (np.asarray(v, dtype=np.uint64) for v in c)
    k0, k1 = (np.asarray(v, dtype=np.uint64) for v in k)
    for _ in range(10):
        p0 = c0 * np.uint64(M0)           # < 2^64: exact
        p1 = c2 * np.uint64(M1)
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & MASK32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & MASK32
        k0 = (k0 + np.uint64(W0)) & MASK32
        k1 = (k1 + np.uint64(W1)) & MASK32
    return c0, c1, c2, c3


def keep_threshold(p):
    return int(np.rint(np.float64(np.float32(p)) * 65536.0))


def keep_bits_ref(seed, L, N, W, p):
    """the contract of mgcn_dropout_keep_bits restated: int32 [L, N, W]"""
    s = np.uint64(seed & 0xFFFFFFFFFFFFFFFF)
    k = (s & MASK32, s >> np.uint64(32))
    t = np.uint64(keep_threshold(p))
    l, n, w = np.meshgrid(np.arange(L, dtype=np.uint64), np.arange(N, dtype=np.uint64), np.arange(W, dtype=np.uint64),
                          indexing="ij")
    bits = np.zeros((L, N, W), dtype=np.uint64)
    for j in range(4):
        r = philox4x32_10((n, l, np.uint64(4) * w + np.uint64(j), np.zeros_like(n)), k)
        for i, ri in enumerate(r):
            bits |= ((ri & np.uint64(0xFFFF)) >= t).astype(np.uint64) << np.uint64(8 * j + 2 * i)
            bits |= ((ri >> np.uint64(16)) >= t).astype(np.uint64) << np.uint64(8 * j + 2 * i + 1)
    return bits.astype(np.uint32).view(np.int32)


def unpack(keep, H):
    """int32 [L, N, W] -> float32 0/1 [L, N, H]"""
    u = np.asarray(keep).view(np.uint32)
    b = (u[..., None] >> np.arange(32, dtype=np.uint32)) & 1
    return torch.from_numpy(b.reshape(u.shape[0], u.shape[1], -1)[..., :H].astype(np.float32))


# ------------------------------------------------------------------------------------------------ host
def test_philox_known_answers():
    """Random123's known-answer vectors for philox4x32 with 10 rounds"""
    cases = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
             ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
             ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
              (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for c, k, want in cases:
        assert tuple(int(v) for v in philox4x32_10(c, k)) == want


def test_stack_eligibility_with_dropout():
    m = GCNModel(**BOTNET)
    ei = torch.zeros(2, 0, dtype=torch.int64)
    assert m.train()._stack_eligible(ei, None, None)            # the reference's default p = 0.5, training
    assert m.eval()._stack_eligible(ei, None, None)
    assert GCNModel(**dict(BOTNET, dropout=0.0)).train()._stack_eligible(ei, None, None)
    one = GCNModel(**dict(BOTNET, dropout=1.0))
    assert not one.train()._stack_eligible(ei, None, None)      # torch's dropout returns zeros: per-layer path
    assert one.eval()._stack_eligible(ei, None, None)
    # the round-1 hidden-32 kernels (x that requires grad) take no dropout: the stack declines before any launch
    x = torch.ones(5, 1, requires_grad=True)
    params = [(torch.zeros(1, 32), torch.zeros(32, 1), torch.zeros(32))] + [
        (torch.zeros(32, 32), torch.zeros(32, 32), torch.zeros(32))] * 2
    assert fused.residual_gcn_stack(x, None, None, None, params, False, dropout=0.5) is None
    with pytest.raises(ValueError):
        fused.residual_gcn_stack(x, None, None, None, params, False, dropout=1.0)


def test_keep_bits_arguments_without_device():
    lib = _lib.load()
    assert lib.mgcn_dropout_keep_bits(None, 3, 10, 1, 1.0, None, None) == _lib_err("SHAPE")      # t = 65536
    assert lib.mgcn_dropout_keep_bits(None, 3, 10, 1, -0.1, None, None) == _lib_err("SHAPE")
    assert lib.mgcn_dropout_keep_bits(None, 3, 10, 1, float("nan"), None, None) == _lib_err("SHAPE")
    assert lib.mgcn_dropout_keep_bits(None, 3, 10, 0, 0.5, None, None) == _lib_err("SHAPE")
    assert lib.mgcn_dropout_keep_bits(None, 3, 10, 1, 0.5, None, None) == _lib_err("NULL")
    assert lib.mgcn_dropout_keep_bits(None, 0, 10, 1, 0.5, None, None) == 0                     # nothing to do
    assert lib.mgcn_dropout_apply(None, None, 10, 30, 1, 2.0, None) == _lib_err("SHAPE")        # H % 4
    assert lib.mgcn_dropout_apply(None, None, 10, 64, 1, 2.0, None) == _lib_err("SHAPE")        # W < H / 32
    with pytest.raises(RuntimeError, match="CPU"):
        torch.ops.mgcn.dropout_keep_bits(torch.zeros(1, dtype=torch.int64), 1, 4, 1, 0.5)


def _lib_err(name):
    return {"NULL": -1, "SHAPE": -3}[name]


# ------------------------------------------------------------------------------------------------ generator on the GPU
def _seed(v=SEED):
    return torch.tensor([v], dtype=torch.int64, device=DEV)


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
@pytest.mark.parametrize("W", [1, 2, 4])
def test_keep_bits_match_restatement(W, p):
    L, N = 3, 1013                      # N not a multiple of 32
    got = ops.dropout_keep_bits_impl(_seed(), L, N, W, p)
    assert_bitexact(got, keep_bits_ref(SEED, L, N, W, p), f"keep bits W={W} p={p}")
    assert_bitexact(torch.ops.mgcn.dropout_keep_bits(_seed(), L, N, W, p), got, "torch.ops.mgcn.dropout_keep_bits")


def _column_counts(words):
    """kept count per column c of int32 words [...]: sum over all words of bit c"""
    return torch.stack([((words >> c) & 1).sum(dtype=torch.int64) for c in range(32)]).double()


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_keep_bits_statistics(p):
    L, N = 12, 1_000_000
    keep = ops.dropout_keep_bits_impl(_seed(), L, N, 1, p).view(L, N)
    q = 1.0 - keep_threshold(p) / 65536.0
    var = q * (1 - q)

    def within(frac, n, what):
        sigma = (var / n) ** 0.5
        assert abs(frac - q) <= 6 * sigma, f"{what}: {frac:.6f} vs {q:.6f} ({abs(frac - q) / sigma:.1f} sigma)"

    cols = _column_counts(keep).cpu().numpy()
    within(cols.sum() / (L * N * 32), L * N * 32, "overall")
    for c in range(32):
        within(cols[c] / (L * N), L * N, f"column {c}")
    for layer in range(L):
        within(float(_column_counts(keep[layer]).sum()) / (N * 32), N * 32, f"layer {layer}")
    # two layers' masks are independent draws: they agree with probability q^2 + (1-q)^2
    agree = float(_column_counts(~(keep[0] ^ keep[1])).sum()) / (N * 32)
    a = q * q + (1 - q) * (1 - q)
    assert abs(agree - a) <= 6 * (a * (1 - a) / (N * 32)) ** 0.5, (agree, a)
    other = ops.dropout_keep_bits_impl(_seed(SEED + 1), L, N, 1, p).view(L, N)
    assert not torch.equal(keep, other)


# ------------------------------------------------------------------------------------------------ training steps
class _MaskedDropout(nn.Module):
    """the oracle's nn.Dropout with the stack's masks: the k-th call multiplies by layer k's mask x scale"""

    def __init__(self, keep, H, p):
        super().__init__()
        self.masks = unpack(keep, H)
        self.scale = torch.tensor(1.0 / (1.0 - p), dtype=torch.float32)
        self.calls = 0

    def forward(self, x):
        m = (self.masks[self.calls] * self.scale).to(x.dtype)
        self.calls += 1
        return x * m


def _pin_seed(monkeypatch, seed=SEED):
    """the stack's seed fixed; returns the list of the forwards that asked for one"""
    calls = []

    def pinned(device):
        calls.append(device)
        return torch.tensor([seed], dtype=torch.int64, device=device)
    monkeypatch.setattr(fused, "dropout_seed", pinned)
    return calls


def _graph(seed=4, num_nodes=20000, edge_entries=220000, evil=1500):
    from meta_gcn_b200.data import synth_botnet_graph
    return synth_botnet_graph(seed=seed, num_nodes=num_nodes, edge_entries=edge_entries, evil=evil)


def _c1_graph():
    from meta_gcn_b200.data import synth_botnet_graph
    return synth_botnet_graph(seed=0)


def _wide_input(g):
    return torch.randn(g["x"].shape[0], 32, generator=torch.Generator().manual_seed(3))


# parity cases: (config, graph, 32-wide input or None for the botnet input ones[N,1], mask seed per p).  The mask seeds
# are inputs like the graph seeds: a ReLU whose exact input lies within rounding of zero has a derivative decided by the
# order of the fp32 sums, and that one element moves many gradients past 1e-5 of their norm whichever side is right
# (scripts/relu_boundary_check.py, __graft_entry__.smoke()).  scripts/dropout_boundary_check.py measures each
# (case, p, mask seed) against the fp64 oracle (profiles/dropout_boundary_check.log): at most seeds the stack is within
# 2e-6 of fp64; at the others one such element puts the stack, or the fp32 oracle, 1e-5 .. 2e-4 away (the 32-wide
# input without dropout too).  The seeds below are ones where both are at fp32 accuracy.
MASK_SEED = 0x2
CASES = {
    "botnet": (dict(BOTNET), _graph, None, {0.5: MASK_SEED, 0.1: MASK_SEED}),
    "rw": (dict(BOTNET, enc_sizes=[32] * 4, deg_norm="rw"), _graph, None, {0.5: SEED}),
    "wide": (dict(BOTNET, in_channels=32, enc_sizes=[32] * 4), _graph, _wide_input, {0.5: MASK_SEED}),
    "generic": (dict(BOTNET, enc_sizes=[64] * 4, bias=True), _graph, None, {0.5: SEED}),
    "c1": (dict(BOTNET), _c1_graph, None, {0.5: MASK_SEED}),
}


def case_inputs(case, p):
    """(config, graph, layer input) of a parity case"""
    cfg, graph, wide, _ = CASES[case]
    g = graph()
    x_in = wide(g) if wide else torch.from_numpy(g["x"][:, 0:1].copy())
    return dict(cfg, dropout=p), g, x_in


def _parity_vs_oracle(monkeypatch, case, p, arbitrated=False):
    """logits, loss and every gradient against the fp32 oracle with the same masks (arbitrated: entries that miss rtol
    1e-5 are judged against fp64, as the full-graph test of tests/test_gpu_bench_shapes.py does), logits against fp64"""
    from test_gpu_bench_shapes import assert_parity_arbitrated
    cfg, g, xin = case_inputs(case, p)
    mask_seed = CASES[case][3][p]
    calls = _pin_seed(monkeypatch, mask_seed)
    torch.manual_seed(0)
    ref = port.OracleGCNModel(**cfg)
    model = GCNModel(**cfg)
    model.load_state_dict(ref.state_dict())
    model.to(DEV).train()
    x = torch.from_numpy(g["x"])
    ei = torch.from_numpy(g["edge_index"])
    y = torch.from_numpy(g["y"]).long()
    deg = x[:, 1].contiguous()
    N, L, H = x.size(0), len(cfg["enc_sizes"]), max(cfg["enc_sizes"])
    keep = keep_bits_ref(mask_seed, L, N, (H + 31) // 32, p)
    ref.dropout = _MaskedDropout(keep, H, p)
    out_r = ref(xin, ei, deg)
    loss_r = nn.CrossEntropyLoss()(out_r, y)
    loss_r.backward()
    assert ref.dropout.calls == L
    out = model(xin.to(DEV), ei.to(DEV), deg_K=deg.to(DEV))
    loss = nn.CrossEntropyLoss()(out, y.to(DEV))
    loss.backward()
    assert len(calls) == 1, "the forward did not take the fused stack"
    ref64 = port.OracleGCNModel(**cfg)
    ref64.load_state_dict(ref.state_dict())
    ref64 = ref64.double()
    ref64.dropout = _MaskedDropout(keep, H, p)
    out64 = ref64(xin.double(), ei, deg.double())
    if arbitrated:
        nn.CrossEntropyLoss()(out64, y).backward()
        assert_parity_arbitrated(out, out_r, out64, "logits")
    else:
        assert_parity(out, out_r, "logits")
    assert abs(loss.item() - loss_r.item()) < 1e-5
    for (k, prm), (_, pr), (_, p64) in zip(model.named_parameters(), ref.named_parameters(), ref64.named_parameters()):
        if arbitrated:
            assert_parity_arbitrated(prm.grad, pr.grad, p64.grad, "grad." + k)
        else:
            assert_parity(prm.grad, pr.grad, "grad." + k)
    assert_parity(out, out64.detach(), "logits vs fp64")


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.5, 0.1])
def test_botnet_stack_with_dropout_vs_oracle(monkeypatch, p):
    """the 12-layer botnet model on the 20k-node hub graph (first layer: the streaming pass, then k_gcn_fwd_tc <0>/<1>)"""
    _parity_vs_oracle(monkeypatch, "botnet", p)


@pytest.mark.gpu
def test_rw_normalisation_with_dropout_vs_oracle(monkeypatch):
    """deg_norm='rw': no per-target factor, the backward's scale vector is the dropout scale alone"""
    _parity_vs_oracle(monkeypatch, "rw", 0.5)


@pytest.mark.gpu
def test_wide_input_with_dropout_vs_oracle(monkeypatch):
    """a 32-wide input that does not require grad: every layer through k_gcn_fwd_tc, none through the first-layer pass"""
    _parity_vs_oracle(monkeypatch, "wide", 0.5)


@pytest.mark.gpu
def test_generic_stack_with_bias_and_dropout_vs_oracle(monkeypatch):
    """hidden 64 with node-model bias: the generic stack, k_dropout_apply on the saved h (two words per row)"""
    _parity_vs_oracle(monkeypatch, "generic", 0.5)


@pytest.mark.gpu
def test_full_c1_graph_with_dropout_vs_oracle(monkeypatch):
    """the full C1 graph: its fp32 oracle sits 4e-6 .. 7e-6 of the gradients' norm from fp64 by itself, so fp64
    arbitrates the entries that miss (the bar of the dropout-free C1 test)"""
    _parity_vs_oracle(monkeypatch, "c1", 0.5, arbitrated=True)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["zero_degree", "x_requires_grad"])
def test_round1_stack_inputs_take_the_per_layer_path(monkeypatch, case):
    """inputs for which the stack would pick the round-1 hidden-32 kernels train with dropout on the per-layer path"""
    def refuse(*args, **kwargs):
        raise AssertionError("the round-1 stack was entered with dropout")
    monkeypatch.setattr(fused._ResidualGCNStack32, "apply", refuse)
    g = _graph()
    torch.manual_seed(0)
    model = GCNModel(**dict(BOTNET, enc_sizes=[32] * 4)).to(DEV).train()
    x = torch.from_numpy(g["x"]).to(DEV)
    deg = x[:, 1].clone()
    xin = x[:, 0:1].clone()
    if case == "zero_degree":
        deg[::7] = 0.0
    else:
        xin.requires_grad_(True)
    out = model(xin, torch.from_numpy(g["edge_index"]).to(DEV), deg_K=deg)
    loss = nn.CrossEntropyLoss()(out, torch.from_numpy(g["y"]).long().to(DEV))
    loss.backward()
    assert torch.isfinite(loss)
    for k, prm in model.named_parameters():
        assert torch.isfinite(prm.grad).all(), k
    if case == "x_requires_grad":
        assert torch.isfinite(xin.grad).all()


def _step(model, x, ei, deg, y):
    for prm in model.parameters():
        prm.grad = None
    loss = nn.CrossEntropyLoss()(model(x, ei, deg_K=deg), y)
    loss.backward()
    return loss.detach().clone(), [prm.grad.clone() for prm in model.parameters()]


def _inputs(g):
    x = torch.from_numpy(g["x"]).to(DEV)
    return (x[:, 0:1].contiguous(), torch.from_numpy(g["edge_index"]).to(DEV), x[:, 1].contiguous(),
            torch.from_numpy(g["y"]).long().to(DEV))


@pytest.mark.gpu
def test_eval_and_zero_p_are_unchanged(monkeypatch):
    """eval() with p = 0.5 and a training step at p = 0 run exactly the code of a dropout=0.0 model: same bits, same
    launches, no seed drawn"""
    def no_draw(device):
        raise AssertionError("a seed was drawn")
    monkeypatch.setattr(fused, "dropout_seed", no_draw)
    g = _graph()
    inputs = _inputs(g)
    torch.manual_seed(0)
    a = GCNModel(**BOTNET).to(DEV)
    b = GCNModel(**dict(BOTNET, dropout=0.0)).to(DEV)
    b.load_state_dict(a.state_dict())
    with torch.no_grad():
        assert_bitexact(a.eval()(*inputs[:2], deg_K=inputs[2]), b.eval()(*inputs[:2], deg_K=inputs[2]), "eval")
    a.train().dropout.p = 0.0
    b.train()
    c0 = _lib.launch_count()
    la, ga = _step(a, *inputs)
    c1 = _lib.launch_count()
    lb, gb = _step(b, *inputs)
    assert _lib.launch_count() - c1 == c1 - c0
    assert_bitexact(la, lb, "loss")
    for u, v in zip(ga, gb):
        assert_bitexact(u, v, "grad")


@pytest.mark.gpu
def test_same_rng_state_same_step_and_new_masks_per_step(monkeypatch):
    seeds = []
    real = fused.dropout_seed
    monkeypatch.setattr(fused, "dropout_seed", lambda device: seeds.append(real(device)) or seeds[-1])
    g = _graph()
    inputs = _inputs(g)
    torch.manual_seed(0)
    model = GCNModel(**dict(BOTNET, enc_sizes=[32] * 4)).to(DEV).train()
    state = torch.cuda.get_rng_state()
    l1, g1 = _step(model, *inputs)
    torch.cuda.set_rng_state(state)
    l2, g2 = _step(model, *inputs)
    l3, _ = _step(model, *inputs)
    assert_bitexact(l1, l2, "loss")
    for u, v in zip(g1, g2):
        assert_bitexact(u, v, "grad")
    assert torch.equal(seeds[0], seeds[1]) and not torch.equal(seeds[1], seeds[2])
    k1 = ops.dropout_keep_bits_impl(seeds[1], 4, inputs[0].size(0), 1, 0.5)
    k2 = ops.dropout_keep_bits_impl(seeds[2], 4, inputs[0].size(0), 1, 0.5)
    assert not torch.equal(k1, k2)
    assert l3.item() != l2.item()


@pytest.mark.gpu
def test_graphed_step_with_dropout_replays_the_rng_state():
    """a captured step draws its seed on the device: restoring the CUDA RNG state before an eager step and before a
    replay gives the same loss and gradients bit for bit, and two consecutive replays draw different masks"""
    from meta_gcn_b200 import functional as F
    from meta_gcn_b200.graphed import GraphedCall
    g = _graph(seed=5, num_nodes=6000, edge_entries=50000, evil=400)
    x0, ei, deg, y = _inputs(g)
    torch.manual_seed(0)
    model = GCNModel(**dict(BOTNET, enc_sizes=[32] * 4)).to(DEV).train()
    params = list(model.parameters())
    for prm in params:
        prm.grad = torch.zeros_like(prm)

    def fwd_loss_bwd():
        for prm in params:
            prm.grad.zero_()
        loss = F.cross_entropy(model(x0, ei, deg_K=deg), y, "sum")
        loss.backward()
        return loss

    graphed = GraphedCall(fwd_loss_bwd)
    state = torch.cuda.get_rng_state()
    loss_e = float(fwd_loss_bwd())
    grads_e = [prm.grad.clone() for prm in params]
    torch.cuda.set_rng_state(state)
    loss_g = float(graphed())
    assert loss_g == loss_e
    for prm, ge in zip(params, grads_e):
        assert torch.equal(prm.grad, ge)
    loss_g2 = float(graphed())
    assert loss_g2 != loss_g
