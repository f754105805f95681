"""The gated oracle (tests/gated_oracle.py) against the goldens the unmodified reference wrote for edge_gate='proj'
(tests/golden/gcn_meta_gate_proj*.npz), in fp32 and fp64; host only."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from gated_oracle import GatedOracle
from util import golden

CFG = dict(enc_sizes=[16, 16, 16], num_classes=2, residual_hop=1, dropout=0.0, final_type="proj", bias=True)


@pytest.mark.parametrize("name, cfg, ew", [
    ("gcn_meta_gate_proj", dict(in_channels=1, aggr="add", deg_norm="sm"), False),
    ("gcn_meta_gate_proj_mean_ew", dict(in_channels=5, aggr="mean", deg_norm="rw"), True),
])
def test_gated_oracle_matches_reference_golden(name, cfg, ew):
    """the gated restatement in fp32 and fp64 against goldens written by the unmodified reference"""
    g = golden(name)
    full = dict(CFG, **cfg)
    for dtype, tol in ((torch.float32, 1e-5), (torch.float64, 1e-5)):
        model = GatedOracle(**full)
        model.load_state_dict({k[6:]: torch.from_numpy(np.asarray(a)) for k, a in g.items() if k.startswith("param.")})
        model = model.to(dtype)
        x = torch.from_numpy(g["x"]).to(dtype)
        ei = torch.from_numpy(g["edge_index"])
        deg = torch.from_numpy(g["deg"]).to(dtype)
        ewt = torch.from_numpy(g["edge_weight"]).to(dtype) if ew else None
        out = model(x, ei, deg, ewt)
        loss = nn.CrossEntropyLoss()(out, torch.from_numpy(g["y"]))
        loss.backward()
        ref = torch.from_numpy(g["out"]).double()
        assert torch.allclose(out.double(), ref, rtol=tol, atol=tol), (dtype, (out.double() - ref).abs().max())
        assert abs(loss.item() - float(g["loss"])) <= tol * max(1.0, abs(float(g["loss"])))
        for k, prm in model.named_parameters():
            r = torch.from_numpy(g["grad." + k]).double()
            assert torch.allclose(prm.grad.double(), r, rtol=1e-4, atol=1e-6), (dtype, k)
