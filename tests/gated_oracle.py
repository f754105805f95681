"""EdgeGateProj (gcn_base_models.py:322-369) restated on top of oracle/port.py: the gated additive node model and
OracleGCNModel with a gate on every node model, in fp32 or, after .double(), fp64.  Pinned to the reference goldens
by tests/test_oracle_gate.py."""
import torch
import torch.nn as nn

from oracle import port


def gated_node_model(x, edge_index, weight_node, bias, u, v, c, deg=None, edge_weight=None, deg_norm="sm", aggr="add"):
    """NodeModelAdditive.forward with edge_gate='proj' (gcn_base_models.py:199-243, 322-369): the message
    (x W)[row] * norm times sigmoid(linsrc(x W)[row] + lintgt(x W)[col] + bias), summed (or averaged) per target"""
    xw = torch.matmul(x, weight_node)
    row, col = edge_index
    gate = torch.sigmoid(torch.index_select(xw @ u.t(), 0, row) + torch.index_select(xw @ v.t(), 0, col) + c)
    if deg_norm is None:
        x_j = torch.index_select(xw, 0, row)
    else:
        norm = port.degnorm_const(edge_index, xw.size(0), deg, edge_weight, deg_norm)
        if deg_norm == "rw" and edge_weight is None:
            x_j = torch.index_select(xw * norm.view(-1, 1).to(xw.dtype), 0, row)
        else:
            x_j = torch.index_select(xw, 0, row) * norm.view(-1, 1).to(xw.dtype)
    out = port.scatter_rows(aggr, x_j * gate, col, xw.size(0))
    return out + bias if bias is not None else out


class _Gate(nn.Module):
    def __init__(self, cout):
        super().__init__()
        self.linsrc = nn.Linear(cout, 1, bias=False)
        self.lintgt = nn.Linear(cout, 1, bias=False)
        self.bias = nn.Parameter(torch.zeros(1))
        for lin in (self.linsrc, self.lintgt):
            nn.init.uniform_(lin.weight, -0.1, 0.1)


class GatedOracle(port.OracleGCNModel):
    """OracleGCNModel with an EdgeGateProj per node model (parameter names of the reference:
    gcn_net.N.gcn.node_models.0.edge_gate.{linsrc.weight, lintgt.weight, bias}); fp32 or, after .double(), fp64"""

    def __init__(self, **cfg):
        super().__init__(**cfg)
        for layer, cout in zip(self.gcn_net, self.sizes[1:]):
            layer.gcn.node_models[0].edge_gate = _Gate(cout)

    def forward(self, x, edge_index, deg=None, edge_weight=None, batch_slices_x=None):
        xr, hop = None, self.residual_hop
        for n, layer in enumerate(self.gcn_net):
            nm = layer.gcn.node_models[0]
            eg = nm.edge_gate
            dg = deg.to(x.dtype) if deg is not None else None
            xo = gated_node_model(x, edge_index, nm.weight_node, nm.bias, eg.linsrc.weight, eg.lintgt.weight, eg.bias,
                                  dg, edge_weight, self.deg_norm, self.aggr)
            xo = self.dropout(self._act(self.act_layer, xo))
            if n % hop == 0 and n // hop < len(self.residuals):
                xr = self.residuals[n // hop](x)
            xo = self._act(self.act_res, xo + xr) if n < self.num_layers - 1 else xo + xr
            x = xo
        return self.final(x)
