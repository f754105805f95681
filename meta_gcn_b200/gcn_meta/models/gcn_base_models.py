"""Mirror of src/gcn_meta/models/gcn_base_models.py for the hot path: ``NodeModelBase.degnorm_const``
(gcn_base_models.py:65-146) and ``NodeModelAdditive`` (gcn_base_models.py:163-243) on libmgcn.

Same constructor arguments and parameter names (``weight_node``, ``weight_edge``, ``bias``) as the
reference, so pickled reference models load.  The forward never materialises [E,H]: X·W runs in the
narrow FMA transform, and gather * norm -> scatter_add is one row-owned aggregation whose per-edge
weight dis[row]*edge_weight*dis[col] is formed in the reference's rounding order inside the kernel.
Edge gates (EdgeGateProj / EdgeGateFree, gcn_base_models.py:322-397) multiply that per-edge weight and receive their
gradient through a per-edge dot product (mgcn_edge_dot).  NodeModelMLP is outside the hot path."""
import torch
import torch.nn as nn
from torch.nn import Parameter

from ... import functional as F_mgcn
from ... import ops
from ...compat.torch_geometric.nn.inits import glorot, zeros
from ...graph import structure_of

_NORM_MODE = {"sm": 0, "rw": 1}


class NodeModelBase(nn.Module):
    def __init__(self, in_channels, out_channels, in_edgedim=None, deg_norm=None, edge_gate=None,
                 aggr="add", *args, **kwargs):
        assert deg_norm in [None, "sm", "rw"]
        assert edge_gate in [None, "proj", "free"]
        assert aggr in ["add", "mean", "max"]
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.in_edgedim = in_edgedim
        self.deg_norm = deg_norm
        self.aggr = aggr
        if edge_gate == "proj":                                           # gcn_base_models.py:57-63
            self.edge_gate = EdgeGateProj(out_channels, in_edgedim=in_edgedim, bias=True)
        elif edge_gate == "free":
            assert "num_edges" in kwargs
            self.edge_gate = EdgeGateFree(kwargs["num_edges"])
        else:
            self.register_parameter("edge_gate", None)

    @staticmethod
    def degree_factors(edge_index, num_nodes, deg=None, edge_weight=None, method="sm"):
        """dis[N] = deg^-1/2 ('sm') or deg^-1 ('rw'), inf -> 0; deg defaults to the (weighted)
        out-degree over edge_index[0] (gcn_base_models.py:119-135)."""
        if edge_weight is not None:
            deg = structure_of(edge_index, num_nodes).weighted_out_degree(edge_weight.view(-1))
        elif deg is None:
            deg = structure_of(edge_index, num_nodes).out_degree()
        return ops.gcn_norm_impl(deg, _NORM_MODE[method])

    @staticmethod
    def degnorm_const(edge_index=None, num_nodes=None, deg=None, edge_weight=None, method="sm",
                      device=None):
        """Reference-shaped result: norm[E] for 'sm' (and 'rw' with weights), dis[N] for 'rw'
        without weights (gcn_base_models.py:137-146).  The model path does not call this — it
        passes ``degree_factors`` to the aggregation kernel instead of materialising norm[E]."""
        assert method in ["sm", "rw"]
        dis = NodeModelBase.degree_factors(edge_index, num_nodes, deg, edge_weight, method)
        if method == "rw" and edge_weight is None:
            return dis
        row, col = edge_index
        if method == "sm":
            if edge_weight is None:
                return dis[row] * dis[col]
            return dis[row] * edge_weight.view(-1) * dis[col]
        return dis[row] * edge_weight.view(-1)

    def forward(self, x, edge_index, edge_attr=None, deg=None, *args, **kwargs):
        return x

    def num_parameters(self):
        if not hasattr(self, "num_para"):
            self.num_para = sum(p.nelement() for p in self.parameters())
        return self.num_para

    def __repr__(self):
        return ("{} (in_channels: {}, out_channels: {}, in_edgedim: {}, deg_norm: {}, edge_gate: {},"
                "aggr: {} | number of parameters: {})").format(
                    self.__class__.__name__, self.in_channels, self.out_channels, self.in_edgedim,
                    self.deg_norm, self.edge_gate.__class__.__name__, self.aggr, self.num_parameters())


class NodeModelAdditive(NodeModelBase):
    def __init__(self, in_channels, out_channels, in_edgedim=None, deg_norm="sm", edge_gate=None,
                 aggr="add", bias=True, **kwargs):
        super().__init__(in_channels, out_channels, in_edgedim, deg_norm, edge_gate, aggr, **kwargs)
        self.weight_node = Parameter(torch.Tensor(in_channels, out_channels))
        if in_edgedim is not None:
            self.weight_edge = Parameter(torch.Tensor(in_edgedim, out_channels))
        if bias:
            self.bias = Parameter(torch.Tensor(out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot(self.weight_node)
        if self.in_edgedim is not None:
            glorot(self.weight_edge)
        if self.bias is not None:
            zeros(self.bias)

    def forward(self, x, edge_index, edge_attr=None, deg=None, edge_weight=None, **kwargs):
        """x [N,C_in] -> [N,C_out]; ``_act`` / ``_dis`` are private hints from GCNLayer / GCNModel
        (fused ReLU epilogue, degree factors shared by all layers)."""
        act = kwargs.get("_act")
        n = x.size(0)
        graph = structure_of(edge_index, n)
        xw = F_mgcn.linear(x, self.weight_node)                       # gcn_base_models.py:201
        nbr_scale = row_scale = None
        if self.deg_norm is not None:
            dis = kwargs.get("_dis")
            if dis is None:
                dis = self.degree_factors(edge_index, n, deg, edge_weight, self.deg_norm)
            nbr_scale = dis
            row_scale = dis if self.deg_norm == "sm" else None
        eg = None
        if self.edge_gate is not None:                                    # gcn_base_models.py:230-232
            eg = self.edge_gate(xw, edge_index, edge_attr=edge_attr, edge_weight=edge_weight).view(-1)
        if self.aggr == "max":
            # gcn_base_models.py:209-237 with scatter_('max'): max over the incoming edges of (x W)[row] * norm_e,
            # norm_e formed exactly as degnorm_const does (one factor per edge, same roundings)
            norm_e = None
            if self.deg_norm is not None:
                dis = nbr_scale
                row, col = edge_index
                if self.deg_norm == "sm":
                    norm_e = dis[row] * dis[col] if edge_weight is None else dis[row] * edge_weight.view(-1) * dis[col]
                else:
                    norm_e = dis[row] if edge_weight is None else dis[row] * edge_weight.view(-1)
            if eg is None and edge_attr is None:
                out = F_mgcn.aggregate_max(xw, graph, norm_e)
            else:
                # the maximum is taken over gate_e * (x W [row_e] * norm_e + edge_attr_e W_e): not separable into a
                # per-node and a per-edge part, so the [E,H] messages are formed as the reference does
                # (gcn_base_models.py:223-232) and reduced by the primitive seam's first-maximum kernel
                msg = F_mgcn.gather_rows(xw, edge_index[0])
                if norm_e is not None:
                    msg = msg * norm_e.view(-1, 1)
                if edge_attr is not None:
                    assert self.in_edgedim is not None
                    msg = msg + F_mgcn.linear(edge_attr, self.weight_edge)
                if eg is not None:
                    msg = eg.view(-1, 1) * msg
                out = F_mgcn.scatter_rows_max(msg, edge_index[1], n)[0]
            if self.bias is not None:
                out = out + self.bias
            return torch.relu(out) if act == "relu" else out
        ew = edge_weight.view(-1) if (edge_weight is not None and self.deg_norm is not None) else None
        if eg is not None:
            ew = eg if ew is None else ew * eg                            # gate_e * norm_e: one weight per edge
        if edge_attr is None:
            return F_mgcn.aggregate(xw, graph, nbr_scale, row_scale, ew, self.aggr, self.bias, None, act)
        # per-edge feature messages (gcn_base_models.py:204-206,227): summed by the primitive seam
        assert self.in_edgedim is not None
        x_je = F_mgcn.linear(edge_attr, self.weight_edge)
        if eg is not None:
            x_je = x_je * eg.view(-1, 1)
        out = F_mgcn.aggregate(xw, graph, nbr_scale, row_scale, ew, self.aggr)
        out = out + F_mgcn.scatter_rows(x_je, edge_index[1], n, self.aggr)
        if self.bias is not None:
            out = out + self.bias
        return torch.relu(out) if act == "relu" else out


class EdgeGateProj(nn.Module):
    """gcn_base_models.py:322-369: gate_e = sigmoid(linsrc(x)[row_e] + lintgt(x)[col_e] (+ linedge(edge_attr)_e) + bias);
    the two node projections are [N,1] transforms on libmgcn, the per-edge part is elementwise on [E,1]"""

    def __init__(self, in_channels, in_edgedim=None, bias=False):
        super().__init__()
        self.in_channels, self.in_edgedim = in_channels, in_edgedim
        proj = lambda width: nn.Linear(width, 1, bias=False)     # noqa: E731  one scalar score per node / edge
        self.linsrc, self.lintgt = proj(in_channels), proj(in_channels)
        if in_edgedim is not None:
            self.linedge = proj(in_edgedim)
        self.register_parameter("bias", Parameter(torch.empty(1)) if bias else None)   # one scalar for all edges
        self.reset_parameters()

    def reset_parameters(self, initrange=0.1):
        scored = [self.linsrc, self.lintgt] + ([self.linedge] if self.in_edgedim is not None else [])
        for lin in scored:
            nn.init.uniform_(lin.weight, -initrange, initrange)
        if self.bias is not None:
            nn.init.zeros_(self.bias)

    def forward(self, x, edge_index, edge_attr=None, edge_weight=None):
        score = lambda lin, t: F_mgcn.linear(t, lin.weight, weight_layout="out_in")   # noqa: E731  [*, 1]
        gate = (F_mgcn.gather_rows(score(self.linsrc, x), edge_index[0])
                + F_mgcn.gather_rows(score(self.lintgt, x), edge_index[1]))
        if edge_attr is not None:
            gate = gate + score(self.linedge, edge_attr)
        if self.bias is not None:
            gate = gate + self.bias.view(-1, 1)
        return torch.sigmoid(gate)


class EdgeGateFree(nn.Module):
    """gcn_base_models.py:372-397: one free gate parameter per edge (fixed edge count), initialised to 1"""

    def __init__(self, num_edges):
        super().__init__()
        self.num_edges = num_edges
        self.edge_gates = Parameter(torch.ones(num_edges, 1))

    def reset_parameters(self):
        nn.init.ones_(self.edge_gates)

    def forward(self, *args, **kwargs):
        return torch.sigmoid(self.edge_gates)
