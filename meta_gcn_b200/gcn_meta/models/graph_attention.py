"""Mirror of src/gcn_meta/models/graph_attention.py:11-117 (NodeModelAttention, multi-head soft attention over a
node's neighbourhood) on the libmgcn building blocks — same constructor arguments and parameter names (``weight``,
``att_weight``, ``bias``).

    x      = x W                                   -> [N, heads, C1]                  (mgcn linear)
    alpha  = act( <x_j, a_src> + <x_i, a_tgt> )    per edge and head                  (two [N, heads] projections,
                                                                                       gathered per edge)
    alpha  = softmax over the edges of each target (att_dir='in') / source ('out')   (common.softmax: segment max +
                                                                                       segment sum, csrc/segmax.cu, spmm.cu)
    out_i  = sum_e alpha_e x_j                      per head                           (mgcn aggregation with a
                                                                                       differentiable per-edge weight,
                                                                                       gradient through mgcn_edge_dot)
The reference materialises [E, heads, C1] messages twice; here only [E, heads] scalars exist per edge."""
import torch
import torch.nn as nn
from torch.nn import Parameter

from ... import functional as F_mgcn
from ...compat.torch_geometric.nn.inits import glorot, zeros
from ...graph import structure_of
from .common import activation, softmax
from .gcn_base_models import NodeModelBase


class NodeModelAttention(NodeModelBase):
    _ACTS = ("none", "lrelu", "relu")
    _COMBINE = ("cat", "add", "mean")

    def __init__(self, in_channels, out_channels, in_edgedim=None, nheads=1, att_act="none", att_dropout=0,
                 att_combine="cat", att_dir="in", bias=False, **kwargs):
        if att_act not in self._ACTS or att_combine not in self._COMBINE or att_dir not in ("in", "out"):
            raise AssertionError((att_act, att_combine, att_dir))
        super().__init__(in_channels, out_channels, in_edgedim)     # deg_norm / edge_gate / aggr keep their defaults
        self.nheads, self.att_combine, self.att_dir = nheads, att_combine, att_dir
        concat = att_combine == "cat"
        # 'cat': the heads share out_channels; 'add' / 'mean': every head is out_channels wide (graph_attention.py:31-45)
        self.out_channels_1head = out_channels // nheads if concat else out_channels
        if concat and self.out_channels_1head * nheads != out_channels:
            raise AssertionError("out_channels should be divisible by nheads")
        # parameters in the reference's creation order (same RNG stream -> same initial values)
        self.weight = Parameter(torch.empty(in_channels, self.out_channels_1head * nheads))
        self.att_weight = Parameter(torch.empty(1, nheads, 2 * self.out_channels_1head))
        self.att_act = activation(att_act)
        self.att_dropout = nn.Dropout(p=att_dropout)
        self.register_parameter("bias", Parameter(torch.empty(out_channels)) if bias else None)
        self.reset_parameters()

    def reset_parameters(self):
        for t in (self.weight, self.att_weight):
            glorot(t)
        zeros(self.bias)

    def forward(self, x, edge_index, edge_attr=None, deg=None, edge_weight=None, attn_store=None, **kwargs):
        """'deg' and 'edge_weight' are not used (graph_attention.py:60-62)"""
        act = kwargs.get("_act")
        n, nh, c1 = x.size(0), self.nheads, self.out_channels_1head
        graph = structure_of(edge_index, n)
        xv = F_mgcn.linear(x, self.weight).view(n, nh, c1)                          # :64
        a = self.att_weight.view(nh, 2 * c1)
        s_src = (xv * a[:, :c1]).sum(-1)                                             # <x_j, a_src>   [N, heads]
        s_tgt = (xv * a[:, c1:]).sum(-1)                                             # <x_i, a_tgt>
        row, col = edge_index[0], edge_index[1]
        alpha = self.att_act(F_mgcn.gather_rows(s_src, row) + F_mgcn.gather_rows(s_tgt, col))   # :71   [E, heads]
        alpha = softmax(alpha, row if self.att_dir == "out" else col, num_nodes=n)      # :74-79
        alpha = self.att_dropout(alpha)                                              # :82
        heads = [F_mgcn.aggregate(xv[:, h, :].contiguous(), graph, None, None, alpha[:, h].contiguous(), self.aggr)
                 for h in range(nh)]                                                 # :97-100
        if self.att_combine == "cat":
            out = torch.cat(heads, dim=1) if nh > 1 else heads[0]
        else:
            out = heads[0]
            for o in heads[1:]:
                out = out + o
            if self.att_combine == "mean":
                out = out / nh
        if self.bias is not None:
            out = out + self.bias
        if attn_store is not None:
            attn_store.append(alpha)
        return torch.relu(out) if act == "relu" else out

    def extra_repr(self):
        return (f"{self.in_channels} -> {self.out_channels}, heads={self.nheads}, combine={self.att_combine}, "
                f"dir={self.att_dir}, att_dropout={self.att_dropout.p}")
