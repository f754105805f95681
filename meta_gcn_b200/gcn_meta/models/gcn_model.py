"""Mirror of src/gcn_meta/models/gcn_model.py: ``GCNModel`` (stack of layers + residual Linear every
``residual_hop`` + final projection + optional per-graph mean, gcn_model.py:8-125) and ``GCNLayer``
(gcn_model.py:128-197), with the same constructor kwargs and parameter names
(gcn_net.N.gcn.node_models.K.weight_node, residuals.N.weight/bias, final.weight/bias).

What changes underneath: the edge_index -> row structure build and the degree factors are done once
per forward and shared by all layers; ReLU after the aggregation is fused into its epilogue; the
residual Linear, the add and the outer ReLU are one narrow-transform launch."""
import torch
import torch.nn as nn

from ... import functional as F_mgcn
from ... import fused
from ...graph import all_positive, structure_of
from .common import activation
from .gcn_base_models import NodeModelBase
from .gcn_multi_kernel import GCNMultiKernel


def _stack_gate(nm):
    """edge gate of a node model as the residual stack sees it: None (no gate), True (EdgeGateProj on node scores only,
    with its bias: the stack's gated kernels) or False (any other gate: the per-layer path)"""
    eg = nm.edge_gate
    if eg is None:
        return None
    return type(eg).__name__ == "EdgeGateProj" and eg.in_edgedim is None and eg.bias is not None


class GCNLayer(nn.Module):
    def __init__(self, in_channels, out_channels, in_edgedim=None, deg_norm="sm", edge_gate=None,
                 aggr="add", bias=True, num_kernel=1, nodemodel="additive", non_linear="relu", **kwargs):
        super().__init__()
        self.gcn = GCNMultiKernel(in_channels, out_channels, in_edgedim, deg_norm=deg_norm,
                                  edge_gate=edge_gate, aggr=aggr, bias=bias, num_kernel=num_kernel,
                                  nodemodel=nodemodel, **kwargs)
        self.non_linear = activation(non_linear)
        self._act_name = non_linear

    def reset_parameters(self):
        self.gcn.reset_parameters()

    def forward(self, x, edge_index_K, edge_attr_K=None, deg_K=None, edge_weight_K=None, **kwargs):
        if self._act_name == "relu":
            return self.gcn(x, edge_index_K, edge_attr_K, deg_K, edge_weight_K, _act="relu", **kwargs)
        xo = self.gcn(x, edge_index_K, edge_attr_K, deg_K, edge_weight_K, **kwargs)
        return self.non_linear(xo)


class GCNModel(nn.Module):
    def __init__(self, in_channels, enc_sizes, num_classes, non_linear="relu",
                 non_linear_layer_wise="relu", residual_hop=None, dropout=0.5, final_layer_config=None,
                 final_type="none", pred_on="node", **kwargs):
        assert final_type in ["none", "proj"]
        assert pred_on in ["node", "graph"]
        super().__init__()
        self.in_channels = in_channels
        self.enc_sizes = [in_channels, *enc_sizes]
        self.num_layers = len(self.enc_sizes) - 1
        self.num_classes = num_classes
        self.residual_hop = residual_hop
        self.non_linear_layer_wise = non_linear_layer_wise
        self.final_type = final_type
        self.pred_on = pred_on
        nheads = kwargs.pop("nheads", 1)
        self.nheads = [nheads] * self.num_layers if isinstance(nheads, int) else list(nheads)
        assert len(self.nheads) == self.num_layers
        # attention-only kwargs of the reference CLI are accepted and ignored by the additive model
        pairs = list(zip(self.enc_sizes, self.enc_sizes[1:]))
        layers = []
        for i, (cin, cout) in enumerate(pairs):
            kw = dict(kwargs)
            if final_layer_config is not None and i == len(pairs) - 1:
                assert isinstance(final_layer_config, dict)
                kw.update(final_layer_config)
            layers.append(GCNLayer(cin, cout, nheads=self.nheads[i], non_linear=non_linear_layer_wise, **kw))
        self.gcn_net = nn.ModuleList(layers)
        self.dropout = nn.Dropout(dropout)
        if residual_hop is not None and residual_hop > 0:
            srcs = range(0, len(self.enc_sizes), residual_hop)
            dsts = range(residual_hop, len(self.enc_sizes), residual_hop)
            self.residuals = nn.ModuleList(
                [nn.Linear(self.enc_sizes[i], self.enc_sizes[j]) for i, j in zip(srcs, dsts)])
            self.non_linear = activation(non_linear)
            self._res_act = non_linear
            self.num_residuals = len(self.residuals)
        self.final = nn.Linear(self.enc_sizes[-1], num_classes) if final_type == "proj" else nn.Identity()

    def reset_parameters(self):
        for net in self.gcn_net:
            net.reset_parameters()
        if self.residual_hop is not None:
            for net in self.residuals:
                net.reset_parameters()
        if self.final_type != "none":
            self.final.reset_parameters()

    def _shared_degree_factors(self, x, edge_index_K, deg_K, edge_weight_K):
        """dis[N] once per forward when all layers see one edge set with one degree vector (the
        reference recomputes norm[E] in every layer: gcn_base_models.py:215)."""
        ei = edge_index_K if isinstance(edge_index_K, torch.Tensor) else (
            edge_index_K[0] if len(edge_index_K) == 1 else None)
        if ei is None:
            return None
        nm = self.gcn_net[0].gcn.node_models[0]
        if nm.deg_norm is None:
            return None
        # one vector serves every layer only if every node model normalises the same way (final_layer_config may
        # override deg_norm for the last layer: the reference recomputes norm per layer with that layer's own method,
        # gcn_base_models.py:215); otherwise each layer derives its own factors
        for layer in self.gcn_net:
            if any(getattr(m, "deg_norm", None) != nm.deg_norm for m in layer.gcn.node_models):
                return None
        deg = deg_K if isinstance(deg_K, torch.Tensor) or deg_K is None else deg_K[0]
        ew = edge_weight_K if isinstance(edge_weight_K, torch.Tensor) or edge_weight_K is None \
            else edge_weight_K[0]
        return NodeModelBase.degree_factors(ei, x.size(0), deg, ew, nm.deg_norm)

    def _stack_eligible(self, edge_index_K, edge_attr_K, edge_weight_K):
        """the whole-stack path covers the botnet configuration family (train_botnet.py:200-212):
        one edge set, additive node models, residual every layer, ReLU/ReLU, sum aggregation, dropout p < 1
        (p = 1 drops everything: torch's dropout returns zeros, the per-layer path keeps that)"""
        if self.residual_hop != 1 or getattr(self, "num_residuals", 0) != self.num_layers:
            return False
        if self.non_linear_layer_wise != "relu" or self._res_act != "relu":
            return False
        if self.training and self.dropout.p >= 1:
            return False
        if edge_attr_K is not None or edge_weight_K is not None:
            return False
        if not isinstance(edge_index_K, torch.Tensor):
            if len(edge_index_K) != 1:
                return False
        if any(w not in fused.FUSED_WIDTHS for w in self.enc_sizes[1:]):
            return False
        nms = [layer.gcn.node_models for layer in self.gcn_net]
        if any(len(m) != 1 or layer.gcn.kernel_combine != "add" for m, layer in zip(nms, self.gcn_net)):
            return False
        first = nms[0][0]
        return all(type(m[0]).__name__ == "NodeModelAdditive" and m[0].aggr == "add" and m[0].deg_norm == first.deg_norm and m[0].in_edgedim is None
                   and (m[0].bias is None) == (first.bias is None)
                   and _stack_gate(m[0]) is not False and _stack_gate(m[0]) == _stack_gate(first) for m in nms)

    def _forward_stack(self, x, edge_index, dis, deg=None):
        nm0 = self.gcn_net[0].gcn.node_models[0]
        graph = structure_of(edge_index, x.size(0))
        # the aggregate-then-transform kernels need a non-zero degree factor on every gathered row: true by construction
        # for the graph's own out-degree (a source has an out-edge), checked once per tensor for a caller's deg_K
        aggregate_first = True
        if deg is not None and dis is not None:
            aggregate_first = all_positive(deg) is True
        pre = dis
        post = dis if nm0.deg_norm == "sm" else None
        has_bias = nm0.bias is not None
        gated = _stack_gate(nm0) is True
        params = []
        for layer, lin in zip(self.gcn_net, self.residuals):
            nm = layer.gcn.node_models[0]
            eg = nm.edge_gate
            params.append((nm.weight_node,) + ((nm.bias,) if has_bias else ())
                          + ((eg.linsrc.weight, eg.lintgt.weight, eg.bias) if gated else ()) + (lin.weight, lin.bias))
        # None: the stack chosen for these inputs does not take dropout or gates (fused.residual_gcn_stack)
        return fused.residual_gcn_stack(x, graph, pre, post, params, has_bias, aggregate_first=aggregate_first,
                                        dropout=self.dropout.p if self.training else 0.0, gated=gated)

    def forward(self, x, edge_index_K, edge_attr_K=None, deg_K=None, edge_weight_K=None, **kwargs):
        hidden = kwargs.pop("_hidden", False)        # forward_loss: stop before the output layer
        dis = self._shared_degree_factors(x, edge_index_K, deg_K, edge_weight_K)
        if self._stack_eligible(edge_index_K, edge_attr_K, edge_weight_K) and not kwargs.get("_no_stack"):
            ei = edge_index_K if isinstance(edge_index_K, torch.Tensor) else edge_index_K[0]
            deg = deg_K if isinstance(deg_K, torch.Tensor) or deg_K is None else deg_K[0]
            out = self._forward_stack(x, ei, dis, deg)
            if out is not None:
                return out if hidden else self._head(out, kwargs)
        kwargs.pop("_no_stack", None)
        hop = self.residual_hop
        xr_src, add_xr_at, res_idx = None, -1, -1
        for n, net in enumerate(self.gcn_net):
            xo = net(x, edge_index_K, edge_attr_K, deg_K, edge_weight_K, _dis=dis, **kwargs)
            xo = self.dropout(xo)
            if hop is not None and hop > 0:
                if n % hop == 0 and (n // hop) < self.num_residuals:
                    xr_src, res_idx = x, n // hop     # residual branch reads this layer's input
                    add_xr_at = n + hop - 1
                if n == add_xr_at:
                    lin = self.residuals[res_idx]
                    last = n == self.num_layers - 1
                    fuse_relu = (not last) and self._res_act == "relu"
                    # relu(xo + Linear(x)) in one launch (gcn_model.py:96-105)
                    xo = F_mgcn.linear(xr_src, lin.weight, lin.bias, add=xo,
                                       act="relu" if fuse_relu else None, weight_layout="out_in")
                    if not last and not fuse_relu:
                        xo = self.non_linear(xo)
            x = xo
        return x if hidden else self._head(x, kwargs)

    def forward_loss(self, x, edge_index_K, target, edge_attr_K=None, deg_K=None, edge_weight_K=None,
                     reduction="mean", confusion=False, **kwargs):
        """forward + ``nn.CrossEntropyLoss(reduction)`` in one call: for node-level models with a 'proj' output layer
        the output Linear, the loss and (``confusion=True``) the binary counters of optim/metrics.py run as ONE launch
        (functional.head_cross_entropy; train_botnet.py:286-305 makes five passes and five host reads of them).
        Returns (loss, logits[, counts]) — same values as ``forward`` followed by the loss."""
        fusable = (self.final_type == "proj" and self.pred_on == "node" and self.final.in_features in (16, 32, 64, 128)
                   and self.final.out_features <= 8)
        if not fusable:
            out = self.forward(x, edge_index_K, edge_attr_K, deg_K, edge_weight_K, **kwargs)
            loss = F_mgcn.cross_entropy(out, target, reduction)
            if confusion:
                from ... import ops
                return loss, out, ops.binary_confusion_impl(target, logits=out.detach())
            return loss, out
        h = self.forward(x, edge_index_K, edge_attr_K, deg_K, edge_weight_K, _hidden=True, **kwargs)
        return F_mgcn.head_cross_entropy(h, self.final, target, reduction, confusion)

    def _head(self, x, kwargs):
        if self.final_type == "proj":
            x = F_mgcn.linear(x, self.final.weight, self.final.bias, weight_layout="out_in")
        if self.pred_on == "graph":
            assert "batch_slices_x" in kwargs
            sl = kwargs["batch_slices_x"]
            if torch.is_tensor(sl) and sl.is_cuda:
                offsets = sl.to(torch.int32)           # device offsets: no host traffic, capture-safe
            else:
                # the boundaries of a batch as a device vector, uploaded once per distinct batch (a pageable copy per
                # forward would synchronise the step and cannot be captured in a CUDA graph)
                key = (tuple(int(v) for v in sl), x.device)
                cache = self.__dict__.setdefault("_offsets_cache", {})
                offsets = cache.get(key)
                if offsets is None:
                    if len(cache) >= 8:
                        cache.pop(next(iter(cache)))
                    offsets = torch.as_tensor(key[0], dtype=torch.int32).to(x.device)
                    cache[key] = offsets
            x = F_mgcn.segment_pool(x, offsets, "mean")
        return x
