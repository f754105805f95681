"""Differentiable wrappers over the mgcn kernels (what the model classes call).

Each Function's forward/backward launches libmgcn kernels only; the backward of the aggregation is
the same row-owned kernel on the structure grouped by the other endpoint (no atomics, so gradients
are deterministic — the reference's CUDA autograd uses index_add_/atomicAdd, SURVEY.md §2.2 K4).
"""
import torch

from . import ops
from .graph import GraphStructure, structure_of, structure_of_index

_ACT = {None: 0, "none": 0, "relu": 1, 0: 0, 1: 1}
_REDUCE = {"add": 0, "sum": 0, "mean": 1}


class _Aggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, bias, residual, graph, nbr_scale, row_scale, ev_fwd, ev_bwd, reduce, act, edge_weight=None):
        # edge_weight (edge_index order) is passed only when its gradient is wanted (edge gates); ev_fwd / ev_bwd are
        # its row-order copies for the two structures
        out = ops.spmm_impl(graph.fwd if ev_fwd is not None else graph.fwd_plain, x, False, ev_fwd, nbr_scale, row_scale, reduce, bias,
                            residual, act)
        ctx.graph = graph
        ctx.cfg = (reduce, act, bias is not None, residual is not None)
        want_dw = edge_weight is not None and edge_weight.requires_grad
        ctx.want_dw = want_dw
        ctx.save_for_backward(out if act else None, nbr_scale, row_scale, ev_bwd, x if want_dw else None)
        return out

    @staticmethod
    def backward(ctx, g):
        out, nbr_scale, row_scale, ev_bwd, x = ctx.saved_tensors
        reduce, act, has_bias, has_res = ctx.cfg
        graph = ctx.graph
        g = g.contiguous()
        if act:
            g = ops.relu_backward_impl(g, out)
        d_bias = g.sum(0) if (has_bias and ctx.needs_input_grad[1]) else None
        d_res = g if (has_res and ctx.needs_input_grad[2]) else None
        dx = d_ew = None
        gg = g
        if reduce == 1 and (ctx.needs_input_grad[0] or ctx.want_dw):
            gg = g / graph.in_degree().clamp(min=1).unsqueeze(1)
        if ctx.needs_input_grad[0]:
            # transpose: rows = sources; the per-target factor is now gathered, the per-source
            # factor scales the row
            dx = ops.spmm_impl(graph.bwd if ev_bwd is not None else graph.bwd_plain, gg, False, ev_bwd, row_scale, nbr_scale, 0, None,
                               None, 0)
        if ctx.want_dw:
            # d w_e = nbr_scale[row_e] * row_scale[col_e] * <g[col_e], x[row_e]>
            d_ew = ops.edge_dot_impl(graph.edge_index, gg, x, nbr_scale, row_scale)
        return dx, d_bias, d_res, None, None, None, None, None, None, None, d_ew


def aggregate(x, graph, nbr_scale=None, row_scale=None, edge_weight=None, reduce="add", bias=None,
              residual=None, act=None, loop_value=1.0):
    """out_i = act( reduce_{e: target(e)=i}  x[source(e)] * w_e  + bias + residual_i ),
    w_e = nbr_scale[source] * edge_weight[e] * row_scale[target]   (gcn_base_models.py:138-139,
    223-240).  ``graph`` is a GraphStructure; edge_weight is in edge_index order and may require grad (edge
    gates, gcn_base_models.py:230-232)."""
    ev_fwd = ev_bwd = None
    if edge_weight is not None:
        ev_fwd, ev_bwd = graph.edge_values(edge_weight.detach(), loop_value)
    return _Aggregate.apply(x, bias, residual, graph, nbr_scale, row_scale, ev_fwd, ev_bwd,
                            _REDUCE[reduce], _ACT[act],
                            edge_weight if (edge_weight is not None and edge_weight.requires_grad) else None)


class _AggregateMax(torch.autograd.Function):
    """out_i = max_e x[source(e)] * w_e over the edges into i (0 for a node without edges); gradient to the first
    maximal edge (torch_scatter scatter_max), accumulated per source by a row-owned pass over the by-source
    structure"""

    @staticmethod
    def forward(ctx, x, graph, ev_fwd, ev_bwd, fill):
        out, arg = ops.segment_max_impl(graph.fwd, x, False, ev_fwd, fill)
        ctx.graph = graph
        ctx.save_for_backward(arg, ev_bwd)
        ctx.mark_non_differentiable(arg)
        return out, arg

    @staticmethod
    def backward(ctx, g, _garg):
        arg, ev_bwd = ctx.saved_tensors
        dx = ops.segment_max_bwd_impl(ctx.graph.bwd, g.contiguous(), arg, ev_bwd) if ctx.needs_input_grad[0] else None
        return dx, None, None, None, None


def aggregate_max(x, graph, edge_weight=None, loop_value=1.0, fill=-1e38):
    """NodeModelAdditive(aggr='max') (gcn_base_models.py:223-237): max over incoming edges of x[row] * norm_e;
    edge_weight = the per-edge factor norm[E] in edge_index order (or None).  As scatter_('max') of common.py:54-64,
    an entry <= fill (-1e38) never wins, and a (node, column) without a winner is 0 and receives no gradient."""
    ev_fwd = ev_bwd = None
    if edge_weight is not None:
        ev_fwd, ev_bwd = graph.edge_values(edge_weight, loop_value)
    return _AggregateMax.apply(x, graph, ev_fwd, ev_bwd, fill)[0]


class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, bias, add, w_out_in, act):
        y = ops.linear_impl(x, w, w_out_in, bias, add, act)
        ctx.cfg = (w_out_in, act, bias is not None, add is not None)
        ctx.save_for_backward(x, w, y if act else None)
        return y

    @staticmethod
    def backward(ctx, g):
        x, w, y = ctx.saved_tensors
        w_out_in, act, has_bias, has_add = ctx.cfg
        g = g.contiguous()
        if act:
            g = ops.relu_backward_impl(g, y)
        dx = dw = db = dadd = None
        if ctx.needs_input_grad[0]:
            # dX = G W^T: the same kernel with the weight read through swapped strides
            dx = ops.linear_impl(g, w, not w_out_in, None, None, 0)
        if ctx.needs_input_grad[1] or (has_bias and ctx.needs_input_grad[2]):
            dw, db_ = ops.linear_wgrad_impl(x, g, w_out_in, has_bias)
            db = db_ if has_bias else None
        if has_add and ctx.needs_input_grad[3]:
            dadd = g
        return dx, dw, db, dadd, None, None


class _HeadCrossEntropy(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, target, mean, want_counts):
        x = x.contiguous()
        logits, loss, counts, _bad = ops.head_cross_entropy_fwd_impl(x, weight, bias, target, mean, want_counts)
        ctx.mean = bool(mean)
        ctx.has_bias = bias is not None
        ctx.save_for_backward(x, logits, weight, target)
        # one call: each call replaces the set of non-differentiable outputs
        if counts is not None:
            ctx.mark_non_differentiable(logits, counts)
            return loss.view(()), logits, counts
        ctx.mark_non_differentiable(logits)
        return loss.view(()), logits

    @staticmethod
    def backward(ctx, g, *_unused):
        x, logits, weight, target = ctx.saved_tensors
        dx, dw, db = ops.head_cross_entropy_bwd_impl(x, logits, weight, target, ctx.mean, g.contiguous().view(1),
                                                     ctx.needs_input_grad[0])
        return dx, dw, db if ctx.has_bias else None, None, None, None


def head_cross_entropy(x, linear, target, reduction="mean", confusion=False):
    """``CrossEntropyLoss(reduction)(linear(x), target)`` with the output layer, the loss and (optionally) the binary
    counters TP / FP / TN / FN / correct of optim/metrics.py:8-24 in one forward and one backward launch
    (csrc/head.cu; gcn_model.py:73,108 + train_botnet.py:287,296-305).  ``linear``: an nn.Linear(H, C), H in
    {16,32,64,128}, C <= 8.  Returns (loss, logits[, counts int64[5]]); the logits are detached (the loss carries the
    gradient to x and to the layer's parameters).  A label outside [0, C) (-100 included) makes the loss NaN and that
    row's gradient NaN, and the counters skip the row; the mean over no rows is NaN (include/mgcn.h)."""
    if reduction not in ("mean", "sum"):
        raise ValueError("reduction must be 'mean' or 'sum'")
    return _HeadCrossEntropy.apply(x, linear.weight, linear.bias, target, reduction == "mean", bool(confusion))


class _BatchNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, training, momentum, eps):
        y, mean, rstd = ops.batchnorm_fwd_impl(x, gamma, beta, running_mean, running_var, training, momentum, eps)
        ctx.training = bool(training)
        ctx.save_for_backward(x, gamma, mean, rstd)
        return y

    @staticmethod
    def backward(ctx, g):
        x, gamma, mean, rstd = ctx.saved_tensors
        dx, dgamma, dbeta = ops.batchnorm_bwd_impl(x, g.contiguous(), gamma, mean, rstd, ctx.training,
                                                   ctx.needs_input_grad[0])
        return (dx, dgamma if gamma is not None else None, dbeta if gamma is not None else None, None, None, None,
                None, None)


def batch_norm(x, bn, training=None):
    """torch.nn.BatchNorm1d ``bn`` applied to x [N,H] by the fixed-order kernels of csrc/batchnorm.cu (kernel/gin.py:15);
    running statistics and num_batches_tracked are updated as torch does in training mode"""
    training = bn.training if training is None else training
    use_batch = training or not bn.track_running_stats
    momentum = 0.0 if bn.momentum is None else bn.momentum
    if training and bn.track_running_stats:
        bn.num_batches_tracked += 1
        if bn.momentum is None:
            momentum = 1.0 / float(bn.num_batches_tracked)
    return _BatchNorm.apply(x, bn.weight, bn.bias, bn.running_mean if bn.track_running_stats else None,
                            bn.running_var if bn.track_running_stats else None, use_batch, momentum, bn.eps)


def linear(x, weight, bias=None, add=None, act=None, weight_layout="in_out"):
    """y = act(x @ W + bias + add).  weight_layout 'in_out': weight_node [Hi,Ho]
    (gcn_base_models.py:201); 'out_in': nn.Linear.weight [Ho,Hi] (gcn_model.py:64,73)."""
    return _Linear.apply(x, weight, bias, add, weight_layout == "out_in", _ACT[act])


class _SegmentReduce(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, offsets, mode):
        ctx.mode = mode
        ctx.n = x.size(0)
        ctx.save_for_backward(offsets)
        return ops.segment_reduce_impl(x, offsets, mode)

    @staticmethod
    def backward(ctx, g):
        (offsets,) = ctx.saved_tensors
        return ops.segment_broadcast_impl(g.contiguous(), offsets, ctx.n, ctx.mode), None, None


def segment_pool(x, offsets, reduce="mean"):
    """per-graph sum/mean over contiguous node ranges (global_mean_pool, kernel/gcn.py:29)"""
    return _SegmentReduce.apply(x, offsets, _REDUCE[reduce])


def pool_by_batch(x, batch, size=None, reduce="mean"):
    """global_{mean,add}_pool(x, batch, size): batch is sorted ascending (Batch.from_data_list)."""
    if size is None:
        size = int(batch.max().item()) + 1 if batch.numel() else 0  # same host sync as PyG
    offsets = ops.batch_to_offsets_impl(batch, size)
    return segment_pool(x, offsets, reduce)


class _ScatterRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, graph, index, reduce):
        out = ops.spmm_impl(graph.fwd, src, True, None, None, None, reduce, None, None, 0)
        ctx.graph = graph
        ctx.reduce = reduce
        ctx.save_for_backward(index)
        return out

    @staticmethod
    def backward(ctx, g):
        (index,) = ctx.saved_tensors
        if ctx.reduce == 1:
            g = g / ctx.graph.in_degree().clamp(min=1).unsqueeze(1)
        return g.index_select(0, index), None, None, None


class _ScatterRowsMax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, graph, fill):
        out, arg = ops.segment_max_impl(graph.fwd, src, True, None, fill)
        ctx.n_src = src.size(0)
        ctx.save_for_backward(arg)
        ctx.mark_non_differentiable(arg)
        return out, arg

    @staticmethod
    def backward(ctx, g, _garg):
        (arg,) = ctx.saved_tensors
        return ops.scatter_max_bwd_impl(arg, g.contiguous(), ctx.n_src), None, None


def scatter_rows_max(src, index, dim_size=None, fill=-1e38):
    """scatter_('max', src, index, dim_size) (common.py:54-64) -> (out, argmax) with torch_scatter's fill rule: an
    entry <= fill never wins; a (row, column) without a winner (no entries, or all <= fill) is 0 / -1.  The default is
    common.py's fill; other callers pass the fill of the call they stand for."""
    squeeze = src.dim() == 1
    src2 = src.unsqueeze(1) if squeeze else src.reshape(src.size(0), -1)
    if dim_size is None:
        dim_size = int(index.max().item()) + 1 if index.numel() else 0
    graph = structure_of_index(index, dim_size)
    out, arg = _ScatterRowsMax.apply(src2, graph, fill)
    if squeeze:
        return out.squeeze(1), arg.squeeze(1).long()
    return out.reshape(dim_size, *src.shape[1:]), arg.reshape(dim_size, *src.shape[1:]).long()


def scatter_rows(src, index, dim_size=None, reduce="add"):
    """Primitive seam: scatter_('add'|'mean', src[E,H], index[E], dim_size) (common.py:37-66) as a
    deterministic row-owned gather-sum over a stable sort of ``index``."""
    squeeze = src.dim() == 1
    src2 = src.unsqueeze(1) if squeeze else src
    if src2.dim() != 2:
        src2 = src2.reshape(src2.size(0), -1)
    if dim_size is None:
        dim_size = int(index.max().item()) + 1 if index.numel() else 0
    graph = structure_of_index(index, dim_size)
    out = _ScatterRows.apply(src2, graph, index, _REDUCE[reduce])
    if squeeze:
        return out.squeeze(1)
    return out.reshape(dim_size, *src.shape[1:])


class _GatherRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, index):
        ctx.n_src = src.size(0)
        ctx.save_for_backward(index)
        return src.index_select(0, index)

    @staticmethod
    def backward(ctx, g):
        (index,) = ctx.saved_tensors
        return scatter_rows(g.contiguous(), index, ctx.n_src, "add") if ctx.needs_input_grad[0] else None, None


def gather_rows(src, index):
    """src.index_select(0, index) whose gradient is summed per source row by the row-owned scatter kernel
    (scatter_rows) instead of index_select's atomicAdd backward: deterministic, and the same for int32 and int64
    indices.  Used for per-edge gathers of node tensors that require grad (edge-gate scores, attention scores,
    the messages of the 'max' aggregation with gates or edge features)."""
    return _GatherRows.apply(src, index)


class _CrossEntropy(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, target, mean):
        loss, _bad = ops.cross_entropy_fwd_impl(logits, target, mean)
        ctx.mean = mean
        ctx.save_for_backward(logits, target)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        logits, target = ctx.saved_tensors
        return ops.cross_entropy_bwd_impl(logits, target, ctx.mean, g.contiguous()), None, None


def cross_entropy(logits, target, reduction="mean"):
    """nn.CrossEntropyLoss(reduction=...)(logits, target) over node logits (train_botnet.py:225,287)
    as two deterministic kernels; target is int64 class ids.  A label outside [0, C) (-100 included: there is no
    ignore_index) makes the loss NaN and that row's gradient NaN, without a host synchronisation; the mean over no
    rows is NaN, as torch's."""
    if reduction not in ("mean", "sum"):
        raise ValueError("reduction must be 'mean' or 'sum'")
    return _CrossEntropy.apply(logits, target, reduction == "mean")
