"""ORACLE / TEST INFRASTRUCTURE ONLY — never imported by the product path (meta_gcn_b200/).

CPU restatement of the torch_scatter 1.3/1.4 API surface the reference calls
(src/gcn_meta/models/common.py:56-59,85-90; gcn_base_models.py:126; data_procs/data_add_degree.py:62-63).
torch_scatter is an un-vendored, un-pinned dependency of the reference (no requirements file); the
1.x Python source defines scatter_add as `out.scatter_add_(dim, index, src)` after broadcasting a
1-D index along `dim`, scatter_mean as add / count.clamp(min=1), and scatter_max as a custom
kernel returning (out, argmax).  Restated here with plain torch ops, CPU, deterministic.
"""
import torch


def _gen(src, index, dim, out, dim_size, fill_value):
    dim = dim if dim >= 0 else src.dim() + dim
    if index.dim() == 1:
        shape = [1] * src.dim()
        shape[dim] = src.size(dim)
        index = index.view(shape).expand_as(src)
    if out is None:
        size = list(src.size())
        if dim_size is not None:
            size[dim] = dim_size
        else:
            size[dim] = int(index.max()) + 1 if index.numel() > 0 else 0
        out = src.new_full(size, fill_value)
    return src, out, index, dim


def scatter_add(src, index, dim=-1, out=None, dim_size=None, fill_value=0):
    src, out, index, dim = _gen(src, index, dim, out, dim_size, fill_value)
    return out.scatter_add_(dim, index, src)


def scatter_mean(src, index, dim=-1, out=None, dim_size=None, fill_value=0):
    out = scatter_add(src, index, dim, out, dim_size, fill_value)
    count = scatter_add(torch.ones_like(src), index, dim, None, out.size(dim))
    return out / count.clamp(min=1)


class _ScatterMax(torch.autograd.Function):
    """torch_scatter 1.x ScatterMax: forward (out, arg) by a custom kernel, backward
    grad_src = 0; grad_src[arg[valid]] = grad_out[valid]  (the first maximal entry receives the gradient).
    `out` is not saved, so the caller may modify it in place (common.py:63-64 does)."""

    @staticmethod
    def forward(ctx, out, src, index, dim):
        init = out
        out = out.scatter_reduce(dim, index, src, reduce="amax", include_self=True)
        # argmax: first position attaining the max, -1 for untouched rows (torch_scatter 1.x); the running maximum
        # starts at the initial value and only a strictly greater entry replaces it, so an entry equal to the
        # initial value (fill_value) is never the argmax
        hit = (src == out.gather(dim, index)) & (src > init.gather(dim, index))
        pos_shape = [1] * src.dim()
        pos_shape[dim] = src.size(dim)
        pos = torch.arange(src.size(dim), device=src.device).view(pos_shape).expand_as(src)
        big = src.size(dim)
        cand = torch.where(hit, pos, torch.full_like(pos, big))
        first = index.new_full(out.size(), big).scatter_reduce(dim, index, cand, reduce="amin", include_self=True)
        arg = torch.where(first < big, first, index.new_full(out.size(), -1))
        ctx.mark_non_differentiable(arg)
        ctx.dim, ctx.src_size = dim, src.size()
        ctx.save_for_backward(arg)
        return out, arg

    @staticmethod
    def backward(ctx, grad_out, _grad_arg):
        (arg,) = ctx.saved_tensors
        valid = arg >= 0
        grad_src = grad_out.new_zeros(ctx.src_size)
        grad_src.scatter_(ctx.dim, torch.where(valid, arg, torch.zeros_like(arg)),
                          torch.where(valid, grad_out, torch.zeros_like(grad_out)), reduce="add")
        return None, grad_src, None, None


def scatter_max(src, index, dim=-1, out=None, dim_size=None, fill_value=None):
    if fill_value is None:
        fill_value = torch.finfo(src.dtype).min if src.is_floating_point() else torch.iinfo(src.dtype).min
    src, out, index, dim = _gen(src, index, dim, out, dim_size, fill_value)
    return _ScatterMax.apply(out, src, index, dim)
