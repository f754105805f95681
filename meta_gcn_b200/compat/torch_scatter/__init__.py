"""``torch_scatter`` names used on the hot path (common.py:56-59, gcn_base_models.py:126), on libmgcn.
dim must be 0 (the only use in the reference); CUDA only."""
from ... import functional as F_mgcn


def _check(dim, out, fill_value):
    if dim not in (0,):
        raise NotImplementedError("mgcn scatter ops aggregate along dim 0 only")
    if fill_value != 0:
        raise NotImplementedError("fill_value != 0 is only used by scatter_max (out of scope)")


def scatter_add(src, index, dim=-1, out=None, dim_size=None, fill_value=0):
    if src.dim() == 1 and dim == -1:
        dim = 0
    _check(dim, out, fill_value)
    res = F_mgcn.scatter_rows(src, index, dim_size if out is None else out.size(0), "add")
    return res if out is None else out + res


def scatter_mean(src, index, dim=-1, out=None, dim_size=None, fill_value=0):
    if src.dim() == 1 and dim == -1:
        dim = 0
    _check(dim, out, fill_value)
    if out is not None:
        raise NotImplementedError("scatter_mean(out=...) is not used by the reference")
    return F_mgcn.scatter_rows(src, index, dim_size, "mean")


def scatter_max(src, index, dim=-1, out=None, dim_size=None, fill_value=None):
    """torch_scatter 1.x scatter_max along dim 0 -> (out, argmax): out = max(fill_value, entries), argmax = the first
    entry strictly greater than fill_value that attains it, -1 (and out = fill_value) where no entry exceeds fill_value
    (common.py:56-57 passes -1e38 and zeroes those rows afterwards)"""
    import torch
    if src.dim() == 1 and dim == -1:
        dim = 0
    if dim != 0:
        raise NotImplementedError("mgcn scatter ops aggregate along dim 0 only")
    if out is not None:
        raise NotImplementedError("scatter_max(out=...) is not used by the reference")
    if fill_value is None:
        fill_value = torch.finfo(src.dtype).min
    res, arg = F_mgcn.scatter_rows_max(src, index, dim_size, fill=fill_value)
    return torch.where(arg < 0, torch.full_like(res, fill_value), res), arg
