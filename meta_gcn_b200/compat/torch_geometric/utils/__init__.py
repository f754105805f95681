"""``torch_geometric.utils`` names on the hot path: ``scatter_`` (graph_attention.py:5 imports it at
module load; PyG's MessagePassing uses it) and ``degree`` (kernel/datasets.py:16)."""
from .... import functional as F_mgcn
from .... import ops
from ....graph import structure_of_index


def scatter_(name, src, index, dim_size=None):
    """PyG 1.3 utils.scatter_: 'add' | 'mean' | 'max' along dim 0; 'max' is torch_scatter's scatter_max from the fill
    value -1e9, whose untouched entries are then replaced by 0 — what the first-maximum kernel with that fill writes"""
    assert name in ["add", "mean", "max"]
    if name == "max":
        return F_mgcn.scatter_rows_max(src, index, dim_size, fill=-1e9)[0]
    return F_mgcn.scatter_rows(src, index, dim_size, name)


def degree(index, num_nodes=None, dtype=None):
    if num_nodes is None:
        num_nodes = int(index.max().item()) + 1 if index.numel() else 0
    deg = ops.degree_impl(structure_of_index(index, num_nodes).fwd.rowptr)
    return deg if dtype is None else deg.to(dtype)
