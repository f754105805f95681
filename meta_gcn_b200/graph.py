"""Row-owned adjacency structures of one ``edge_index`` and a small identity-keyed cache.

The reference walks COO ``edge_index`` with index_select / scatter_add in every layer
(gcn_base_models.py:223-237).  Here the COO list is turned ONCE per batch into two int32
structures — grouped by target (forward aggregation) and grouped by source (backward, the
transpose) — by ``mgcn_csr_build``; all layers of the model then share them.
"""
from collections import OrderedDict

import torch

from . import ops

Csr = ops.Csr

LOOPS_KEEP = 0      # edge_index used as given (gcn_meta: loops are already in the data, loop.py:13-17)
LOOPS_REMOVE = 1    # PyG remove_self_loops (GINConv)
LOOPS_ADD_REMAINING = 2  # PyG add_remaining_self_loops (GCNConv.norm, SAGEConv)


# set False to always build the by-source structure (tests compare both)
USE_SYMMETRY = True
# set False to always sort (tests compare the sort-free build of already ordered lists with it)
USE_PRESORTED = True


class GraphStructure:
    """Lazily built forward (by target) and backward (by source) structures of an edge_index."""

    def __init__(self, edge_index, num_nodes, loop_mode=LOOPS_KEEP,
                 hub_threshold=ops.DEFAULT_HUB_THRESHOLD, segments=None, recycle=None):
        if not edge_index.is_cuda:
            raise RuntimeError("GraphStructure needs a CUDA edge_index (no CPU fallback)")
        self.edge_index = edge_index
        self.num_nodes = int(num_nodes)
        self.num_edges = int(edge_index.size(1))
        self.loop_mode = int(loop_mode)
        self.hub_threshold = int(hub_threshold)
        self._fwd = None
        self._bwd = None
        self._symmetric = None
        self._facts = None
        # batch boundaries (cumulative node and edge counts per graph, host lists) when the caller knows them
        # (GraphBatch / DeviceLoader): lets an ordered batch be recognised graph by graph
        self._segments_host = segments if segments is not None and len(segments[0]) > 2 else None
        self._segments = None
        self._deg = {}
        # buffers of a dead structure of the same shape ({by: Csr}), overwritten instead of allocating (loader slots)
        self._recycle = recycle or {}

    @property
    def facts(self):
        """symmetry and order of the edge list: one device pass pair and ONE host read per edge_index
        (ops.edge_layout_impl)"""
        if self._facts is None:
            self._facts = ops.edge_layout_impl(self.edge_index, self.num_nodes, self.segments)
        return self._facts

    @property
    def segments(self):
        if self._segments is None and self._segments_host is not None:
            dev = self.edge_index.device
            self._segments = tuple(torch.tensor(list(v), dtype=torch.int32).to(dev, non_blocking=True)
                                   for v in self._segments_host)
        return self._segments

    def _build(self, by):
        layout = 0
        if USE_PRESORTED and self.loop_mode == LOOPS_KEEP and self.num_edges > 0:
            f = self.facts
            # a list in (src,dst) order groups by source without a sort; by target too when it is symmetric
            # (a batch described graph by graph: by source only — the mirror search of the by-target build is per list)
            if f["layout"] and (by == 0 or (f["symmetric"] and self.segments is None)):
                layout = f["layout"]
        # only the "+ loops" layouts need the graph boundaries: a batch whose graphs are each sorted, with their ids in
        # their own node ranges, is sorted as one list (node ids ascend from graph to graph)
        segments = self.segments if layout & 3 == 2 else None
        return ops.csr_build_impl(self.edge_index, self.num_nodes, by, self.loop_mode,
                                  self.hub_threshold, layout, segments, reuse=self._recycle.pop(by, None))

    def built(self):
        """the structures built so far (Csr objects)"""
        return [c for c in (self._fwd, self._bwd) if c is not None]

    @property
    def fwd(self):
        """rows = targets (edge_index[1]), nbr = sources: out_i = sum over incoming edges"""
        if self._fwd is None:
            self._fwd = self._build(1)
        return self._fwd

    @property
    def fwd_plain(self):
        """Structure for forward aggregations WITHOUT per-edge values or edge ids: row contents in the order of `fwd`,
        `perm` unspecified.  For a list that is in (src,dst) order and symmetric (every botnet graph of the
        reference's preprocessing) the by-source grouping has exactly these rows — sources ascending, the appended loop
        last — and needs neither a sort nor the mirror search of the exact by-target build (1.3 ms against 3.6 ms
        at the botnet batch); it is also the exact `bwd`."""
        if self._fwd is not None:
            return self._fwd
        if USE_PRESORTED and USE_SYMMETRY and self.loop_mode == LOOPS_KEEP and self.num_edges > 0:
            f = self.facts
            if f["layout"] and f["symmetric"]:
                return self.bwd
        return self.fwd

    @property
    def bwd(self):
        """rows = sources (edge_index[0]), nbr = targets: the transpose, used by autograd"""
        if self._bwd is None:
            self._bwd = self._build(0)
        return self._bwd

    @property
    def symmetric(self):
        """every (u, v) occurs as often as (v, u) — true for the reference's botnet data
        (data_procs/undirected.py:6-35).  Checked once per edge_index on the device (ops.edge_symmetry_impl)."""
        if self._symmetric is None:
            self._symmetric = USE_SYMMETRY and self.facts["symmetric"]
        return self._symmetric

    @property
    def bwd_plain(self):
        """Structure for transposed aggregations WITHOUT per-edge values: rows = sources, neighbour multisets
        only.  For a symmetric edge list that is the forward structure (same multisets per row, another order
        inside a row), so the second sort is skipped; `bwd` keeps the exact by-source structure with `perm`."""
        if self._bwd is not None:
            return self._bwd
        if self.symmetric:
            return self.fwd_plain
        return self.bwd

    def has_self_loops(self):
        """True iff edge_index holds an (i, i) entry — one device reduction and one host read per edge_index, cached"""
        if "loops" not in self._deg:
            ei = self.edge_index
            self._deg["loops"] = bool((ei[0] == ei[1]).any().item()) if self.num_edges else False
        return self._deg["loops"]

    def out_degree(self):
        """float degree over edge_index[0] (after loop handling): gcn_base_models.py:126"""
        if "out" not in self._deg:
            rowptr = self.bwd.rowptr if (self._bwd is not None or not self.symmetric) else self.fwd_plain.rowptr
            self._deg["out"] = ops.degree_impl(rowptr)
        return self._deg["out"]

    def in_degree(self):
        if "in" not in self._deg:
            self._deg["in"] = ops.degree_impl(self.fwd_plain.rowptr)
        return self._deg["in"]

    def weighted_out_degree(self, edge_weight, loop_weight=1.0):
        return ops.weighted_degree_impl(self.bwd, edge_weight, loop_weight)

    def edge_values(self, edge_weight, loop_value=1.0):
        """edge weights (input edge order) -> (forward row order, backward row order)"""
        return (ops.permute_edge_values_impl(self.fwd, edge_weight, loop_value),
                ops.permute_edge_values_impl(self.bwd, edge_weight, loop_value))

    def check_indices(self):
        """host-synchronising validation (debug entry point): raises on out-of-range endpoints"""
        if int(self.fwd.bad.item()) != 0:
            raise IndexError("edge_index contains node ids outside [0, num_nodes)")


def _version_of(t):
    """in-place modification counter; tensors created under torch.inference_mode() have none"""
    try:
        return t._version
    except RuntimeError:
        return None


class _StructureCache:
    """Keeps the structures of the last few edge_index tensors (keyed on storage identity and version counter), so
    that the L layers of a model and its backward build them once.  Each entry pins its edge_index and ~30 bytes of
    int32 structure per edge on the device, so the cache stays small: an entry is dropped as soon as the SAME
    storage shows up with a new version (a loader slot that was refilled), and at most `capacity` distinct storages
    are kept (the current batch and the one a prefetching loader is filling).  Tensors without a version counter
    (inference mode) are not cached."""

    def __init__(self, capacity=3):
        self.capacity = capacity
        self._items = OrderedDict()

    def get(self, edge_index, num_nodes, loop_mode, hub_threshold=ops.DEFAULT_HUB_THRESHOLD, segments=None,
            recycle=False):
        """recycle: when this storage was rewritten in place (a loader slot), the new structure overwrites the buffers
        of the old one instead of allocating — the caller guarantees that nothing enqueued LATER still needs the old
        structure (DeviceLoader: a slot is refilled only after its batch's step)."""
        version = _version_of(edge_index)
        if version is None:
            return GraphStructure(edge_index, num_nodes, loop_mode, hub_threshold, segments)
        ident = (edge_index.data_ptr(), edge_index.device.index)
        key = (ident, tuple(edge_index.shape), version, int(num_nodes), int(loop_mode), int(hub_threshold))
        hit = self._items.get(key)
        if hit is not None:
            self._items.move_to_end(key)
            return hit
        dead = {}
        for stale in [k for k in self._items if k[0] == ident and (k[1] != key[1] or k[2] != version)]:
            old = self._items.pop(stale)    # the storage was rewritten: its old structures are dead
            if recycle and stale[1] == key[1] and stale[3:] == key[3:]:
                if old._fwd is not None:
                    dead[1] = old._fwd
                if old._bwd is not None:
                    dead[0] = old._bwd
        gs = GraphStructure(edge_index, num_nodes, loop_mode, hub_threshold, segments, recycle=dead)
        self._items[key] = gs  # holds edge_index alive, so the data_ptr cannot be recycled
        while len(self._items) > self.capacity:
            self._items.popitem(last=False)
        return gs

    def clear(self):
        self._items.clear()


_CACHE = _StructureCache()


def structure_of(edge_index, num_nodes, loop_mode=LOOPS_KEEP,
                 hub_threshold=ops.DEFAULT_HUB_THRESHOLD, segments=None, recycle=False):
    """the (cached) GraphStructure of an edge_index.  segments = (cumulative node counts, cumulative edge counts) of
    the graphs of a batch, when known (GraphBatch.structure / DeviceLoader pass them): only consulted when the
    structure object is created"""
    return _CACHE.get(edge_index, num_nodes, loop_mode, hub_threshold, segments, recycle)


_INDEX_CACHE = OrderedDict()


def structure_of_index(index, dim_size, hub_threshold=ops.DEFAULT_HUB_THRESHOLD):
    """Structure for the primitive seam scatter_(name, src, index): rows = values of ``index``,
    perm = positions in ``index`` (a stable sort).  Cached on the identity of ``index``."""
    version = _version_of(index)
    if version is None:
        return GraphStructure(torch.stack([index, index]), dim_size, LOOPS_KEEP, hub_threshold)
    key = (index.data_ptr(), index.numel(), version, int(dim_size), int(hub_threshold),
           index.device.index)
    hit = _INDEX_CACHE.get(key)
    if hit is not None:
        _INDEX_CACHE.move_to_end(key)
        return hit[1]
    gs = GraphStructure(torch.stack([index, index]), dim_size, LOOPS_KEEP, hub_threshold)
    _INDEX_CACHE[key] = (index, gs)
    while len(_INDEX_CACHE) > 3:
        _INDEX_CACHE.popitem(last=False)
    return gs


def clear_structure_cache():
    _CACHE.clear()
    _INDEX_CACHE.clear()


_POSITIVE = OrderedDict()


def all_positive(t):
    """every entry of a device vector is > 0 and finite — one host read per (storage, version), cached.  Used by the
    hidden-32 stack: its aggregate-then-transform kernels store activations scaled by the per-source degree factor and
    need that factor to be non-zero on every gathered row, which a user-supplied degree vector (deg_K) need not give.
    Inside a CUDA-graph capture only the cached answer is available (None = unknown)."""
    version = _version_of(t)
    key = (t.data_ptr(), t.numel(), version, t.device.index)
    if version is not None and key in _POSITIVE:
        _POSITIVE.move_to_end(key)
        return _POSITIVE[key]
    if torch.cuda.is_current_stream_capturing():
        return None
    ok = bool(((t > 0) & torch.isfinite(t)).all().item())
    if version is not None:
        _POSITIVE[key] = ok
        while len(_POSITIVE) > 16:
            _POSITIVE.popitem(last=False)
    return ok
