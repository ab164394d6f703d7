"""Edge builders - the reference's plugin interface for the edge-construction path.

Mirrors /root/reference/src/anemoi/graphs/edges/builder.py (``BaseEdgeBuilder`` :42-156,
``NodeMaskingMixin`` :159-193, ``KNNEdges`` :196-270, ``CutOffEdges`` :273-371, ``MultiScaleEdges``
:374-462): same constructor arguments, assertion messages, method names and graph side effects.  The
sklearn / networkx internals are replaced by the CUDA kernels behind ``ops`` (cube-sphere cell-binned
neighbour search, count-scan-fill cut-off, CSR frontier expansion on the icosphere).

Differences a caller can observe, all inside what the reference leaves unspecified:
* edge ORDER within an edge set (KNN: by target, then ascending (distance, source); cut-off: by target,
  cell-scan order; multi-scale: sorted by (target, source)) - the reference's orders are sklearn tree /
  networkx insertion orders;
* exact float64 distance ties at the k-th KNN boundary go to the lower source index (the reference keeps
  whichever its ball tree visits first, sklearn/utils/_heap.pyx:46);
* tensors are returned on the device the node coordinates live on (CPU in, CPU out).
"""

from __future__ import annotations

import logging
from abc import ABC

import numpy as np
import torch

from .. import EARTH_RADIUS
from .. import device as _device
from .. import ops
from ..config import DotDict
from ..config import instantiate
from ..utils import concat_edges_device
from ..utils import get_grid_reference_distance

LOGGER = logging.getLogger(__name__)


class BaseEdgeBuilder(ABC):
    """Base class for edge builders."""

    def __init__(
        self,
        source_name: str,
        target_name: str,
        source_mask_attr_name: str | None = None,
        target_mask_attr_name: str | None = None,
    ):
        self.source_name = source_name
        self.target_name = target_name
        self.source_mask_attr_name = source_mask_attr_name
        self.target_mask_attr_name = target_mask_attr_name

    @property
    def name(self) -> tuple[str, str, str]:
        """Name of the edge subgraph."""
        return self.source_name, "to", self.target_name

    _agx_device_aware = True

    def compute_edge_index(self, source_nodes, target_nodes) -> torch.Tensor:
        """CUDA int32 (2, E): row 0 source index, row 1 target index (edges/builder.py:86-87).

        The package's builders override this.  A builder written for the REFERENCE's plugin contract - a subclass that
        provides ``get_adjacency_matrix(source_nodes, target_nodes)`` returning a scipy COO matrix (targets x sources,
        edges/builder.py:63) - works unchanged: its matrix is turned into the edge list the way the reference does
        (``edge_index = [col; row]``, :86-87) and uploaded."""
        if type(self).get_adjacency_matrix is BaseEdgeBuilder.get_adjacency_matrix:
            raise NotImplementedError(
                f"{type(self).__name__} must implement compute_edge_index (device) or get_adjacency_matrix (reference contract)."
            )
        _device.flush()  # the plugin reads host tensors
        adjmat = self.get_adjacency_matrix(source_nodes, target_nodes)
        adjmat = adjmat.tocoo() if hasattr(adjmat, "tocoo") else adjmat
        edge_index = torch.from_numpy(np.stack([adjmat.col, adjmat.row], axis=0).astype(np.int32))
        return edge_index.to(_device.compute_device())

    def get_adjacency_matrix(self, source_nodes, target_nodes):
        """scipy COO (targets x sources) connectivity - the reference's intermediate form
        (edges/builder.py:63); kept for callers that use it directly."""
        from scipy.sparse import coo_matrix

        ei = self.compute_edge_index(source_nodes, target_nodes).cpu().numpy()
        shape = (int(target_nodes["x"].shape[0]), int(source_nodes["x"].shape[0]))
        return coo_matrix((np.ones(ei.shape[1]), (ei[1], ei[0])), shape=shape)

    def prepare_node_data(self, graph):
        """Prepare node information and get source and target nodes."""
        return graph[self.source_name], graph[self.target_name]

    # May this builder run on a node set that is still in provisional numbering (``device.Provisional``)?  Only if
    # its result does not depend on how the nodes are numbered; ``_provisional_ok`` is raised per call by
    # ``register_edges`` when nothing else (masks, a merge with existing edges) needs final indices.
    provisional_source_ok = True
    provisional_target_ok = True
    _provisional_ok = False

    def get_edge_index_device(self, graph) -> torch.Tensor:
        source_nodes, target_nodes = self.prepare_node_data(graph)
        return self.compute_edge_index(source_nodes, target_nodes)

    def get_edge_index(self, graph) -> torch.Tensor:
        """Edge indices (2, num_edges) int32 of source and target nodes (edges/builder.py:69-87)."""
        self._provisional_ok = False
        dev = self.get_edge_index_device(graph)
        out = _device.like_input(dev, graph[self.target_name]["x"], _device.edge_shard(dev), dim=1)
        _device.maybe_flush()
        return out

    def register_edges(self, graph):
        """Register edges in the graph (edges/builder.py:89-115)."""
        store = graph[self.name]
        self._provisional_ok = "edge_index" not in store  # a merge sorts by index: final numbering only
        try:
            edge_dev = self.get_edge_index_device(graph)
        finally:
            self._provisional_ok = False
        edge_type = type(self).__name__
        x = graph[self.target_name]["x"]

        if "edge_index" in store:
            # Expand current edge indices: sorted unique columns (utils.concat_edges)
            if _device.sharded_output():
                raise NotImplementedError(
                    "several edge builders on one node pair are merged on complete edge lists: build this recipe in the "
                    "default output mode (AGX_OUTPUT=gather / device.set_sharded_output(False))"
                )
            edge_dev = concat_edges_device(
                _device.device_edge_index(store), edge_dev, int(graph[self.source_name]["x"].shape[0]), int(x.shape[0])
            )
            if edge_type not in store["edge_type"]:
                store["edge_type"] = store["edge_type"] + "," + edge_type
        else:
            store["edge_type"] = edge_type

        out = _device.edge_index_like_input(edge_dev, x)
        store["edge_index"] = out
        _device.remember_edge_index(store, out, edge_dev)
        shard = _device.edge_shard(edge_dev)
        if shard is not None and x.is_cuda:
            store["edge_shard"] = shard.describe()  # a device-resident sharded graph: which block this rank holds
        _device.maybe_flush()
        return graph

    def register_attributes(self, graph, config: DotDict):
        """Register attributes in the edges of the graph (edges/builder.py:117-134).

        An ``EdgeLength`` and an ``EdgeDirection`` of the same edge set are evaluated by ONE fused kernel
        pass; any other attribute object goes through its own ``compute``."""
        from .attributes import compute_attributes

        attrs = {attr_name: instantiate(attr_config) for attr_name, attr_config in config.items()}
        for attr_name, values in compute_attributes(graph, self.name, attrs).items():
            graph[self.name][attr_name] = values
        _device.maybe_flush()
        return graph

    def update_graph(self, graph, attrs_config: DotDict | None = None):
        """Update the graph with the edges (edges/builder.py:136-156)."""
        with _device.deferred():
            graph = self.register_edges(graph)

            if attrs_config is not None:
                graph = self.register_attributes(graph, attrs_config)

        return graph


class NodeMaskingMixin:
    """Mixin class for masking source/target nodes when building edges (edges/builder.py:159-193).

    Row selection is a device gather; the compact->original index map (the reference's python-dict ``np.vectorize``
    remap) is applied by the search kernels as they write (``masked_outputs``), so no pass over the edge list follows.
    ``undo_masking`` itself remains for callers that hold compact indices."""

    # A reversed builder searches the other way round: the TARGETS are indexed and every source node is a query.  Its
    # searches write the query side to row 0 (``swap_rows``), so the edge list still reads (source, target).
    _reversed = False

    def search_roles(self, of_source, of_target) -> tuple:
        """``(indexed side, query side)`` of a (source, target) pair - and, applied to that, the (source, target) pair."""
        return (of_target, of_source) if self._reversed else (of_source, of_target)

    @staticmethod
    def _selection(nodes, mask_attr_name: str | None, device) -> torch.Tensor | None:
        if mask_attr_name is None:
            return None
        mask = nodes[mask_attr_name]
        if not isinstance(mask, torch.Tensor):
            mask = torch.as_tensor(np.asarray(mask))
        mask = mask.squeeze().to(device=device, dtype=torch.bool)
        return torch.nonzero(mask, as_tuple=False).squeeze(1)

    def get_node_coordinates(self, source_nodes, target_nodes):
        """Device coordinates of the (masked) source and target nodes and the row selections."""
        masked = self.source_mask_attr_name is not None or self.target_mask_attr_name is not None
        ok = self._provisional_ok and not masked
        src_st = _device.node_state(source_nodes, provisional_ok=ok and self.provisional_source_ok)
        dst_st = _device.node_state(target_nodes, provisional_ok=ok and self.provisional_target_ok)
        self._row_provs = (src_st.prov, dst_st.prov)  # rows of the result that will be in provisional numbering
        self._node_states = (src_st, dst_st)  # the indexed side's index is shared between the builders of a recipe
        src, dst = src_st.x, dst_st.x
        src_sel = self._selection(source_nodes, self.source_mask_attr_name, src.device)
        dst_sel = self._selection(target_nodes, self.target_mask_attr_name, dst.device)
        if src_sel is not None:
            src = src[src_sel]
        if dst_sel is not None:
            dst = dst[dst_sel]
        return src, dst, src_sel, dst_sel

    @staticmethod
    def masked_outputs(ref_sel, query_sel, lo: int, hi: int):
        """``with self.masked_outputs(ref_sel, query_sel, lo, hi):`` - searches over the query rows [lo, hi) of the masked
        coordinates write ORIGINAL node indices (``undo_masking`` fused into the kernels' stores, ``ops.output_maps``)."""
        return ops.output_maps(ref_sel, None if query_sel is None else query_sel[lo:hi].contiguous())

    @staticmethod
    def undo_masking(edge_index: torch.Tensor, src_sel, dst_sel) -> torch.Tensor:
        if src_sel is None and dst_sel is None:
            return edge_index
        src = edge_index[0] if src_sel is None else src_sel[edge_index[0].long()].to(torch.int32)
        dst = edge_index[1] if dst_sel is None else dst_sel[edge_index[1].long()].to(torch.int32)
        return torch.stack([src, dst])


def _gather_blocks(full: torch.Tensor, counts: list[int], rank: int, masked: bool) -> torch.Tensor:
    """All-gather the per-rank column blocks of ``full`` (2, E).  Without node masks the exchange is asynchronous
    and ``full`` remembers which columns this rank produced itself (``device.edge_meta(full).local``), so the attribute kernel can
    start on them while the other ranks' blocks are still in flight."""
    if masked:
        return _device.all_gather_v(full, counts, dim=1)  # undo_masking reads every column next
    _device.all_gather_v(full, counts, dim=1, async_op=True)
    lo = sum(counts[:rank])
    _device.edge_meta(full, create=True).local = (lo, lo + counts[rank], list(counts))
    return full


class KNNEdges(BaseEdgeBuilder, NodeMaskingMixin):
    """Computes KNN based edges and adds them to the graph (edges/builder.py:196-270).

    Attributes
    ----------
    source_name : str
        The name of the source nodes.
    target_name : str
        The name of the target nodes.
    num_nearest_neighbours : int
        Number of nearest neighbours.
    source_mask_attr_name : str | None
        The name of the source mask attribute to filter edge connections.
    target_mask_attr_name : str | None
        The name of the target mask attribute to filter edge connections.
    """

    def __init__(
        self,
        source_name: str,
        target_name: str,
        num_nearest_neighbours: int,
        source_mask_attr_name: str | None = None,
        target_mask_attr_name: str | None = None,
    ) -> None:
        super().__init__(source_name, target_name, source_mask_attr_name, target_mask_attr_name)
        assert isinstance(num_nearest_neighbours, int), "Number of nearest neighbours must be an integer"
        assert num_nearest_neighbours > 0, "Number of nearest neighbours must be positive"
        self.num_nearest_neighbours = num_nearest_neighbours
        self.stats = None  # optional CUDA int64[4]: {float64-refined, tied at the k-th boundary, widened, 0}

    # Ties at the k-th boundary go to the lower index of the indexed side (the SOURCES; the targets for
    # ReversedKNNEdges), so the result depends on the final numbering of that side - but only for the queries that have
    # such a tie.  With a provisionally numbered indexed side the search runs at once, flags those queries
    # (agx_knn_flagged), and re-decides exactly them when the order is known (``_redecide_ties``); everything else is a
    # relabel.
    provisional_source_ok = True

    @staticmethod
    def _redecide_ties(prov, index, out: torch.Tensor, tie_list, queries: torch.Tensor, k: int, swap_rows: bool) -> None:
        """Runs inside ``Provisional.resolve`` before the rows are relabelled: ``index`` is the one the search used
        (provisional labels); ties go to the lower FINAL label ``prov.rank[label]``, provisional labels are written."""
        index.knn_redecide_list(queries, k, out, tie_list[0], tie_list[1], rank=prov.rank, order=prov.order_dev,
                                swap_rows=swap_rows)  # fmt: skip
        meta = _device.edge_meta(out)
        if meta is not None:
            meta.fixup = None

    def compute_edge_index(self, source_nodes, target_nodes) -> torch.Tensor:
        src, dst, src_sel, dst_sel = self.get_node_coordinates(source_nodes, target_nodes)
        assert self.num_nearest_neighbours is not None, "number of neighbors required for knn encoder"
        rev = self._reversed
        LOGGER.info(
            "Using %sKNN-Edges (with %d nearest neighbours) between %s and %s.",
            "Reversed-" if rev else "",
            self.num_nearest_neighbours,
            self.source_name,
            self.target_name,
        )
        k = self.num_nearest_neighbours
        ref, qry = self.search_roles(src, dst)
        ref_sel, qry_sel = self.search_roles(src_sel, dst_sel)
        ref_state = self.search_roles(*self._node_states)[0]
        nq = int(qry.shape[0])
        # sharded output mode: this rank's queries only and nothing to exchange, so sharding always pays; otherwise
        # every rank needs the complete list and small searches are replicated (``shard_world``)
        sharded_out = _device.sharded_output()
        rank, w = _device.world() if sharded_out else _device.shard_world(nq)
        ref_prov, qry_prov = self.search_roles(*self._row_provs)
        if ref_prov is not None and ((w > 1 and not sharded_out) or qry_prov is not None):
            # flag-and-redecide is built for final query numbering and rank-local results: order first
            ref, qry = self.search_roles(_device.node_state(source_nodes).x, _device.node_state(target_nodes).x)
            self._row_provs = (None, None)
            ref_prov = qry_prov = None
        lo, hi = _device.shard_range(nq, rank, w)
        shard = None
        if sharded_out:
            shard = _device.Shard(rank, w, [(b - a) * k for a, b in (_device.shard_range(nq, r, w) for r in range(w))])
        if ref_prov is not None:
            q = qry[lo:hi]  # all queries on one rank
            flags = torch.zeros(hi - lo, dtype=torch.uint8, device=qry.device)
            with _device.neighbour_index(ref_state, ref, hint_k=k) as index:
                out = index.knn(q, k, dst_base=lo, stats=self.stats, tie_flags=flags, swap_rows=rev)
            out = _device.tag_rows(out, *self.search_roles(ref_prov, None))
            meta = _device.edge_meta(out, create=True)
            tie_list = ops.compact_flags(flags)  # ascending ids of the tied queries, count on the device: no read-back
            meta.fixup, meta.shard = ref_prov, shard
            if not rev:
                # the attribute kernel evaluates the un-flagged targets' edges before the re-decision; its flag modes
                # are keyed by row-1 targets, so a reversed list (flagged SOURCES) leaves them unset: its attributes
                # are evaluated on the final edges
                meta.tie_flags, meta.tie_list, meta.regular_k = flags, tie_list, k
                meta.flag_base = lo  # ``flags`` is indexed by target id - lo
                meta.regular_targets = not sharded_out and (lo, hi) == (0, nq)  # unmasked by construction
            # ``index`` stays alive in the closure: the re-decision searches it again, no second index
            ref_prov.add_fixup(lambda prov, index=index, out=out, tl=tie_list, q=q, k=k: self._redecide_ties(prov, index, out, tl, q, k, rev))  # fmt: skip
            return out
        if sharded_out:
            # rank-local block, global query ids; no exchange
            with _device.neighbour_index(ref_state if ref_sel is None else None, ref, hint_k=k) as index:
                with self.masked_outputs(ref_sel, qry_sel, lo, hi):
                    out = index.knn(qry[lo:hi], k, dst_base=lo, stats=self.stats, swap_rows=rev)
            out = _device.tag_rows(out, *self._row_provs)
            meta = _device.edge_meta(out, create=True)
            meta.shard = shard
            if not rev:
                meta.regular_k = k
            return out
        with _device.neighbour_index(ref_state if ref_sel is None else None, ref, hint_k=k) as index:
            out = torch.empty((2, nq * k), dtype=torch.int32, device=qry.device)
            masked = src_sel is not None or dst_sel is not None
            if w > 1 and not masked and _device.VMM_PUSH:
                # opt-in: chunks pushed into peer-mapped staging buffers by the copy engines while the next chunk is
                # searched (device.VmmGather)
                n_chunks = _device.n_query_chunks(nq, w)
                ranges = [_device.query_chunks(*_device.shard_range(nq, r, w), n_chunks) for r in range(w)]
                gather = _device.make_gather(out, [[(b - a) * k for a, b in rr] for rr in ranges])
                lib, marks = ops.load_library(), []
                try:
                    for c, (a, b) in enumerate(ranges[rank]):
                        if b > a:
                            index.knn(qry[a:b], k, dst_base=a, stats=self.stats, out=out, out_offset=a * k, swap_rows=rev)
                            if c == 0:  # the first chunk decided the query order (one sync): pin it for the rest
                                lib.agx_set_query_order_mode(lib.agx_last_query_order())
                        marks.append(gather.mark())
                        if c > 0:
                            gather.chunk_done(c - 1, marks[c - 1])
                    gather.chunk_done(n_chunks - 1, marks[-1])
                finally:
                    lib.agx_set_query_order_mode(-1)
                gather.finish()
                w = 1  # complete on every rank
            else:
                # equal blocks: one in-place NCCL all-gather after the search (640 GB/s per rank; chunking the search
                # to overlap an NCCL exchange was measured and does not pay: the persistent search kernel leaves no
                # room for the collective's CTAs until it ends - 40 M queries, N = 2: 4.8 ms chunked against 4.5 ms)
                with self.masked_outputs(ref_sel, qry_sel, lo, hi):  # original node indices straight from the kernel
                    index.knn(qry[lo:hi], k, dst_base=lo, stats=self.stats, out=out, out_offset=lo * k, swap_rows=rev)
        if w > 1:
            counts = [(b - a) * k for a, b in (_device.shard_range(nq, r, w) for r in range(w))]
            out = _gather_blocks(out, counts, rank, src_sel is not None or dst_sel is not None)
        local = _device.edge_meta(out).local if _device.edge_meta(out) is not None else None
        out = _device.tag_rows(out, *self._row_provs)
        meta = _device.edge_meta(out, create=True)
        meta.local = local
        if not rev:
            meta.regular_k = k  # k edges per target, target after target: attributes walk it by target
            meta.regular_targets = src_sel is None and dst_sel is None  # complete list, row 1 = column // k
        return out


class ReversedKNNEdges(KNNEdges):
    """KNN edges in the other direction: for every (masked) source node, its k nearest (masked) target nodes.

    The same edges as ``KNNEdges(target_name, source_name, ...)`` with its two rows swapped (and the masks swapped with
    them), column for column: the targets are indexed and the sources are the queries, grouped by source, k columns per
    source.  Exact float64 distance ties at the k-th boundary go to the lower TARGET index.  The class of newer
    anemoi-graphs releases; parity with them is unverified (the pinned reference has no such class).

    Attributes
    ----------
    source_name : str
        The name of the source nodes.
    target_name : str
        The name of the target nodes.
    num_nearest_neighbours : int
        Number of nearest target nodes of each source node.
    source_mask_attr_name : str | None
        The name of the source mask attribute to filter edge connections.
    target_mask_attr_name : str | None
        The name of the target mask attribute to filter edge connections.
    """

    _reversed = True


class CutOffEdges(BaseEdgeBuilder, NodeMaskingMixin):
    """Computes cut-off based edges and adds them to the graph (edges/builder.py:273-371).

    Attributes
    ----------
    source_name : str
        The name of the source nodes.
    target_name : str
        The name of the target nodes.
    cutoff_factor : float
        Factor to multiply the grid reference distance to get the cut-off radius.
    source_mask_attr_name : str | None
        The name of the source mask attribute to filter edge connections.
    target_mask_attr_name : str | None
        The name of the target mask attribute to filter edge connections.
    max_num_neighbours : int | None
        At most this many edges per target node: a target with more source nodes within the radius keeps its
        ``max_num_neighbours`` nearest, exact float64 distance ties at the boundary going to the lower source index.
        None (default): no cap.  The argument of newer anemoi-graphs releases, whose default is 64 as far as is known;
        parity with them is unverified (DESIGN.md section 4).
    """

    def __init__(
        self,
        source_name: str,
        target_name: str,
        cutoff_factor: float,
        source_mask_attr_name: str | None = None,
        target_mask_attr_name: str | None = None,
        max_num_neighbours: int | None = None,
    ):
        super().__init__(source_name, target_name, source_mask_attr_name, target_mask_attr_name)
        assert isinstance(cutoff_factor, (int, float)), "Cutoff factor must be a float"
        assert cutoff_factor > 0, "Cutoff factor must be positive"
        check_max_num_neighbours(max_num_neighbours)
        self.cutoff_factor = cutoff_factor
        self.max_num_neighbours = max_num_neighbours
        # optional CUDA int64[4]: {pairs decided in float64, pairs within 2^-40 of the radius, queries capped at
        # max_num_neighbours, capped queries with a tie at the boundary}
        self.stats = None

    def get_cutoff_radius(self, graph, mask_attr: torch.Tensor | None = None) -> float:
        """Cut-off radius = reference distance of the query nodes x cut-off factor (edges/builder.py:312-334): the
        TARGET nodes, the sources for ``ReversedCutOffEdges``."""
        query_nodes = graph[self.search_roles(self.source_name, self.target_name)[1]]
        mask = query_nodes[mask_attr] if mask_attr is not None else None
        # the reference distance does not depend on the numbering of the nodes
        state = _device.node_state(query_nodes, provisional_ok=True)
        query_grid_reference_distance = get_grid_reference_distance(state.x, mask, state=state)
        radius = query_grid_reference_distance * self.cutoff_factor
        return radius

    def prepare_node_data(self, graph):
        """Prepare node information and get source and target nodes."""
        self.radius = self.get_cutoff_radius(graph)
        return super().prepare_node_data(graph)

    def compute_edge_index(self, source_nodes, target_nodes) -> torch.Tensor:
        src, dst, src_sel, dst_sel = self.get_node_coordinates(source_nodes, target_nodes)
        rev = self._reversed
        LOGGER.info(
            "Using %sCutOff-Edges (with radius = %.1f km) between %s and %s.",
            "Reversed-" if rev else "",
            self.radius * EARTH_RADIUS,
            self.source_name,
            self.target_name,
        )
        ref, qry = self.search_roles(src, dst)
        ref_sel, qry_sel = self.search_roles(src_sel, dst_sel)
        cap_m = self.max_num_neighbours
        ref_prov, qry_prov = self.search_roles(*self._row_provs)
        if cap_m is not None and ref_prov is not None:
            # the nearest-M pick breaks ties by the numbering of the indexed side: final numbering first (provisional
            # numbering implies no masks)
            ref = _device.node_state(self.search_roles(source_nodes, target_nodes)[0]).x
            self._row_provs = self.search_roles(None, qry_prov)
        nq = int(qry.shape[0])
        sharded_out = _device.sharded_output()
        rank, w = _device.world() if sharded_out else _device.shard_world(nq)
        lo, hi = _device.shard_range(nq, rank, w)

        def count(index, q):
            """``(offsets, total, cap)``: ``cap`` the keyword arguments ``radius_fill`` takes for query rows [a, b)."""
            if cap_m is None:
                return (*index.radius_count(q, self.radius), lambda a, b: {})
            offsets, total, counts = index.radius_capped(q, self.radius, cap_m)
            return offsets, total, lambda a, b: {"counts": counts[a:b], "max_neighbours": cap_m}

        if sharded_out:
            # this rank's queries only; the blocks stay where they are (global query ids), only the counts travel
            with ops.NeighbourIndex(ref, hint_radius=self.radius) as index:
                q = qry[lo:hi]
                offsets, total, cap = count(index, q)
                out = torch.empty((2, total), dtype=torch.int32, device=qry.device)
                with self.masked_outputs(ref_sel, qry_sel, lo, hi):
                    index.radius_fill(q, self.radius, offsets, total, out, 0, dst_base=lo, stats=self.stats, swap_rows=rev,
                                      **cap(0, hi - lo))  # fmt: skip
            counts = _device.exchange_counts(total, qry.device)
            out = _device.tag_rows(out, *self._row_provs)
            _device.edge_meta(out, create=True).shard = _device.Shard(rank, w, counts)
            return out
        with ops.NeighbourIndex(ref, hint_radius=self.radius) as index:
            q = qry[lo:hi]
            offsets, total, cap = count(index, q)
            masked = src_sel is not None or dst_sel is not None
            if w > 1 and not masked and torch.distributed.get_backend() == "nccl":
                # uneven blocks: padded equal-block all-gathers, chunk by chunk (device.ChunkedGather); per-chunk pair
                # counts from the count pass
                n_chunks = _device.n_query_chunks(nq, w)
                chunks = _device.query_chunks(0, hi - lo, n_chunks)
                bounds = offsets[[a for a, _ in chunks] + [hi - lo]].tolist()  # pair offsets at the chunk boundaries
                mine = [o1 - o0 for o0, o1 in zip(bounds[:-1], bounds[1:])]
                rows = _device.all_gather_count_rows(mine, qry.device)
                counts = [sum(r) for r in rows]
                out = torch.empty((2, sum(counts)), dtype=torch.int32, device=qry.device)
                base = sum(counts[:rank])
                gather = _device.make_gather(out, rows)
                lib, marks = ops.load_library(), []
                lib.agx_set_query_order_mode(lib.agx_last_query_order())  # as the count pass decided: no more syncs
                try:
                    for c, (a, b) in enumerate(chunks):
                        if mine[c]:
                            # the offsets keep their block-relative values, so the chunk lands at its final columns
                            index.radius_fill(q[a:b], self.radius, offsets[a : b + 1], mine[c], out, base,
                                              dst_base=lo + a, stats=self.stats, swap_rows=rev, **cap(a, b))  # fmt: skip
                        marks.append(gather.mark())
                        if c > 0:
                            gather.chunk_done(c - 1, marks[c - 1])
                    gather.chunk_done(n_chunks - 1, marks[-1])
                finally:
                    lib.agx_set_query_order_mode(-1)
                gather.finish()
                _device.edge_meta(out, create=True).local = (base, base + counts[rank], list(counts))
                w = 1  # complete on every rank
            else:
                counts = _device.all_gather_counts(total, qry.device) if w > 1 else [total]
                out = torch.empty((2, sum(counts)), dtype=torch.int32, device=qry.device)
                base = sum(counts[:rank])
                with self.masked_outputs(ref_sel, qry_sel, lo, hi):  # original node indices straight from the kernel
                    index.radius_fill(q, self.radius, offsets, total, out, base, dst_base=lo, stats=self.stats,
                                      swap_rows=rev, **cap(0, hi - lo))  # fmt: skip
        if w > 1:
            out = _gather_blocks(out, counts, rank, src_sel is not None or dst_sel is not None)
        return _device.tag_rows(out, *self._row_provs)


class ReversedCutOffEdges(CutOffEdges):
    """Cut-off edges in the other direction: every (masked) (source, target) pair with the target within the cut-off
    radius of the source, grouped by source.

    The radius is ``cutoff_factor`` x the grid reference distance of the SOURCE nodes (the query side, as the targets
    are for ``CutOffEdges``), with the same inclusive test, so the edges are those of ``CutOffEdges(target_name,
    source_name, ...)`` with its two rows swapped, column for column.  The class of newer anemoi-graphs releases;
    parity with them is unverified (the pinned reference has no such class).

    Attributes
    ----------
    source_name : str
        The name of the source nodes.
    target_name : str
        The name of the target nodes.
    cutoff_factor : float
        Factor to multiply the grid reference distance of the source nodes to get the cut-off radius.
    source_mask_attr_name : str | None
        The name of the source mask attribute to filter edge connections.
    target_mask_attr_name : str | None
        The name of the target mask attribute to filter edge connections.
    max_num_neighbours : int | None
        At most this many edges per SOURCE node (the query side), chosen as for ``CutOffEdges``.  None (default): no cap.
    """

    _reversed = True


def check_max_num_neighbours(max_num_neighbours) -> None:
    """The ``max_num_neighbours`` argument of the cut-off builders: None (no cap) or a positive int."""
    if max_num_neighbours is None:
        return
    assert isinstance(max_num_neighbours, int) and not isinstance(max_num_neighbours, bool), (
        "Maximum number of neighbours must be an integer"
    )
    assert max_num_neighbours > 0, "Maximum number of neighbours must be positive"


MULTISCALE_MAX_LEVELS = 16  # MS_MAX_LEVELS of the multi-scale edge kernel (agx_mesh.cu)


def scale_levels(scale_resolutions) -> list[int] | None:
    """The refinement levels a ``MultiScaleEdges(scale_resolutions=...)`` argument names, ascending and distinct: an int
    ``n`` names 1..n, a list its own entries, None every level of the node set (returned as None)."""
    assert not isinstance(scale_resolutions, str), "The scale_resolutions argument is not valid."
    if scale_resolutions is None:
        return None
    if isinstance(scale_resolutions, int) and not isinstance(scale_resolutions, bool):
        assert scale_resolutions > 0, "The scale_resolutions argument only supports positive integers."
        return list(range(1, scale_resolutions + 1))
    assert isinstance(scale_resolutions, (list, tuple)) and len(scale_resolutions) > 0, (
        "The scale_resolutions argument is not valid."
    )
    assert all(isinstance(r, int) and not isinstance(r, bool) and r > 0 for r in scale_resolutions), (
        "The scale_resolutions argument only supports positive integers."
    )
    return sorted(set(scale_resolutions))


def check_scale_levels(levels: list[int], finest: int | None) -> None:
    """Levels the multi-scale edge kernel can build on a node set whose finest level is ``finest`` (None: not known
    yet); raised before any kernel runs."""
    if len(levels) > MULTISCALE_MAX_LEVELS:
        raise NotImplementedError(
            f"MultiScaleEdges: {len(levels)} scale_resolutions > {MULTISCALE_MAX_LEVELS} levels is not built"
        )
    if finest is not None and max(levels) > finest:
        raise ValueError(f"MultiScaleEdges: scale_resolutions {levels} go past the finest level {finest} of the nodes")


class MultiScaleEdges(BaseEdgeBuilder):
    """Multi-scale edges in the nodes of a refined icosahedron (edges/builder.py:374-462).

    Attributes
    ----------
    source_name : str
        The name of the source nodes.
    target_name : str
        The name of the target nodes.
    x_hops : int
        Number of hops (in the refined icosahedron) between two nodes to connect
        them with an edge.
    scale_resolutions : int | list[int] | None
        Refinement levels that contribute edges: ``n`` for the levels 1..n, a list for exactly those levels, None
        (default) for every level of the node set (its ``_resolutions``).  As in newer anemoi-graphs releases, as far
        as is known (the pinned reference has no such argument).
    """

    VALID_NODES = ["TriNodes", "HexNodes", "LimitedAreaTriNodes", "LimitedAreaHexNodes", "StretchedTriNodes"]

    def __init__(
        self, source_name: str, target_name: str, x_hops: int, scale_resolutions: int | list[int] | None = None, **kwargs
    ):
        super().__init__(source_name, target_name)
        assert source_name == target_name, f"{self.__class__.__name__} requires source and target nodes to be the same."
        assert isinstance(x_hops, int), "Number of x_hops must be an integer"
        assert x_hops > 0, "Number of x_hops must be positive"
        self.x_hops = x_hops
        self.scale_resolutions = scale_levels(scale_resolutions)

    def levels(self, nodes) -> list[int]:
        """The refinement levels whose edges are built on ``nodes``."""
        if self.scale_resolutions is None:
            return nodes["_resolutions"]
        check_scale_levels(self.scale_resolutions, max(int(r) for r in nodes["_resolutions"]))
        return self.scale_resolutions

    def compute_edge_index(self, source_nodes, target_nodes) -> torch.Tensor:
        from ..generate import tri_icosahedron

        node_type = source_nodes["node_type"]
        resolutions = self.levels(source_nodes)
        if node_type in ("TriNodes", "LimitedAreaTriNodes"):
            return tri_icosahedron.multiscale_edges(
                source_nodes,
                resolutions=resolutions,
                x_hops=self.x_hops,
                area_mask_builder=source_nodes.get("_area_mask_builder", None),
                allow_provisional=self._provisional_ok,
            )
        if node_type == "StretchedTriNodes":
            from ..generate.masks import KNNAreaMaskBuilder

            # edges/builder.py:422-432: a level-r vertex is valid iff it lies within 1 km of an existing node
            all_points_mask_builder = KNNAreaMaskBuilder("all_nodes", 1.0)
            all_points_mask_builder.fit_coords(_device.node_state(source_nodes).x)
            return tri_icosahedron.multiscale_edges(
                source_nodes,
                resolutions=resolutions,
                x_hops=self.x_hops,
                area_mask_builder=all_points_mask_builder,
            )
        if node_type in ("HexNodes", "LimitedAreaHexNodes"):
            from ..generate import hex_icosahedron

            # the graph's nodes are the cells of the node set's finest level, whichever levels contribute edges
            finest = None if self.scale_resolutions is None else max(int(r) for r in source_nodes["_resolutions"])
            return hex_icosahedron.multiscale_edges(source_nodes, resolutions=resolutions, x_hops=self.x_hops, finest=finest)
        raise ValueError(f"Invalid node type {node_type}")

    def get_edge_index_device(self, graph) -> torch.Tensor:
        out = super().get_edge_index_device(graph)
        if _device.sharded_output():
            # replicas only (SURVEY 8e): every rank computes the whole (small) set; a host-resident graph receives 1/W
            # of its columns from each rank
            rank, w = _device.world()
            _device.edge_meta(out, create=True).shard = _device.Shard(rank, w, [int(out.shape[1])], replicated=True)
        return out

    def update_graph(self, graph, attrs_config: DotDict | None = None):
        node_type = graph[self.source_name].node_type
        assert node_type in self.VALID_NODES, f"{self.__class__.__name__} requires {','.join(self.VALID_NODES)} nodes."

        return super().update_graph(graph, attrs_config)
