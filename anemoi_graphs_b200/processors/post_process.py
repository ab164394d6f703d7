"""Graph post-processors (/root/reference/src/anemoi/graphs/processors/post_process.py:22-149).

``RemoveUnconnectedNodes`` keeps the reference's constructor, ``compute_mask`` / ``update_graph`` contract and
results; the per-edge work - marking connected nodes and rewriting every edge endpoint through the old -> new
index map, which the reference does with a python dict and ``Tensor.apply_`` - runs on the GPU
(``agx_mark_nodes`` -> ``agx_exclusive_scan`` -> ``agx_relabel_nodes``).

``RestrictEdgeLength``, ``SortEdgeIndexBySourceNodes`` and ``SortEdgeIndexByTargetNodes`` carry the names of the
post-processors of newer anemoi-graphs releases.  Each computes an index list on the GPU (``agx_restrict_flags`` ->
``agx_compact_flags``, or ``agx_sort_edges``) and applies it to ``edge_index`` and every per-edge attribute in one
launch per eight arrays (``agx_gather_edge_columns``).  An endpoint outside its node set raises ``ValueError`` before
the graph changes; a sharded block of a device-resident graph raises ``NotImplementedError``.

Tensors come back where they were (CPU in, CPU out), with their dtypes.
"""

from __future__ import annotations

import logging
from abc import ABC
from abc import abstractmethod

import torch

from .. import EARTH_RADIUS
from .. import device as _device
from .. import ops
from .._cabi import check, current_stream, load_library, ptr

LOGGER = logging.getLogger(__name__)


class PostProcessor(ABC):
    _agx_device_aware = True

    @abstractmethod
    def update_graph(self, graph):
        raise NotImplementedError(f"The {self.__class__.__name__} class does not implement the method update_graph().")


def _row_int32(row: torch.Tensor) -> torch.Tensor:
    """One edge_index row as a contiguous CUDA int32 tensor (the row itself when it already is one)."""
    return _device.to_device(row.contiguous(), torch.int32)


class BaseMaskingProcessor(PostProcessor, ABC):
    """Base class for mask based processor."""

    def __init__(self, nodes_name: str, save_mask_indices_to_attr: str | None = None) -> None:
        self.nodes_name = nodes_name
        self.save_mask_indices_to_attr = save_mask_indices_to_attr
        self.mask: torch.Tensor = None
        self._flags_dev: torch.Tensor | None = None  # CUDA int32 keep flags behind ``mask``

    def removing_nodes(self, graph):
        """Remove nodes based on the mask passed."""
        nodes = graph[self.nodes_name]
        for attr_name in nodes.node_attrs():
            value = nodes[attr_name]
            nodes[attr_name] = value[self.mask.to(value.device)]
        return graph

    def create_indices_mapper_from_mask(self) -> dict[int, int]:
        return dict(zip(torch.where(self.mask)[0].tolist(), list(range(int(self.mask.sum())))))

    def update_edge_indices(self, graph):
        """Update the edge indices to the new position of the nodes (post_process.py:49-60)."""
        lib = load_library()
        flags = self._flags_dev
        if flags is None:
            flags = _device.to_device(self.mask, torch.int32)
        n_nodes = int(flags.shape[0])
        new_index = torch.empty(n_nodes + 1, dtype=torch.int64, device=flags.device)
        stream = current_stream()
        check(lib.agx_exclusive_scan(ptr(flags), n_nodes, ptr(new_index), None, stream))
        for edges_name in graph.edge_types:
            for row, name in ((0, edges_name[0]), (1, edges_name[2])):
                if name != self.nodes_name:
                    continue
                edge_index = graph[edges_name].edge_index
                dev_row = _row_int32(edge_index[row])
                check(lib.agx_relabel_nodes(ptr(dev_row), int(dev_row.shape[0]), ptr(new_index), stream))
                edge_index[row] = dev_row.to(device=edge_index.device, dtype=edge_index.dtype)
        return graph

    @abstractmethod
    def compute_mask(self, graph) -> torch.Tensor: ...

    def add_attribute(self, graph):
        """Add an attribute of the mask indices as node attribute."""
        if self.save_mask_indices_to_attr is not None:
            LOGGER.info(
                f"An attribute {self.save_mask_indices_to_attr} has been added with the indices to mask the nodes from the original graph."
            )
            mask_indices = torch.where(self.mask)[0].reshape((graph[self.nodes_name].num_nodes, -1))
            graph[self.nodes_name][self.save_mask_indices_to_attr] = mask_indices
        return graph

    def update_graph(self, graph):
        """Post-process the graph."""
        self.mask = self.compute_mask(graph)
        LOGGER.info(f"Removing {(~self.mask).sum()} nodes from {self.nodes_name}.")
        graph = self.removing_nodes(graph)
        graph = self.update_edge_indices(graph)
        graph = self.add_attribute(graph)
        self._flags_dev = None
        return graph


class RemoveUnconnectedNodes(BaseMaskingProcessor):
    """Remove unconnected nodes in the graph.

    Attributes
    ----------
    nodes_name: str
        Name of the unconnected nodes to remove.
    ignore: str, optional
        Name of an attribute to ignore when removing nodes. Nodes with
        this attribute set to True will not be removed.
    save_mask_indices_to_attr: str, optional
        Name of the attribute to save the mask indices. If provided,
        the indices of the kept nodes will be saved in this attribute.
    """

    def __init__(
        self,
        nodes_name: str,
        save_mask_indices_to_attr: str | None = None,
        ignore: str | None = None,
    ) -> None:
        super().__init__(nodes_name, save_mask_indices_to_attr)
        self.ignore = ignore

    def compute_mask(self, graph) -> torch.Tensor:
        """Compute the mask of connected nodes (post_process.py:133-149): bool (num_nodes,), on the device ``x``
        lives on."""
        nodes = graph[self.nodes_name]
        n_nodes = int(nodes.num_nodes)
        dev = _device.compute_device()
        flags = torch.zeros(n_nodes, dtype=torch.int32, device=dev)

        if self.ignore is not None:
            LOGGER.info(f"The nodes with {self.ignore}=True will not be removed.")
            flags[nodes[self.ignore].bool().squeeze().to(dev)] = 1

        lib = load_library()
        stream = current_stream()
        for (source_name, _, target_name), edges in graph.edge_items():
            for row, name in ((0, source_name), (1, target_name)):
                if name != self.nodes_name:
                    continue
                dev_row = _row_int32(edges.edge_index[row])
                check(lib.agx_mark_nodes(ptr(dev_row), int(dev_row.shape[0]), n_nodes, ptr(flags), stream))

        self._flags_dev = flags
        return flags.bool().to(nodes["x"].device)


# ------------------------------------------------------------------------------------------------
# edge post-processors: every one ends in ONE int32 index list applied to each per-edge tensor of an edge set
# ------------------------------------------------------------------------------------------------
def _check_gathered(name, store) -> None:
    if "edge_shard" in store:
        _refuse_sharded(name)


def _refuse_sharded(name) -> None:
    raise NotImplementedError(
        f"edge set {name} is a sharded block of a device-resident graph: the edge post-processors work on complete "
        "edge lists - build this recipe in the default output mode (AGX_OUTPUT=gather / "
        "device.set_sharded_output(False))"
    )


def _select_edges(store, index: torch.Tensor, ei_dev: torch.Tensor) -> None:
    """Replace ``edge_index`` and every per-edge tensor of ``store`` (``edge_attrs()``) by its columns / rows at the
    CUDA int32 positions ``index`` - one ``agx_gather_edge_columns`` launch per eight arrays.  ``ei_dev`` is the CUDA
    int32 copy of ``edge_index``.  Each tensor keeps its dtype and comes back on the device it was on."""
    m = int(index.numel())
    pairs, results = [], {}
    for name in store.edge_attrs():
        t = store[name]
        if name == "edge_index":
            src = ei_dev if t.dtype == torch.int32 else _device.to_device(t)
            out = torch.empty((2, m), dtype=t.dtype, device=src.device)
            pairs += [(src[0], out[0]), (src[1], out[1])]
        else:
            src = _device.to_device(t)
            out = torch.empty((m, *t.shape[1:]), dtype=t.dtype, device=src.device)
            pairs.append((src, out))
        results[name] = out
    ops.gather_rows(pairs, index)
    for name, out in results.items():
        was = store[name]
        store[name] = out if was.is_cuda else out.to(was.device)
    if not store["edge_index"].is_cuda and results["edge_index"].dtype == torch.int32:
        _device.remember_edge_index(store, store["edge_index"], results["edge_index"])


def _node_mask(graph, nodes_name: str, attr_name: str | None) -> torch.Tensor | None:
    """CUDA uint8 (N,) of a bool node attribute of shape (N,) or (N, 1); None without an attribute name."""
    if attr_name is None:
        return None
    nodes = graph[nodes_name]
    mask = nodes[attr_name]
    n = nodes.num_nodes
    if not isinstance(mask, torch.Tensor) or mask.dtype != torch.bool or mask.shape not in ((n,), (n, 1)):
        what = f"{mask.dtype} {tuple(mask.shape)}" if isinstance(mask, torch.Tensor) else type(mask).__name__
        raise ValueError(f"The mask attribute '{attr_name}' of {nodes_name} must be a bool tensor of shape ({n},) or ({n}, 1), got {what}.")
    return _device.to_device(mask.reshape(n)).view(torch.uint8)


class RestrictEdgeLength(PostProcessor):
    """Remove the edges of one edge set that are longer than a length.

    An edge of ``(source_name, "to", target_name)`` is subject to the restriction when its source is True in
    ``source_mask_attr_name`` and its target is True in ``target_mask_attr_name`` (each mask optional: a bool node
    attribute of shape (N,) or (N, 1)).  Such an edge is removed iff it is longer than ``max_length_km``, by exactly
    the test ``CutOffEdges`` applies: it is kept iff its haversine ``rdist`` (float64 on the float32 coordinates) is
    at most ``sin^2(r / 2)``, r = max_length_km / EARTH_RADIUS - so an edge exactly at the limit stays, and a cut-off
    edge set restricted to its own radius is unchanged.

    ``edge_index`` and every per-edge attribute are filtered with one selection; kept edges keep their relative order.
    Attributes are filtered, not re-normalised: normalised values keep the scale of the unrestricted edge set.

    Attributes
    ----------
    source_name: str
        Name of the source nodes of the edge set.
    target_name: str
        Name of the target nodes of the edge set.
    max_length_km: int | float
        Longest edge kept, in km.
    source_mask_attr_name: str, optional
        Bool source node attribute: only edges from these sources are restricted.
    target_mask_attr_name: str, optional
        Bool target node attribute: only edges into these targets are restricted.
    """

    def __init__(
        self,
        source_name: str,
        target_name: str,
        max_length_km: float,
        source_mask_attr_name: str | None = None,
        target_mask_attr_name: str | None = None,
    ) -> None:
        assert isinstance(max_length_km, (int, float)), "Maximum edge length must be a number"
        assert max_length_km > 0, "Maximum edge length must be positive"
        self.source_name = source_name
        self.target_name = target_name
        self.max_length_km = max_length_km
        self.source_mask_attr_name = source_mask_attr_name
        self.target_mask_attr_name = target_mask_attr_name

    def update_graph(self, graph):
        name = (self.source_name, "to", self.target_name)
        if name not in graph.edge_types:
            raise ValueError(f"{self.__class__.__name__}: the graph has no edge set {name}.")
        store = graph[name]
        _check_gathered(name, store)
        ei_dev = _device.device_edge_index(store)
        src_mask = _node_mask(graph, self.source_name, self.source_mask_attr_name)
        dst_mask = _node_mask(graph, self.target_name, self.target_mask_attr_name)
        src_x = _device.node_state(graph[self.source_name]).x
        dst_x = _device.node_state(graph[self.target_name]).x
        radius = float(self.max_length_km) / EARTH_RADIUS
        keep = ops.restrict_flags(ei_dev, src_x, dst_x, radius, src_mask, dst_mask)
        index, count = ops.compact_flags(keep)
        n_kept = int(count.item())
        LOGGER.info(f"Removing {int(ei_dev.shape[1]) - n_kept} edges longer than {self.max_length_km} km from {name}.")
        _select_edges(store, index[:n_kept], ei_dev)
        return graph


class BaseSortEdgeIndex(PostProcessor, ABC):
    """Sort the columns of every edge set lexicographically by (key row, other row) and permute every per-edge
    attribute with them.  The sort is stable: columns equal in both rows keep their order, so the result is unique."""

    key_row: int

    def __init__(self, descending: bool = True) -> None:
        assert isinstance(descending, bool), "descending must be a bool"
        self.descending = descending

    def update_graph(self, graph):
        items = graph.edge_items()
        for name, store in items:
            _check_gathered(name, store)
        # every permutation (and its endpoint check) first: an invalid edge set leaves the whole graph unchanged
        perms = []
        for (source_name, _, target_name), store in items:
            ei_dev = _device.device_edge_index(store)
            n_nodes = (graph[source_name].num_nodes, graph[target_name].num_nodes)
            k, o = self.key_row, 1 - self.key_row
            perms.append((ei_dev, ops.sort_permutation(ei_dev[k], ei_dev[o], n_nodes[k], n_nodes[o], self.descending)))
        for (_, store), (ei_dev, perm) in zip(items, perms):
            _select_edges(store, perm, ei_dev)
        return graph


class SortEdgeIndexBySourceNodes(BaseSortEdgeIndex):
    """Sort every edge set by source node, then target node (``descending`` applies to both; default True as in the
    upstream class as far as is known - unverified here).  Stable: duplicate columns keep their order.

    Attributes
    ----------
    descending: bool
        Sort in descending order (default True).
    """

    key_row = 0


class SortEdgeIndexByTargetNodes(BaseSortEdgeIndex):
    """Sort every edge set by target node, then source node (``descending`` applies to both; default True as in the
    upstream class as far as is known - unverified here).  Stable: duplicate columns keep their order.
    ``SortEdgeIndexByTargetNodes(descending=False)`` gives numpy's ``lexsort((edge_index[0], edge_index[1]))`` order.

    Attributes
    ----------
    descending: bool
        Sort in descending order (default True).
    """

    key_row = 1
