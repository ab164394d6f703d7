"""Edge sets as sparse matrices: the ``export_to_sparse`` command of newer anemoi-graphs releases, as far as is known.

The pinned reference has no such command, so upstream parity is unverified.  The layout is the reference's own
intermediate form, ``BaseEdgeBuilder.get_adjacency_matrix`` (edges/builder.py:63): rows are targets, columns sources.
For an edge set ``(S, "to", T)`` and an optional edge attribute ``a`` the matrix has shape
``(num_nodes[T], num_nodes[S])`` and ``M[dst_e, src_e] += v_e``, with ``v_e = a[e]`` or 1 - the CSR that
``scipy.sparse.coo_matrix((v, (edge_index[1], edge_index[0])), shape).tocsr()`` followed by ``sum_duplicates()`` gives:
int64 ``indptr``, int32 ``indices`` ascending within each row, duplicate pairs summed in the order their columns appear
(bool: OR).  Values keep the attribute's dtype (float32 or bool); without an attribute they are float32 ones.

The CSR arrays are built on the GPU (``ops.edges_to_csr``: ``agx_sort_edges`` + ``agx_edges_to_csr``).  A
device-resident graph gets a CUDA ``torch.sparse_csr_tensor``; a host-resident one a ``scipy.sparse.csr_matrix``.
"""

from __future__ import annotations

import logging
import warnings
from pathlib import Path

import torch

from . import device as _device
from . import ops
from .processors.post_process import _check_gathered

LOGGER = logging.getLogger(__name__)


def _edge_values(store, edges_name, edge_attribute_name: str | None, n_edges: int) -> torch.Tensor | None:
    """The attribute as an (E,) float32 / bool tensor where it lives, or None for ones."""
    if edge_attribute_name is None:
        return None
    value = store[edge_attribute_name]
    if not isinstance(value, torch.Tensor) or value.shape not in ((n_edges,), (n_edges, 1)):
        what = f"shape {tuple(value.shape)}" if isinstance(value, torch.Tensor) else type(value).__name__
        raise ValueError(
            f"The edge attribute '{edge_attribute_name}' of {edges_name} must have one value per edge, shape "
            f"({n_edges},) or ({n_edges}, 1); got {what}."
        )
    if value.dtype not in (torch.float32, torch.bool):
        raise ValueError(f"The edge attribute '{edge_attribute_name}' of {edges_name} must be float32 or bool, got {value.dtype}.")
    return value.reshape(n_edges)


def edge_set_to_sparse(graph, edges_name, edge_attribute_name: str | None = None):
    """The (num target nodes x num source nodes) matrix of one edge set, ``M[target, source]`` = the attribute
    ``edge_attribute_name`` (summed over duplicate edges), or 1 per edge without one.

    A CUDA ``torch.sparse_csr_tensor`` (int32 ``crow_indices`` / ``col_indices``) when ``edge_index`` is on the GPU, a
    ``scipy.sparse.csr_matrix`` when it is on the host (built on the GPU and copied back).

    Raises ``ValueError`` for an attribute that is not float32 / bool with shape (E,) or (E, 1) and for an endpoint
    outside its node set, ``NotImplementedError`` for a sharded block of a device-resident graph, ``KeyError`` for an
    edge set or attribute the graph does not have.
    """
    name = _edge_type(edges_name)
    if name not in graph.edge_types:
        raise KeyError(f"The graph has no edge set {name}; it has {graph.edge_types}.")
    store = graph[name]
    _check_gathered(name, store)
    if edge_attribute_name is not None and edge_attribute_name not in store:
        raise KeyError(f"The edge set {name} has no attribute '{edge_attribute_name}'.")
    edge_index = store["edge_index"]
    n_edges = int(edge_index.shape[1])
    n_dst, n_src = int(graph[name[2]].num_nodes), int(graph[name[0]].num_nodes)
    values = _edge_values(store, name, edge_attribute_name, n_edges)
    _device.flush()  # every node set in its final numbering, every pending copy and collective complete
    values = None if values is None else _device.to_device(values)
    indptr, indices, data = ops.edges_to_csr(_device.to_device(edge_index, torch.int32), n_dst, n_src, values)
    if edge_index.is_cuda:
        return torch.sparse_csr_tensor(indptr.to(torch.int32), indices, data, size=(n_dst, n_src), check_invariants=False)
    from scipy.sparse import csr_matrix

    return csr_matrix((data.cpu().numpy(), indices.cpu().numpy(), indptr.cpu().numpy()), shape=(n_dst, n_src))


def _edge_type(name) -> tuple[str, str, str]:
    name = tuple(name)
    if len(name) == 2:
        return name[0], "to", name[1]
    if len(name) == 3 and name[1] == "to":
        return name
    raise ValueError(f"An edge set is named (source, target) or (source, 'to', target), got {name}.")


class GraphExporter:
    """Write edge sets as scipy sparse matrices, one compressed ``.npz`` file per edge set
    (``output_path/<source>_to_<target>.npz``, ``scipy.sparse.save_npz``); see ``edge_set_to_sparse``.

    Attributes
    ----------
    graph : str | Path | graph
        A graph saved as ``.pt`` or a graph object.
    output_path : str | Path
        Directory of the files (created if missing).
    edges_name : list, optional
        The edge sets, as (source, target) pairs or (source, "to", target) keys; None = every edge set.
    edge_attribute_name : str, optional
        Edge attribute that gives the values; None = 1 per edge.  Edge sets without it are skipped with a warning.
    """

    def __init__(self, graph, output_path, edges_name=None, edge_attribute_name: str | None = None) -> None:
        self.graph = graph
        self.output_path = Path(output_path)
        self.edges_name = None if edges_name is None else [_edge_type(n) for n in edges_name]
        self.edge_attribute_name = edge_attribute_name

    def export(self) -> list[Path]:
        """Write the files; returns their paths."""
        from scipy.sparse import csr_matrix
        from scipy.sparse import save_npz

        graph = self.graph
        if isinstance(graph, (str, Path)):
            from .describe import load_graph

            graph = load_graph(graph)
        names = graph.edge_types if self.edges_name is None else self.edges_name
        for name in names:
            if name not in graph.edge_types:
                raise KeyError(f"The graph has no edge set {name}; it has {graph.edge_types}.")
        attr = self.edge_attribute_name
        skipped = [name for name in names if attr is not None and attr not in graph[name]]
        if skipped:
            warnings.warn(f"Edge sets without the attribute '{attr}' are skipped: {skipped}", stacklevel=2)
        self.output_path.mkdir(parents=True, exist_ok=True)
        written = []
        for name in names:
            if name in skipped:
                continue
            matrix = edge_set_to_sparse(graph, name, attr)
            if isinstance(matrix, torch.Tensor):
                matrix = csr_matrix(
                    (matrix.values().cpu().numpy(), matrix.col_indices().cpu().numpy(), matrix.crow_indices().cpu().numpy()),
                    shape=tuple(matrix.shape),
                )  # fmt: skip
            path = self.output_path / f"{name[0]}_to_{name[2]}.npz"
            save_npz(path, matrix)
            LOGGER.info(f"Edge set {name} written to {path} ({matrix.nnz} entries).")
            written.append(path)
        return written
