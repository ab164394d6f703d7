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
``EdgeSetOperator`` keeps the CUDA arrays and applies the matrix to node fields (``ops.csr_spmm``: ``agx_csr_spmm``).
"""

from __future__ import annotations

import logging
import warnings
from pathlib import Path
from typing import NamedTuple

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
    csr = _device_csr(graph, edges_name, edge_attribute_name)
    if csr.on_device:
        return torch.sparse_csr_tensor(csr.indptr.to(torch.int32), csr.indices, csr.data, size=csr.shape, check_invariants=False)
    from scipy.sparse import csr_matrix

    return csr_matrix((csr.data.cpu().numpy(), csr.indices.cpu().numpy(), csr.indptr.cpu().numpy()), shape=csr.shape)


class _DeviceCSR(NamedTuple):
    name: tuple[str, str, str]
    shape: tuple[int, int]  # (num target nodes, num source nodes)
    indptr: torch.Tensor
    indices: torch.Tensor
    data: torch.Tensor
    on_device: bool  # edge_index lives on the GPU


def _device_csr(graph, edges_name, edge_attribute_name: str | None) -> _DeviceCSR:
    """The CUDA CSR arrays of ``edge_set_to_sparse``, with its checks."""
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
    return _DeviceCSR(name, (n_dst, n_src), indptr, indices, data, bool(edge_index.is_cuda))


class EdgeSetOperator:
    """The matrix of one edge set (``edge_set_to_sparse``) as an operator on node fields: ``op(x)`` maps a field on
    the source nodes to one on the target nodes, ``y[t] = sum over the entries (t, s) of M[t, s] * x[s]``.  With
    ``GaussianDistanceWeights`` on a KNN edge set the rows sum to 1 and ``op`` interpolates.

    The CSR is built once on the GPU (``ops.edges_to_csr``) and kept there; every call is one ``agx_csr_spmm``.
    Each element of ``y`` is a float32 sum over its row in ascending source order, ``acc = fmaf(M[t, s], x[s], acc)``
    from +0, rounded once to x's dtype (float32 or bfloat16): bit-identical from call to call, and between host- and
    device-resident graphs.  An empty row gives +0; NaN and inf reach only the rows that reference them.

    Attributes
    ----------
    shape : tuple[int, int]
        ``(num_nodes[target], num_nodes[source])``.

    Raises ``ValueError`` for a bool attribute (a bool matrix is not an operator) and for the attribute errors of
    ``edge_set_to_sparse``, ``KeyError`` for an edge set or attribute the graph does not have, ``NotImplementedError``
    for a sharded block of a device-resident graph.
    """

    def __init__(self, graph, edges_name, edge_attribute_name: str | None = None) -> None:
        csr = _device_csr(graph, edges_name, edge_attribute_name)
        if csr.data.dtype == torch.bool:
            raise ValueError(
                f"The edge attribute '{edge_attribute_name}' of {csr.name} is bool: a bool matrix is not an operator; "
                "use a float32 attribute."
            )
        self.name = csr.name
        self.shape = csr.shape
        self._indptr, self._indices, self._data = csr.indptr, csr.indices, csr.data

    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        """``M x`` for a float32 or bfloat16 field ``x`` of shape (num_nodes[source], F) or (num_nodes[source],), on
        the GPU or the host; ``y`` has shape (num_nodes[target], F) or (num_nodes[target],), x's dtype, and lives
        where x lives (a host x is uploaded and the result copied back).  ValueError for an x of another dtype, of more
        than two dimensions, or whose first dimension is not num_nodes[source]."""
        if x.dim() not in (1, 2):
            raise ValueError(f"{self.name}: a node field has shape (N,) or (N, F), got {tuple(x.shape)}.")
        if x.dtype not in ops.SPMM_DTYPES:
            raise ValueError(f"{self.name}: a node field must be float32 or bfloat16, got {x.dtype}.")
        if x.shape[0] != self.shape[1]:
            raise ValueError(f"{self.name}: x has {x.shape[0]} rows, the source node set has {self.shape[1]} nodes.")
        y = ops.csr_spmm(self._indptr, self._indices, self._data, x.to(self._indptr.device), self.shape[0])
        return y.to(x.device)


def apply_edge_set(graph, edges_name, x: torch.Tensor, edge_attribute_name: str | None = None) -> torch.Tensor:
    """``EdgeSetOperator(graph, edges_name, edge_attribute_name)(x)``: one field through an edge set's matrix.  To
    apply one edge set to several fields, build the operator once."""
    return EdgeSetOperator(graph, edges_name, edge_attribute_name)(x)


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
