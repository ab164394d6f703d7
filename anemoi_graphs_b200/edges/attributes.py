"""Edge attributes (/root/reference/src/anemoi/graphs/edges/attributes.py:24-157).

``EdgeLength`` and ``EdgeDirection`` keep the reference's constructor arguments and ``compute(graph,
edges_name)`` contract (float32 ``(E, 1)`` / ``(E, 2)`` tensors, normalised over the whole edge set).
Raw values, the global reduction for the normalisation and the final float32 cast are one fused CUDA
kernel pair (``ops.edge_attributes``); when both attributes are requested for an edge set
(``compute_attributes``) they share a single pass over ``edge_index``.

``Azimuth``, ``GaussianDistanceWeights``, ``AttributeFromSourceNode`` and ``AttributeFromTargetNode`` carry the names
of edge attributes of newer anemoi-graphs releases, which the pinned reference does not have: their semantics follow
the upstream classes as far as is known, unverified against their source (DESIGN.md).  They need the final node
numbering (a canonical order by target, or rows of a node attribute) and are evaluated after ``EdgeLength`` /
``EdgeDirection`` of the same edge set.
"""

from __future__ import annotations

import math
from abc import ABC

import torch

from .. import device as _device
from .. import ops
from .._cabi import NORM_CODES
from ..processors.post_process import _refuse_sharded


def _check_norm(norm) -> None:
    if norm not in NORM_CODES:
        # normalise.py:53-55
        raise ValueError(
            f"Attribute normalisation \"{norm}\" is not valid. Options are: 'l1', 'l2', 'unit-max' or 'unit-std'."
        )


class BaseEdgeAttribute(ABC):
    """Base class for edge attributes."""

    _agx_device_aware = True

    def __init__(self, norm: str | None = None) -> None:
        self.norm = norm

    def _kernel_args(self) -> dict:
        raise NotImplementedError

    def _pick(self, length, direction) -> torch.Tensor:
        raise NotImplementedError

    def compute(self, graph, edges_name: tuple[str, str, str], *args, **kwargs) -> torch.Tensor:
        """Compute the edge attributes."""
        out = compute_attributes(graph, edges_name, {"value": self})["value"]
        _device.maybe_flush()
        return out


class EdgeDirection(BaseEdgeAttribute):
    """Edge direction feature (edges/attributes.py:56-104).

    1. Rotated features: the target nodes are rotated to the north pole to compute the edge direction.
    2. Non-rotated features: difference in latitude and longitude between the source and target nodes.

    Attributes
    ----------
    norm : Optional[str]
        Normalisation method. Options: None, "l1", "l2", "unit-max", "unit-range", "unit-std".
    luse_rotated_features : bool
        Whether to use rotated features.
    """

    def __init__(self, norm: str | None = None, luse_rotated_features: bool = True) -> None:
        super().__init__(norm)
        self.luse_rotated_features = luse_rotated_features

    def _kernel_args(self) -> dict:
        return dict(direction=True, direction_norm=self.norm, direction_rotated=bool(self.luse_rotated_features))

    def _pick(self, length, direction):
        return direction


class EdgeLength(BaseEdgeAttribute):
    """Edge length feature: haversine distance on the unit sphere (edges/attributes.py:107-157).

    Attributes
    ----------
    norm : Optional[str]
        Normalisation method. Options: None, "l1", "l2", "unit-max", "unit-range", "unit-std".
    invert : bool
        Whether to invert the edge lengths, i.e. 1 - edge_length. Defaults to False.
    """

    def __init__(self, norm: str | None = None, invert: bool = False) -> None:
        super().__init__(norm)
        self.invert = invert

    def _kernel_args(self) -> dict:
        return dict(length=True, length_norm=self.norm, length_invert=bool(self.invert))

    def _pick(self, length, direction):
        return length


def _check_nodes(graph, edges_name) -> tuple[str, str]:
    source_name, _, target_name = edges_name
    assert (
        source_name in graph.node_types
    ), f"Node \"{source_name}\" not found in graph. Optional nodes are {', '.join(graph.node_types)}."
    assert (
        target_name in graph.node_types
    ), f"Node \"{target_name}\" not found in graph. Optional nodes are {', '.join(graph.node_types)}."
    return source_name, target_name


def compute_attributes(graph, edges_name: tuple[str, str, str], attrs: dict) -> dict:
    """Evaluate a set of attribute objects on one edge set.

    Pairs one ``EdgeLength`` with one ``EdgeDirection`` per kernel pass; foreign attribute objects (anything
    with a ``compute(graph, edges_name)`` method) are called as the reference would call them
    (edges/builder.py:133).  The edge-list attributes (``EdgeListAttribute``) follow, in final numbering."""
    listed = {k: a for k, a in attrs.items() if isinstance(a, EdgeListAttribute)}
    if not listed:
        return _fused_attributes(graph, edges_name, attrs)
    if _device.sharded_output() or "edge_shard" in graph[tuple(edges_name)]:
        _refuse_sharded(tuple(edges_name))
    _check_nodes(graph, edges_name)
    out = _fused_attributes(graph, edges_name, {k: a for k, a in attrs.items() if k not in listed})
    out.update(_edge_list_attributes(graph, edges_name, listed))
    return {k: out[k] for k in attrs}  # the recipe's order


def _fused_attributes(graph, edges_name: tuple[str, str, str], attrs: dict) -> dict:
    """``EdgeLength`` / ``EdgeDirection`` (K5) and foreign attribute objects."""
    ours = {k: a for k, a in attrs.items() if isinstance(a, (EdgeLength, EdgeDirection))}
    out: dict = {}
    for k, a in attrs.items():
        if k not in ours:
            # a foreign (reference-style plugin) attribute may read ``x`` / ``edge_index`` on the host: give every
            # provisional node set its final order and wait for the pending device->host copies first
            _device.flush()
            out[k] = a.compute(graph, edges_name)
    if not ours:
        return out
    source_name, target_name = _check_nodes(graph, edges_name)
    for a in ours.values():
        _check_norm(a.norm)
    store = graph[tuple(edges_name)]
    edge_index = _device.device_edge_index(store)
    host_side = not store["edge_index"].is_cuda
    # A row of the edge list may still be in the provisional numbering of its node set (device.Provisional): the
    # attributes depend on coordinates only, so they are evaluated right away against the matching (provisional)
    # node records.  Anything else - final rows against a provisional node set - needs the final order first.
    meta = _device.edge_meta(edge_index)
    # KNN edges whose index-order ties are re-decided when the node order resolves: evaluated NOW (the trigonometry
    # runs in the shadow of the host sort) with the re-decided targets' edges kept out of the statistics; those edges
    # are evaluated again after the re-decision and the normalisation is applied then (``_deferred_attributes``)
    pending = meta.fixup if meta is not None else None
    if pending is not None and pending.done:
        pending = None
    _, w = _device.world()
    if pending is not None and ((w > 1 and not _device.sharded_output()) or meta.tie_flags is None or len(ours) > 2):
        pending.resolve()
        pending = None
    tags = _device.row_tags(edge_index)
    for row, name in ((0, source_name), (1, target_name)):
        prov = _device.active_provisional(graph[name])
        if prov is not None and tags[row] is not prov:
            prov.resolve()
    if source_name == target_name and tags[0] is not tags[1]:
        for prov in tags:
            if prov is not None:
                prov.resolve()
    src = _device.node_tables(graph[source_name], provisional_ok=True)
    dst = _device.node_tables(graph[target_name], provisional_ok=True)
    lengths = [(k, a) for k, a in ours.items() if isinstance(a, EdgeLength)]
    dirs = [(k, a) for k, a in ours.items() if isinstance(a, EdgeDirection)]
    if pending is not None and len(lengths) <= 1 and len(dirs) <= 1:
        out.update(_deferred_attributes(pending, meta, edge_index, src, dst, lengths, dirs, host_side))
        return {k: out[k] for k in attrs}
    if pending is not None:
        pending.resolve()
        src = _device.node_tables(graph[source_name], provisional_ok=True)
        dst = _device.node_tables(graph[target_name], provisional_ok=True)
    local = meta.local if meta is not None else None  # set by a sharded builder: this rank's own columns
    while lengths or dirs:
        kl = lengths.pop(0) if lengths else None
        kd = dirs.pop(0) if dirs else None
        shard = meta.shard if (meta is not None and _device.sharded_output()) else None
        args = dict(length=False, direction=False, sharded=w > 1, local=local, shard=shard,
                    regular_k=meta.regular_k if meta is not None else 0)
        if kl:
            args.update(kl[1]._kernel_args())
        if kd:
            args.update(kd[1]._kernel_args())
        ln, dr = ops.edge_attributes(edge_index, src, dst, **args)
        if kl:
            out[kl[0]] = _device.to_host(ln, shard) if host_side else ln
        if kd:
            out[kd[0]] = _device.to_host(dr, shard) if host_side else dr
    return {k: out[k] for k in attrs}  # the recipe's order


def _deferred_attributes(prov, meta, edge_index, src, dst, lengths, dirs, host_side: bool) -> dict:
    """One EdgeLength and/or one EdgeDirection of an edge set that still waits for a KNN tie re-decision: raw pass now,
    the re-decided edges again when the order resolves (a fixup: still provisional numbering, the same node records),
    scaling and host copies after that (a finalizer).  Returns the tensors the graph stores: device tensors that are
    complete in stream order, or pinned host tensors that are complete at ``flush()``."""
    args = dict(length=False, direction=False)
    for _, a in lengths + dirs:
        args.update(a._kernel_args())
    flag_list, flag_count = meta.tie_list if meta.tie_list is not None else (None, None)
    job = ops.DeferredEdgeAttributes(
        edge_index, src, dst, meta.tie_flags, flag_list=flag_list, flag_count=flag_count, regular_k=meta.regular_k,
        flag_base=meta.flag_base, shard=meta.shard, **args
    )
    job.raw()
    prov.add_fixup(lambda p, job=job: job.patch())  # registered after the builder's re-decision: runs after it
    results, host_targets = {}, []
    for name, _ in lengths:
        results[name] = job.out_len
    for name, _ in dirs:
        results[name] = job.out_dir
    if host_side:
        shard = meta.shard if (meta.shard is not None and _device.sharded_output()) else None
        for name, dev_out in list(results.items()):
            if shard is None:
                host = dest = torch.empty(dev_out.shape, dtype=dev_out.dtype, pin_memory=True)
            else:  # the complete array in the shared host buffer; this rank fills its rows
                host = _device.host_tensor((shard.total, int(dev_out.shape[1])), dev_out.dtype, require_shared=True)
                dest = host[shard.offset : shard.offset + int(dev_out.shape[0])]
            host_targets.append((dev_out, dest))
            results[name] = host

    def finalize(p, job=job, host_targets=host_targets):
        job.apply()
        for dev_out, dest in host_targets:
            _device.to_host_into(dev_out, dest)

    prov.add_finalizer(finalize)
    return results


# ------------------------------------------------------------------------------------------------
# attributes of newer anemoi-graphs releases: evaluated on the complete edge list in final numbering
# ------------------------------------------------------------------------------------------------
class EdgeListAttribute(BaseEdgeAttribute):
    """An edge attribute that reads the complete device edge list of its edge set in final node numbering."""

    def evaluate(self, graph, edges_name, edge_index: torch.Tensor) -> torch.Tensor:
        """The CUDA result for the CUDA int32 (2, E) ``edge_index`` (final numbering, not yet checked)."""
        raise NotImplementedError


def _check_endpoints(edge_index: torch.Tensor, n_src: int, n_dst: int) -> None:
    """ValueError unless every source is in [0, n_src) and every target in [0, n_dst) - one read-back."""
    if edge_index.shape[1] == 0:
        return
    lo, hi = torch.aminmax(edge_index, dim=1)
    (s_lo, d_lo), (s_hi, d_hi) = torch.stack([lo, hi]).tolist()
    if s_lo < 0 or d_lo < 0 or s_hi >= n_src or d_hi >= n_dst:
        raise ValueError("an edge endpoint is outside [0, num_nodes) of its node set")


def _edge_list_attributes(graph, edges_name, attrs: dict) -> dict:
    source_name, _, target_name = edges_name
    store = graph[tuple(edges_name)]
    reference_input = store["edge_index"]
    edge_index = _device.device_edge_index(store)  # before the order resolves: it relabels this very tensor
    meta = _device.edge_meta(edge_index)
    for prov in (meta.fixup if meta is not None else None, *_device.row_tags(edge_index),
                 _device.active_provisional(graph[source_name]), _device.active_provisional(graph[target_name])):  # fmt: skip
        if prov is not None:
            prov.resolve()
    _device.wait_for(edge_index)
    return {k: _device.like_input(a.evaluate(graph, edges_name, edge_index), reference_input) for k, a in attrs.items()}


class Azimuth(EdgeListAttribute):
    """Initial bearing at the target node towards the source node, in radians, clockwise from north, in [-pi, pi]:
    ``atan2(sin(dlon) cos(lat_s), cos(lat_t) sin(lat_s) - sin(lat_t) cos(lat_s) cos(dlon))``, dlon = lon_s - lon_t,
    in float64 from the float32 coordinates, stored as float32 (E, 1).  As the upstream ``Azimuth.compute(x_i, x_j)``
    with i = target, j = source, as far as is known.

    Attributes
    ----------
    norm : Optional[str]
        Normalisation over the whole edge set, as for ``EdgeLength``. Options: None, "l1", "l2", "unit-max",
        "unit-range", "unit-std".
    """

    def __init__(self, norm: str | None = None) -> None:
        _check_norm(norm)
        super().__init__(norm)

    def evaluate(self, graph, edges_name, edge_index):
        source_name, _, target_name = edges_name
        src_x = _device.node_state(graph[source_name]).x
        dst_x = _device.node_state(graph[target_name]).x
        return ops.edge_azimuth(edge_index, src_x, dst_x, self.norm)


class GaussianDistanceWeights(EdgeListAttribute):
    """Gaussian weights of the edge lengths, normalised per target node: w = exp(-d^2 / (2 sigma^2)), d the float32
    ``EdgeLength(norm=None)`` value on the unit sphere, in float64; ``norm`` is applied to the edges of each target
    node as normalise.py applies it to a whole array (a NaN weight makes its group NaN; under "unit-std" a group of
    bit-equal weights is left unnormalised), rounded to float32 (E, 1) once.  The result does not depend on the order
    of the columns of ``edge_index``.  As the upstream class, as far as is known.

    Attributes
    ----------
    sigma : float
        Width of the Gaussian, in radians. Default 1.0.
    norm : Optional[str]
        Normalisation per target node. Options: None, "l1", "l2", "unit-max", "unit-range", "unit-std". Default "l1".
    """

    def __init__(self, sigma: float = 1.0, norm: str | None = "l1") -> None:
        assert isinstance(sigma, (int, float)) and not isinstance(sigma, bool), "sigma must be a number"
        assert sigma > 0, "sigma must be positive"
        _check_norm(norm)
        super().__init__(norm)
        self.sigma = sigma

    def evaluate(self, graph, edges_name, edge_index):
        source_name, _, target_name = edges_name
        n_src, n_dst = int(graph[source_name].num_nodes), int(graph[target_name].num_nodes)
        perm = None
        if self.norm is None:
            _check_endpoints(edge_index, n_src, n_dst)
        else:  # the canonical order; checks the endpoints
            perm = ops.sort_permutation(edge_index[1], edge_index[0], n_dst, n_src, descending=False)
        meta = _device.edge_meta(edge_index)
        src = _device.node_tables(graph[source_name])
        dst = _device.node_tables(graph[target_name])
        lengths, _ = ops.edge_attributes(edge_index, src, dst, length=True, length_norm=None, direction=False,
                                         regular_k=meta.regular_k if meta is not None else 0)  # fmt: skip
        return ops.gaussian_weights(edge_index, n_src, n_dst, lengths, self.sigma, self.norm, perm)


class _AttributeFromNode(EdgeListAttribute):
    row: int

    def __init__(self, node_attr_name: str) -> None:
        assert isinstance(node_attr_name, str), "node_attr_name must be a str"
        super().__init__(None)
        self.node_attr_name = node_attr_name

    def evaluate(self, graph, edges_name, edge_index):
        nodes_name = edges_name[0] if self.row == 0 else edges_name[2]
        nodes = graph[nodes_name]
        n = int(nodes.num_nodes)
        value = nodes.get(self.node_attr_name, None) if hasattr(nodes, "get") else None
        if not isinstance(value, torch.Tensor) or value.dim() == 0 or value.shape[0] != n:
            what = f"shape {tuple(value.shape)}" if isinstance(value, torch.Tensor) else "missing"
            raise ValueError(f"The node attribute '{self.node_attr_name}' of {nodes_name} must be a tensor with {n} rows ({what}).")
        _check_endpoints(edge_index, int(graph[edges_name[0]].num_nodes), int(graph[edges_name[2]].num_nodes))
        rows = _device.to_device(value.reshape(n, math.prod(value.shape[1:]))).bool().view(torch.uint8).contiguous()
        out = torch.empty((int(edge_index.shape[1]), int(rows.shape[1])), dtype=torch.bool, device=edge_index.device)
        ops.gather_rows([(rows, out.view(torch.uint8))], edge_index[self.row])
        return out


class AttributeFromSourceNode(_AttributeFromNode):
    """The source node's row of a node attribute, as a bool edge attribute: ``graph[source][node_attr_name]`` at
    ``edge_index[0]``, (E, 1) for an (N,) attribute and (E, M) for an (N, M) one, cast as ``Tensor.bool()`` casts.
    As the upstream class (a mask such as CutOutMask carried onto the edges), as far as is known.

    Attributes
    ----------
    node_attr_name : str
        Name of the source node attribute.
    """

    row = 0


class AttributeFromTargetNode(_AttributeFromNode):
    """The target node's row of a node attribute, as a bool edge attribute: ``graph[target][node_attr_name]`` at
    ``edge_index[1]``, (E, 1) for an (N,) attribute and (E, M) for an (N, M) one, cast as ``Tensor.bool()`` casts.
    As the upstream class, as far as is known.

    Attributes
    ----------
    node_attr_name : str
        Name of the target node attribute.
    """

    row = 1
