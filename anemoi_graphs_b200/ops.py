"""Device-level operations: thin, typed wrappers over the C ABI working on CUDA tensors.

These are the calls the builders (``edges/builder.py``, ``edges/attributes.py``, ``nodes/builders.py``)
make; PyTorch is used only to own device memory and streams.  Everything here requires a CUDA
device - there is no CPU fallback.
"""

from __future__ import annotations

import ctypes
import math
from ctypes import byref, c_double, c_int, c_int32, c_int64, c_void_p

import torch

from . import _cabi
from ._cabi import NORM_CODES, check, current_stream, load_library, ptr


class Timeline:
    """CUDA-event stopwatch around the C-ABI calls (``bench.py`` switches it on to time each kernel live,
    on the stream the kernel is launched on).  ``spans[name]`` collects (start, end) event pairs."""

    def __init__(self) -> None:
        self.spans: dict[str, list] = {}
        self.units: dict[str, float] = {}

    def record(self, name: str, start, end, units: float = 0.0) -> None:
        self.spans.setdefault(name, []).append((start, end))
        self.units[name] = self.units.get(name, 0.0) + units

    def totals_ms(self) -> dict[str, float]:
        torch.cuda.synchronize()
        return {k: sum(a.elapsed_time(b) for a, b in v) for k, v in self.spans.items()}

    def counts(self) -> dict[str, int]:
        return {k: len(v) for k, v in self.spans.items()}


timeline: Timeline | None = None


class _span:
    def __init__(self, name: str, units: float = 0.0) -> None:
        self.name, self.units = name, units

    def __enter__(self):
        if timeline is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.start.record()
        return self

    def __exit__(self, *exc):
        if timeline is not None:
            end = torch.cuda.Event(enable_timing=True)
            end.record()
            timeline.record(self.name, self.start, end, self.units)


def _dev_x(x: torch.Tensor) -> torch.Tensor:
    """float32 (n, 2) contiguous CUDA coordinates."""
    _cabi.require_cuda()
    if not x.is_cuda:
        x = x.cuda(non_blocking=True)
    if x.dtype != torch.float32:
        x = x.to(torch.float32)
    assert x.dim() == 2 and x.shape[1] == 2, f"coordinates must have shape (N, 2), got {tuple(x.shape)}"
    return x.contiguous()


def _row_ptrs(out: torch.Tensor, col: int, swap_rows: bool) -> tuple[int, int]:
    """Addresses of column ``col`` of the rows the search writes its reference points and its queries to: rows 0 and 1
    of the (2, E) int32 ``out``, or rows 1 and 0."""
    row0 = out.data_ptr() + 4 * col
    row1 = row0 + 4 * out.shape[1]
    return (row1, row0) if swap_rows else (row0, row1)


class NeighbourIndex:
    """Cell-binned reference point set - the stand-in for a fitted ``NearestNeighbors(metric="haversine")``
    (/root/reference/src/anemoi/graphs/edges/builder.py:259-260, 364-365)."""

    def __init__(self, x: torch.Tensor, cells_per_face: int = 0, hint_k: int = 0, hint_radius: float = 0.0) -> None:
        self.lib = load_library()
        self.x = _dev_x(x)  # kept alive: the index reads it during float64 refinement
        self.n = int(self.x.shape[0])
        handle = c_void_p()
        with _span("index_build", self.n):
            check(
                self.lib.agx_index_build(
                    ptr(self.x), self.n, int(cells_per_face), int(hint_k), float(hint_radius), current_stream(),
                    byref(handle),
                )
            )  # fmt: skip
        self.handle = handle

    @property
    def cells_per_face(self) -> int:
        n, c = c_int64(), c_int()
        check(self.lib.agx_index_info(self.handle, byref(n), byref(c)))
        return c.value

    def close(self) -> None:
        if getattr(self, "handle", None):
            self.lib.agx_index_free(self.handle, current_stream())
            self.handle = None

    def __del__(self) -> None:  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self) -> "NeighbourIndex":
        return self

    def __exit__(self, *exc) -> None:
        self.close()

    # ------------------------------------------------------------------------------------------
    def knn(
        self,
        q: torch.Tensor,
        k: int,
        dst_base: int = 0,
        return_rdist: bool = False,
        stats: torch.Tensor | None = None,
        out: torch.Tensor | None = None,
        out_offset: int = 0,
        tag: str = "knn",
        max_radius: float = 0.0,
        tie_flags: torch.Tensor | None = None,
        swap_rows: bool = False,
    ):
        """``edge_index`` (2, nq*k) int32 - row 0 the k nearest reference points of each query, row 1
        ``dst_base + query`` - and optionally the float64 ``rdist`` (nq, k).  With ``out`` (a larger
        contiguous (2, E) int32 buffer) the block is written at column ``out_offset`` instead.  Each query's k sources
        are a SET; only with ``return_rdist`` is a row ordered, ascending (rdist, index).  ``max_radius`` (radians,
        0 = unlimited) bounds the search: exact for queries whose k-th neighbour is within it; any other query gets
        every point within it, and -1 / +inf or points beyond it in the other slots (``agx_b200.h``).  ``tie_flags``
        (zeroed uint8 (nq,)) marks the queries whose result depends on the numbering of the reference points
        (``agx_knn_flagged``).  ``swap_rows``: the kernel writes the queries to row 0 and the reference points to row 1
        (reversed edge builders: the queries are the sources)."""
        q = _dev_x(q)
        nq = int(q.shape[0])
        if out is None:
            out = torch.empty((2, nq * k), dtype=torch.int32, device=q.device)
            out_offset = 0
        assert out.dim() == 2 and out.shape[0] == 2 and out.dtype == torch.int32 and out.is_contiguous()
        assert 0 <= out_offset and out_offset + nq * k <= out.shape[1]
        rdist = torch.empty((nq, k), dtype=torch.float64, device=q.device) if return_rdist else None
        ref_row, q_row = _row_ptrs(out, out_offset, swap_rows)
        with _span(tag, nq * k):
            check(
                self.lib.agx_knn_flagged(
                    self.handle, ptr(q), nq, int(k), float(max_radius), ref_row, q_row, int(dst_base), ptr(rdist),
                    ptr(stats), ptr(tie_flags), current_stream(),
                )
            )  # fmt: skip
        return (out, rdist) if return_rdist else out

    def knn_redecide(
        self, q: torch.Tensor, k: int, out: torch.Tensor, tie_flags: torch.Tensor, rank: torch.Tensor | None = None,
        order: torch.Tensor | None = None,
    ) -> None:  # fmt: skip
        """Search only the queries flagged in ``tie_flags`` and overwrite their sources in row 0 of ``out``
        (``agx_knn_redecide``).  With ``rank`` / ``order`` (CUDA int64 inverse permutations) this index is still the
        one over the PROVISIONALLY numbered points: ties go to the lower final label ``rank[label]`` and provisional
        labels are written back (``agx_knn_redecide_ranked``) - no second index over the re-ordered points."""
        q = _dev_x(q)
        nq = int(q.shape[0])
        assert out.shape == (2, nq * k) and out.dtype == torch.int32 and out.is_contiguous()
        assert tie_flags.shape == (nq,) and tie_flags.dtype == torch.uint8
        assert tie_flags.is_cuda and tie_flags.is_contiguous()  # the library checks the 16-byte alignment
        with _span("knn_ties", nq):
            if rank is None:
                check(self.lib.agx_knn_redecide(self.handle, ptr(q), nq, int(k), 0.0, out.data_ptr(), ptr(tie_flags), current_stream()))
            else:
                assert rank.dtype == torch.int64 and order.dtype == torch.int64 and rank.numel() >= self.n and order.numel() >= self.n
                check(
                    self.lib.agx_knn_redecide_ranked(
                        self.handle, ptr(q), nq, int(k), 0.0, out.data_ptr(), ptr(tie_flags), ptr(rank), ptr(order),
                        current_stream(),
                    )
                )

    def knn_redecide_list(
        self, q: torch.Tensor, k: int, out: torch.Tensor, flag_list: torch.Tensor, flag_count: torch.Tensor,
        rank: torch.Tensor | None = None, order: torch.Tensor | None = None, swap_rows: bool = False,
    ) -> None:  # fmt: skip
        """``knn_redecide`` driven by the ascending list of flagged query ids (``compact_flags``): one thread per
        listed query (``agx_knn_redecide_list``).  ``swap_rows``: ``out`` came from ``knn(..., swap_rows=True)``, its
        reference points are row 1."""
        q = _dev_x(q)
        nq = int(q.shape[0])
        assert out.shape == (2, nq * k) and out.dtype == torch.int32 and out.is_contiguous()
        assert flag_list.dtype == torch.int32 and flag_count.dtype == torch.int64
        with _span("knn_ties", nq):
            check(
                self.lib.agx_knn_redecide_list(
                    self.handle, ptr(q), nq, int(k), 0.0, _row_ptrs(out, 0, swap_rows)[0], ptr(flag_list),
                    ptr(flag_count), ptr(rank), ptr(order), current_stream(),
                )
            )  # fmt: skip

    def radius_count(self, q: torch.Tensor, radius: float) -> tuple[torch.Tensor, int]:
        """Pass 1 of the cut-off search: ``(offsets (nq+1,) int64, total)``."""
        q = _dev_x(q)
        nq = int(q.shape[0])
        counts = torch.empty(nq, dtype=torch.int32, device=q.device)
        offsets = torch.empty(nq + 1, dtype=torch.int64, device=q.device)
        stream = current_stream()
        with _span("radius_count", nq):
            check(self.lib.agx_radius_count(self.handle, ptr(q), nq, float(radius), ptr(counts), stream))
        total = c_int64()
        check(self.lib.agx_exclusive_scan(ptr(counts), nq, ptr(offsets), byref(total), stream))
        return offsets, int(total.value)

    def radius_capped(self, q: torch.Tensor, radius: float, max_neighbours: int) -> tuple[torch.Tensor, int, torch.Tensor]:
        """Pass 1 of the capped cut-off search: ``(offsets (nq+1,) int64, total, counts (nq,) int32)`` - the offsets
        and total of at most ``max_neighbours`` pairs per query, and the uncapped counts ``radius_fill`` takes with
        them."""
        q = _dev_x(q)
        nq = int(q.shape[0])
        counts = torch.empty(nq, dtype=torch.int32, device=q.device)
        capped = torch.empty(nq, dtype=torch.int32, device=q.device)
        offsets = torch.empty(nq + 1, dtype=torch.int64, device=q.device)
        stream = current_stream()
        with _span("radius_count", nq):
            check(self.lib.agx_radius_count(self.handle, ptr(q), nq, float(radius), ptr(counts), stream))
        check(self.lib.agx_radius_cap_counts(ptr(counts), nq, int(max_neighbours), ptr(capped), stream))
        total = c_int64()
        check(self.lib.agx_exclusive_scan(ptr(capped), nq, ptr(offsets), byref(total), stream))
        return offsets, int(total.value), counts

    def radius_fill(
        self, q: torch.Tensor, radius: float, offsets: torch.Tensor, total: int, out: torch.Tensor, out_offset: int = 0,
        dst_base: int = 0, stats: torch.Tensor | None = None, swap_rows: bool = False,
        counts: torch.Tensor | None = None, max_neighbours: int | None = None,
    ) -> torch.Tensor:  # fmt: skip
        """Pass 2: write the ``total`` pairs at column ``out_offset`` of the contiguous (2, E) int32 ``out``; with
        ``swap_rows`` the queries go to row 0 and the reference points to row 1.  With ``max_neighbours`` (and the
        ``counts`` and ``offsets`` of ``radius_capped``) a query with more candidates keeps its ``max_neighbours``
        nearest, ties at the boundary to the lower reference index (``agx_radius_select``)."""
        q = _dev_x(q)
        assert out.dim() == 2 and out.shape[0] == 2 and out.dtype == torch.int32 and out.is_contiguous()
        assert 0 <= out_offset and out_offset + total <= out.shape[1]
        if total:
            ref_row, q_row = _row_ptrs(out, out_offset, swap_rows)
            nq, stream = int(q.shape[0]), current_stream()
            if max_neighbours is None:
                with _span("radius_fill", total):
                    check(
                        self.lib.agx_radius_fill(
                            self.handle, ptr(q), nq, float(radius), ptr(offsets), ref_row, q_row, int(dst_base),
                            ptr(stats), stream,
                        )
                    )  # fmt: skip
                return out
            assert counts is not None and counts.dtype == torch.int32 and counts.shape == (nq,)
            with _span("radius_fill", total):
                check(
                    self.lib.agx_radius_fill_capped(
                        self.handle, ptr(q), nq, float(radius), ptr(counts), int(max_neighbours), ptr(offsets),
                        ref_row, q_row, int(dst_base), ptr(stats), stream,
                    )
                )  # fmt: skip
            with _span("radius_select", nq):
                check(
                    self.lib.agx_radius_select(
                        self.handle, ptr(q), nq, float(radius), ptr(counts), int(max_neighbours), ptr(offsets),
                        ref_row, q_row, int(dst_base), ptr(stats), stream,
                    )
                )  # fmt: skip
        return out

    def radius(self, q: torch.Tensor, radius: float, dst_base: int = 0, stats: torch.Tensor | None = None) -> torch.Tensor:
        """``edge_index`` (2, E) int32 of every (reference, query) pair within ``radius`` (inclusive)."""
        q = _dev_x(q)
        offsets, total = self.radius_count(q, radius)
        out = torch.empty((2, total), dtype=torch.int32, device=q.device)
        return self.radius_fill(q, radius, offsets, total, out, 0, dst_base, stats)


class output_maps:
    """``with output_maps(src_sel, dst_sel):`` - the searches launched inside write ``src_sel[reference index]`` /
    ``dst_sel[query index]`` (CUDA int64, ascending: the row selections of masked node sets) instead of compact indices:
    ``NodeMaskingMixin.undo_masking`` fused into the kernels' stores (``agx_set_output_maps``)."""

    def __init__(self, src_sel: torch.Tensor | None, dst_sel: torch.Tensor | None) -> None:
        for sel in (src_sel, dst_sel):
            assert sel is None or (sel.is_cuda and sel.dtype == torch.int64 and sel.is_contiguous())
        self.src_sel, self.dst_sel = src_sel, dst_sel

    def __enter__(self):
        if self.src_sel is not None or self.dst_sel is not None:
            load_library().agx_set_output_maps(ptr(self.src_sel), ptr(self.dst_sel))
        return self

    def __exit__(self, *exc) -> None:
        load_library().agx_set_output_maps(None, None)


def search_vectors(x: torch.Tensor) -> torch.Tensor:
    """float32 (n, 3) unit vectors the neighbour search filters with (see ``agx_search_vectors``)."""
    x = _dev_x(x)
    out = torch.empty((x.shape[0], 3), dtype=torch.float32, device=x.device)
    check(load_library().agx_search_vectors(ptr(x), int(x.shape[0]), ptr(out), current_stream()))
    return out


def new_stats(device) -> torch.Tensor:
    return torch.zeros(4, dtype=torch.int64, device=device)


def haversine_rdist_host(lat1: float, lon1: float, lat2: float, lon2: float) -> float:
    """sklearn ``HaversineDistance64.rdist`` with the C library's sin/cos - the same libm calls sklearn's
    compiled code makes, so the value is bit-identical to the reference's."""
    s0 = math.sin(0.5 * (lat1 - lat2))
    s1 = math.sin(0.5 * (lon1 - lon2))
    return s0 * s0 + math.cos(lat1) * math.cos(lat2) * s1 * s1


REFDIST_K = 7  # self + 6: every neighbour that can tie for "nearest" on a degree-6 mesh or a regular grid
REFDIST_MAX_CANDIDATES = 4096


REFDIST_INDEX_HINT_K = 3  # cell width of the index the self query runs on: the one a KNN-3 decoder over the same nodes uses


def grid_reference_distance(x: torch.Tensor, state=None) -> float:
    """``utils.get_grid_reference_distance`` (/root/reference/src/anemoi/graphs/utils.py:44-63): the largest
    strictly positive nearest-neighbour distance of a node set (column 1 of a k = 2 self query).

    The search and the float64 distances run on the GPU: a k = 7 self query, per node the smallest of its six
    neighbour distances (the value of "column 1" whichever of several equidistant neighbours sklearn's heap keeps),
    the maximum of those.  The nodes within rounding (1e-13 relative; CUDA's sin/cos differ from glibc's by <= 2 ulp)
    of that maximum are then re-evaluated on the host with libm and the reference's exact-compare semantics
    (``agx_host_reference_rdist``), so the returned float64 carries the bits sklearn produces (it becomes the
    cut-off radius).  Nothing here depends on how the nodes are numbered."""
    xd = _dev_x(x)
    lib = load_library()
    n = int(xd.shape[0])
    k = min(REFDIST_K, n)
    if k < 2:
        raise ValueError("zero-size array to reduction operation maximum which has no identity")
    from . import device as _device

    # the k = 7 self query of a node set is a small search whatever the cell width: it runs on the index a KNN-3
    # decoder over the same nodes will use, so a recipe bins its hidden nodes once (device.neighbour_index)
    with _device.neighbour_index(state, xd, hint_k=min(REFDIST_INDEX_HINT_K, k)) as index:
        ei, rdist = index.knn(xd, k, return_rdist=True, tag="knn_refdist")
    nearest = rdist[:, 1:].min(dim=1).values  # 0 where a duplicate point exists (excluded like ``dists > 0``)
    top = nearest.max()
    cand = torch.nonzero((nearest >= top * (1.0 - 1.0e-13)) & (nearest > 0.0), as_tuple=False).squeeze(1)
    cand = cand[:REFDIST_MAX_CANDIDATES]
    if cand.numel() == 0:
        raise ValueError("zero-size array to reduction operation maximum which has no identity")
    nb = ei[0].view(n, k)[cand, 1:].long()
    q_host = xd[cand].cpu().contiguous()
    nb_host = xd[nb.reshape(-1)].cpu().contiguous()
    value = c_double()
    check(lib.agx_host_reference_rdist(q_host.data_ptr(), nb_host.data_ptr(), int(cand.numel()), k - 1, byref(value)))
    return 2.0 * math.asin(math.sqrt(value.value))


# node sets with more nodes than this are NOT tabulated for the attribute kernel: it evaluates their per-node quantities
# per edge from the 8-byte coordinates (a table costs 32 B written + 32 B gathered per node and role; the hidden mesh
# of a recipe stays tabulated - 5 MB, L2-resident).  AGX_ATTR_COORD_MIN_NODES overrides (0: never tabulate).
ATTR_COORD_MIN_NODES = int(float(__import__("os").environ.get("AGX_ATTR_COORD_MIN_NODES", "1e6")))


class NodeTables:
    """Per-node inputs of the attribute kernel.  Small node sets: one 32-byte record per role, built on first use:

    * ``src_rec`` float32 (n, 8): (x, y, z, cos lat, lat, lon, 0, 0) - the node as an edge SOURCE;
    * ``dst_rec`` float64 (n, 4): (quat x, quat y, quat w, bits(lat, lon)) - the node as an edge TARGET
      (rotation to the north pole, edges/directional.py:19-37).

    Large node sets (``n > ATTR_COORD_MIN_NODES``): no table - ``source_inputs()`` / ``target_inputs()`` hand the
    kernel the coordinates and it evaluates the same quantities per edge (bit-identical results).

    ``with_rotation`` is accepted for compatibility; the target record always carries the quaternion."""

    def __init__(self, x: torch.Tensor, with_rotation: bool = True, tabulate: bool | None = None) -> None:
        self.x = _dev_x(x)
        self.n = int(self.x.shape[0])
        self.tabulate = (self.n <= ATTR_COORD_MIN_NODES) if tabulate is None else bool(tabulate)
        self._src = None
        self._dst = None

    def _build(self, want_src: bool, want_dst: bool) -> None:
        dev = self.x.device
        src = torch.empty((self.n, 8), dtype=torch.float32, device=dev) if want_src else None
        dst = torch.empty((self.n, 4), dtype=torch.float64, device=dev) if want_dst else None
        with _span("node_tables", self.n):
            check(load_library().agx_node_tables(ptr(self.x), self.n, ptr(src), ptr(dst), current_stream()))
        if want_src:
            self._src = src
        if want_dst:
            self._dst = dst

    def prepare(self, as_source: bool = False, as_target: bool = False) -> "NodeTables":
        """Build the missing records of the requested roles in ONE kernel launch."""
        need_src, need_dst = as_source and self._src is None, as_target and self._dst is None
        if self.n and (need_src or need_dst):
            self._build(need_src, need_dst)
        elif need_src or need_dst:  # empty node set
            if need_src:
                self._src = torch.empty((0, 8), dtype=torch.float32, device=self.x.device)
            if need_dst:
                self._dst = torch.empty((0, 4), dtype=torch.float64, device=self.x.device)
        return self

    def source_inputs(self) -> tuple:
        """``(record pointer or None, coordinate pointer or None)`` for the kernel's source side."""
        return (ptr(self.src_rec), None) if self.tabulate else (None, ptr(self.x))

    def target_inputs(self) -> tuple:
        return (ptr(self.dst_rec), None) if self.tabulate else (None, ptr(self.x))

    @property
    def src_rec(self) -> torch.Tensor:
        return self.prepare(as_source=True)._src

    @property
    def dst_rec(self) -> torch.Tensor:
        return self.prepare(as_target=True)._dst

    @property
    def xyzc(self) -> torch.Tensor:
        """float32 (n, 4) view: unit vector and cos(lat) with numpy's float32 bits."""
        return self.src_rec[:, :4]

    @property
    def quat(self) -> torch.Tensor:
        return self.dst_rec


def _node_inputs(src: NodeTables, dst: NodeTables) -> tuple:
    """The four node pointers of an attribute call: (src_rec, src_latlon, dst_rec, dst_latlon)."""
    if src is dst and src.tabulate:
        src.prepare(as_source=True, as_target=True)
    return (*src.source_inputs(), *dst.target_inputs())


_workspace: dict = {}


def _attr_workspace(device) -> torch.Tensor:
    key = (device.type, device.index)
    if key not in _workspace:
        n = int(load_library().agx_edge_attrs_workspace())
        _workspace[key] = torch.empty(n, dtype=torch.float64, device=device)
    return _workspace[key]


# below this many edges a multi-GPU build evaluates the attributes on every rank instead of sharding them: the
# statistics exchange and the two all-gathers (12 bytes per edge to every rank) cost more than the kernel, and the
# device->host copies of a host-resident graph queue behind them (O1280 decoder, 19.8 M edges, N = 2: 22.2 ms
# host-to-host sharded vs 14.0 ms replicated).  AGX_ATTR_SHARD_MIN_EDGES overrides.
ATTR_SHARD_MIN_EDGES = int(float(__import__("os").environ.get("AGX_ATTR_SHARD_MIN_EDGES", "64e6")))


def edge_attributes(
    edge_index: torch.Tensor,
    src: NodeTables,
    dst: NodeTables,
    length: bool = True,
    length_norm: str | None = None,
    length_invert: bool = False,
    direction: bool = True,
    direction_norm: str | None = None,
    direction_rotated: bool = True,
    sharded: bool = False,
    local: tuple[int, int, list[int]] | None = None,
    shard=None,
    regular_k: int = 0,
):
    """Fused EdgeLength / EdgeDirection: returns ``(len (E, 1) float32 | None, dir (E, 2) float32 | None)``.

    ``sharded=True`` (multi-GPU): this rank evaluates only a contiguous range of the edges, the per-rank
    normalisation statistics are exchanged (and folded in rank order inside the kernel) and the attribute blocks
    all-gathered asynchronously, so every rank ends with the complete arrays (complete once ``device.wait_for`` /
    ``device.flush`` has run).  ``local = (lo, hi, counts)`` names the range this rank's own builder produced
    (its columns of ``edge_index`` are valid before the edge all-gather has finished) and every rank's block
    size; without it the edges are split evenly.  ``shard`` (``device.Shard``, sharded output mode): ``edge_index`` is
    this rank's own block and so are the results - only the statistics are exchanged.  ``regular_k`` > 0: the edges of the
    i-th target are the columns [i k, (i + 1) k) (a KNN result) - evaluated by target instead of by edge.

    A NaN attribute value (an antipodal pair's length: ``a > 1`` in float32) makes every normalised value of that
    attribute NaN, whatever the norm, as in the reference."""
    from . import device as _device

    for norm in (length_norm, direction_norm):
        if norm not in NORM_CODES:
            raise ValueError(
                f"Attribute normalisation \"{norm}\" is not valid. Options are: 'l1', 'l2', 'unit-max' or 'unit-std'."
            )
    assert edge_index.is_cuda and edge_index.dtype == torch.int32 and edge_index.dim() == 2 and edge_index.shape[0] == 2
    assert edge_index.is_contiguous(), "edge_index must be a contiguous (2, E) int32 tensor"
    n_edges = int(edge_index.shape[1])
    dev = edge_index.device
    out_len = torch.empty((n_edges, 1), dtype=torch.float32, device=dev) if length else None
    out_dir = torch.empty((n_edges, 2), dtype=torch.float32, device=dev) if direction else None
    lib = load_library()
    nodes = _node_inputs(src, dst)
    len_code = NORM_CODES[length_norm] if length else -1
    dir_code = NORM_CODES[direction_norm] if direction else -1
    rank, w = _device.world() if sharded else (0, 1)
    # sharded output mode: ``edge_index`` IS this rank's block, and the attribute blocks stay on their ranks
    own_block = shard is not None and shard.world > 1 and not shard.replicated
    if shard is not None and not own_block:
        w = 1  # a replicated set in sharded output mode: every rank evaluates all of it
    if w > 1 and not own_block and local is None and n_edges < ATTR_SHARD_MIN_EDGES:
        w = 1  # small edge set: every rank evaluates all of it (identical results, no exchange)
    ws = _attr_workspace(dev)
    stream = current_stream()
    if w == 1 and not own_block:
        _device.wait_for(edge_index)
        with _span("edge_attrs", n_edges):
            check(
                lib.agx_edge_attrs(
                    edge_index[0].data_ptr(), edge_index[1].data_ptr(), n_edges, *nodes, len_code,
                    int(bool(length_invert)), ptr(out_len), dir_code, int(bool(direction_rotated)), ptr(out_dir),
                    ptr(ws), int(regular_k), stream,
                )
            )  # fmt: skip
        return out_len, out_dir
    # this rank's block [lo, hi) of the edges and of the outputs; ``counts``: every rank's block size (all-gathered)
    n_global, counts = n_edges, None
    if own_block:
        lo, hi, n_global, w = 0, n_edges, shard.total, shard.world
    elif local is not None:
        lo, hi, counts = local
        assert sum(counts) == n_edges and hi - lo == counts[rank]
    else:
        _device.wait_for(edge_index)
        lo, hi = _device.shard_range(n_edges, rank, w)
        counts = [b - a for a, b in (_device.shard_range(n_edges, r, w) for r in range(w))]
    m = hi - lo
    e_src, e_dst = edge_index[0].data_ptr() + 4 * lo, edge_index[1].data_ptr() + 4 * lo
    o_len = out_len.data_ptr() + 4 * lo if length else None
    o_dir = out_dir.data_ptr() + 8 * lo if direction else None
    if len_code > 0 or dir_code > 0:
        # one pass over the block: raw float32 values + the block's statistics; then every rank's statistics (folded
        # in rank order inside the kernel) and the scaling in place
        stats = torch.empty(8, dtype=torch.float64, device=dev)
        with _span("edge_attrs_stats", m):
            check(
                lib.agx_edge_attrs_stats(
                    e_src, e_dst, m, *nodes, int(length), int(direction), int(bool(direction_rotated)), o_len, o_dir,
                    ptr(stats), ptr(ws), None, 0, None, None, 0, stream,
                )
            )  # fmt: skip
        stats = _device.all_gather_stats_raw(stats)
        with _span("edge_attrs_apply", m):
            check(
                lib.agx_edge_attrs_apply(
                    m, len_code, int(bool(length_invert)), o_len, dir_code, int(bool(direction_rotated)), o_dir,
                    ptr(stats), w, n_global, ptr(ws), stream,
                )
            )  # fmt: skip
    else:
        with _span("edge_attrs_apply", m):  # no statistics: the raw pass writes the final values
            check(
                lib.agx_edge_attrs(
                    e_src, e_dst, m, *nodes, len_code, int(bool(length_invert)), o_len, dir_code,
                    int(bool(direction_rotated)), o_dir, ptr(ws), 0, stream,
                )
            )  # fmt: skip
    if counts is not None:
        if length:
            _device.all_gather_v(out_len, counts, 0, async_op=True)
        if direction:
            _device.all_gather_v(out_dir, counts, 0, async_op=True)
    return out_len, out_dir


def relabel_rows(rows: list[torch.Tensor], new_index: torch.Tensor) -> None:
    """``row[i] = new_index[row[i]]`` in place for every CUDA int32 row (views allowed when contiguous), eight rows per
    launch (``agx_relabel_rows``)."""
    lib = load_library()
    rows = [r for r in rows if r.numel()]
    for a in range(0, len(rows), 8):
        part = rows[a : a + 8]
        for r in part:
            assert r.is_cuda and r.dtype == torch.int32 and r.is_contiguous()
        ptrs = (c_void_p * len(part))(*[r.data_ptr() for r in part])
        lens = (c_int64 * len(part))(*[int(r.numel()) for r in part])
        with _span("relabel", sum(int(r.numel()) for r in part)):
            check(lib.agx_relabel_rows(ptrs, lens, len(part), ptr(new_index), current_stream()))


ATTR_FLAGS_SKIP, ATTR_FLAGS_ONLY = 1, 2


def compact_flags(flags: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    """``(list, count)``: the ascending positions of the non-zero bytes of a CUDA uint8 array and their number (CUDA
    int32 (n,) / int64 (1,); nothing is read back - consumers take the count from device memory)."""
    assert flags.is_cuda and flags.dtype == torch.uint8 and flags.is_contiguous()
    n = int(flags.numel())
    out = torch.empty(max(n, 1), dtype=torch.int32, device=flags.device)
    count = torch.empty(1, dtype=torch.int64, device=flags.device)
    with _span("flag_list", n):
        check(load_library().agx_compact_flags(ptr(flags), n, ptr(out), ptr(count), current_stream()))
    return out, count


def restrict_flags(
    edge_index: torch.Tensor, src_x: torch.Tensor, dst_x: torch.Tensor, max_radius: float,
    src_mask: torch.Tensor | None = None, dst_mask: torch.Tensor | None = None,
) -> torch.Tensor:  # fmt: skip
    """CUDA uint8 (E,): 0 for the edges of the CUDA int32 (2, E) ``edge_index`` that are subject to the restriction
    (``src_mask[source]`` and ``dst_mask[target]``, CUDA uint8 per node, each optional) and longer than ``max_radius``
    (radians) by CutOffEdges' test, 1 for the others (``agx_restrict_flags``).  ValueError for an endpoint outside
    its node set."""
    assert edge_index.is_cuda and edge_index.dtype == torch.int32 and edge_index.dim() == 2 and edge_index.shape[0] == 2
    edge_index = edge_index.contiguous()
    src_x, dst_x = _dev_x(src_x), _dev_x(dst_x)
    for mask, x in ((src_mask, src_x), (dst_mask, dst_x)):
        assert mask is None or (mask.is_cuda and mask.dtype == torch.uint8 and mask.shape == (x.shape[0],))
    n = int(edge_index.shape[1])
    keep = torch.empty(n, dtype=torch.uint8, device=edge_index.device)
    with _span("restrict_flags", n):
        check(
            load_library().agx_restrict_flags(
                ptr(edge_index[0]), ptr(edge_index[1]), n, ptr(src_x), int(src_x.shape[0]), ptr(dst_x),
                int(dst_x.shape[0]), ptr(src_mask), ptr(dst_mask), float(max_radius), ptr(keep), current_stream(),
            )
        )  # fmt: skip
    return keep


def sort_permutation(key_row: torch.Tensor, other_row: torch.Tensor, n_key_nodes: int, n_other_nodes: int,
                     descending: bool) -> torch.Tensor:  # fmt: skip
    """CUDA int32 (E,): the stable permutation that orders the columns (key_row, other_row) lexicographically
    (``agx_sort_edges``).  ValueError for an endpoint outside its node set."""
    for row in (key_row, other_row):
        assert row.is_cuda and row.dtype == torch.int32 and row.is_contiguous() and row.shape == key_row.shape
    n = int(key_row.numel())
    perm = torch.empty(n, dtype=torch.int32, device=key_row.device)
    with _span("sort_edges", n):
        check(
            load_library().agx_sort_edges(
                ptr(key_row), ptr(other_row), n, int(n_key_nodes), int(n_other_nodes), int(bool(descending)), ptr(perm),
                current_stream(),
            )
        )  # fmt: skip
    return perm


CSR_VALUE_KINDS = {None: 0, torch.float32: 1, torch.bool: 2}


def edges_to_csr(edge_index: torch.Tensor, n_dst_nodes: int, n_src_nodes: int,
                 values: torch.Tensor | None = None) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor]:  # fmt: skip
    """CUDA ``(indptr int64 (n_dst + 1,), indices int32 (nnz,), data (nnz,))``: the canonical CSR of the targets x
    sources matrix ``M[edge_index[1, e], edge_index[0, e]] += values[e]`` of the CUDA int32 (2, E) ``edge_index``
    (``agx_sort_edges`` by (target, source), then ``agx_edges_to_csr``; one read-back).  ``values``: CUDA float32 or
    bool (E,), or None for float32 ones; duplicates are summed in column order (bool: OR).  ValueError for an endpoint
    outside its node set and for E >= 2^31."""
    assert edge_index.is_cuda and edge_index.dtype == torch.int32 and edge_index.dim() == 2 and edge_index.shape[0] == 2
    edge_index = edge_index.contiguous()
    n = int(edge_index.shape[1])
    if n >= 2**31:
        raise ValueError(f"edges_to_csr: {n} edges; an edge set must have fewer than 2^31 edges")
    dtype = torch.float32 if values is None else values.dtype
    assert values is None or (values.is_cuda and values.dtype in CSR_VALUE_KINDS and values.is_contiguous() and values.shape == (n,))
    perm = sort_permutation(edge_index[1], edge_index[0], n_dst_nodes, n_src_nodes, descending=False)
    dev = edge_index.device
    indptr = torch.empty(int(n_dst_nodes) + 1, dtype=torch.int64, device=dev)
    indices = torch.empty(n, dtype=torch.int32, device=dev)
    data = torch.empty(n, dtype=dtype, device=dev)
    nnz = c_int64(0)
    with _span("edges_to_csr", n):
        check(
            load_library().agx_edges_to_csr(
                ptr(edge_index[0]), ptr(edge_index[1]), n, int(n_dst_nodes), ptr(perm), ptr(values),
                CSR_VALUE_KINDS[None if values is None else dtype], ptr(indptr), ptr(indices), ptr(data), byref(nnz),
                current_stream(),
            )
        )  # fmt: skip
    m = int(nnz.value)
    if m < n:  # duplicate pairs: keep only the nnz entries
        indices, data = indices[:m].clone(), data[:m].clone()
    return indptr, indices, data


SPMM_DTYPES = {torch.float32: 0, torch.bfloat16: 1}  # AGX_SPMM_FLOAT32, AGX_SPMM_BFLOAT16


def csr_spmm(indptr: torch.Tensor, indices: torch.Tensor, data: torch.Tensor, x: torch.Tensor, n_rows: int) -> torch.Tensor:
    """``y = M x`` for the CSR ``(indptr, indices, data)`` of ``edges_to_csr`` (CUDA int64 / int32 / float32) and the
    CUDA float32 or bfloat16 field ``x`` of shape (n_cols, F) or (n_cols,): ``y[t, f]`` is the float32 sum, left to
    right in CSR order, of ``fmaf(data[j], x[indices[j], f], acc)`` from +0, rounded once to x's dtype
    (``agx_csr_spmm``; one read-back, the index check).  ``y`` has shape (n_rows, F) or (n_rows,) and x's dtype.
    ValueError for an index outside [0, n_cols)."""
    assert indptr.is_cuda and indptr.dtype == torch.int64 and indptr.shape == (int(n_rows) + 1,)
    assert indices.is_cuda and indices.dtype == torch.int32 and data.is_cuda and data.dtype == torch.float32
    assert indices.dim() == 1 and indices.shape == data.shape
    assert x.is_cuda and x.dtype in SPMM_DTYPES and x.dim() in (1, 2)
    x = x.contiguous()
    n_features = int(x.shape[1]) if x.dim() == 2 else 1
    y = torch.empty((int(n_rows), *x.shape[1:]), dtype=x.dtype, device=x.device)
    if y.numel() == 0:
        return y
    if indices.numel() == 0:  # no entries: every row is empty
        return y.zero_()
    with _span("csr_spmm", int(indices.numel()) * n_features):
        check(
            load_library().agx_csr_spmm(
                ptr(indptr), ptr(indices), ptr(data), int(n_rows), int(x.shape[0]), ptr(x), n_features, SPMM_DTYPES[x.dtype],
                ptr(y), current_stream(),
            )
        )  # fmt: skip
    return y


def gather_rows(pairs: list[tuple[torch.Tensor, torch.Tensor]], index: torch.Tensor) -> None:
    """``dst[j] = src[index[j]]`` along dim 0 for every (src, dst) pair of contiguous CUDA tensors of one dtype and row
    shape, eight pairs per launch (``agx_gather_edge_columns``)."""
    assert index.is_cuda and index.dtype == torch.int32 and index.is_contiguous()
    m = int(index.numel())
    pairs = [(s, d) for s, d in pairs if d.numel()]
    lib = load_library()
    for a in range(0, len(pairs), 8):
        part = pairs[a : a + 8]
        for s, d in part:
            assert s.is_cuda and d.is_cuda and s.is_contiguous() and d.is_contiguous() and s.dtype == d.dtype
            assert d.shape[0] == m and s.shape[1:] == d.shape[1:]
        srcs = (c_void_p * len(part))(*[s.data_ptr() for s, _ in part])
        dsts = (c_void_p * len(part))(*[d.data_ptr() for _, d in part])
        row_bytes = (c_int64 * len(part))(*[d.numel() // m * d.element_size() for _, d in part])
        with _span("gather_edges", m * len(part)):
            check(lib.agx_gather_edge_columns(len(part), srcs, dsts, row_bytes, ptr(index), m, current_stream()))


def edge_azimuth(edge_index: torch.Tensor, src_x: torch.Tensor, dst_x: torch.Tensor, norm: str | None) -> torch.Tensor:
    """CUDA float32 (E, 1): the bearing at each edge's target towards its source, clockwise from north, in radians,
    normalised over the whole edge set as ``EdgeLength`` is (``agx_edge_azimuth``).  ValueError for an endpoint outside
    its node set."""
    assert edge_index.is_cuda and edge_index.dtype == torch.int32 and edge_index.dim() == 2 and edge_index.shape[0] == 2
    edge_index = edge_index.contiguous()
    src_x, dst_x = _dev_x(src_x), _dev_x(dst_x)
    n = int(edge_index.shape[1])
    out = torch.empty((n, 1), dtype=torch.float32, device=edge_index.device)
    with _span("edge_azimuth", n):
        check(
            load_library().agx_edge_azimuth(
                ptr(edge_index[0]), ptr(edge_index[1]), n, ptr(src_x), int(src_x.shape[0]), ptr(dst_x),
                int(dst_x.shape[0]), NORM_CODES[norm], ptr(out), ptr(_attr_workspace(edge_index.device)), current_stream(),
            )
        )  # fmt: skip
    return out


def gaussian_weights(edge_index: torch.Tensor, n_src_nodes: int, n_dst_nodes: int, lengths: torch.Tensor, sigma: float,
                     norm: str | None, perm: torch.Tensor | None) -> torch.Tensor:  # fmt: skip
    """CUDA float32 (E, 1): exp(-d^2 / (2 sigma^2)) of the float32 lengths d (E, 1), normalised within each target's
    edges (``agx_gaussian_weights``).  ``perm``: ``sort_permutation(edge_index[1], edge_index[0], ..., False)`` (which
    checks the endpoints); None with ``norm=None``."""
    assert edge_index.is_cuda and edge_index.dtype == torch.int32 and edge_index.dim() == 2 and edge_index.shape[0] == 2
    edge_index = edge_index.contiguous()
    n = int(edge_index.shape[1])
    assert lengths.is_cuda and lengths.dtype == torch.float32 and lengths.is_contiguous() and lengths.numel() == n
    assert (perm is None) == (norm is None) and (perm is None or (perm.is_cuda and perm.dtype == torch.int32 and perm.numel() == n))
    lib = load_library()
    out = torch.empty((n, 1), dtype=torch.float32, device=edge_index.device)
    scratch = None
    if norm is not None and n:
        size = int(lib.agx_gaussian_weights_scratch_bytes(n, int(n_dst_nodes)))
        scratch = torch.empty(size, dtype=torch.uint8, device=edge_index.device)
    with _span("gaussian_weights", n):
        check(
            lib.agx_gaussian_weights(
                ptr(edge_index[0]), ptr(edge_index[1]), n, int(n_src_nodes), int(n_dst_nodes), ptr(lengths),
                float(sigma), NORM_CODES[norm], ptr(perm), ptr(out), ptr(scratch), current_stream(),
            )
        )  # fmt: skip
    return out


class DeferredEdgeAttributes:
    """EdgeLength / EdgeDirection of an edge set whose sources of a FEW targets are still to be re-decided (KNN edges
    searched while the source numbering was provisional; ``dst_flags`` marks those targets).

    ``raw()`` evaluates every edge now - the trigonometry of the whole set runs in the shadow of the host sort - but
    keeps the flagged targets' edges out of the statistics; after the re-decision ``patch()`` evaluates exactly those
    edges again (statistics set 2) and ``apply()`` derives the normalisation from both sets and scales in place.
    Single rank only (a sharded build orders the nodes first)."""

    def __init__(self, edge_index, src: NodeTables, dst: NodeTables, dst_flags: torch.Tensor, length=True,
                 length_norm=None, length_invert=False, direction=True, direction_norm=None, direction_rotated=True,
                 flag_list=None, flag_count=None, regular_k: int = 0, flag_base: int = 0, shard=None):  # fmt: skip
        """``flag_list`` / ``flag_count`` (``compact_flags(dst_flags)``) with ``regular_k`` (the edges of target t are
        columns [t k, (t + 1) k): a KNN result) let ``patch()`` touch the listed targets' edges only."""
        assert edge_index.is_cuda and edge_index.dtype == torch.int32 and edge_index.is_contiguous()
        assert dst_flags.dtype == torch.uint8 and dst_flags.is_cuda
        self.edge_index, self.flags = edge_index, dst_flags
        self.flag_list, self.flag_count, self.regular_k = flag_list, flag_count, int(regular_k)
        # flags[t - flag_base] belongs to target t; ``shard``: this is one rank's block, the statistics of all blocks
        # are exchanged before the scaling
        self.flag_base = int(flag_base)
        self.shard = shard if (shard is not None and shard.world > 1 and not shard.replicated) else None
        self.n_edges = int(edge_index.shape[1])
        dev = edge_index.device
        self.length, self.direction, self.rotated, self.invert = bool(length), bool(direction), bool(direction_rotated), bool(length_invert)
        self.len_code = NORM_CODES[length_norm] if length else -1
        self.dir_code = NORM_CODES[direction_norm] if direction else -1
        self.out_len = torch.empty((self.n_edges, 1), dtype=torch.float32, device=dev) if length else None
        self.out_dir = torch.empty((self.n_edges, 2), dtype=torch.float32, device=dev) if direction else None
        self.nodes = _node_inputs(src, dst)
        self._keep = (src, dst)  # the tables / coordinates the pointers refer to
        self.stats = torch.tensor([[0.0, 0.0, 1e300, -1e300] * 2] * 2, dtype=torch.float64, device=dev)  # "no value"
        self.ws = _attr_workspace(dev)

    def _stats(self, which: int, tag: str, work: int, mode: int, regular_k: int, listed: bool = False) -> None:
        """Raw values + statistics set ``which``; ``listed``: the flagged targets are ``flag_list`` / ``flag_count``."""
        if self.n_edges == 0:
            return
        ei = self.edge_index
        flags = None if listed else self.flags.data_ptr() - self.flag_base
        with _span(tag, work):
            check(
                load_library().agx_edge_attrs_stats(
                    ei[0].data_ptr(), ei[1].data_ptr(), self.n_edges, *self.nodes,
                    int(self.length), int(self.direction), int(self.rotated), ptr(self.out_len), ptr(self.out_dir),
                    self.stats[which].data_ptr(), ptr(self.ws), flags, mode, ptr(self.flag_list) if listed else None,
                    ptr(self.flag_count) if listed else None, regular_k, current_stream(),
                )
            )

    def raw(self) -> None:
        self._stats(0, "edge_attrs_raw", self.n_edges, ATTR_FLAGS_SKIP, self.regular_k)

    def patch(self) -> None:
        listed = self.flag_list is not None and self.regular_k > 0
        self._stats(1, "edge_attrs_patch", 0, ATTR_FLAGS_ONLY, self.regular_k if listed else 0, listed)

    def apply(self) -> None:
        from . import device as _device

        stats, n_global = self.stats, self.n_edges
        if self.shard is not None:
            # every rank's two statistics sets, in rank order (a collective: also ranks without edges take part)
            stats, n_global = _device.all_gather_stats_raw(self.stats), self.shard.total
        if self.n_edges == 0:
            return
        with _span("edge_attrs_scale", self.n_edges):
            check(
                load_library().agx_edge_attrs_apply(
                    self.n_edges, self.len_code, int(self.invert), ptr(self.out_len), self.dir_code, int(self.rotated),
                    ptr(self.out_dir), ptr(stats), stats.numel() // 8, n_global, ptr(self.ws), current_stream(),
                )
            )


# ----------------------------------------------------------------------------------------------
# icosphere + multi-scale edges
# ----------------------------------------------------------------------------------------------
def ico_num_vertices(level: int) -> int:
    return 10 * 4**level + 2


def ico_num_faces(level: int) -> int:
    return 20 * 4**level


def ico_face_offset(level: int) -> int:
    return 20 * ((4**level - 1) // 3)


class Icosphere:
    """All levels 0..max_level of ``trimesh.creation.icosphere`` on the device."""

    def __init__(self, max_level: int, device=None) -> None:
        _cabi.require_cuda()
        device = torch.device("cuda") if device is None else device
        self.max_level = int(max_level)
        nv = ico_num_vertices(self.max_level)
        self.vertices = torch.empty((nv, 3), dtype=torch.float64, device=device)
        self.faces_all = torch.empty((ico_face_offset(self.max_level + 1), 3), dtype=torch.int32, device=device)
        self.latlon = torch.empty((nv, 2), dtype=torch.float32, device=device)
        with _span("icosphere", nv):
            check(
                load_library().agx_icosphere(
                    self.max_level, ptr(self.vertices), ptr(self.faces_all), ptr(self.latlon), current_stream()
                )
            )

    def faces(self, level: int) -> torch.Tensor:
        o = ico_face_offset(level)
        return self.faces_all[o : o + ico_num_faces(level)]


def multiscale_tri_edges(ico: Icosphere, levels: list[int], x_hops: int, node_ordering: torch.Tensor) -> torch.Tensor:
    """MultiScaleEdges for global TriNodes: (2, E) int32 sorted by (dst, src).

    ``node_ordering[p]`` is the icosphere vertex at graph position ``p``."""
    lib = load_library()
    dev = ico.vertices.device
    nv = ico_num_vertices(ico.max_level)
    order = node_ordering.to(device=dev, dtype=torch.int32).contiguous()
    assert order.shape == (nv,), f"node_ordering must list all {nv} vertices of level {ico.max_level}"
    rank = torch.empty(nv, dtype=torch.int32, device=dev)
    rank[order.long()] = torch.arange(nv, dtype=torch.int32, device=dev)
    lv = (c_int32 * len(levels))(*[int(v) for v in levels])
    per_node = int(lib.agx_multiscale_scratch_per_node(len(levels), int(x_hops)))
    if x_hops > 8:
        raise NotImplementedError(f"x_hops = {x_hops} > 8 is not built yet")
    scratch = torch.empty(per_node * nv, dtype=torch.int32, device=dev)
    counts = torch.empty(nv, dtype=torch.int32, device=dev)
    offsets = torch.empty(nv + 1, dtype=torch.int64, device=dev)
    stream = current_stream()
    with _span("multiscale_count", nv):
        check(
            lib.agx_multiscale_tri_count(
                ico.max_level, ptr(ico.faces_all), lv, len(levels), int(x_hops), ptr(order), ptr(rank), ptr(counts),
                ptr(scratch), stream,
            )
        )  # fmt: skip
    total = c_int64()
    check(lib.agx_exclusive_scan(ptr(counts), nv, ptr(offsets), byref(total), stream))
    out = torch.empty((2, total.value), dtype=torch.int32, device=dev)
    if total.value:
        check(
            lib.agx_multiscale_tri_fill(
                nv, ptr(counts), ptr(offsets), ptr(scratch), per_node, out[0].data_ptr(), out[1].data_ptr(), stream
            )
        )
    return out


def multiscale_tri_edges_mapped(
    ico: Icosphere, levels: list[int], x_hops: int, n_nodes: int, vertex_map: torch.Tensor
) -> torch.Tensor:
    """MultiScaleEdges for limited-area / stretched TriNodes: (2, E) int32 sorted by (dst, src).

    ``vertex_map[v]`` is the graph position of icosphere vertex ``v`` of the finest level, or -1 if the
    vertex is masked out (lower levels are prefixes, so the same map serves every level)."""
    lib = load_library()
    dev = ico.vertices.device
    if x_hops > 8:
        raise NotImplementedError(f"x_hops = {x_hops} > 8 is not built yet")
    vmap = vertex_map.to(device=dev, dtype=torch.int32).contiguous()
    assert vmap.shape == (ico_num_vertices(ico.max_level),)
    node_vertex = torch.full((len(levels), n_nodes), -1, dtype=torch.int32, device=dev)
    for i, level in enumerate(levels):
        nv = ico_num_vertices(int(level))
        v = torch.nonzero(vmap[:nv] >= 0, as_tuple=False).squeeze(1)
        node_vertex[i, vmap[v].long()] = v.to(torch.int32)
    lv = (c_int32 * len(levels))(*[int(v) for v in levels])
    per_node = int(lib.agx_multiscale_scratch_per_node(len(levels), int(x_hops)))
    scratch = torch.empty(per_node * max(n_nodes, 1), dtype=torch.int32, device=dev)
    counts = torch.zeros(n_nodes, dtype=torch.int32, device=dev)
    offsets = torch.empty(n_nodes + 1, dtype=torch.int64, device=dev)
    stream = current_stream()
    check(
        lib.agx_multiscale_tri_count_mapped(
            ico.max_level, ptr(ico.faces_all), lv, len(levels), int(x_hops), n_nodes, ptr(vmap), ptr(node_vertex),
            ptr(counts), ptr(scratch), stream,
        )
    )  # fmt: skip
    total = c_int64()
    check(lib.agx_exclusive_scan(ptr(counts), n_nodes, ptr(offsets), byref(total), stream))
    out = torch.empty((2, total.value), dtype=torch.int32, device=dev)
    if total.value:
        check(
            lib.agx_multiscale_tri_fill(
                n_nodes, ptr(counts), ptr(offsets), ptr(scratch), per_node, out[0].data_ptr(), out[1].data_ptr(), stream
            )
        )
    return out


# ----------------------------------------------------------------------------------------------
# hexagonal (H3) mesh
# ----------------------------------------------------------------------------------------------
def hex_num_cells(res: int) -> int:
    """H3's ``numHexagons(res)`` = 2 + 120 * 7**res."""
    n = int(load_library().agx_hex_num_cells(int(res)))
    if n < 0:
        raise ValueError(f"H3 resolutions are 0..15, got {res}")
    return n


class HexCells:
    """All cells of one H3 resolution on the device: ``latlon`` float64 (n, 2) radians - the values the reference
    obtains as ``np.deg2rad(h3.h3_to_geo(idx))`` (generate/hex_icosahedron.py:47) - in (face, i, j) order, and the
    ``pentagon`` flags.  ``neighbours()`` gives the edge-adjacency table (one ring of ``h3.k_ring``)."""

    def __init__(self, res: int, device=None) -> None:
        _cabi.require_cuda()
        device = torch.device("cuda") if device is None else device
        self.res = int(res)
        self.n = hex_num_cells(self.res)
        self.latlon = torch.empty((self.n, 2), dtype=torch.float64, device=device)
        self.pentagon = torch.empty(self.n, dtype=torch.uint8, device=device)
        with _span("hex_cells", self.n):
            check(load_library().agx_hex_cells(self.res, ptr(self.latlon), ptr(self.pentagon), current_stream()))
        self._latlon32 = None
        self._nb = None

    @property
    def latlon32(self) -> torch.Tensor:
        if self._latlon32 is None:
            self._latlon32 = self.latlon.to(torch.float32)
        return self._latlon32

    def neighbours(self) -> tuple[torch.Tensor, torch.Tensor]:
        """``(nb (n, 6) int32, -1 padded; deg (n,) int32)``: the cells sharing an edge with each cell."""
        if self._nb is None:
            x = self.latlon32
            with NeighbourIndex(x, hint_k=7) as index:
                knn7 = index.knn(x, 7, tag="knn_hex_adjacency")[0]
            nb = torch.empty((self.n, 6), dtype=torch.int32, device=x.device)
            deg = torch.empty(self.n, dtype=torch.int32, device=x.device)
            check(load_library().agx_hex_adjacency(knn7.data_ptr(), ptr(self.pentagon), self.n, ptr(nb), ptr(deg), current_stream()))
            self._nb = (nb, deg)
        return self._nb


def multiscale_adj_edges(levels: list[tuple], x_hops: int, walk_all: bool, n_nodes: int) -> torch.Tensor:
    """Multi-scale edges over explicit adjacency tables: (2, E) int32 sorted by (dst, src).

    ``levels`` lists, per mesh level, ``(nb (n, 6) int32, deg (n,) int32, cell_node (n,) int32, node_cell
    (n_nodes,) int32)`` - see ``agx_multiscale_adj_count``."""
    lib = load_library()
    if x_hops > 8:
        raise NotImplementedError(f"x_hops = {x_hops} > 8 is not built yet")
    dev = levels[0][0].device
    n_levels = len(levels)
    tables = [[t.contiguous() for t in lv] for lv in levels]
    for nb, deg, cell_node, node_cell in tables:
        assert nb.dtype == deg.dtype == cell_node.dtype == node_cell.dtype == torch.int32
        assert nb.shape == (deg.shape[0], 6) and cell_node.shape == deg.shape and node_cell.shape == (n_nodes,)
    arrays = [(c_void_p * n_levels)(*[lv[i].data_ptr() for lv in tables]) for i in range(4)]
    per_node = int(lib.agx_multiscale_scratch_per_node(n_levels, int(x_hops)))
    scratch = torch.empty(per_node * max(n_nodes, 1), dtype=torch.int32, device=dev)
    counts = torch.zeros(n_nodes, dtype=torch.int32, device=dev)
    offsets = torch.empty(n_nodes + 1, dtype=torch.int64, device=dev)
    stream = current_stream()
    with _span("multiscale_count", n_nodes):
        check(
            lib.agx_multiscale_adj_count(
                n_levels, arrays[0], arrays[1], arrays[2], arrays[3], int(x_hops), int(bool(walk_all)), n_nodes,
                ptr(counts), ptr(scratch), stream,
            )
        )  # fmt: skip
    total = c_int64()
    check(lib.agx_exclusive_scan(ptr(counts), n_nodes, ptr(offsets), byref(total), stream))
    out = torch.empty((2, total.value), dtype=torch.int32, device=dev)
    if total.value:
        check(
            lib.agx_multiscale_tri_fill(
                n_nodes, ptr(counts), ptr(offsets), ptr(scratch), per_node, out[0].data_ptr(), out[1].data_ptr(), stream
            )
        )
    return out


def healpix_nodes(resolution: int, device=None) -> torch.Tensor:
    """float32 (12 * 4**resolution, 2) (lat, lon) radians of the HEALPix pixel centres in nested order
    (``agx_healpix_nodes``; nodes/builders/from_healpix.py:61-66)."""
    _cabi.require_cuda()
    device = torch.device("cuda") if device is None else device
    out = torch.empty((12 * 4 ** int(resolution), 2), dtype=torch.float32, device=device)
    check(load_library().agx_healpix_nodes(int(resolution), ptr(out), current_stream()))
    return out


def gaussian_latitudes(n: int, device=None) -> torch.Tensor:
    """float64 (2n,) Gaussian latitudes in degrees, north to south: the roots of the Legendre polynomial P_2n
    (``agx_gaussian_latitudes``).  ValueError for n < 1 or a grid O<n> past int32 node indices."""
    _cabi.require_cuda()
    device = torch.device("cuda") if device is None else device
    out = torch.empty(max(2 * int(n), 0), dtype=torch.float64, device=device)
    check(load_library().agx_gaussian_latitudes(int(n), ptr(out), current_stream()))
    return out


def octahedral_nodes(n: int, device=None) -> torch.Tensor:
    """float32 (4n(n+9), 2) (lat, lon) radians of the octahedral reduced Gaussian grid O<n>, north to south and west to
    east from 0 degrees (``agx_octahedral_nodes``); ``grids.latlon_deg_to_x(*grids.octahedral_grid(n))`` on the device."""
    lat = gaussian_latitudes(n, device)  # checks n before the output is allocated
    n = int(n)
    out = torch.empty((4 * n * (n + 9), 2), dtype=torch.float32, device=lat.device)
    check(load_library().agx_octahedral_nodes(n, ptr(lat), ptr(out), current_stream()))
    return out


# ----------------------------------------------------------------------------------------------
# spherical Voronoi cell areas
# ----------------------------------------------------------------------------------------------
VORONOI_SMALL_N = 64  # up to this many generators unclosed cells go through the exhaustive spherical form
VORONOI_K = (17, 33, 64)  # neighbours tried in turn (self included): a regular grid's cells close within the first 16
VORONOI_WIDE_MAX_EDGES = 1024  # polygon capacity of the wide pass (agx_voronoi_areas_wide)
# what the last voronoi_areas call handed to the wide pass: cells, rounds of vertex queries, candidates per final cell,
# and the generator ids of those cells (CUDA int32, None when the pass did not run)
voronoi_wide: dict = {}


def voronoi_areas(x: torch.Tensor, radius: float = 1.0) -> torch.Tensor:
    """float64 (n,) areas of the spherical Voronoi cells of a node set - ``SphericalVoronoi(points, radius)
    .calculate_areas()`` of nodes/attributes.py:199-221 - on the device.  Generators whose cell is not closed by
    their 16 nearest neighbours are retried with 32, then 63; the cells still open after that (a coarse generator
    next to a much finer region) go through the wide pass, which grows each cell's candidates from the neighbours of
    its vertices (``voronoi_wide`` records what it did)."""
    voronoi_wide.update(cells=0, rounds=0, max_candidates=0, mean_candidates=0.0, generators=None)
    xd = _dev_x(x)
    n = int(xd.shape[0])
    lib = load_library()
    if n < 4:
        raise ValueError("SphericalVoronoi needs at least 4 generators")
    areas = torch.zeros(n, dtype=torch.float64, device=xd.device)
    subset = None  # None = all generators
    stream = current_stream()
    with NeighbourIndex(xd, hint_k=VORONOI_K[0]) as index:
        for k in VORONOI_K:
            k = min(k, n)
            q = xd if subset is None else xd[subset.long()]
            m = int(q.shape[0])
            knn = index.knn(q, k, tag="knn_voronoi")[0]
            status = torch.empty(m, dtype=torch.int32, device=xd.device)
            with _span("voronoi_areas", m):
                check(
                    lib.agx_voronoi_areas(
                        ptr(xd), n, knn.data_ptr(), k, int(k == n), ptr(subset), m, float(radius), ptr(areas),
                        ptr(status), stream,
                    )
                )
            worst = int(status.max().item())
            if worst == 0:
                return areas
            if worst == 3:
                raise ValueError("Duplicate generators present.")  # scipy's message
            retry = torch.nonzero(status > 0, as_tuple=False).squeeze(1).to(torch.int32)
            subset = retry if subset is None else subset[retry.long()]
            if k == n:
                break
        if n > VORONOI_SMALL_N:
            # cells next to a much finer region: grown from their vertices' neighbours until certified
            m = int(subset.numel())
            seeds = knn.view(-1, k)[retry.long()].contiguous()
            stats = (c_int64 * 6)()
            with _span("voronoi_areas_wide", m):
                check(
                    lib.agx_voronoi_areas_wide(
                        index.handle, ptr(xd), n, ptr(subset), m, ptr(seeds), k, float(radius), ptr(areas), stats,
                        stream,
                    )
                )  # fmt: skip
            voronoi_wide.update(
                cells=m, rounds=stats[0], max_candidates=stats[2], mean_candidates=stats[3] / m, generators=subset
            )
            failed = stats[4]
            if failed & (1 << 3):
                raise ValueError("Duplicate generators present.")
            if failed & (1 << 5):
                raise NotImplementedError(f"a Voronoi cell with more than {VORONOI_WIDE_MAX_EDGES} edges is not built")
            if failed & (1 << 6):
                raise NotImplementedError(
                    "a Voronoi vertex is not certified by its 32 nearest generators (float32 generators denser than "
                    "~1e-3 rad around it)"
                )
            if stats[1] and not stats[5]:
                raise NotImplementedError(f"{stats[1]} Voronoi cells are still open after {stats[0]} rounds of the wide pass")
            if not failed and not stats[1]:
                return areas
            # a cell still touching the initial square: not inside its open hemisphere (a limited-area set on its own)
    if n <= VORONOI_SMALL_N:
        # a handful of generators: cells wider than a hemisphere do not fit the gnomonic plane - exhaustive form on the
        # sphere (every pair of bisector planes), the reference's range from 4 generators up
        m = int(subset.numel())
        status = torch.empty(m, dtype=torch.int32, device=xd.device)
        with _span("voronoi_areas_small", m):
            check(lib.agx_voronoi_areas_small(ptr(xd), n, ptr(subset), m, float(radius), ptr(areas), ptr(status), stream))
        worst = int(status.max().item())
        if worst == 0:
            return areas
        if worst == 3:
            raise ValueError("Duplicate generators present.")
    raise NotImplementedError(
        f"{int(subset.numel())} Voronoi cells are not closed by their {VORONOI_K[-1] - 1} nearest neighbours "
        "(fewer than ~8 generators per hemisphere, or an extremely anisotropic point set)"
    )


def isolatitude_areas(x: torch.Tensor) -> tuple[torch.Tensor, int]:
    """float64 (n,) isolatitude area weights of a node set and its number of latitude rows (``agx_isolatitude_areas``):
    every node gets the unit-sphere area of its latitude band - bounded by the midpoints to the neighbouring rows and by
    the poles - over the number of nodes in its row, a row being one float32 latitude (-0.0 and +0.0 one row).
    ValueError for a latitude that is NaN or beyond +-float32(pi/2)."""
    xd = _dev_x(x)
    n = int(xd.shape[0])
    areas = torch.empty(n, dtype=torch.float64, device=xd.device)
    n_rows = c_int32(0)
    with _span("isolatitude_areas", n):
        check(load_library().agx_isolatitude_areas(ptr(xd), n, ptr(areas), byref(n_rows), current_stream()))
    return areas, int(n_rows.value)


__all__ = [
    "multiscale_tri_edges_mapped",
    "relabel_rows",
    "output_maps",
    "DeferredEdgeAttributes",
    "voronoi_areas",
    "isolatitude_areas",
    "HexCells",
    "hex_num_cells",
    "multiscale_adj_edges",
    "NeighbourIndex",
    "NodeTables",
    "Icosphere",
    "edge_attributes",
    "grid_reference_distance",
    "multiscale_tri_edges",
    "haversine_rdist_host",
    "new_stats",
]

_ = ctypes  # keep the import for type users
