"""Device residency, deferred device->host copies and the multi-GPU shard context.

The reference keeps every tensor on the CPU (``graph[name].x``, ``edge_index``, attributes) and the
builders hand numpy arrays to sklearn.  Here the arithmetic runs on the GPU, so the builders need

* a device copy of the node coordinates and of what is derived from ONE node set (the float32 xyz
  table, the rotation quaternions) that survives from one builder to the next - kept on the node
  storage under ``_agx_state`` (private, removed by ``GraphCreator.clean`` like every ``_`` attribute,
  /root/reference/src/anemoi/graphs/create.py:108-112);
* the device copy of an ``edge_index`` the builder has just produced, so the attribute kernel does not
  re-upload it - kept on the edge storage under ``_agx_edge_index``;
* device->host copies that do not stall the stream: outputs go to pinned host tensors with
  ``non_blocking=True`` and are awaited once, at the end of the outermost ``deferred()`` scope
  (``GraphCreator.update_graph`` opens one; a builder used on its own flushes before it returns).

Residency rule: tensors come back where the coordinates live.  A graph whose ``x`` tensors are CUDA
tensors gets CUDA ``edge_index`` / attributes and nothing crosses PCIe.

Multi-GPU: when ``torch.distributed`` is initialised with more than one rank every rank runs the same
recipe; query nodes (and, for attributes, edges) are split into contiguous per-rank ranges and the
per-rank blocks are concatenated in rank order with an all-gather (``all_gather_v``), so every rank
ends with the complete graph, in the same order as a single-GPU build.
"""

from __future__ import annotations

import contextlib
import os
from dataclasses import dataclass, field

import torch

from . import _cabi

_defer_depth = 0
_pending: list[torch.cuda.Event] = []
_works: dict[int, list] = {}  # storage pointer -> outstanding asynchronous collectives writing into that storage
_resident = False


def set_resident(flag: bool) -> bool:
    """Device-resident graphs: node builders place ``x`` on the GPU, so every edge tensor stays there too
    (nothing crosses PCIe until the caller asks).  Returns the previous setting."""
    global _resident
    prev, _resident = _resident, bool(flag)
    return prev


def is_resident() -> bool:
    return _resident


# Multi-GPU output mode.  "gather" (default): every rank ends with the complete graph (per-rank edge blocks are
# all-gathered over NCCL).  "sharded": nothing is exchanged between the GPUs - a device-resident graph keeps each rank's
# own block of every sharded edge set (global node ids, attributes normalised with the global statistics), and a
# host-resident graph is assembled in ONE shared page-locked host buffer that every rank writes its block into over
# its own PCIe link (``shm.HostArena``), so rank 0 - and every other rank - ends with the complete graph on the host.
_sharded_output = __import__("os").environ.get("AGX_OUTPUT", "gather") == "sharded"
_force_single = False
_shared_host_used = False


def set_sharded_output(flag: bool) -> bool:
    global _sharded_output
    prev, _sharded_output = _sharded_output, bool(flag)
    return prev


def sharded_output() -> bool:
    """Sharded output mode is on AND this build runs on more than one rank."""
    return _sharded_output and world()[1] > 1


@contextlib.contextmanager
def single_rank():
    """Build as if this process were alone (parity checks of a sharded build against the one-GPU result)."""
    global _force_single
    prev, _force_single = _force_single, True
    try:
        yield
    finally:
        _force_single = prev


@dataclass
class Shard:
    """How an edge set is spread over the ranks: ``counts[r]`` edges on rank ``r`` (blocks in rank order make the
    single-GPU order), or ``replicated`` (every rank holds all of it: small sets are computed everywhere)."""

    rank: int
    world: int
    counts: list
    replicated: bool = False

    @property
    def total(self) -> int:
        return int(self.counts[0]) if self.replicated else int(sum(self.counts))

    @property
    def offset(self) -> int:
        return 0 if self.replicated else int(sum(self.counts[: self.rank]))

    def describe(self) -> dict:
        return {"rank": self.rank, "world": self.world, "counts": [int(c) for c in self.counts], "replicated": self.replicated}


def host_tensor(shape, dtype: torch.dtype, require_shared: bool = False) -> torch.Tensor:
    """Page-locked host tensor for a result: from the node-wide shared arena in sharded output mode (same bytes on
    every rank), else this process's own pinned memory.  ``require_shared``: the caller will fill only THIS rank's part
    (a sharded edge set) - without a common arena (ranks on several nodes) that cannot give a complete tensor."""
    if sharded_output():
        from . import shm

        arena = shm.arena()
        if arena is not None:
            global _shared_host_used
            _shared_host_used = True
            return arena.tensor(shape, dtype)
        if require_shared:
            raise NotImplementedError(
                "sharded output with host-resident graphs needs all ranks on one node (a common /dev/shm); keep the graph "
                "on the devices (device.set_resident(True)) or use the gathered output mode"
            )
    return torch.empty(tuple(shape), dtype=dtype, pin_memory=True)


def exchange_counts(count: int, device: torch.device) -> list[int]:
    """Every rank's ``count`` in rank order: through the shared-memory control block when the ranks share a node (a
    host-side rendezvous of microseconds, the GPU queues keep running), else an NCCL all-gather + read-back."""
    from . import shm

    group = shm.local_group()
    if group is not None:
        return [row[0] for row in group.all_gather([int(count)])]
    return all_gather_counts(int(count), device)


def compute_device(like: torch.Tensor | None = None) -> torch.device:
    """The CUDA device this process computes on (raises without one: there is no CPU fallback)."""
    _cabi.require_cuda()
    if like is not None and like.is_cuda:
        return like.device
    return torch.device("cuda", torch.cuda.current_device())


def to_device(t: torch.Tensor, dtype: torch.dtype | None = None) -> torch.Tensor:
    dev = compute_device(t)
    if not t.is_cuda:
        t = t.to(dev, non_blocking=True)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


@contextlib.contextmanager
def deferred():
    """Scope inside which device->host copies are only awaited at exit."""
    global _defer_depth
    _defer_depth += 1
    try:
        yield
    finally:
        _defer_depth -= 1
        if _defer_depth == 0:
            flush()


def deferring() -> bool:
    """Inside a ``deferred()`` scope (results are only complete when the scope exits)?"""
    return _defer_depth > 0


def flush() -> None:
    """Give every provisionally numbered node set its final order, then wait for every outstanding collective
    (``all_gather_v(async_op=True)``) and device->host copy (``to_host``)."""
    for prov in list(_provisionals):
        prov.resolve()
    wait_copies()
    _early_rows.clear()  # rows no builder adopted
    _prefetch_events.clear()
    global _shared_host_used
    if _shared_host_used:
        # the shared host buffers are complete when EVERY rank's copies have landed
        _shared_host_used = False
        from . import shm

        group = shm.local_group()
        if group is not None:
            import time

            last_trace["copies_done"] = time.perf_counter()
            group.barrier()
            last_trace["node_barrier_done"] = time.perf_counter()


def wait_copies() -> None:
    """Wait for the outstanding collectives and device->host copies only (provisional node sets stay provisional)."""
    for key in list(_works):
        for work in _works.pop(key):
            work.wait()  # NCCL: orders the current stream behind the collective; gloo: blocks the host
    while _pending:
        _pending.pop().synchronize()


def _storage_key(t: torch.Tensor) -> int:
    return t.untyped_storage().data_ptr()


def wait_for(t: torch.Tensor | None) -> None:
    """Order the current stream behind the asynchronous collectives still filling ``t``'s storage."""
    if t is None or not _works:
        return
    for work in _works.pop(_storage_key(t), []):
        work.wait()


def is_device_aware(obj) -> bool:
    """One of this package's own builders / attributes / processors (they work from the cached device copies and
    know about provisional numbering).  Anything else - a reference-style plugin named by a recipe ``_target_`` - may
    read ``graph[n].x`` / ``edge_index`` on the host, so callers ``flush()`` before handing the graph to it."""
    return bool(getattr(type(obj), "_agx_device_aware", False))


def flush_for(obj) -> None:
    """``flush()`` unless ``obj`` is one of the package's device-aware classes."""
    if not is_device_aware(obj):
        flush()


def maybe_flush() -> None:
    if _defer_depth == 0:
        flush()


_copy_streams: dict = {}
_order_streams: dict = {}


def _order_stream(device: torch.device) -> torch.cuda.Stream:
    """The stream a ``Provisional``'s worker thread uploads its index arrays and launches the resolve kernel on."""
    key = device.index if device.index is not None else torch.cuda.current_device()
    if key not in _order_streams:
        _order_streams[key] = torch.cuda.Stream(device=device, priority=-1)
    return _order_streams[key]


def _copy_stream(device: torch.device) -> torch.cuda.Stream:
    key = device.index if device.index is not None else torch.cuda.current_device()
    if key not in _copy_streams:
        _copy_streams[key] = torch.cuda.Stream(device=device)
    return _copy_streams[key]


def to_host(t: torch.Tensor, shard: Shard | None = None, dim: int = 0) -> torch.Tensor:
    """Asynchronous copy of a CUDA tensor into a pinned host tensor (awaited by ``flush``).

    The copy runs on a dedicated stream behind an event recorded on the producing stream, so the PCIe transfer
    of one edge set overlaps the kernels of the next.  With ``shard`` (sharded output mode) ``t`` is this rank's block
    along ``dim`` - or a replicated tensor, of which this rank copies its 1/W slice - and the result is the COMPLETE
    tensor in the node-wide shared host buffer: every rank writes its part over its own PCIe link."""
    if not t.is_cuda:
        return t
    wait_for(t)
    if shard is not None and shard.world > 1 and sharded_output():
        full_shape = list(t.shape)
        if shard.replicated:
            lo, hi = shard_range(int(t.shape[dim]), shard.rank, shard.world)
            src = t.narrow(dim, lo, hi - lo)
        else:
            full_shape[dim] = shard.total
            lo, hi = shard.offset, shard.offset + int(t.shape[dim])
            src = t
        full = host_tensor(full_shape, t.dtype, require_shared=True)
        if hi > lo:
            dst = full.narrow(dim, lo, hi - lo)
            if dst.is_contiguous() and src.is_contiguous():
                to_host_into(src, dst)
            else:  # column block of a (R, E) row-major tensor: one contiguous run per row
                assert t.dim() == 2 and dim == 1
                for r in range(int(t.shape[0])):
                    to_host_into(src[r], dst[r])
        return full
    return to_host_into(t, torch.empty(t.shape, dtype=t.dtype, pin_memory=True))


def copy_replicated_to_host(t: torch.Tensor, out: torch.Tensor) -> None:
    """Copy a tensor every rank holds identically into ``out``: all of it, or - when ``out`` lives in the shared host
    arena (sharded output mode) - this rank's 1/W slice along dim 0."""
    if sharded_output() and _is_shared_host(out):
        rank, w = world()
        lo, hi = shard_range(int(t.shape[0]), rank, w)
        if hi > lo:
            to_host_into(t[lo:hi], out[lo:hi])
        return
    to_host_into(t, out)


def _is_shared_host(t: torch.Tensor) -> bool:
    from . import shm

    arena = shm._arena
    if arena is None:
        return False
    p = t.data_ptr()
    return any(base <= p < base + size for base, size in ((seg.data_ptr(), seg.numel()) for seg in arena.segments.values()))


copy_trace: list | None = None  # tools/copy_timeline.py: (bytes, ready, begin, done) timing events of every host copy


def to_host_into(t: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """``to_host`` into an existing pinned host tensor (or a view of one)."""
    wait_for(t)
    if t.numel() == 0:
        return out
    timing = copy_trace is not None
    ready = torch.cuda.Event(enable_timing=timing)
    ready.record()
    side = _copy_stream(t.device)
    with torch.cuda.stream(side):
        side.wait_event(ready)
        if timing:
            begin = torch.cuda.Event(enable_timing=True)
            begin.record(side)
        out.copy_(t, non_blocking=True)
        done = torch.cuda.Event(enable_timing=timing)
        done.record(side)
    if timing:
        copy_trace.append((t.numel() * t.element_size(), ready, begin, done))
    t.record_stream(side)
    _pending.append(done)
    return out


def like_input(result: torch.Tensor, reference_input: torch.Tensor, shard: Shard | None = None, dim: int = 0) -> torch.Tensor:
    """Return ``result`` (CUDA) on the device the caller's input lives on."""
    return result if reference_input.is_cuda else to_host(result, shard, dim)


# --------------------------------------------------------------------------------------------------
# per-node-set device state
# --------------------------------------------------------------------------------------------------
def _key(t: torch.Tensor) -> tuple:
    return (t.data_ptr(), t._version, tuple(t.shape), str(t.device))


@dataclass
class NodeState:
    key: tuple
    x: torch.Tensor  # CUDA float32 (n, 2)
    tables: object | None = None  # ops.NodeTables
    extras: dict = field(default_factory=dict)
    prov: object | None = None  # Provisional: ``x`` is in provisional numbering until it resolves


STATE_ATTR = "_agx_state"
EDGE_ATTR = "_agx_edge_index"


def node_state(nodes, provisional_ok: bool = False) -> NodeState:
    """Device copy of ``nodes.x`` (uploaded once per node set; re-uploaded if ``x`` was replaced or modified).

    A node set whose final order is still being computed (``Provisional``) is given that order first, unless the
    caller states that it works in the provisional numbering and tags what it produces (``provisional_ok``)."""
    x = nodes["x"]
    st = nodes.get(STATE_ATTR, None) if hasattr(nodes, "get") else None
    if isinstance(st, NodeState) and st.prov is not None:
        if provisional_ok:
            return st
        st.prov.resolve()
        st = nodes[STATE_ATTR]
    if isinstance(st, NodeState) and st.key == _key(x):
        uploaded = st.extras.pop("uploaded", None)  # prefetch_coordinates: the copy runs on a side stream
        if uploaded is not None:
            torch.cuda.current_stream().wait_event(uploaded)
        return st
    wait_copies()  # x may be a pinned tensor one of our own copies is still filling
    st = NodeState(key=_key(x), x=upload_replicated(x))
    nodes[STATE_ATTR] = st
    return st


_upload_streams: dict = {}
_prefetch_events: list = []  # uploads of this build still (possibly) in flight; forgotten at flush
PREFETCH_MIN_BYTES = 1 << 20


def prefetch_coordinates(nodes) -> None:
    """Start the upload of a host node set's coordinates NOW, on a side stream: ``GraphCreator.update_graph`` calls it for
    the node sets a graph arrives with and the recipe's edges name.  The copy engine works while the first kernels of
    the build run (node generation, the reference distance of the OTHER node set); the first ``node_state(nodes)`` orders
    the calling stream behind it.  53 MB of O1280 coordinates: 1 ms that no longer precedes the first search.
    Pinned float32 inputs only (a pageable source is staged synchronously by the driver: nothing to overlap); sharded
    output mode has its own sliced upload."""
    if not torch.cuda.is_available() or sharded_output():
        return
    x = nodes.get("x", None) if hasattr(nodes, "get") else None
    if not isinstance(x, torch.Tensor) or x.is_cuda or x.dtype != torch.float32 or x.dim() != 2 or not x.is_pinned():
        return
    if x.numel() * x.element_size() < PREFETCH_MIN_BYTES or not x.is_contiguous():
        return
    st = nodes.get(STATE_ATTR, None)
    if isinstance(st, NodeState) and (st.prov is not None or st.key == _key(x)):
        return
    dev = compute_device()
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _upload_streams:
        _upload_streams[key] = torch.cuda.Stream(device=dev)
    side = _upload_streams[key]
    x_dev = torch.empty(x.shape, dtype=torch.float32, device=dev)
    side.wait_stream(torch.cuda.current_stream())  # the block may have been freed by work still queued on this stream
    with torch.cuda.stream(side):
        x_dev.copy_(x, non_blocking=True)
        uploaded = torch.cuda.Event()
        uploaded.record(side)
    x_dev.record_stream(side)
    st = NodeState(key=_key(x), x=x_dev)
    st.extras["uploaded"] = uploaded
    nodes[STATE_ATTR] = st
    _prefetch_events.append(uploaded)


# host node sets from this many bytes are uploaded once per NODE in a sharded multi-GPU build (each rank 1/W over its
# own PCIe link, the rest over NVLink) instead of once per GPU
SLICED_UPLOAD_MIN_BYTES = int(float(__import__("os").environ.get("AGX_SLICED_UPLOAD_MIN_BYTES", "4e6")))


def upload_replicated(x: torch.Tensor) -> torch.Tensor:
    """Device float32 copy of host node coordinates that every rank holds identically (every rank runs the same recipe
    on the same inputs).  Sharded output mode on one node: every rank uploads only ITS 1/W of the rows and the ranks
    all-gather the rest over NVLink - W uploads of the whole array (424 MB for O1280 on 8 GPUs) would queue on the
    host's DMA ceiling before any search can start."""
    if x.is_cuda or not sharded_output() or x.numel() * x.element_size() < SLICED_UPLOAD_MIN_BYTES:
        return to_device(x, torch.float32)
    import torch.distributed as dist

    if dist.get_backend() != "nccl":
        return to_device(x, torch.float32)
    rank, w = world()
    dev = compute_device()
    n = int(x.shape[0])
    per = (n + w - 1) // w  # equal blocks (the last one padded): NCCL's in-place all-gather
    full = torch.empty((per * w,) + tuple(x.shape[1:]), dtype=torch.float32, device=dev)
    lo, hi = min(rank * per, n), min((rank + 1) * per, n)
    if hi > lo:
        full[lo:hi].copy_(x[lo:hi], non_blocking=True)  # dtype conversion (if any) on the device side of the copy
    dist.all_gather_into_tensor(full, full[rank * per : (rank + 1) * per])
    return full[:n]


# node sets up to this size keep their neighbour index on the node state (``NodeState.extras``), so the builders of
# one recipe that search the same set with the same cell width share ONE build (reference distance + KNN decoder over
# the hidden nodes); larger sets (106 MB of records for an O1280 grid) are binned per search and freed at once
INDEX_CACHE_MAX_NODES = int(float(__import__("os").environ.get("AGX_INDEX_CACHE_MAX_NODES", "2e6")))


class _Borrowed:
    """Context manager handing out a cached index without closing it."""

    def __init__(self, index) -> None:
        self.index = index

    def __enter__(self):
        return self.index

    def __exit__(self, *exc) -> None:
        return None


def neighbour_index(st: NodeState | None, x: torch.Tensor, hint_k: int = 0, hint_radius: float = 0.0):
    """``with neighbour_index(state, x, hint_k=k) as index`` - the cell-binned index over ``x``; shared through the
    node state when ``x`` IS the state's coordinate tensor (no mask) and the set is small, else built for this search
    and freed when the block exits."""
    from . import ops

    if st is None or x is not st.x or int(x.shape[0]) > INDEX_CACHE_MAX_NODES:
        return ops.NeighbourIndex(x, hint_k=hint_k, hint_radius=hint_radius)
    cache = st.extras.setdefault("index", {})
    key = (int(hint_k), float(hint_radius))
    hit = cache.get(key)
    if hit is None or hit.handle is None:
        hit = cache[key] = ops.NeighbourIndex(x, hint_k=hint_k, hint_radius=hint_radius)
    return _Borrowed(hit)


def seed_node_state(nodes, x_dev: torch.Tensor) -> NodeState:
    """Install an already-resident device copy of ``nodes.x`` (e.g. coordinates generated on the GPU)."""
    st = NodeState(key=_key(nodes["x"]), x=x_dev.contiguous())
    nodes[STATE_ATTR] = st
    return st


def node_tables(nodes, with_rotation: bool = True, provisional_ok: bool = False):
    from . import ops

    st = node_state(nodes, provisional_ok)
    if st.tables is None:
        st.tables = ops.NodeTables(st.x)
    return st.tables


# --------------------------------------------------------------------------------------------------
# provisional numbering: edge construction that overlaps the host-side node ordering
# --------------------------------------------------------------------------------------------------
_provisionals: list = []
_prov_seq = 0
SHARED_NODE_ORDER = __import__("os").environ.get("AGX_SHARED_ORDER", "1") != "0"
_order_pool = None
last_trace: dict = {}  # host timestamps of the most recent provisional node set (tools/step_timeline.py)
# AGX_LAZY_ORDER=0 restores the serial "sort, then build" order of operations (A/B measurements)
LAZY_NODE_ORDER = __import__("os").environ.get("AGX_LAZY_ORDER", "1") != "0"


# The thread that runs the node-order sort is pinned to one CPU of the process's affinity set (the last one, minus the
# local rank) when several ranks share the host: the scheduler then does not migrate it while the other ranks' threads
# are busy (N = 2, O1280 -> res 7: 6.05 -> 5.73 ms/step; no effect on a single process, where it stays off).
# AGX_PIN_SORT=0 / 1 forces it off / on.
PIN_SORT_THREAD = __import__("os").environ.get("AGX_PIN_SORT", "auto")
_sort_thread_pinned = False


def _pin_sort_thread(follower: bool) -> None:
    global _sort_thread_pinned
    want = PIN_SORT_THREAD == "1" or (PIN_SORT_THREAD == "auto" and world()[1] > 1)
    if not want or _sort_thread_pinned or follower:
        return
    import os

    try:
        cpus = sorted(os.sched_getaffinity(0))
        local = int(os.environ.get("LOCAL_RANK", "0"))
        os.sched_setaffinity(0, {cpus[-1 - (local % len(cpus))]})
        _sort_thread_pinned = True
    except (AttributeError, OSError):
        pass


_upload_pool = None
# AGX_UPLOAD_HANDOVER=1: the sorting thread hands every index array but the last to a helper thread for its pinned copy
# + upload.  Measured (tools/tail_ab.py): the 0.15 ms leave the sorting thread, the step does not get shorter
# (5.22 / 5.24 ms, host-resident 14.2 / 14.3 ms: the helper competes with the main thread's launches) - off by default.
UPLOAD_HANDOVER = os.environ.get("AGX_UPLOAD_HANDOVER", "0") == "1"


def _upload_helper():
    global _upload_pool
    if _upload_pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _upload_pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="agx-order-upload")
    return _upload_pool


# Everything that follows the node order (upload of the index arrays, agx_order_resolve, tie re-decision, relabel,
# scaling pass, device -> host copies) is queued on the main stream BEFORE the sort has ended, behind stream gates
# (agx_gate_wait) that the sorting thread opens with a plain store the moment an index array lies in page-locked host
# memory: the host's launch work (0.25 ms) leaves the critical path.  Only the CPU opens a gate and the sorting thread
# needs no GPU after its coordinates have arrived, so a waiting stream can never wait for work queued behind itself.
# Measured on B200 (tools/tail_ab.py, modes interleaved in one process, O1280 -> res 7): device-resident build
# 5.22 -> 5.05 ms per step; host-resident build 14.2 -> 14.45 ms (the build is bound by the device -> host DMA queue there
# and the early queueing disturbs it).  "auto": on for device-resident graphs only; "1" / "0": always / never.
PRELAUNCH_TAIL = os.environ.get("AGX_PRELAUNCH_TAIL", "auto")


def _prelaunch_wanted() -> bool:
    mode = PRELAUNCH_TAIL
    if isinstance(mode, bool):
        return mode
    return mode == "1" or (mode == "auto" and _resident)


_gate_ring = None
_gate_next = 0
GATE_RING = 256


def _new_gates(count: int) -> torch.Tensor:
    """``count`` consecutive closed gates (int32 words of page-locked host memory, from a ring that outlives every build)."""
    global _gate_ring, _gate_next
    if _gate_ring is None:
        _gate_ring = torch.zeros(GATE_RING, dtype=torch.int32, pin_memory=True)
    if _gate_next % GATE_RING + count > GATE_RING:
        _gate_next += GATE_RING - _gate_next % GATE_RING
    lo = _gate_next % GATE_RING
    _gate_next += count
    gates = _gate_ring[lo : lo + count]
    gates.zero_()
    return gates


def _pool():
    global _order_pool
    if _order_pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _order_pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="agx-node-order")
    return _order_pool


class Provisional:
    """A node set whose FINAL order is still being computed on a host thread.

    The order of icosahedral nodes is defined by two unstable numpy argsorts on the host
    (``generate.utils.get_coordinates_ordering``, DESIGN.md H4: 4.4 ms for 164 k nodes, more than all the GPU
    work of the O1280 graph).  Edge sets whose content does not depend on how the nodes are numbered - cut-off
    and multi-scale edges, every attribute - are therefore built right away in the generator's own numbering
    (``x_prov``), while a worker thread sorts; each index row they produce is registered here (``add_row``) and
    rewritten ``v -> rank[v]`` (``agx_relabel_nodes``) once the order is known, before it is copied to the host.
    Anything that does depend on the numbering (KNN's lower-index tie rule on the source side, masks, merged
    builders, a caller reading ``x``) asks for the final order first: ``node_state(nodes)`` / ``flush()``.

    Only a permutation is supported (same node count before and after)."""

    def __init__(self, x_prov: torch.Tensor, sorter, combine) -> None:
        """``sorter(lat, lon, emit)`` runs on the worker thread on contiguous host float32 columns, calls ``emit(array)``
        for every int64 index array as soon as it is final and returns them all; ``combine`` turns them into the order
        (CUDA int64: generator index at every graph position) on the device - ``"latlon"``: the two argsorts of
        ``get_coordinates_ordering``, combined by ``agx_order_resolve`` which the WORKER launches on its own stream the
        moment the second sort returns (no hand-over to the main thread in between); else a callable
        ``combine(*device_copies)``."""
        import time

        self.x_prov = x_prov.contiguous()
        n = int(x_prov.shape[0])
        self.n = n
        dev = x_prov.device
        self.combine = combine
        self.x_final = torch.empty((n, 2), dtype=torch.float32, device=dev)
        self.x_host = None  # pinned (n, 2) float32 when the graph lives on the host
        self.order_host = host_tensor((n,), torch.int64)  # ``_node_ordering`` (shared host buffer in sharded output mode)
        # everything the resolution needs exists before the sort ends
        self.order_dev = torch.empty(n, dtype=torch.int64, device=dev)
        self.rank = torch.empty(n + 1, dtype=torch.int64, device=dev)  # final position of every provisional label
        self.rows: list = []
        self.fixups: list = []
        self.finalizers: list = []
        self.nodes = None
        self.state = None
        self.on_resolved = None
        self.done = False
        self._order_ready = None  # event on the worker's stream: order / rank / x_final are complete
        # the worker needs the coordinates on the host, as two contiguous columns: one async copy behind the
        # kernel that produced them
        columns = self.x_prov.t().contiguous()
        staged = torch.empty((2, n), dtype=torch.float32, pin_memory=True)
        ready = torch.cuda.Event()
        ready.record()
        side = _copy_stream(dev)
        with torch.cuda.stream(side):
            side.wait_event(ready)
            staged.copy_(columns, non_blocking=True)
            copied = torch.cuda.Event()
            copied.record(side)
        columns.record_stream(side)
        self.trace = {"created": time.perf_counter()}
        max_parts = 2
        # More than one rank on this node: ONE rank sorts, the index arrays travel through the shared page-locked host
        # arena (every rank uploads them from there), the others' workers wait on a stamp in the control block - one
        # host sort per node instead of one per GPU (8 AVX-512 sorts side by side slow each other down).
        group, prov_seq = None, 0
        if SHARED_NODE_ORDER and world()[1] > 1:
            from . import shm

            group = shm.local_group()
        if group is not None:
            global _prov_seq
            global _shared_host_used
            _shared_host_used = True  # flush() ends with the node-wide barrier
            prov_seq, _prov_seq = _prov_seq, _prov_seq + 1
            parts_pinned = shm.arena().tensor((max_parts, n), torch.int64)
            stamps = group.order[prov_seq % shm.RING]
        else:
            parts_pinned = torch.empty((max_parts, n), dtype=torch.int64, pin_memory=True)
        parts_dev = torch.empty((max_parts, n), dtype=torch.int64, device=dev)
        follower = group is not None and group.rank != 0
        ostream = _order_stream(dev)
        for t in (parts_dev, self.order_dev, self.rank, self.x_final, self.x_prov):
            t.record_stream(ostream)
        import threading

        gates = None
        if _prelaunch_wanted() and combine == "latlon" and _cabi.load_library().agx_gate_supported():
            gates = _new_gates(max_parts)
        gates_np = gates.numpy() if gates is not None else None
        self._gates, self._parts_pinned, self._parts_dev, self._group = gates, parts_pinned, parts_dev, group
        self._coords_ready = threading.Event()  # the worker needs nothing from the GPU any more

        def work():
            from ._cabi import check, load_library

            torch.cuda.set_device(dev)  # the device context is per thread
            _pin_sort_thread(follower)
            self.trace["worker_start"] = time.perf_counter()
            copied.synchronize()  # the coordinates are on the host (and complete on the device)
            self._coords_ready.set()
            self.trace["coords_on_host"] = time.perf_counter()
            cols = staged.numpy()
            sent = []

            def upload(i: int, part) -> None:  # pinned copy (node-wide when the order is shared) and upload
                if part is not None:
                    parts_pinned[i].numpy()[:] = part
                    if group is not None:
                        stamps[i] = prov_seq + 1  # the followers may read part i now ...
                        group.wake_followers()  # ... and are asleep in read(2): one byte each
                if gates_np is not None:
                    gates_np[i] = 1  # the main stream's queued upload of part i may start (x86: stores stay in order)
                    return
                with torch.cuda.stream(ostream):
                    parts_dev[i].copy_(parts_pinned[i], non_blocking=True)

            handed_over = []

            def emit(part) -> None:  # an index array is final
                i = len(sent)
                self.trace[f"part{i}_ready"] = time.perf_counter()
                if i < max_parts:
                    if UPLOAD_HANDOVER and part is not None and i + 1 < max_parts:
                        # not the last array: its 0.15 ms of copy + upload go to a helper thread, the next sort (the
                        # critical path of the whole build) starts at once
                        handed_over.append(_upload_helper().submit(upload, i, part))
                    else:
                        for f in handed_over:  # uploads are queued on the order stream in order, failures surface here
                            f.result()
                        upload(i, part)
                sent.append(part)
                self.trace[f"part{i}_sent"] = time.perf_counter()

            if follower:
                from . import shm

                # the sorting rank's arrays, as they appear.  The first wait is long and of unknown length: asleep in
                # read(2) until the wake-up byte.  Every later array takes about as long as the first did (the same sort
                # on the same number of keys), so the follower sleeps 80 % of that and then polls the stamp - it picks
                # the array up within microseconds instead of a scheduler wake-up (~0.1 ms on the critical path).
                t_start = time.perf_counter()
                t_first = None
                for i in range(max_parts):
                    if i == 0 or t_first is None:
                        group.sleep_until_woken()
                    else:
                        time.sleep(max(0.0, 0.8 * t_first - (time.perf_counter() - t_prev)))
                        while int(stamps[i]) not in (prov_seq + 1, -(prov_seq + 1)):
                            time.sleep(0)
                        group.drain_wakeups()
                    if int(stamps[i]) == -(prov_seq + 1):
                        raise RuntimeError("the rank that sorts the node order failed; see its traceback")
                    shm._spin(lambda i=i: int(stamps[i]) == prov_seq + 1, f"part {i} of node order {prov_seq}")
                    t_prev = time.perf_counter()
                    if i == 0:
                        t_first = t_prev - t_start
                    emit(None)
                out = (None, None)
            else:
                try:
                    out = sorter(cols[0], cols[1], emit)
                except BaseException:
                    if group is not None:  # do not leave the followers asleep: a negative stamp tells them to give up
                        stamps[:] = -(prov_seq + 1)
                        for _ in range(max_parts):
                            group.wake_followers()
                    raise
                out = out if isinstance(out, tuple) else (out,)
            self.trace["sorted"] = time.perf_counter()
            if gates_np is not None:
                if len(sent) != max_parts:
                    raise RuntimeError(f"node order: the sorter emitted {len(sent)} index arrays, {max_parts} were queued for")
                return None  # the upload and agx_order_resolve are (being) queued by resolve() behind the gates
            if self.combine == "latlon" and len(out) == 2 and len(sent) == 2:
                # order, its inverse and the re-ordered coordinates in one kernel, launched from here
                check(
                    load_library().agx_order_resolve(
                        parts_dev[0].data_ptr(), parts_dev[1].data_ptr(), n, self.x_prov.data_ptr(),
                        self.x_final.data_ptr(), self.order_dev.data_ptr(), self.rank.data_ptr(), ostream.cuda_stream,
                    )
                )
                done = torch.cuda.Event()
                done.record(ostream)
                self._order_ready = done
                if group is not None:
                    _pending.append(done)  # awaited before the end-of-build barrier: the shared arrays have been read
                self.trace["order_launched"] = time.perf_counter()
                return None
            assert not follower, "a shared node order needs the 'latlon' combine"
            return out

        def guarded():
            try:
                return work()
            except BaseException:
                # never leave the device waiting for index arrays that will not come: valid (identity) arrays, gates open;
                # resolve() re-raises this failure
                self._coords_ready.set()
                if gates_np is not None:
                    import numpy as np

                    parts_pinned.numpy()[:] = np.arange(n, dtype=np.int64)
                    gates_np[:] = 1
                raise

        self.future = _pool().submit(guarded)
        _provisionals.append(self)

    def __getstate__(self):  # never pickled with its worker future / pinned buffers
        return {"done": True, "n": self.n}

    def attach(self, nodes, state: NodeState) -> None:
        self.nodes, self.state = nodes, state
        state.prov = self
        state.x = self.x_prov

    def add_row(self, tensor: torch.Tensor, row: int, host_row: torch.Tensor | None, cols: tuple | None = None) -> None:
        """``tensor[row]`` (CUDA int32 (2, E)) holds provisional indices of this node set; ``host_row`` is the pinned
        1-D destination of the final ones (None: the graph is device-resident) - of the whole row, or of its columns
        ``cols = (lo, hi)`` (a replicated edge set in sharded output mode: every rank copies a slice)."""
        self.rows.append((tensor, row, host_row, cols))

    def add_fixup(self, fn) -> None:
        """``fn(self)`` runs when the order resolves (``self.rank`` / ``self.order_dev`` are known), BEFORE the
        registered rows are relabelled: everything is still in provisional numbering (KNN re-decides its index-order
        ties there, the attributes of the re-decided edges are evaluated again)."""
        self.fixups.append(fn)

    def add_finalizer(self, fn) -> None:
        """``fn(self)`` runs after every fixup, CONCURRENTLY with the relabel of the registered rows (which happens on a
        side stream): it must not read index rows - it is the normalisation of attributes whose statistics waited for
        a re-decision, and their host copies."""
        self.finalizers.append(fn)

    def resolve(self) -> None:
        if self.done:
            return
        self.done = True
        if self in _provisionals:
            _provisionals.remove(self)
        import time

        self.trace["resolve_enter"] = time.perf_counter()
        dev = self.x_prov.device
        order_dev, rank = self.order_dev, self.rank
        gated = self._gates is not None
        if gated:
            from ._cabi import check, load_library

            lib = load_library()
            self._coords_ready.wait()  # from here on only the CPU stands between the device and an open gate
            main = torch.cuda.current_stream()
            for i in range(int(self._gates.numel())):
                check(lib.agx_gate_wait(self._gates.data_ptr() + 4 * i, main.cuda_stream))
                self._parts_dev[i].copy_(self._parts_pinned[i], non_blocking=True)
            if self._group is not None:
                uploaded = torch.cuda.Event()
                uploaded.record(main)
                _pending.append(uploaded)  # awaited before the end-of-build barrier: the shared arrays have been read
            check(
                lib.agx_order_resolve(
                    self._parts_dev[0].data_ptr(), self._parts_dev[1].data_ptr(), self.n, self.x_prov.data_ptr(),
                    self.x_final.data_ptr(), order_dev.data_ptr(), rank.data_ptr(), main.cuda_stream,
                )
            )
            self.trace["order_launched"] = time.perf_counter()
        else:
            parts = self.future.result()  # None: the worker has launched the resolve kernel itself
            self.trace["resolve_got_order"] = time.perf_counter()
        if gated:
            pass  # order / rank / x_final are produced in stream order by what was just queued
        elif parts is None:
            torch.cuda.current_stream().wait_event(self._order_ready)
        else:
            staged = torch.empty((len(parts), self.n), dtype=torch.int64, pin_memory=True)
            for i, part in enumerate(parts):
                staged[i].numpy()[:] = part
            parts_dev = staged.to(dev, non_blocking=True)
            order_dev = self.combine(*[parts_dev[i] for i in range(int(parts_dev.shape[0]))]).contiguous()
            rank[order_dev] = torch.arange(self.n, dtype=torch.int64, device=dev)
            torch.index_select(self.x_prov, 0, order_dev, out=self.x_final)
        self.order_dev = order_dev
        self.rank = rank
        fixups, self.fixups = self.fixups, []
        for fn in fixups:
            fn(self)
        from . import ops

        for tensor, row, host_row, cols in self.rows:
            wait_for(tensor)  # a sharded builder's all-gather may still be filling it
        # The relabel of every provisional row (one launch, gather-latency-bound: 30 % of the DRAM rate) runs on a side
        # stream WHILE the finalizers - the HBM-bound scaling pass of the attributes whose statistics waited for the tie
        # re-decision - run on the main stream: different data, and the fixups that still read provisional labels are
        # all enqueued before this point.
        main = torch.cuda.current_stream()
        side = _order_stream(dev)
        fixed = torch.cuda.Event()
        fixed.record(main)
        with torch.cuda.stream(side):
            side.wait_event(fixed)
            ops.relabel_rows([tensor[row] for tensor, row, host_row, cols in self.rows], rank)  # one launch for all rows
            relabelled = torch.cuda.Event()
            relabelled.record(side)
        for tensor, row, host_row, cols in self.rows:
            tensor.record_stream(side)
        rank.record_stream(side)
        finalizers, self.finalizers = self.finalizers, []
        for fn in finalizers:
            fn(self)
        main.wait_event(relabelled)
        for tensor, row, host_row, cols in self.rows:
            if host_row is not None and host_row.numel():
                to_host_into(tensor[row] if cols is None else tensor[row, cols[0] : cols[1]], host_row)
        self.rows = []
        # host copies that nothing on the device waits for go last: ``_node_ordering`` and (host-resident graphs) ``x``
        # are complete at flush like every host copy
        copy_replicated_to_host(order_dev, self.order_host)
        if self.x_host is not None:
            copy_replicated_to_host(self.x_final, self.x_host)
        if gated:
            self.trace["tail_queued"] = time.perf_counter()
            self.future.result()  # the sort (a failure surfaces here; its handler has opened the gates)
            self.trace["resolve_got_order"] = time.perf_counter()
        if self.state is not None:
            st = self.state
            st.prov = None
            st.x = self.x_final
            st.tables = None  # built from the provisional coordinates
            st.extras = {}
            if self.nodes is not None:
                st.key = _key(self.nodes["x"])
        if self.on_resolved is not None:
            self.on_resolved(self)
        self.trace["resolve_done"] = time.perf_counter()
        global last_trace
        last_trace = self.trace


def active_provisional(nodes):
    """The unresolved ``Provisional`` of a node set, or None."""
    st = nodes.get(STATE_ATTR, None) if hasattr(nodes, "get") else None
    return st.prov if isinstance(st, NodeState) else None


# Bookkeeping about a freshly built CUDA edge_index (which rows are provisional, a pending tie re-decision, which
# columns this rank produced).  It lives in a side table keyed by the tensor's identity, NOT on the tensor: torch
# pickles a tensor's ``__dict__``, and a device-resident graph stores these very tensors, so attributes holding a
# ``Provisional`` (a ``Future``, pinned buffers) would break ``torch.save(graph)`` and keep the buffers alive.
class EdgeMeta:
    __slots__ = ("prov", "fixup", "local", "tie_flags", "tie_list", "regular_k", "shard", "flag_base", "regular_targets")

    def __init__(self) -> None:
        self.prov = (None, None)  # (source row, target row): the Provisional whose numbering the row is in
        self.fixup = None  # Provisional that still has to re-decide KNN ties of this edge list ...
        self.tie_flags = None  # ... and the CUDA uint8 flag per TARGET node naming the queries it will re-decide
        self.tie_list = None  # (list, count) = ops.compact_flags(tie_flags)
        self.regular_k = 0  # k when the edges of target t are the columns [t k, (t + 1) k) (a KNN result)
        self.regular_targets = False  # ... and row 1 is exactly t = column // k for ALL targets (unmasked, one rank)
        self.flag_base = 0  # tie_flags[t - flag_base] belongs to target t (a rank's block starts at its first target)
        self.shard = None  # Shard: sharded output mode - this tensor is the rank's own block (or a replicated set)
        self.local = None  # (lo, hi, counts): this rank's own columns of a sharded edge list


_edge_meta: dict[int, tuple] = {}


def edge_meta(edge_index: torch.Tensor, create: bool = False) -> EdgeMeta | None:
    import weakref

    key = id(edge_index)
    hit = _edge_meta.get(key)
    if hit is not None and hit[0]() is edge_index:
        return hit[1]
    if not create:
        return None
    meta = EdgeMeta()
    _edge_meta[key] = (weakref.ref(edge_index, lambda _r, key=key: _edge_meta.pop(key, None)), meta)
    return meta


def tag_rows(edge_index: torch.Tensor, src_prov, dst_prov) -> torch.Tensor:
    """Mark which rows of a freshly built CUDA (2, E) edge_index are in provisional numbering."""
    if src_prov is not None or dst_prov is not None:
        edge_meta(edge_index, create=True).prov = (src_prov, dst_prov)
    return edge_index


def row_tags(edge_index: torch.Tensor) -> tuple:
    meta = edge_meta(edge_index)
    tags = meta.prov if meta is not None else (None, None)
    return tuple(p if (p is not None and not p.done) else None for p in tags)


def edge_shard(edge_index: torch.Tensor) -> Shard | None:
    meta = edge_meta(edge_index)
    return meta.shard if meta is not None else None


# The target row of an unmasked KNN edge list is known before any search has run: target t owns the columns
# [t k, (t + 1) k).  For a host-resident graph ``GraphCreator.update_graph`` has it written and sent on its way the moment
# the node builders are queued (``emit_regular_target_row``): 79 MB of the O1280 decoder cross PCIe while the device->host
# copy queue would otherwise wait 1.9 ms for the first search result; the builder's ``edge_index_like_input`` adopts the
# host tensor and copies the source row only.  AGX_EARLY_TARGET_ROW=0 disables.
EARLY_TARGET_ROW = os.environ.get("AGX_EARLY_TARGET_ROW", "1") != "0"
_early_rows: dict = {}  # (n_targets, k) -> pinned int32 (2, n_targets k) whose row 1 is complete at flush


def emit_regular_target_row(n_targets: int, k: int) -> None:
    e = int(n_targets) * int(k)
    if not EARLY_TARGET_ROW or e <= 0 or e >= 2**31 or (n_targets, k) in _early_rows or sharded_output():
        return
    dev = compute_device()
    host = torch.empty((2, e), dtype=torch.int32, pin_memory=True)
    row = torch.div(torch.arange(e, dtype=torch.int32, device=dev), int(k), rounding_mode="floor")
    # behind the coordinate uploads: the two directions share the host's DMA rate, and the upload gates the first search
    # (measured: started together, the upload takes twice as long and the first result appears 1.3 ms later)
    side = _copy_stream(dev)
    for uploaded in _prefetch_events:
        side.wait_event(uploaded)
    to_host_into(row, host[1])
    _early_rows[(int(n_targets), int(k))] = host


def _adopt_early_row(edge_dev: torch.Tensor) -> torch.Tensor | None:
    """The pinned (2, E) host tensor whose target row was emitted ahead for exactly this edge list, or None."""
    meta = edge_meta(edge_dev)
    if not _early_rows or meta is None or not meta.regular_targets or not meta.regular_k or edge_dev.dtype != torch.int32:
        return None
    return _early_rows.pop((int(edge_dev.shape[1]) // meta.regular_k, meta.regular_k), None)


def edge_index_like_input(edge_dev: torch.Tensor, reference_input: torch.Tensor) -> torch.Tensor:
    """``like_input`` for an edge_index that may carry provisional rows: final rows are copied (or returned) now,
    provisional rows are registered with their node set and complete when it resolves.  In sharded output mode the host
    result is the complete (2, E) list in the shared host buffer; this rank fills its own columns."""
    tags = row_tags(edge_dev)
    shard = edge_shard(edge_dev)
    if shard is not None and not (shard.world > 1 and sharded_output()):
        shard = None
    if tags == (None, None):
        early = _adopt_early_row(edge_dev) if (shard is None and not reference_input.is_cuda) else None
        if early is None:
            return like_input(edge_dev, reference_input, shard, dim=1)
        to_host_into(edge_dev[0], early[0])  # the target row is in flight since the top of the build
        return early
    if reference_input.is_cuda:
        for row, prov in enumerate(tags):
            if prov is not None:
                prov.add_row(edge_dev, row, None)
        return edge_dev
    early = None
    if shard is None:
        if tags[1] is None:
            early = _adopt_early_row(edge_dev)
        out = early if early is not None else torch.empty(edge_dev.shape, dtype=edge_dev.dtype, pin_memory=True)
        lo, hi, cols = 0, int(edge_dev.shape[1]), None
    else:
        out = host_tensor((2, shard.total), edge_dev.dtype, require_shared=True)
        if shard.replicated:
            lo, hi = shard_range(int(edge_dev.shape[1]), shard.rank, shard.world)
            cols = (lo, hi)  # of the (complete) device tensor
        else:
            lo, hi, cols = shard.offset, shard.offset + int(edge_dev.shape[1]), None
    for row, prov in enumerate(tags):
        host_row = out[row, lo:hi]
        if prov is None:
            if row == 1 and early is not None:
                continue  # the target row is in flight since the top of the build
            if hi > lo:
                to_host_into(edge_dev[row] if cols is None else edge_dev[row, cols[0] : cols[1]], host_row)
        else:
            prov.add_row(edge_dev, row, host_row, cols)
    return out


def remember_edge_index(store, host_or_dev: torch.Tensor, dev: torch.Tensor) -> None:
    store[EDGE_ATTR] = (_key(host_or_dev), dev)


def device_edge_index(store) -> torch.Tensor:
    """CUDA int32 (2, E) copy of ``store.edge_index``."""
    ei = store["edge_index"]
    if ei.is_cuda:
        return ei if ei.dtype == torch.int32 and ei.is_contiguous() else ei.to(torch.int32).contiguous()
    cached = store.get(EDGE_ATTR, None) if hasattr(store, "get") else None
    if cached is not None and cached[0] == _key(ei):
        return cached[1]
    flush()
    dev = to_device(ei, torch.int32)
    remember_edge_index(store, ei, dev)
    return dev


# --------------------------------------------------------------------------------------------------
# multi-GPU shard context
# --------------------------------------------------------------------------------------------------
def world() -> tuple[int, int]:
    """(rank, world_size) of the sharded build; (0, 1) when torch.distributed is not initialised."""
    import torch.distributed as dist

    if not _force_single and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


# A multi-GPU build shards a neighbour search over its QUERY nodes only when there are at least this many of them:
# every rank needs the complete result, so a sharded edge set is all-gathered (20 bytes per edge to every rank, a
# handful of collective launches), which costs more than it saves while one GPU does the whole search in well under
# a millisecond.  Below the threshold every rank computes the (identical) full edge set.  Measured on O1280 -> res 7
# (6.6 M queries, 0.44 ms on one B200) at N = 2: searches and attributes sharded 6.4 ms/step and 22.2 ms host-to-host
# (the device->host copies queue behind the all-gathers), everything replicated 6.3 / 14.0 ms = the single-GPU
# numbers.  AGX_SHARD_MIN_QUERIES=0 AGX_ATTR_SHARD_MIN_EDGES=0 force sharding (tools/dist_check.py, tools/sweep.py).
SHARD_MIN_QUERIES = int(float(__import__("os").environ.get("AGX_SHARD_MIN_QUERIES", "16e6")))


def shard_world(n_queries: int) -> tuple[int, int]:
    """``world()`` for a search over ``n_queries`` query nodes: (0, 1) - every rank does all of it - when the set is
    too small for sharding to pay."""
    rank, w = world()
    if w > 1 and n_queries < SHARD_MIN_QUERIES:
        return 0, 1
    return rank, w


def shard_range(n: int, rank: int | None = None, world_size: int | None = None) -> tuple[int, int]:
    """Contiguous range of ``n`` units owned by ``rank``: ``[rank*n//W, (rank+1)*n//W)``."""
    if rank is None or world_size is None:
        rank, world_size = world()
    return (rank * n) // world_size, ((rank + 1) * n) // world_size


def all_gather_counts(count: int, device: torch.device) -> list[int]:
    import torch.distributed as dist

    _, w = world()
    mine = torch.tensor([count], dtype=torch.int64, device=device)
    out = torch.empty(w, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(out, mine)
    return [int(v) for v in out.tolist()]


def all_gather_v(full: torch.Tensor, counts: list[int], dim: int, async_op: bool = False) -> torch.Tensor:
    """In-place variable-length all-gather along ``dim``.

    ``full`` is the complete output buffer; this rank has already written its own block (the slice at
    offset ``sum(counts[:rank])`` of length ``counts[rank]``) - the kernels write straight into it, so
    there is no staging copy.  NCCL moves every rank's block into every other rank's buffer.

    ``async_op=True`` only enqueues the transfers: the other ranks' blocks are complete after ``wait_for(full)``
    (issued automatically by ``to_host`` and ``flush``), so the exchange overlaps the kernels of the next edge set.
    """
    import torch.distributed as dist

    rank, w = world()
    if w == 1:
        return full
    offs = [0]
    for c in counts:
        offs.append(offs[-1] + c)
    if dim == 0 or full.shape[0] == 1:
        rows = [full]
    else:  # (R, E) row-major: each row is its own contiguous gather
        rows = [full[r] for r in range(full.shape[0])]
        dim = 0
    backend = dist.get_backend()
    equal = len(set(counts)) == 1 and counts[0] > 0
    works = []
    for row in rows:
        views = [row.narrow(dim, offs[r], counts[r]) for r in range(w)]
        if equal and row.is_contiguous():
            # equal blocks: NCCL's in-place all-gather (send buffer = this rank's slot of the receive buffer)
            works.append(dist.all_gather_into_tensor(row, views[rank], async_op=async_op))
        elif backend == "nccl":
            # unequal sizes: one NCCL group of point-to-point transfers, every block straight into its place on every
            # peer (ProcessGroupNCCL's own uneven all_gather is one broadcast per rank, one after the other:
            # 245 GB/s per rank for the 100 M-query cut-off at N = 4 against 640 GB/s for the equal-block gather)
            ops = []
            for peer in range(w):
                if peer == rank:
                    continue
                if counts[rank]:
                    ops.append(dist.P2POp(dist.isend, views[rank], peer))
                if counts[peer]:
                    ops.append(dist.P2POp(dist.irecv, views[peer], peer))
            reqs = dist.batch_isend_irecv(ops) if ops else []
            if async_op:
                works.extend(reqs)
            else:
                for req in reqs:
                    req.wait()
        else:  # gloo (CPU tests): broadcasts
            for r in range(w):
                if counts[r]:
                    works.append(dist.broadcast(views[r], src=r, async_op=async_op))
    if async_op:
        _works.setdefault(_storage_key(full), []).extend(wk for wk in works if wk is not None)
    return full


# --------------------------------------------------------------------------------------------------
# chunked exchange: the all-gather of per-rank edge blocks overlapped with the search that produces them
# --------------------------------------------------------------------------------------------------
GATHER_CHUNK_QUERIES = int(float(__import__("os").environ.get("AGX_GATHER_CHUNK_QUERIES", "4e6")))


def query_chunks(lo: int, hi: int, n_chunks: int) -> list[tuple[int, int]]:
    """The query range [lo, hi) cut into ``n_chunks`` nearly equal pieces (some may be empty)."""
    n = hi - lo
    return [(lo + (i * n) // n_chunks, lo + ((i + 1) * n) // n_chunks) for i in range(n_chunks)]


def n_query_chunks(nq: int, world_size: int) -> int:
    """How many chunks every rank cuts its query range into (the same number on all ranks)."""
    per_rank = (nq + world_size - 1) // world_size
    return max(1, min(16, (per_rank + GATHER_CHUNK_QUERIES - 1) // GATHER_CHUNK_QUERIES))


_gather_pg = None


def _gather_group():
    """A process group of all ranks whose NCCL kernels run on a HIGH-PRIORITY stream: the exchange of a finished
    chunk must get its few CTAs while the (persistent, SM-filling) search kernel of the next chunk is running."""
    global _gather_pg
    import torch.distributed as dist

    if _gather_pg is None:
        opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        _gather_pg = dist.new_group(backend="nccl", pg_options=opts)
    return _gather_pg


class ChunkedGather:
    """All-gather of a sharded (2, E) edge list that runs WHILE the search fills it.

    Every rank searches its query range in the same number of chunks.  When a chunk's kernels have written their
    columns (main stream), a second stream packs them into the rank's slot of a padded (W, 2, max) buffer, runs
    NCCL's equal-block in-place all-gather on it (640 GB/s per rank over NVLink, against ~260 GB/s for an uneven
    exchange) and unpacks the other ranks' slots into their final columns of ``full`` - while the main stream is
    already searching the next chunk.  ``finish`` orders the main stream behind the last unpack.  The collectives
    are issued in chunk order on every rank; empty chunks are skipped consistently (the count matrix is global).

    ``counts[r][c]`` = number of columns rank ``r`` produces in its chunk ``c``; rank ``r``'s block starts at column
    ``sum(counts[:r])`` and its chunks follow each other inside it."""

    def __init__(self, full: torch.Tensor, counts: list[list[int]]) -> None:
        self.rank, self.w = world()
        self.full = full
        self.counts = counts
        self.offsets = []
        col = 0
        for r in range(self.w):
            row = []
            for c in counts[r]:
                row.append(col)
                col += c
            self.offsets.append(row)
        assert col == full.shape[1], (col, tuple(full.shape))
        self.on_device = full.is_cuda
        if self.on_device:
            self.side = torch.cuda.Stream(device=full.device, priority=-1)
            self.group = _gather_group()
        else:  # host tensors (gloo, the CPU tests of the bookkeeping): same steps, inline, default group
            self.side = None
            self.group = None

    def mark(self):
        """Event after the kernels of the chunk just enqueued on the current stream."""
        if not self.on_device:
            return None
        ready = torch.cuda.Event()
        ready.record()
        return ready

    def _exchange(self, c: int, widest: int) -> None:
        import torch.distributed as dist

        full, rank = self.full, self.rank
        slots = torch.empty((self.w, 2, widest), dtype=full.dtype, device=full.device)
        mine, o = self.counts[rank][c], self.offsets[rank][c]
        if mine:
            slots[rank, :, :mine].copy_(full[:, o : o + mine])
        dist.all_gather_into_tensor(slots.view(-1), slots[rank].reshape(-1), group=self.group)
        for r in range(self.w):
            n, o = self.counts[r][c], self.offsets[r][c]
            if r != rank and n:
                full[:, o : o + n].copy_(slots[r, :, :n])
        return slots

    def chunk_done(self, c: int, ready=None) -> None:
        """Exchange chunk ``c`` once ``ready`` (default: everything enqueued so far) has completed.  Call it AFTER
        enqueuing the search of chunk c + 1, so that the main stream never waits for this host work."""
        widest = max(self.counts[r][c] for r in range(self.w))
        if widest == 0:
            return
        if not self.on_device:
            self._exchange(c, widest)
            return
        if ready is None:
            ready = self.mark()
        with torch.cuda.stream(self.side):
            self.side.wait_event(ready)
            slots = self._exchange(c, widest)
            slots.record_stream(self.side)

    def finish(self) -> None:
        if not self.on_device:
            return
        done = torch.cuda.Event()
        done.record(self.side)
        torch.cuda.current_stream().wait_event(done)
        self.full.record_stream(self.side)


# --------------------------------------------------------------------------------------------------
# VMM push (default of the gathered mode on one node; AGX_VMM_PUSH=0 disables): the exchange over peer-mapped memory, by the copy engines
# --------------------------------------------------------------------------------------------------
def _vmm_push_default() -> bool:
    """The peer-mapped exchange is the default of the GATHERED output mode wherever it can work: all ranks on one node
    (file descriptors travel over Unix sockets) and the CUDA driver bindings importable - conditions that are the same
    on every rank.  Measured at N = 4, 100 M queries (gathered mode): KNN-3 7.4 -> 5.7 ms, KNN-16 33.4 -> 22.8 ms,
    cut-off 22.2 -> 14.3 ms, bit-identical graphs (tools/dist_check.py).  AGX_VMM_PUSH=0 / 1 forces it off / on."""
    import importlib.util
    import os

    env = os.environ.get("AGX_VMM_PUSH", "auto")
    if env in ("0", "1"):
        return env == "1"
    same_node = os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")) == os.environ.get("WORLD_SIZE", "1")
    try:
        have_driver = importlib.util.find_spec("cuda.bindings.driver") is not None
    except (ImportError, ValueError):
        have_driver = False
    return same_node and have_driver


VMM_PUSH = _vmm_push_default()


class _VmmHeap:
    """One persistent staging buffer per rank, allocated with the driver's virtual-memory API (cuMemCreate), exported
    as a POSIX file descriptor, passed to every other rank of the box over Unix sockets and mapped there for access
    from THAT rank's device (cuMemMap + cuMemSetAccess).  A copy into such a mapping is a device-to-device DMA over
    NVLink: 771 GB/s per rank with both ranks of a pair pushing (tools/vmm_probe.py), against 26 GB/s through
    PyTorch's legacy CUDA-IPC tensor sharing (tools/ipc_probe.py); mapping a 1 GiB peer allocation takes 0.3 ms and
    is done once."""

    def __init__(self) -> None:
        self.size = 0
        self.own = None
        self.own_va = 0
        self.peer_va: dict[int, int] = {}
        self._peer_handles: list = []

    @staticmethod
    def _ck(res):
        from cuda.bindings import driver as cu

        if res[0] != cu.CUresult.CUDA_SUCCESS:
            raise _cabi.AgxError(f"CUDA driver call failed: {res[0]}")
        return res[1] if len(res) == 2 else None

    def _map(self, handle, size: int, device_index: int) -> int:
        from cuda.bindings import driver as cu

        va = self._ck(cu.cuMemAddressReserve(size, 0, 0, 0))
        self._ck(cu.cuMemMap(va, size, 0, handle, 0))
        acc = cu.CUmemAccessDesc()
        acc.location.type = cu.CUmemLocationType.CU_MEM_LOCATION_TYPE_DEVICE
        acc.location.id = device_index
        acc.flags = cu.CUmemAccess_flags.CU_MEM_ACCESS_FLAGS_PROT_READWRITE
        self._ck(cu.cuMemSetAccess(va, size, [acc], 1))
        return int(va)

    def ensure(self, nbytes: int, device: torch.device) -> None:
        """Collective: every rank calls it with the same ``nbytes``."""
        if nbytes <= self.size:
            return
        import os
        import socket
        import time

        import torch.distributed as dist
        from cuda.bindings import driver as cu

        rank, w = world()
        dev = device.index if device.index is not None else torch.cuda.current_device()
        torch.cuda.synchronize()
        dist.barrier()  # nobody still uses the old buffers
        fd_type = cu.CUmemAllocationHandleType.CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR
        prop = cu.CUmemAllocationProp()
        prop.type = cu.CUmemAllocationType.CU_MEM_ALLOCATION_TYPE_PINNED
        prop.location.type = cu.CUmemLocationType.CU_MEM_LOCATION_TYPE_DEVICE
        prop.location.id = dev
        prop.requestedHandleTypes = fd_type
        gran = self._ck(cu.cuMemGetAllocationGranularity(prop, cu.CUmemAllocationGranularity_flags.CU_MEM_ALLOC_GRANULARITY_MINIMUM))
        size = (int(nbytes * 1.25) + gran - 1) // gran * gran
        # (the previous, smaller buffers stay mapped until the process ends: growth is rare and they are small)
        self.own = self._ck(cu.cuMemCreate(size, prop, 0))
        self.own_va = self._map(self.own, size, dev)
        fd = int(self._ck(cu.cuMemExportToShareableHandle(self.own, fd_type, 0)))
        # every rank listens, then sends its descriptor to every other rank (SCM_RIGHTS).  The sockets live in the
        # abstract namespace under a random token that rank 0 draws and broadcasts through the process group, the
        # peer is checked with SO_PEERCRED (same user) and must name a rank nobody else has claimed
        import secrets
        import struct

        token = [secrets.token_hex(16) if rank == 0 else None]
        dist.broadcast_object_list(token, src=0)
        name = lambda r: f"\0agx_vmm_{token[0]}_{r}"  # noqa: E731
        srv = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        srv.bind(name(rank))
        srv.listen(w)
        srv.settimeout(60.0)
        dist.barrier()
        outgoing = []
        for p in range(w):
            if p == rank:
                continue
            c = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
            for attempt in range(200):
                try:
                    c.connect(name(p))
                    break
                except OSError:
                    if attempt == 199:
                        raise _cabi.AgxError(f"VMM exchange: rank {rank} cannot reach rank {p}'s descriptor socket") from None
                    time.sleep(0.01)
            socket.send_fds(c, [bytes([rank])], [fd])
            outgoing.append(c)
        self.peer_va = {}
        for _ in range(w - 1):
            conn, _addr = srv.accept()
            _pid, uid, _gid = struct.unpack("3i", conn.getsockopt(socket.SOL_SOCKET, socket.SO_PEERCRED, struct.calcsize("3i")))
            msg, fds, _flags, _a = socket.recv_fds(conn, 16, 1)
            peer = int(msg[0]) if msg else -1
            if uid != os.getuid() or not (0 <= peer < w) or peer == rank or peer in self.peer_va or len(fds) != 1:
                raise _cabi.AgxError(f"VMM exchange: unexpected peer (uid {uid}, rank byte {peer}) on rank {rank}'s socket")
            handle = self._ck(cu.cuMemImportFromShareableHandle(fds[0], fd_type))
            self._peer_handles.append(handle)
            self.peer_va[peer] = self._map(handle, size, dev)
            os.close(fds[0])
            conn.close()
        dist.barrier()
        for c in outgoing:
            c.close()
        srv.close()
        os.close(fd)
        self.size = size


_vmm_heap = _VmmHeap()


class VmmGather:
    """``ChunkedGather`` with the copy engines instead of a collective: every finished chunk of the rank's block is
    pushed into the same byte range of every peer's staging buffer (``_VmmHeap``) on a second stream while the main
    stream searches the next chunk; after one stream-ordered barrier each rank copies the other ranks' blocks from
    its own staging buffer into ``full``.  No SMs are used by the exchange, so - unlike an NCCL kernel - it runs
    while the persistent search kernels occupy the whole GPU.  Validated at N = 2 and N = 4 (bit-identical graphs)."""

    def __init__(self, full: torch.Tensor, counts: list[list[int]]) -> None:
        import torch.distributed as dist

        self.rank, self.w = world()
        self.full = full
        self.counts = counts
        self.offsets = []
        col = 0
        for r in range(self.w):
            row = []
            for c in counts[r]:
                row.append(col)
                col += c
            self.offsets.append(row)
        assert col == full.shape[1] and full.is_contiguous()
        self.row_bytes = int(full.shape[1]) * full.element_size()
        _vmm_heap.ensure(int(full.shape[0]) * self.row_bytes, full.device)
        self.side = torch.cuda.Stream(device=full.device, priority=-1)
        self._token = torch.zeros(1, dtype=torch.int32, device=full.device)
        dist.all_reduce(self._token)  # every rank has finished reading its staging buffer from the previous build
        start = torch.cuda.Event()
        start.record()
        self.side.wait_event(start)

    def mark(self):
        ready = torch.cuda.Event()
        ready.record()
        return ready

    def chunk_done(self, c: int, ready=None) -> None:
        from cuda.bindings import driver as cu

        n, o = self.counts[self.rank][c], self.offsets[self.rank][c]
        if n == 0:
            return
        if ready is None:
            ready = self.mark()
        self.side.wait_event(ready)
        es = self.full.element_size()
        for step in range(1, self.w):  # a different first peer on every rank: all links busy at once
            peer = (self.rank + step) % self.w
            for row in range(int(self.full.shape[0])):
                off = row * self.row_bytes + o * es
                _VmmHeap._ck(cu.cuMemcpyDtoDAsync(_vmm_heap.peer_va[peer] + off, self.full.data_ptr() + off, n * es, self.side.cuda_stream))

    def finish(self) -> None:
        import torch.distributed as dist
        from cuda.bindings import driver as cu

        done = torch.cuda.Event()
        done.record(self.side)
        main = torch.cuda.current_stream()
        main.wait_event(done)
        dist.all_reduce(self._token)  # stream-ordered barrier: every rank's pushes have landed
        es = self.full.element_size()
        for r in range(self.w):
            n = sum(self.counts[r])
            if r == self.rank or n == 0:
                continue
            o = self.offsets[r][0]
            for row in range(int(self.full.shape[0])):
                off = row * self.row_bytes + o * es
                _VmmHeap._ck(cu.cuMemcpyDtoDAsync(self.full.data_ptr() + off, _vmm_heap.own_va + off, n * es, main.cuda_stream))
        self.full.record_stream(self.side)


def make_gather(full: torch.Tensor, counts: list[list[int]]):
    """The exchange object of a sharded edge set: ``VmmGather`` (``VMM_PUSH``), else ``ChunkedGather``."""
    if VMM_PUSH and full.is_cuda:
        return VmmGather(full, counts)
    return ChunkedGather(full, counts)


def all_gather_count_rows(mine: list[int], device: torch.device) -> list[list[int]]:
    """Every rank's list of per-chunk counts: (W x C) nested list."""
    import torch.distributed as dist

    _, w = world()
    t = torch.tensor(mine, dtype=torch.int64, device=device)
    out = torch.empty((w, len(mine)), dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(out.view(-1), t)
    return [[int(v) for v in row] for row in out.tolist()]


def all_gather_stats_raw(stats: torch.Tensor) -> torch.Tensor:
    """Per-rank attribute statistics stacked in rank order: (W, n) float64 for the n doubles of ``stats`` (one or more
    sets of 8).  The attribute kernel folds the sets in that order (``agx_edge_attrs_apply``), so every rank applies
    bit-identical constants."""
    import torch.distributed as dist

    n = stats.numel()
    assert n % 8 == 0, "attribute statistics come in sets of 8 doubles"
    _, w = world()
    if w == 1:
        return stats.reshape(1, n)
    allst = torch.empty((w, n), dtype=stats.dtype, device=stats.device)
    dist.all_gather_into_tensor(allst, stats.reshape(1, n))
    return allst
