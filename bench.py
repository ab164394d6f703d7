#!/usr/bin/env python
"""Headline benchmark: O1280 -> TriNodes(7) encoder / processor / decoder graph, edges per second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

One STEP = one complete pass of the edge-construction path over the workload: hidden TriNodes generation
(icosphere subdivision kernels + the host node ordering the reference defines), CutOffEdges 0.6 encoder
(data -> hidden), MultiScaleEdges x_hops=1 processor, KNNEdges k=3 decoder (hidden -> data), EdgeLength +
EdgeDirection (unit-std) on all three edge sets - through the reference-facing builder API
(``GraphCreator.update_graph``), i.e. the recipe ``anemoi-graphs create`` would run.  Data-node coordinates are
synthetic (octahedral reduced Gaussian grid, ``anemoi_graphs_b200.grids``) and are an INPUT of the step.

* ``value``: edges/s with the data coordinates already resident in HBM and every output left in HBM
  (CUDA events around exactly K steps; max over ranks).
* ``e2e``: the same step with HOST buffers - coordinates in pinned host memory are uploaded and all
  ``edge_index`` / attribute tensors are copied back to pinned host memory inside the timed region.
* ``roofline``: the dominant kernel, timed live with CUDA events on its launch stream during the timed steps.
* ``cpu_baseline``: the oracle port (``oracle/ref_path.py``: the reference's own sklearn / scipy / networkx calls)
  timed on this host's cores on a bounded sample of the same workload, with its error against a full pass stated.
* ``--impl reference``: ONE full, unsampled pass of the UNMODIFIED reference (``oracle/_ref``, vendored byte for byte by
  ``oracle/build_ref.py``) through its own ``GraphCreator.update_graph`` on the box's host cores.
* ``--dump-outputs DIR``: what the last timed ``value`` step returned, as ``DIR/<name>.npy`` (``dump_outputs``), so two
  builds of the project can be compared output for output on identical inputs.

Multi-GPU (torchrun, one rank per GPU): sharded OUTPUT mode - query (target) nodes are sharded by rank, reference nodes
replicated, nothing is exchanged between the GPUs except the attribute statistics (8 doubles per rank).  ``value``
leaves every rank's block in its own HBM; ``e2e`` has every rank copy its block over its own PCIe link into ONE shared
page-locked host buffer, so the host ends with the complete graph.  Total work is fixed => "scaling": "strong".
"""

from __future__ import annotations

import argparse
import json
import os
import pathlib
import statistics
import subprocess
import sys
import threading
import time

REPO = pathlib.Path(__file__).resolve().parent
if str(REPO) not in sys.path:
    sys.path.insert(0, str(REPO))

import numpy as np  # noqa: E402
import torch  # noqa: E402

T = "anemoi.graphs."
METRIC = "O1280->ico7 graph edges/sec (CutOff encoder + MultiScale processor + KNN-3 decoder + EdgeLength/EdgeDirection)"
WORKLOADS = {
    # name: (data grid, hidden TriNodes resolution)
    "o1280_res7": ("o1280", 7),
    "n320_res6": ("n320", 6),
    "o96_res5": ("o96", 5),
}
CUTOFF_FACTOR = 0.6
KNN_K = 3
X_HOPS = 1
NORM = "unit-std"
# algorithmic HBM bytes per output unit, SURVEY.md section 8(d) / DESIGN.md
ALGO_BYTES = {
    "knn": lambda nq, nr, e: 8.0 * nq + 8.0 * nr + 8.0 * e,
    "radius_fill": lambda nq, nr, e: 8.0 * nq + 8.0 * nr + 8.0 * e,
    "edge_attrs": lambda nq, nr, e: 20.0 * e,
}


def attrs_cfg():
    return {
        "edge_length": {"_target_": T + "edges.attributes.EdgeLength", "norm": NORM},
        "edge_dirs": {"_target_": T + "edges.attributes.EdgeDirection", "norm": NORM},
    }


def recipe(resolution: int) -> dict:
    return {
        "nodes": {"hidden": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": resolution}}},
        "edges": [
            {"source_name": "data", "target_name": "hidden", "attributes": attrs_cfg(),
             "edge_builders": [{"_target_": T + "edges.CutOffEdges", "cutoff_factor": CUTOFF_FACTOR}]},
            {"source_name": "hidden", "target_name": "hidden", "attributes": attrs_cfg(),
             "edge_builders": [{"_target_": T + "edges.MultiScaleEdges", "x_hops": X_HOPS}]},
            {"source_name": "hidden", "target_name": "data", "attributes": attrs_cfg(),
             "edge_builders": [{"_target_": T + "edges.KNNEdges", "num_nearest_neighbours": KNN_K}]},
        ],
    }  # fmt: skip


EDGE_KEYS = [("data", "to", "hidden"), ("hidden", "to", "hidden"), ("hidden", "to", "data")]


def data_coordinates(grid: str) -> torch.Tensor:
    from anemoi_graphs_b200 import grids

    lat, lon = grids.named_grid(grid)
    return grids.latlon_deg_to_x(lat, lon)


# ----------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = (
        "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
        "clocks_event_reasons.sw_power_cap"
    )

    def __init__(self, gpu_index: int) -> None:
        self.gpu_index = gpu_index
        self.lines: list[str] = []
        self.proc = None

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.gpu_index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )  # fmt: skip
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self) -> None:
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            f = [c.strip() for c in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(smax) if smax else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


# ----------------------------------------------------------------------------------------------------
# the GPU arm
# ----------------------------------------------------------------------------------------------------
def run_step(creator, data_x: torch.Tensor):
    from anemoi_graphs_b200.graph import HeteroData

    graph = HeteroData()
    graph["data"].x = data_x
    graph["data"].node_type = "LatLonNodes"
    return creator.update_graph(graph)


def edge_set_sizes(graph) -> dict:
    """GLOBAL number of edges of every edge set (a device-resident sharded graph holds one rank's block and says so in
    ``edge_shard``)."""
    sizes = {}
    for k in EDGE_KEYS:
        info = graph[k].get("edge_shard", None)
        if info is None:
            sizes[k] = int(graph[k].edge_index.shape[1])
        else:
            sizes[k] = int(info["counts"][0] if info["replicated"] else sum(info["counts"]))
    return sizes


def output_bytes(graph) -> int:
    n = 0
    for k in EDGE_KEYS:
        for name in ("edge_index", "edge_length", "edge_dirs"):
            t = graph[k][name]
            n += t.numel() * t.element_size()
    return n


DUMP_EDGES_PER_SET = 1 << 19  # 28 bytes per dumped edge: the three edge sets stay below 64 MB together
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(graph, out_dir: pathlib.Path) -> None:
    """Write the graph one step returned as ``out_dir/<name>.npy``: the hidden node coordinates and, for every edge set,
    ``<src>_to_<dst>_edge_index`` (float64, exact for int32 ids), ``_edge_length`` and ``_edge_dirs`` (float32).  Edges
    are in canonical (target, source) order, so the files do not depend on the order the kernels emit an edge set in; a
    set larger than ``DUMP_EDGES_PER_SET`` is sampled at fixed seeded positions of that order."""
    arrays = {"hidden_x": graph["hidden"].x.cpu().numpy()}
    for key in EDGE_KEYS:
        store = graph[key]
        ei = store.edge_index
        order = torch.argsort(ei[1].long() * graph[key[0]].x.shape[0] + ei[0].long())
        n = int(order.numel())
        if n > DUMP_EDGES_PER_SET:
            pick = np.sort(np.random.default_rng(0).choice(n, size=DUMP_EDGES_PER_SET, replace=False))
            order = order[torch.from_numpy(pick).to(order.device)]
        name = f"{key[0]}_to_{key[2]}"
        arrays[f"{name}_edge_index"] = ei[:, order].cpu().numpy().astype(np.float64)
        arrays[f"{name}_edge_length"] = store["edge_length"][order].cpu().numpy()
        arrays[f"{name}_edge_dirs"] = store["edge_dirs"][order].cpu().numpy()
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a)


def sharding_note(world: int) -> str:
    if world == 1:
        return "single GPU"
    return (
        f"sharded output over {world} ranks: cut-off and KNN searches and their attributes by query (target) node, "
        "reference nodes replicated, multi-scale edges and node generation replicated (SURVEY 8e); one rank sorts the "
        "hidden nodes, the order reaches the others through shared host memory; no edge data crosses NVLink: `value` "
        "leaves every rank's block in its HBM, `e2e` has every rank copy its block over its own PCIe link into one "
        "shared page-locked host buffer (the complete graph on the host); attribute statistics are all-gathered (8 "
        "doubles per rank, NCCL)"
    )


def knn_probe(x_dev: torch.Tensor, res: int, lo: int, hi: int) -> dict:
    """Counters of the dominant kernel on this rank's queries (one extra launch outside the timed region): (query, candidate)
    pairs of the staged scans (`stats[3]`), float64 re-decisions, ties."""
    from anemoi_graphs_b200 import ops

    ico = ops.Icosphere(res, x_dev.device)
    stats = ops.new_stats(x_dev.device)
    with ops.NeighbourIndex(ico.latlon, hint_k=KNN_K) as index:
        index.knn(x_dev[lo:hi], KNN_K, stats=stats, tag="knn_probe")
    torch.cuda.synchronize()
    st = [int(v) for v in stats.cpu().tolist()]
    return {"refined_f64": st[0], "tied": st[1], "widened": st[2], "pairs": st[3]}


def bench_b200(args) -> dict:
    import torch.distributed as dist

    from anemoi_graphs_b200 import _cabi, ops
    from anemoi_graphs_b200 import device as agx_device
    from anemoi_graphs_b200.create import GraphCreator

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs a single process: a sharded device-resident graph holds one rank's block")
    torch.cuda.set_device(local_rank)
    shared_host = True
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        agx_device.set_sharded_output(True)
        from anemoi_graphs_b200 import shm

        if shm.local_group() is None:  # ranks on several nodes, or a /dev/shm too small for the result buffers
            shared_host = False
            agx_device.set_sharded_output(False)
    if world != args.gpus and rank == 0:
        print(f"note: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)

    grid, res = WORKLOADS[args.workload]
    x_host = data_coordinates(grid).pin_memory()
    x_dev = x_host.cuda()
    creator = GraphCreator(recipe(res))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        """CUDA-event time of `steps` calls, max over ranks (ms)."""
        barrier()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        out = None
        for _ in range(steps):
            out = None  # drop the previous step's graph first: one live output set, as in the warm-up
            out = fn()
        end.record()
        torch.cuda.synchronize()
        ms = start.elapsed_time(end)
        if world > 1:
            mine = torch.tensor([ms], dtype=torch.float64, device="cuda")
            every = torch.empty(world, dtype=torch.float64, device="cuda")
            dist.all_gather_into_tensor(every, mine)
            by_rank.append([round(float(v) / steps, 4) for v in every.tolist()])
            ms = float(every.max().item())
        barrier()
        return ms, out

    by_rank: list = []  # per timed region: ms per step of every rank (the reported time is the maximum)

    # ---- device-resident: `value` -------------------------------------------------------------------
    agx_device.set_resident(True)
    graph = None
    for _ in range(args.warmup):
        graph = None
        graph = run_step(creator, x_dev)
    sizes = edge_set_sizes(graph)
    n_edges = sum(sizes.values())
    graph = None
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ops.timeline = ops.Timeline()
    launches0 = _cabi.launch_count()
    ms_total, graph = timed(lambda: run_step(creator, x_dev), args.steps)
    launches = _cabi.launch_count() - launches0
    spans = ops.timeline.totals_ms()
    span_counts = ops.timeline.counts()
    ops.timeline = None
    clock_info = clocks.stop() if rank == 0 else {}
    ms_per_step = ms_total / args.steps
    value = n_edges / (ms_per_step * 1e-3)
    n_data, n_hidden = int(x_dev.shape[0]), int(graph["hidden"].x.shape[0])
    if args.dump_outputs:
        dump_outputs(graph, pathlib.Path(args.dump_outputs))
    del graph
    if world > 1:
        t = torch.tensor([launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(t)
        launches = int(t.item())

    # ---- end to end with host buffers: `e2e` ---------------------------------------------------------
    agx_device.set_resident(False)
    for _ in range(args.warmup):
        graph = None
        graph = run_step(creator, x_host)
    d2h = output_bytes(graph)  # the complete host graph (at N > 1: each byte written once, by the rank that owns it)
    assert sum(int(graph[k].edge_index.shape[1]) for k in EDGE_KEYS) == n_edges
    graph = None
    e2e_steps = max(1, args.steps)
    ms_e2e, graph = timed(lambda: run_step(creator, x_host), e2e_steps)
    e2e_value = n_edges / (ms_e2e / e2e_steps * 1e-3)
    del graph

    # ---- roofline of the dominant kernel ---------------------------------------------------------------
    # spans: one per C-ABI call, timed with CUDA events on the launch stream during the timed steps (rank 0's).  "knn"
    # is the decoder's k_knn<4> launch alone: THIS RANK's queries (all of them on one GPU, 1/W in sharded mode).
    per_step = {k: spans[k] / args.steps for k in spans}
    per_call = {k: spans[k] / span_counts[k] for k in spans}
    lo, hi = agx_device.shard_range(n_data, rank, world)
    nq_knn, e_knn = hi - lo, (hi - lo) * KNN_K
    kern = "knn"
    algo_bytes = ALGO_BYTES["knn"](nq_knn, n_hidden, e_knn)
    achieved = algo_bytes / (per_call[kern] * 1e-3) / 1e9
    peaks = {}
    peaks_path = REPO / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peaks = json.loads(peaks_path.read_text())
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    traffic = None
    tpath = REPO / "profiles" / "traffic.json"
    if tpath.exists() and world == 1:
        traffic = json.loads(tpath.read_text()).get("k_knn")
    # FP32 FMA-pipe view of the same launch: every staged candidate is tested against all queries of its (half-)tile;
    # 8 flop per (query, candidate) pair (3 sub, 1 mul, 2 fma).  Peak = SMs x 128 lanes x 2 x clock.
    probe = knn_probe(x_dev, res, lo, hi)
    props = torch.cuda.get_device_properties(local_rank)
    sm_mhz = float(clock_info.get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)) if rank == 0 else 1965.0
    fp32_peak = props.multi_processor_count * 128 * 2 * sm_mhz * 1e6 / 1e12
    pairs = probe["pairs"]
    fp32_achieved = pairs * 8 / (per_call[kern] * 1e-3) / 1e12
    roofline = {
        "kernel": "k_knn<4> (KNNEdges decoder, one launch per step" + (f", this rank's 1/{world} of the queries)" if world > 1 else ")"),
        "bound": "hbm",
        "achieved": round(achieved, 2),
        "peak": peak,
        "peak_source": peak_src,
        "unit": "GB/s",
        "frac": round(achieved / peak, 5),
        "traffic": traffic,
        "algorithmic_bytes_per_launch": algo_bytes,
        "ms_per_launch": round(per_call[kern], 4),
        "fp32": {
            "pairs_evaluated": pairs,
            "pairs_per_query": round(pairs / max(nq_knn, 1), 2),
            "flop_per_pair": 8,
            "achieved_tflops": round(fp32_achieved, 3),
            "peak_tflops": round(fp32_peak, 2),
            "peak_source": f"{props.multi_processor_count} SMs x 128 FP32 lanes x 2 x {sm_mhz:.0f} MHz (clock sampled under load)",
            "frac": round(fp32_achieved / fp32_peak, 5),
            "counters": probe,
        },
        "note": "issue-bound (d = 3 distance tests against every staged candidate), neither HBM- nor FMA-bound: see profiles/",
        "stage_ms_per_step": {k: round(v, 4) for k, v in sorted(per_step.items(), key=lambda kv: -kv[1])},
        "stage_launch_groups_per_step": {k: span_counts[k] // args.steps for k in span_counts},
    }

    line = {
        "metric": METRIC,
        "value": round(value, 1),
        "unit": "edges/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": round(ms_per_step, 4),
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f32 filter + f64 decisions, int32 indices",
        "data": "synthetic",
        "config": workload_config(args.workload, n_data, n_hidden, sizes),
        "sharding": sharding_note(world) if shared_host else (
            f"{world} ranks, GATHERED output (every rank ends with the complete graph): no node-wide shared memory available "
            "for the sharded host output (ranks on several nodes, or /dev/shm below AGX_MIN_SHM_FREE_BYTES)"
        ),
        "e2e": {
            "value": round(e2e_value, 1),
            "unit": "edges/s",
            "ms_per_step": round(ms_e2e / e2e_steps, 4),
            "steps": e2e_steps,
            "h2d_bytes_per_step": int(x_host.numel() * 4) * world,  # every rank uploads the (replicated) data coordinates
            "d2h_bytes_per_step": int(d2h),
        },
        "gpu_launches": int(launches),
        "ms_per_step_by_rank": {"value": by_rank[0], "e2e": by_rank[1]} if by_rank else None,
        "roofline": roofline,
        "clocks": clock_info,
    }  # fmt: skip
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_reference(args.workload, n_jobs=4, budget_s=args.cpu_budget)
        line["cpu_baseline"].update(sample_error_note(args.workload, line["cpu_baseline"]))
    if world > 1:
        dist.destroy_process_group()
    return line if rank == 0 else {}


# ----------------------------------------------------------------------------------------------------
# the CPU reference arm (oracle = the reference's own sklearn / scipy / networkx calls)
# ----------------------------------------------------------------------------------------------------
def cpu_reference(workload: str, n_jobs: int, budget_s: float = 20.0, x=None) -> dict:
    """Time the reference path on this host on a bounded sample of the workload and extrapolate to the full
    graph: fixed costs (ball-tree fits, reference distance) are paid in full, per-query / per-edge costs are
    measured on a fraction f of the queries and scaled by 1/f."""
    from oracle import ref_path as R

    grid, res = WORKLOADS[workload]
    dx = (data_coordinates(grid) if x is None else x).numpy()
    t_all = time.perf_counter()
    hx, order = R.tri_nodes(res)
    t_nodes = time.perf_counter() - t_all
    nd, nh = dx.shape[0], hx.shape[0]
    # query fractions sized from the survey's rates (~3e4 KNN queries/s on 4 threads)
    f = min(1.0, max(1.0 / 256, budget_s * 0.3 * 3.0e4 / nd))
    rng = np.random.default_rng(0)
    qd = np.sort(rng.choice(nd, size=max(1, int(nd * f)), replace=False))
    qh = np.sort(rng.choice(nh, size=max(1, int(nh * f)), replace=False))

    from sklearn.neighbors import NearestNeighbors

    t = time.perf_counter()
    radius = R.cutoff_radius(hx, CUTOFF_FACTOR, n_jobs)  # k=2 self query on the hidden nodes (fixed cost)
    t_refdist = time.perf_counter() - t
    t = time.perf_counter()
    nn = NearestNeighbors(metric="haversine", n_jobs=n_jobs).fit(dx)
    t_fit_data = time.perf_counter() - t
    t = time.perf_counter()
    adj = nn.radius_neighbors_graph(hx[qh], radius=radius).tocoo()
    cut = np.stack([adj.col, qh[adj.row]]).astype(np.int32)
    t_cut = time.perf_counter() - t
    del nn
    t = time.perf_counter()
    nn = NearestNeighbors(metric="haversine", n_jobs=n_jobs).fit(hx)
    t_fit_hidden = time.perf_counter() - t
    t = time.perf_counter()
    adj = nn.kneighbors_graph(dx[qd], n_neighbors=KNN_K, mode="distance").tocoo()
    knn = np.stack([adj.col, qd[adj.row]]).astype(np.int32)
    t_knn = time.perf_counter() - t
    # multi-scale: the reference's networkx path on a coarser mesh (cost is linear in the vertex count)
    ms_res = min(res, 5)
    mx, morder = R.tri_nodes(ms_res)
    t = time.perf_counter()
    ms = R.multiscale_edges_tri_networkx(range(ms_res + 1), X_HOPS, morder, mx)
    t_ms = time.perf_counter() - t
    ms_full_edges = sum(60 * 4**r for r in range(res + 1))
    t_ms_full = t_ms * ms_full_edges / ms.shape[1]
    # attributes on the sampled edges
    t = time.perf_counter()
    with np.errstate(all="ignore"):
        for sx, tx, ei in ((dx, hx, cut), (hx, dx, knn)):
            R.edge_length(sx, tx, ei, NORM)
            R.edge_direction(sx, tx, ei, NORM)
    t_attr = time.perf_counter() - t
    attr_rate = (cut.shape[1] + knn.shape[1]) / t_attr
    e_cut, e_knn = cut.shape[1] / f, knn.shape[1] / f
    e_total = e_cut + e_knn + ms_full_edges
    t_full = t_nodes + t_refdist + t_fit_data + t_fit_hidden + t_cut / f + t_knn / f + t_ms_full + e_total / attr_rate
    return {
        "value": round(e_total / t_full, 1),
        "unit": "edges/s",
        "cores": n_jobs if n_jobs > 0 else os.cpu_count(),
        "host_cpus": os.cpu_count(),
        "kind": "port",
        "sample": (
            f"oracle/ref_path.py (the reference's sklearn BallTree / scipy / networkx calls) on {workload}: full tree "
            f"fits + reference distance, a random {f:.4f} of the KNN and cut-off queries, MultiScale via networkx at "
            f"res {ms_res}, attributes on the sampled edges; per-query/per-edge times scaled to the full graph "
            f"({int(e_total)} edges, est. {t_full:.1f} s)"
        ),
        "measured_s": round(time.perf_counter() - t_all, 2),
        "stage_s": {
            "tri_nodes": round(t_nodes, 3), "ref_distance": round(t_refdist, 3), "fit_data_tree": round(t_fit_data, 3),
            "fit_hidden_tree": round(t_fit_hidden, 3), "cutoff_query_sample": round(t_cut, 3),
            "knn_query_sample": round(t_knn, 3), "multiscale_sample": round(t_ms, 3), "attrs_sample": round(t_attr, 3),
        },
        "estimated_full_graph_s": round(t_full, 2),
    }  # fmt: skip


def sample_error_note(workload: str, sampled: dict) -> dict:
    """How far the sampled-and-scaled ``cpu_baseline`` estimate is from a FULL pass of the unmodified reference: against
    the ``--impl reference`` run of this box when it left its result (the driver runs it first), else against the
    full pass committed under profiles/ (another box: the error then includes the host difference)."""
    full, where = None, None
    try:
        cand = json.loads(REFERENCE_RESULT.read_text())
        if cand.get("workload") == workload:
            full, where = cand, "this box (--impl reference, run before this arm)"
    except (OSError, ValueError):
        pass
    if full is None:
        path = REPO / "profiles" / "r02_reference_full_pass.json"
        if path.exists():
            cand = json.loads(path.read_text())
            if cand.get("config", {}).get("workload") == workload:
                full = {"wall_s": cand["ms_per_step"] / 1e3, "value": cand["value"]}
                where = "profiles/r02_reference_full_pass.json (a B200 box of the same pool, earlier run)"
    if full is None:
        return {"full_pass": None}
    est = sampled["estimated_full_graph_s"]
    return {
        "full_pass": {"wall_s": round(full["wall_s"], 2), "value": round(full["value"], 1), "kind": "reference-unmodified",
                      "from": where},
        "sample_error": round(est / full["wall_s"] - 1.0, 4),
        "sample_error_note": "estimated_full_graph_s / full-pass wall_s - 1 (negative: the sample under-estimates the reference's time)",
    }  # fmt: skip


def reference_full_pass(workload: str, x=None) -> dict:
    """ONE unsampled pass of the UNMODIFIED reference (``oracle/_ref``, vendored byte for byte by
    ``oracle/build_ref.py`` and verified against ``oracle/ref_manifest.json``) over the workload: its own
    ``GraphCreator.update_graph`` (create.py:62-92) on the same recipe and the same data coordinates as the GPU
    arm, behind the import shims of ``oracle/shims`` (torch_geometric / hydra / anemoi.utils stand-ins, trimesh's
    icosphere restated).  sklearn runs with the reference's hard-coded ``n_jobs=4`` (edges/builder.py:259,364).
    Stage times come from ``perf_counter`` wrappers around the reference's own methods (no code path changes)."""
    import importlib.util
    import logging
    import warnings

    spec = importlib.util.spec_from_file_location("_agx_build_ref", REPO / "oracle" / "build_ref.py")
    build_ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(build_ref)
    ref_root = build_ref.build()  # copies when /root/reference is here, else verifies the vendored tree
    n_files = len(build_ref.check())
    sys.path[:0] = [str(REPO / "oracle" / "shims"), str(ref_root.parent)]
    from anemoi.graphs import create as ref_create  # the reference's module
    from anemoi.graphs.edges import builder as ref_builder
    from anemoi.graphs.nodes.builders import base as ref_nodes_base
    from anemoi.utils.config import DotDict
    from torch_geometric.data import HeteroData as RefHeteroData

    assert pathlib.Path(ref_create.__file__).resolve().is_relative_to(ref_root.resolve()), ref_create.__file__
    logging.getLogger("anemoi").setLevel(logging.WARNING)
    grid, res = WORKLOADS[workload]
    dx = data_coordinates(grid) if x is None else x

    stage_s: dict[str, float] = {}

    def timed_method(cls, name, label):
        inner = getattr(cls, name)

        def wrapper(self, *a, **kw):
            t = time.perf_counter()
            try:
                return inner(self, *a, **kw)
            finally:
                key = label(self)
                stage_s[key] = stage_s.get(key, 0.0) + time.perf_counter() - t

        setattr(cls, name, wrapper)
        return inner

    saved = [
        (ref_builder.BaseEdgeBuilder, "register_edges",
         timed_method(ref_builder.BaseEdgeBuilder, "register_edges", lambda b: f"{type(b).__name__}.register_edges")),
        (ref_builder.BaseEdgeBuilder, "register_attributes",
         timed_method(ref_builder.BaseEdgeBuilder, "register_attributes", lambda b: f"{type(b).__name__}.register_attributes")),
        (ref_nodes_base.BaseNodeBuilder, "update_graph",
         timed_method(ref_nodes_base.BaseNodeBuilder, "update_graph", lambda b: f"{type(b).__name__}.update_graph")),
    ]  # fmt: skip
    try:
        graph = RefHeteroData()
        graph["data"].x = dx
        graph["data"].node_type = "LatLonNodes"
        creator = ref_create.GraphCreator(DotDict(recipe(res)))
        t0 = time.perf_counter()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            graph = creator.update_graph(graph)
        wall = time.perf_counter() - t0
    finally:
        for cls, name, inner in saved:
            setattr(cls, name, inner)
    sizes = {k: int(graph[k].edge_index.shape[1]) for k in EDGE_KEYS}
    for k in EDGE_KEYS:
        assert graph[k]["edge_length"].shape == (sizes[k], 1) and graph[k]["edge_dirs"].shape == (sizes[k], 2)
    return {
        "wall_s": wall,
        "edges": sizes,
        "n_data": int(dx.shape[0]),
        "n_hidden": int(graph["hidden"].x.shape[0]),
        "stage_s": {k: round(v, 3) for k, v in stage_s.items()},
        "ref_files_verified": n_files,
    }


def workload_config(workload: str, n_data: int, n_hidden: int, sizes: dict) -> dict:
    """The ``config`` object both arms print (identical keys and values for the same workload)."""
    return {
        "workload": workload,
        "data_nodes": n_data,
        "hidden_nodes": n_hidden,
        "edges": {"cutoff": sizes[EDGE_KEYS[0]], "multiscale": sizes[EDGE_KEYS[1]], "knn": sizes[EDGE_KEYS[2]]},
        "cutoff_factor": CUTOFF_FACTOR, "knn_k": KNN_K, "x_hops": X_HOPS, "attribute_norm": NORM,
        "l2": "inputs + outputs (~0.7 GB per step) exceed the 126 MB L2; no explicit flush",
    }  # fmt: skip


REFERENCE_RESULT = pathlib.Path(os.environ.get("AGX_REFERENCE_RESULT", "/tmp/agx_reference_full_pass.json"))


def bench_reference(args) -> dict:
    """``--impl reference``: the reference's own CPU implementation, timed on this box's host cores.

    ONE full, unsampled pass of the unmodified reference per run (a pass takes minutes, so ``--steps`` /
    ``--warmup`` are not repeated: the line says ``steps: 1, warmup: 0`` and echoes what was requested);
    ``value`` = edges of that pass / its wall time, ``ms_per_step`` = the same wall time."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return {}
    res = reference_full_pass(args.workload)
    n_edges = sum(res["edges"].values())
    value = n_edges / res["wall_s"]
    cpu = {
        "value": round(value, 1),
        "unit": "edges/s",
        "cores": 4,
        "host_cpus": os.cpu_count(),
        "kind": "reference-unmodified",
        "sample": (
            f"the whole {args.workload} workload, unsampled: oracle/_ref (the reference's sources, {res['ref_files_verified']} "
            "files verified against oracle/ref_manifest.json) GraphCreator.update_graph over oracle/shims, one pass, "
            "sklearn n_jobs=4 as the reference hard-codes, everything else single-threaded numpy / scipy / networkx"
        ),
        "wall_s": round(res["wall_s"], 2),
        "stage_s": res["stage_s"],
    }
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": round(value, 1),
        "unit": "edges/s",
        "n_gpus": args.gpus,
        "steps": 1,
        "warmup": 0,
        "steps_requested": args.steps,
        "warmup_requested": args.warmup,
        "ms_per_step": round(res["wall_s"] * 1e3, 1),
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f64 (sklearn BallTree haversine), f32/f64 numpy attributes",
        "data": "synthetic",
        "config": workload_config(args.workload, res["n_data"], res["n_hidden"], res["edges"]),
        "sharding": "CPU only: the reference has no GPU or multi-process path (rank 0 runs it, other ranks exit)",
        "cpu_baseline": cpu,
        "e2e": {"value": round(value, 1), "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    try:  # left for the GPU arm's cpu_baseline (same box, run right after): the error of its sampled estimate
        REFERENCE_RESULT.write_text(json.dumps({"workload": args.workload, "wall_s": res["wall_s"], "edges": n_edges,
                                                "value": value, "stage_s": res["stage_s"], "host_cpus": os.cpu_count()}))  # fmt: skip
    except OSError:
        pass
    return line


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="o1280_res7", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=20.0, help="seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's graph as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the b200 arm's outputs")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    line = bench_reference(args) if args.impl == "reference" else bench_b200(args)
    if line:
        print(json.dumps(line))


if __name__ == "__main__":
    main()
