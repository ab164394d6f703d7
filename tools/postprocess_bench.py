#!/usr/bin/env python
"""Edge post-processors on the bench.py O1280 -> TriNodes(7) graph, device-resident, against a pure-torch composition.

    python tools/postprocess_bench.py [--workload o1280_res7] [--reps 10] [--warmup 3]

For the decoder (hidden -> data, KNN-3) and the encoder (data -> hidden, cut-off) edge sets, each processor is timed with
CUDA events after warm-up, alternating in the same process with a torch composition of the same result:
* sort:     stable ``torch.sort`` of int64 packed (key << 32 | other) keys, then ``index_select`` of every per-edge tensor;
* restrict: the float64 haversine rdist in torch, ``<= sin^2(r / 2)``, then boolean indexing of every per-edge tensor.
Both must give identical outputs.  Reported per edge set: milliseconds (median over --reps) and the bytes per edge
each path is charged (what the kernels must read and write: edge_index, attributes, keys / flags / index lists), with
the GPU name and power limit read in the same run.  One JSON line per (edge set, processor).
"""

from __future__ import annotations

import argparse
import json
import math
import pathlib
import statistics
import subprocess
import sys

REPO = pathlib.Path(__file__).resolve().parents[1]
if str(REPO) not in sys.path:
    sys.path.insert(0, str(REPO))

import torch  # noqa: E402

from bench import WORKLOADS, data_coordinates, recipe  # noqa: E402

EDGE_SETS = {"decoder": ("hidden", "to", "data"), "encoder": ("data", "to", "hidden")}


def gpu_info() -> dict:
    try:
        out = subprocess.run(
            ["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
            capture_output=True, text=True, timeout=30,
        ).stdout.strip()  # fmt: skip
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": out}


def clone_store(store) -> dict:
    return {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in store.items() if not k.startswith("_")}


def public(store) -> dict:
    return {k: v for k, v in store.items() if not k.startswith("_")}


def one_set_graph(graph, key, store_dict):
    from anemoi_graphs_b200.graph import HeteroData

    g = HeteroData()
    for name in (key[0], key[2]):
        g[name].x = graph[name].x
    for k, v in store_dict.items():
        g[key][k] = v
    return g


def torch_sort(store: dict, key_row: int, descending: bool) -> dict:
    ei = store["edge_index"]
    keys = (ei[key_row].long() << 32) | ei[1 - key_row].long()
    order = torch.sort(keys, stable=True, descending=descending).indices
    return {k: (v.index_select(-1 if k == "edge_index" else 0, order) if isinstance(v, torch.Tensor) else v) for k, v in store.items()}


def torch_restrict(store: dict, sx: torch.Tensor, tx: torch.Tensor, radius: float) -> dict:
    ei = store["edge_index"].long()
    s, t = sx.double()[ei[0]], tx.double()[ei[1]]
    sin_0 = torch.sin(0.5 * (t[:, 0] - s[:, 0]))
    sin_1 = torch.sin(0.5 * (t[:, 1] - s[:, 1]))
    rd = sin_0 * sin_0 + torch.cos(t[:, 0]) * torch.cos(s[:, 0]) * sin_1 * sin_1
    keep = rd <= math.sin(0.5 * radius) ** 2
    return {k: (v[:, keep] if k == "edge_index" else v[keep]) if isinstance(v, torch.Tensor) else v for k, v in store.items()}


def timed(fn, reps: int, warmup: int) -> tuple[float, object]:
    out = None
    for _ in range(warmup):
        out = fn()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times), out


def same(a: dict, b: dict) -> bool:
    return all(
        a[k].dtype == b[k].dtype and a[k].shape == b[k].shape and torch.equal(a[k].view(torch.uint8), b[k].view(torch.uint8))
        for k in a
        if isinstance(a[k], torch.Tensor)
    )


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="o1280_res7", choices=sorted(WORKLOADS))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--max-km", type=float, default=30.0, help="RestrictEdgeLength limit")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("postprocess_bench needs a CUDA device")

    from anemoi_graphs_b200 import EARTH_RADIUS
    from anemoi_graphs_b200 import device as agx_device
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.graph import HeteroData
    from anemoi_graphs_b200.processors import RestrictEdgeLength, SortEdgeIndexByTargetNodes

    grid, res = WORKLOADS[args.workload]
    agx_device.set_resident(True)
    graph = HeteroData()
    graph["data"].x = data_coordinates(grid).cuda()
    graph["data"].node_type = "LatLonNodes"
    graph = GraphCreator(recipe(res)).update_graph(graph)
    torch.cuda.synchronize()
    info = gpu_info()

    for set_name, key in EDGE_SETS.items():
        base = clone_store(graph[key])
        e = int(base["edge_index"].shape[1])
        attr_bytes = sum(v.element_size() * v.numel() // max(e, 1) for k, v in base.items() if isinstance(v, torch.Tensor) and k != "edge_index")
        ei_bytes = 2 * base["edge_index"].element_size()
        row_bytes = ei_bytes + attr_bytes  # one edge's edge_index column + attributes, read once and written once

        # sort by target, descending (the processor's default)
        def ours_sort():
            return public(SortEdgeIndexByTargetNodes().update_graph(one_set_graph(graph, key, dict(base)))[key])

        ms_ours, out_ours = timed(ours_sort, args.reps, args.warmup)
        ms_torch, out_torch = timed(lambda: torch_sort(base, 1, True), args.reps, args.warmup)
        assert same(out_ours, out_torch), f"{set_name}: sort outputs differ"
        # ours: rows read (8) + keys written / read by the radix passes + permutation + gather of every array
        print(json.dumps({
            "set": set_name, "op": "SortEdgeIndexByTargetNodes", "edges": e, "ms_cuda": round(ms_ours, 3),
            "ms_torch": round(ms_torch, 3), "bytes_per_edge_moved": 2 * row_bytes, **info,
        }), flush=True)  # fmt: skip

        radius = args.max_km / EARTH_RADIUS
        sx, tx = graph[key[0]].x, graph[key[2]].x

        def ours_restrict():
            return public(RestrictEdgeLength(key[0], key[2], args.max_km).update_graph(one_set_graph(graph, key, dict(base)))[key])

        ms_ours, out_ours = timed(ours_restrict, args.reps, args.warmup)
        ms_torch, out_torch = timed(lambda: torch_restrict(base, sx, tx, radius), args.reps, args.warmup)
        assert same(out_ours, out_torch), f"{set_name}: restrict outputs differ"
        kept = int(out_ours["edge_index"].shape[1])
        # ours: edge_index (8) + 2 x 8 coordinates + 1 flag byte + 4 index bytes per kept edge + gather of kept rows
        print(json.dumps({
            "set": set_name, "op": "RestrictEdgeLength", "max_km": args.max_km, "edges": e, "kept": kept,
            "ms_cuda": round(ms_ours, 3), "ms_torch": round(ms_torch, 3),
            "bytes_per_edge_moved": round(ei_bytes + 16 + 1 + (kept / max(e, 1)) * (4 + 2 * row_bytes), 2), **info,
        }), flush=True)  # fmt: skip


if __name__ == "__main__":
    main()
