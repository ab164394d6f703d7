"""Device time of ``CutOffEdges(max_num_neighbours=M)`` on the O1280 encoders, beside a host reference.

    python tools/cutoff_cap_bench.py [--reps 10] [--host] [--out results.json]

Workloads: O1280 -> TriNodes(6) and O1280 -> TriNodes(7), cutoff_factor 0.6, M in {None, 64, 16}.  The device time is
the builder's ``compute_edge_index`` between CUDA events, after a warm-up, median of ``--reps``.  The host reference is
sklearn's ``radius_neighbors`` plus a per-row ``argpartition`` (one run, on the node sets as float64).  The card's name
and power limit are read in the same run."""

from __future__ import annotations

import argparse
import json
import pathlib
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))

from anemoi_graphs_b200 import grids  # noqa: E402
from anemoi_graphs_b200.edges import CutOffEdges  # noqa: E402
from anemoi_graphs_b200.graph import HeteroData  # noqa: E402
from oracle import ref_path as R  # noqa: E402


def card() -> dict:
    q = "name,power.limit"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    name, limit = (out.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return {"gpu": name, "power_limit": limit}


def host_reference(dx: np.ndarray, hx: np.ndarray, radius: float, M: int | None) -> tuple[float, int]:
    from sklearn.neighbors import BallTree

    t = time.perf_counter()
    dist, ind = BallTree(dx.astype(np.float64), metric="haversine").query_radius(hx.astype(np.float64), radius,
                                                                               return_distance=True)  # fmt: skip
    n = 0
    for d, i in zip(dist, ind):
        if M is not None and d.size > M:
            i = i[np.argpartition(d, M - 1)[:M]]
        n += i.size
    return time.perf_counter() - t, n


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--host", action="store_true", help="also time the host reference")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    rows = []
    dx = grids.latlon_deg_to_x(*grids.octahedral_grid(1280))
    for res in (6, 7):
        hx = torch.from_numpy(np.ascontiguousarray(R.tri_nodes(res)[0], dtype=np.float32))
        g = HeteroData()
        g["data"].x, g["hidden"].x = dx.cuda(), hx.cuda()
        for M in (None, 64, 16):
            b = CutOffEdges("data", "hidden", 0.6, max_num_neighbours=M)
            src, dst = b.prepare_node_data(g)
            for _ in range(2):
                b.compute_edge_index(src, dst)
            torch.cuda.synchronize()
            times = []
            for _ in range(args.reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ei = b.compute_edge_index(src, dst)
                e1.record()
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1))
            row = {"encoder": f"O1280->TriNodes({res})", "M": M, "edges": int(ei.shape[1]),
                   "device_ms": float(np.median(times)), "device_ms_min": float(np.min(times))}  # fmt: skip
            if args.host:
                secs, n = host_reference(dx.numpy(), hx.numpy(), b.radius, M)
                assert n == row["edges"], (n, row["edges"])
                row["host_s"] = secs
            rows.append(row)
            print(json.dumps(row), flush=True)
    result = {**card(), "rows": rows}
    print(json.dumps(result))
    if args.out:
        pathlib.Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(args.out).write_text(json.dumps(result, indent=1))
    return 0


if __name__ == "__main__":
    sys.exit(main())
