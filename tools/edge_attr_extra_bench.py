#!/usr/bin/env python
"""Edge attributes of newer releases on the bench.py O1280 -> TriNodes(7) decoder, device-resident, against a pure-torch
composition.

    python tools/edge_attr_extra_bench.py [--workload o1280_res7] [--reps 10] [--warmup 3]

On the decoder edge set (hidden -> data, KNN-3) each attribute is timed through its ``compute(graph, edges_name)`` with
CUDA events after warm-up, alternating in the same process with a torch composition of the same quantity:
* Azimuth:                 float64 gathers of both endpoints' coordinates and the bearing formula, cast to float32;
* GaussianDistanceWeights: float64 haversine, ``exp``, group sums by ``scatter_reduce`` and the division (l1);
* AttributeFrom*Node:      ``mask[edge_index[row]]`` of a bool node attribute.
Outputs are compared: the copies must be equal, the azimuth within 1e-5 (modulo 2 pi).  The weights are checked against
the same torch composition fed with the EdgeLength values the attribute is defined on (1e-6); the float64 haversine of
the timed composition differs from EdgeLength's float32 arithmetic (the reference's) by up to ~1e-5 relative on edges
across the date line near the poles, and the largest such difference is reported.  Reported per attribute: milliseconds (median over --reps), the bytes per edge the result needs at
least (index rows, endpoint coordinates or node rows, the output) and what that gives in GB/s, with the GPU name and
power limit read in the same run.  One JSON line per attribute.
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

KEY = ("hidden", "to", "data")


def gpu_info() -> dict:
    try:
        out = subprocess.run(
            ["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
            capture_output=True, text=True, timeout=30,
        ).stdout.strip()  # fmt: skip
    except (OSError, subprocess.SubprocessError):
        out = ""
    return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": out}


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


def torch_azimuth(ei, sx, tx):
    s, t = sx.double()[ei[0]], tx.double()[ei[1]]
    dl = s[:, 1] - t[:, 1]
    y = torch.sin(dl) * torch.cos(s[:, 0])
    x = torch.cos(t[:, 0]) * torch.sin(s[:, 0]) - torch.sin(t[:, 0]) * torch.cos(s[:, 0]) * torch.cos(dl)
    return torch.atan2(y, x).float().unsqueeze(1)


def torch_gaussian_l1(ei, sx, tx, sigma: float, n_dst: int, d=None):
    if d is None:
        s, t = sx.double()[ei[0]], tx.double()[ei[1]]
        a = torch.sin(0.5 * (t[:, 0] - s[:, 0])) ** 2 + torch.cos(s[:, 0]) * torch.cos(t[:, 0]) * torch.sin(0.5 * (t[:, 1] - s[:, 1])) ** 2
        d = 2 * torch.atan2(torch.sqrt(a), torch.sqrt(1 - a))
    w = torch.exp(-(d * d) / (2 * sigma**2))
    sums = torch.zeros(n_dst, dtype=torch.float64, device=w.device).scatter_reduce(0, ei[1], w, "sum")
    return (w / sums[ei[1]]).float().unsqueeze(1)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="o1280_res7", choices=sorted(WORKLOADS))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sigma", type=float, default=0.01, help="GaussianDistanceWeights sigma (radians)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("edge_attr_extra_bench needs a CUDA device")

    from anemoi_graphs_b200 import device as agx_device
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.edges.attributes import (
        AttributeFromSourceNode,
        AttributeFromTargetNode,
        Azimuth,
        EdgeLength,
        GaussianDistanceWeights,
    )
    from anemoi_graphs_b200.graph import HeteroData

    grid, res = WORKLOADS[args.workload]
    agx_device.set_resident(True)
    graph = HeteroData()
    graph["data"].x = data_coordinates(grid).cuda()
    graph["data"].node_type = "LatLonNodes"
    graph = GraphCreator(recipe(res)).update_graph(graph)
    agx_device.flush()
    for name in ("hidden", "data"):
        graph[name]["north"] = graph[name].x[:, 0] > 0
    torch.cuda.synchronize()
    info = gpu_info()
    ei = graph[KEY].edge_index
    e = int(ei.shape[1])
    ei64 = ei.long()
    sx, tx = graph[KEY[0]].x, graph[KEY[2]].x
    n_dst = int(tx.shape[0])

    cases = [
        ("Azimuth", Azimuth(), lambda: torch_azimuth(ei64, sx, tx), 8 + 16 + 4, 1e-5),
        ("GaussianDistanceWeights", GaussianDistanceWeights(sigma=args.sigma, norm="l1"),
         lambda: torch_gaussian_l1(ei64, sx, tx, args.sigma, n_dst), 8 + 16 + 4, 1e-5),
        ("AttributeFromSourceNode", AttributeFromSourceNode("north"),
         lambda: graph["hidden"]["north"][ei64[0]].unsqueeze(1), 4 + 1 + 1, 0.0),
        ("AttributeFromTargetNode", AttributeFromTargetNode("north"),
         lambda: graph["data"]["north"][ei64[1]].unsqueeze(1), 4 + 1 + 1, 0.0),
    ]  # fmt: skip
    failed = False
    for name, attr, ref, bytes_per_edge, rtol in cases:
        ms_ours, ours = timed(lambda attr=attr: attr.compute(graph, KEY), args.reps, args.warmup)
        ms_torch, theirs = timed(ref, args.reps, args.warmup)
        extra = {}
        if name == "GaussianDistanceWeights":
            extra["max_rel_diff_vs_float64_haversine"] = float(((ours.double() - theirs.double()).abs() / theirs.double().abs()).max())
            lengths = EdgeLength().compute(graph, KEY)[:, 0].double()
            theirs = torch_gaussian_l1(ei64, sx, tx, args.sigma, n_dst, d=lengths)
            rtol = 1e-6
        if rtol == 0.0:
            bad = ours != theirs
        else:
            diff = ours.double() - theirs.double()
            if name == "Azimuth":  # +-pi may flip
                diff = torch.remainder(diff + math.pi, 2 * math.pi) - math.pi
            bad = ~(diff.abs() <= rtol * theirs.double().abs().clamp(min=0.1)) & ~(ours.isnan() & theirs.isnan())
        n_bad = int(bad.sum())
        if n_bad:
            at = torch.nonzero(bad[:, 0])[:5, 0]
            print(json.dumps({"attribute": name, "mismatches": n_bad, "at": at.tolist(), "ours": ours[at, 0].tolist(),
                              "torch": theirs[at, 0].tolist(), "targets": ei64[1, at].tolist(),
                              "sources": ei64[0, at].tolist()}), flush=True)  # fmt: skip
            failed = True
        gbs = lambda ms: round(bytes_per_edge * e / (ms * 1e-3) / 1e9, 1)  # noqa: E731
        print(json.dumps({
            "set": "decoder", "attribute": name, "edges": e, "ms_cuda": round(ms_ours, 3), "ms_torch": round(ms_torch, 3),
            "bytes_min_per_edge": bytes_per_edge, "gbs_cuda": gbs(ms_ours), "gbs_torch": gbs(ms_torch), **extra, **info,
        }), flush=True)  # fmt: skip
    if failed:
        raise SystemExit("outputs differ")


if __name__ == "__main__":
    main()
