#!/usr/bin/env python
"""``IsolatitudeAreaWeights`` on the device, against ``SphericalAreaWeights`` and against a numpy host route.

    python tools/isolatitude_bench.py [--reps 20] [--warmup 3] [--host-reps 3] [--out profiles/isolatitude_bench.jsonl]

Workloads, device-resident float32 coordinates: O1280 (6 599 680 nodes, rows in order) and O2560 (26 306 560), as
``ReducedGaussianGridNodes`` generates them, and HEALPix resolution 10 in nested order (12 582 912 nodes; the
latitudes are not monotone, so the sort does real work).  O1280's 52.8 MB of coordinates fit the 126 MB L2, the
other two do not.  Per workload, one JSON line:
* ``ops.isolatitude_areas`` and ``IsolatitudeAreaWeights().compute`` on a device-resident graph - CUDA events, median
  of --reps after --warmup; at O1280 also ``SphericalAreaWeights().compute`` (k = 17 search included);
* the kernels of one call by name (``torch.profiler``, a separate pass after the timed ones): the share of the sort;
* the numpy route on the same float32 input already on the host (``np.unique``, then the bands:
  ``tests/test_gpu_isolatitude.py``'s reference) - perf_counter, median of --host-reps;
* how many of the two routes' float64 raw values are bit-equal, and the largest relative difference.
The card's name and power limit are read in the same run.
"""

from __future__ import annotations

import argparse
import json
import pathlib
import sys

REPO = pathlib.Path(__file__).resolve().parents[1]
for p in (REPO, REPO / "tools", REPO / "tests"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from edge_attr_extra_bench import gpu_info  # noqa: E402
from reduced_gaussian_bench import event_ms, host_ms  # noqa: E402
from test_gpu_isolatitude import reference  # noqa: E402


def kernel_ms(fn) -> dict[str, float]:
    """Device milliseconds of one call of ``fn`` per kernel name (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out: dict[str, float] = {}
    for evt in prof.key_averages():
        us = getattr(evt, "device_time_total", None)
        if us is None:
            us = getattr(evt, "cuda_time_total", 0.0)
        if us > 0 and not evt.key.startswith(("Memcpy", "Memset", "cuda")):
            if "cub" in evt.key.lower():
                name = "cub_radix_sort" if "Radix" in evt.key else "cub_run_length_encode"
            else:
                name = evt.key.split("(")[0].split("<")[0].split(" ")[-1]
            out[name] = out.get(name, 0.0) + us / 1e3
    return {k: round(v, 4) for k, v in sorted(out.items())}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--out", default=str(REPO / "profiles" / "isolatitude_bench.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("isolatitude_bench needs a CUDA device")

    from anemoi_graphs_b200 import ops
    from anemoi_graphs_b200.graph import HeteroData
    from anemoi_graphs_b200.nodes.attributes import IsolatitudeAreaWeights, SphericalAreaWeights

    info, lines = gpu_info(), []
    workloads = [("O1280", lambda: ops.octahedral_nodes(1280)), ("O2560", lambda: ops.octahedral_nodes(2560)),
                 ("healpix10_nested", lambda: ops.healpix_nodes(10))]  # fmt: skip
    for name, make in workloads:
        x = make()
        n = int(x.shape[0])
        graph = HeteroData()
        graph["data"].x = x
        graph["data"].node_type = name
        line = {"workload": name, "nodes": n}
        line["device_ms_ops"] = round(event_ms(lambda: ops.isolatitude_areas(x), args.reps, args.warmup), 4)
        line["device_ms_isolatitude_compute"] = round(
            event_ms(lambda: IsolatitudeAreaWeights().compute(graph, "data"), args.reps, args.warmup), 4
        )
        if name == "O1280":
            line["device_ms_spherical_compute"] = round(
                event_ms(lambda: SphericalAreaWeights().compute(graph, "data"), max(args.reps // 4, 3), 1), 3
            )
            line["spherical_over_isolatitude"] = round(
                line["device_ms_spherical_compute"] / line["device_ms_isolatitude_compute"], 1
            )
        line["kernels_ms"] = kernel_ms(lambda: ops.isolatitude_areas(x))
        kernels_total = sum(line["kernels_ms"].values())
        line["sort_share"] = round(line["kernels_ms"].get("cub_radix_sort", 0.0) / max(kernels_total, 1e-9), 3)
        device, n_rows = ops.isolatitude_areas(x)
        device = device.cpu().numpy()
        host_x = x.cpu().numpy()
        ms_host, (host, host_rows, _) = host_ms(lambda: reference(host_x), args.host_reps)
        line.update({
            "rows": n_rows, "rows_agree": n_rows == host_rows, "host_ms_numpy": round(ms_host, 1),
            "bit_equal": int((device.view(np.int64) == host.view(np.int64)).sum()),
            "max_rel_diff": float(np.max(np.abs(device - host) / host)), "sum_minus_4pi": float(device.sum() - 4 * np.pi),
            **info,
        })  # fmt: skip
        print(json.dumps(line), flush=True)
        lines.append(line)
        del x, graph, device, host, host_x
        torch.cuda.empty_cache()
    out = pathlib.Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text("".join(json.dumps(line) + "\n" for line in lines))
    if not all(line["rows_agree"] and line["max_rel_diff"] <= 1e-14 for line in lines):
        raise SystemExit("device and host weights differ beyond 1e-14")


if __name__ == "__main__":
    main()
