#!/usr/bin/env python
"""Octahedral grids O<N> (``ReducedGaussianGridNodes``) generated on the device, against the host route.

    python tools/reduced_gaussian_bench.py [--grids 1280 2560] [--reps 20] [--warmup 3] [--host-reps 3]

Per grid, one JSON line:
* device: ``agx_gaussian_latitudes`` and ``agx_octahedral_nodes`` each timed on its own with CUDA events, and
  ``ops.octahedral_nodes`` (both kernels and the allocations) end to end - median of --reps after --warmup; each
  kernel's share of the sum of the two, and the bytes the node kernel writes over its time;
* host: ``grids.octahedral_grid`` (numpy), the float32 cast of ``grids.latlon_deg_to_x`` and the upload of that tensor
  (``Tensor.cuda()`` from pageable memory, synchronised) - perf_counter, median of --host-reps;
* whether the device and host float32 results are equal bit for bit (the exit status is non-zero if not).
The GPU name and power limit are read in the same run.
"""

from __future__ import annotations

import argparse
import json
import pathlib
import statistics
import sys
import time

REPO = pathlib.Path(__file__).resolve().parents[1]
for p in (REPO, REPO / "tools"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import torch  # noqa: E402

from edge_attr_extra_bench import gpu_info  # noqa: E402


def event_ms(fn, reps: int, warmup: int) -> float:
    """Median CUDA-event milliseconds of ``fn`` on the current stream."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def host_ms(fn, reps: int) -> tuple[float, object]:
    """Median perf_counter milliseconds of ``fn`` (which ends in a device synchronise where it touches the device)."""
    times, out = [], None
    for _ in range(reps):
        out = None
        t0 = time.perf_counter()
        out = fn()
        times.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(times), out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--grids", type=int, nargs="+", default=[1280, 2560])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("reduced_gaussian_bench needs a CUDA device")

    from anemoi_graphs_b200 import _cabi, grids, ops

    lib, info, failed = _cabi.load_library(), gpu_info(), False
    for n in args.grids:
        points = 4 * n * (n + 9)
        lat = torch.empty(2 * n, dtype=torch.float64, device="cuda")
        out = torch.empty((points, 2), dtype=torch.float32, device="cuda")
        stream = _cabi.current_stream()
        ms_lat = event_ms(lambda: _cabi.check(lib.agx_gaussian_latitudes(n, _cabi.ptr(lat), stream)), args.reps, args.warmup)
        ms_nodes = event_ms(
            lambda: _cabi.check(lib.agx_octahedral_nodes(n, _cabi.ptr(lat), _cabi.ptr(out), stream)), args.reps, args.warmup
        )
        ms_ops = event_ms(lambda: ops.octahedral_nodes(n), args.reps, args.warmup)
        device_x = ops.octahedral_nodes(n).cpu()
        del lat, out

        ms_numpy, latlon = host_ms(lambda: grids.octahedral_grid(n), args.host_reps)
        ms_cast, host_x = host_ms(lambda: grids.latlon_deg_to_x(*latlon), args.host_reps)

        def upload():
            x = host_x.cuda()
            torch.cuda.synchronize()
            return x

        ms_upload, _ = host_ms(upload, args.host_reps)
        equal = bool(torch.equal(device_x.view(torch.int32), host_x.view(torch.int32)))
        failed |= not equal
        print(json.dumps({
            "grid": f"O{n}", "points": points, "output_bytes": points * 8,
            "device_ms_latitudes": round(ms_lat, 4), "device_ms_nodes": round(ms_nodes, 4),
            "share_latitudes": round(ms_lat / (ms_lat + ms_nodes), 3), "share_nodes": round(ms_nodes / (ms_lat + ms_nodes), 3),
            "nodes_write_gbps": round(points * 8 / (ms_nodes * 1e6), 1), "device_ms_ops_octahedral_nodes": round(ms_ops, 4),
            "host_ms_numpy": round(ms_numpy, 1), "host_ms_float32_cast": round(ms_cast, 1), "host_ms_upload": round(ms_upload, 2),
            "host_ms_total": round(ms_numpy + ms_cast + ms_upload, 1), "bit_equal": equal, **info,
        }), flush=True)  # fmt: skip
        del device_x, host_x, latlon
    if failed:
        raise SystemExit("device and host grids differ")


if __name__ == "__main__":
    main()
