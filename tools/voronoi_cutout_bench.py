#!/usr/bin/env python
"""``SphericalAreaWeights`` on cutout node sets (the wide pass of ``ops.voronoi_areas``), and the global O1280 path
it must not slow down.

    python tools/voronoi_cutout_bench.py [--baseline DIR] [--reps 5] [--out profiles/voronoi_cutout_bench.jsonl]

* Global O1280 (6 599 680 nodes, device-resident): ``SphericalAreaWeights().compute`` - CUDA events, median of --reps
  after one warm-up, in a fresh process per sample.  With --baseline (a built checkout of another revision) the
  samples alternate between that tree and this one, three of each.
* Cutout sets of ``tests/test_gpu_area_weights_cutout.py`` - case A (O48 + O1280 in a 10 degree cap), case B
  (O24 + O2560 in a 3 degree cap) and a realistic cutout, O96 + O1280 in a 15 degree cap: the cells handed to the wide
  pass, its rounds, its candidates per final cell (largest, mean), the time of ``ops.voronoi_areas`` and of its wide
  pass alone (``ops.Timeline`` span), and scipy's ``SphericalVoronoi`` on the host for the same set.
* Case A's regional part on its own, a limited-area set: the rounds and time the wide pass spends before it raises.
The card's name and power limit are read in the same run.
"""

from __future__ import annotations

import argparse
import json
import pathlib
import subprocess
import sys
import time

REPO = pathlib.Path(__file__).resolve().parents[1]


def _o1280_worker(reps: int) -> None:
    import numpy as np
    import torch

    from anemoi_graphs_b200 import ops
    from anemoi_graphs_b200.graph import HeteroData
    from anemoi_graphs_b200.nodes.attributes import SphericalAreaWeights

    x = ops.octahedral_nodes(1280)
    graph = HeteroData()
    graph["data"].x = x
    graph["data"].node_type = "O1280"
    SphericalAreaWeights().compute(graph, "data")
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        SphericalAreaWeights().compute(graph, "data")
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    print(json.dumps({"ms": float(np.median(times))}))


def _sample(root: pathlib.Path, reps: int) -> float:
    code = f"import sys; sys.path.insert(0, {str(root)!r}); sys.path.insert(1, {str(REPO / 'tools')!r}); " \
           f"import voronoi_cutout_bench as b; b._o1280_worker({reps})"  # fmt: skip
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True, cwd=root)
    return json.loads(out.stdout.strip().splitlines()[-1])["ms"]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", default=None, help="a built checkout of the revision to compare the O1280 time with")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=str(REPO / "profiles" / "voronoi_cutout_bench.jsonl"))
    args = ap.parse_args()
    for p in (REPO, REPO / "tools", REPO / "tests"):
        if str(p) not in sys.path:
            sys.path.insert(0, str(p))
    import numpy as np
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("voronoi_cutout_bench needs a CUDA device")
    from edge_attr_extra_bench import gpu_info
    from test_gpu_area_weights_cutout import CASES, _scipy, cutout

    from oracle import ref_path as R

    from anemoi_graphs_b200 import ops

    info, lines = gpu_info(), []
    roots = [("this", REPO)] + ([("baseline", pathlib.Path(args.baseline).resolve())] if args.baseline else [])
    samples: dict[str, list[float]] = {name: [] for name, _ in roots}
    for _ in range(3):
        for name, root in roots[::-1]:
            samples[name].append(round(_sample(root, args.reps), 3))
    line = {"workload": "O1280_spherical_compute", "nodes": 6599680, **{f"ms_{k}": v for k, v in samples.items()}, **info}
    print(json.dumps(line), flush=True)
    lines.append(line)

    sets = {"A": CASES["A"], "B": CASES["B"], "O96+O1280_15deg": (96, 1280, 15.0, 0.3, 50.0, 10.0)}
    for name, spec in sets.items():
        x = cutout(*spec)
        xd = torch.from_numpy(x).cuda()
        got = ops.voronoi_areas(xd)  # warm-up
        times, wide_ms = [], []
        for _ in range(args.reps):
            ops.timeline = ops.Timeline()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            got = ops.voronoi_areas(xd)
            b.record()
            torch.cuda.synchronize()
            times.append(a.elapsed_time(b))
            wide_ms.append(ops.timeline.totals_ms().get("voronoi_areas_wide", 0.0))
            ops.timeline = None
        t0 = time.perf_counter()
        want = R.spherical_area_weights(x, None, "float64")[:, 0]
        host_ms = (time.perf_counter() - t0) * 1e3
        widest = _scipy(x)[2]
        got = got.cpu().numpy()
        line = {
            "workload": name, "nodes": int(x.shape[0]), "spec": spec,
            **{k: v for k, v in ops.voronoi_wide.items() if k != "generators"},
            "ms_voronoi_areas": round(float(np.median(times)), 3), "ms_wide_pass": round(float(np.median(wide_ms)), 3),
            "host_ms_scipy": round(host_ms, 1), "scipy_widest_region": int(widest),
            "max_rel_diff": float(np.max(np.abs(got - want) / want)), **info,
        }  # fmt: skip
        print(json.dumps(line), flush=True)
        lines.append(line)
    # a limited-area set on its own still raises; what the wide pass spends before it does
    x = cutout(*CASES["A"], regional_only=True)
    xd = torch.from_numpy(x).cuda()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    try:
        ops.voronoi_areas(xd)
        raised = ""
    except NotImplementedError as exc:
        raised = str(exc)
    torch.cuda.synchronize()
    line = {"workload": "A_regional_alone", "nodes": int(x.shape[0]), **ops.voronoi_wide, "raised": raised,
            "ms_until_raise": round((time.perf_counter() - t0) * 1e3, 3), **info}  # fmt: skip
    line.pop("generators")
    print(json.dumps(line), flush=True)
    lines.append(line)
    out = pathlib.Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text("".join(json.dumps(line) + "\n" for line in lines))


if __name__ == "__main__":
    main()
