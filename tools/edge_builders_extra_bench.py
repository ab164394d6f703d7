#!/usr/bin/env python
"""ReversedKNNEdges and MultiScaleEdges(scale_resolutions) on the bench.py workload (O1280 -> TriNodes(7)), device-resident.

    python tools/edge_builders_extra_bench.py [--workload o1280_res7] [--reps 10] [--warmup 3]

Timed with CUDA events after warm-up, the two sides of each comparison alternating in the same process (median ms):
* search: ``ReversedKNNEdges(data -> hidden, k = 3).get_edge_index`` against ``KNNEdges(hidden -> data, k = 3)``, the
  same search over final node coordinates; the two edge lists must be each other's row swap, column for column;
* step: the bench.py recipe, and the same recipe with its encoder replaced by ``ReversedKNNEdges(data -> hidden, k = 3)``
  (every data point gets its 3 nearest mesh nodes), with the mesh order sorted on the host while the searches run
  (the default) and sorted first (``LAZY_NODE_ORDER`` off);
* multiscale: ``MultiScaleEdges(hidden -> hidden, x_hops = 1).get_edge_index`` with ``scale_resolutions = 7`` (levels
  1..7) against the default (levels 0..7).
The GPU name and power limit are read in the same run.  One JSON line per comparison.
"""

from __future__ import annotations

import argparse
import copy
import json
import pathlib
import statistics
import sys

REPO = pathlib.Path(__file__).resolve().parents[1]
for p in (REPO, REPO / "tools"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import torch  # noqa: E402

from bench import T, WORKLOADS, data_coordinates, recipe, run_step  # noqa: E402
from edge_attr_extra_bench import gpu_info  # noqa: E402


def alternate(fns: dict, reps: int, warmup: int) -> tuple[dict, dict]:
    """Median CUDA-event ms of each callable, the callables interleaved rep by rep; and each one's last output."""
    outs, times = {}, {name: [] for name in fns}
    for _ in range(warmup):
        for name, fn in fns.items():
            outs[name] = None
            outs[name] = fn()
    torch.cuda.synchronize()
    for _ in range(reps):
        for name, fn in fns.items():
            outs[name] = None
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            outs[name] = fn()
            b.record()
            torch.cuda.synchronize()
            times[name].append(a.elapsed_time(b))
    return {name: round(statistics.median(t), 3) for name, t in times.items()}, outs


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="o1280_res7", choices=sorted(WORKLOADS))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("edge_builders_extra_bench needs a CUDA device")

    from anemoi_graphs_b200 import device as agx_device
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.edges import KNNEdges, MultiScaleEdges, ReversedKNNEdges

    grid, res = WORKLOADS[args.workload]
    info = gpu_info()
    agx_device.set_resident(True)
    x_dev = data_coordinates(grid).cuda()
    graph = run_step(GraphCreator({"nodes": recipe(res)["nodes"]}), x_dev)
    agx_device.flush()
    torch.cuda.synchronize()
    n_data, n_hidden = int(graph["data"].x.shape[0]), int(graph["hidden"].x.shape[0])
    failed = False

    # ---- the search ---------------------------------------------------------------------------------
    ms, out = alternate({
        "reversed_knn": lambda: ReversedKNNEdges("data", "hidden", 3).get_edge_index(graph),
        "knn": lambda: KNNEdges("hidden", "data", 3).get_edge_index(graph),
    }, args.reps, args.warmup)  # fmt: skip
    same = bool(torch.equal(out["reversed_knn"], out["knn"].flip(0)))
    failed |= not same
    print(json.dumps({"case": "search", "workload": args.workload, "k": 3, "queries": n_data, "indexed": n_hidden,
                      "edges": int(out["knn"].shape[1]), "ms_reversed_knn": ms["reversed_knn"], "ms_knn": ms["knn"],
                      "row_swap_equal": same, **info}), flush=True)  # fmt: skip

    # ---- the whole step with a reversed encoder --------------------------------------------------------
    reversed_recipe = copy.deepcopy(recipe(res))
    reversed_recipe["edges"][0]["edge_builders"] = [{"_target_": T + "edges.ReversedKNNEdges", "num_nearest_neighbours": 3}]
    bench_creator, reversed_creator = GraphCreator(recipe(res)), GraphCreator(reversed_recipe)

    def serial(creator):
        prev, agx_device.LAZY_NODE_ORDER = agx_device.LAZY_NODE_ORDER, False
        try:
            return run_step(creator, x_dev)
        finally:
            agx_device.LAZY_NODE_ORDER = prev

    ms, out = alternate({
        "bench_recipe": lambda: run_step(bench_creator, x_dev),
        "reversed_encoder": lambda: run_step(reversed_creator, x_dev),
        "reversed_encoder_order_first": lambda: serial(reversed_creator),
    }, args.reps, args.warmup)  # fmt: skip
    key = ("data", "to", "hidden")
    a, b = out["reversed_encoder"][key], out["reversed_encoder_order_first"][key]
    # the same edges: the same source row, and the same SET of k targets per source (their order within a source
    # follows the index the search ran on)
    same = bool(torch.equal(a.edge_index[0], b.edge_index[0])) and bool(
        torch.equal(a.edge_index[1].view(-1, 3).sort(dim=1).values, b.edge_index[1].view(-1, 3).sort(dim=1).values)
    )
    failed |= not same
    print(json.dumps({"case": "step", "workload": args.workload, "ms_bench_recipe": ms["bench_recipe"],
                      "ms_reversed_encoder": ms["reversed_encoder"],
                      "ms_reversed_encoder_order_first": ms["reversed_encoder_order_first"],
                      "encoder_edges": int(a.edge_index.shape[1]), "lazy_equals_order_first": same, **info}), flush=True)  # fmt: skip
    del out, a, b

    # ---- MultiScaleEdges(scale_resolutions) -------------------------------------------------------------
    ms, out = alternate({
        "default": lambda: MultiScaleEdges("hidden", "hidden", 1).get_edge_index(graph),
        "levels_1_to_7": lambda: MultiScaleEdges("hidden", "hidden", 1, scale_resolutions=res).get_edge_index(graph),
    }, args.reps, args.warmup)  # fmt: skip
    print(json.dumps({"case": "multiscale", "workload": args.workload, "x_hops": 1, "ms_default": ms["default"],
                      "ms_levels_1_to_n": ms["levels_1_to_7"], "edges_default": int(out["default"].shape[1]),
                      "edges_levels_1_to_n": int(out["levels_1_to_7"].shape[1]), **info}), flush=True)  # fmt: skip
    if failed:
        raise SystemExit("outputs differ")


if __name__ == "__main__":
    main()
