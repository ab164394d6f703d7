#!/usr/bin/env python
"""Edge sets as operators (``export.EdgeSetOperator``, ``agx_csr_spmm``) against ``torch.sparse.mm`` on the same CSR.

    python tools/edge_operator_bench.py [--features 1 16 64 256] [--reps 20] [--warmup 3] [--out profiles/edge_operator_bench.jsonl]

Edge sets of the ``bench.py`` O1280 -> TriNodes(7) graph, built once by ``GraphCreator`` on a device-resident graph,
as matrices of ones (no attribute; the values do not change the work):
* ``decoder``: KNN-3, hidden -> data, 6.6 M rows of 3 entries over 163 842 sources;
* ``encoder``: CutOff 0.6, data -> hidden, 163 842 rows of about 63 entries over 6.6 M sources.
One JSON line per (edge set, F, dtype), F in --features, float32 and bfloat16:
* ``op_ms``: one ``op(x)`` call (CUDA events, median of --reps after --warmup), the index check's read-back included;
* ``torch_sparse_mm_ms`` (float32 only): ``torch.sparse.mm`` on the CUDA tensor ``edge_set_to_sparse`` returns,
  timed alternately with the kernel in the same loop, and the largest difference between the two results relative
  to the largest |y|;
* ``bytes``: the compulsory traffic - indptr, indices and values once, x once, y once - and ``hbm_bound_share``, the
  time those bytes take at the 7.7 TB/s of the data sheet over ``op_ms``; ``gathered_bytes``: x read once per entry,
  the traffic of a gather that finds nothing in cache;
* ``csr_build_ms``: the one-off ``EdgeSetOperator`` construction (sort and CSR build; CUDA events, median of 5).
The card's name and power limit are read in the same run.
"""

from __future__ import annotations

import argparse
import json
import pathlib
import statistics
import sys

REPO = pathlib.Path(__file__).resolve().parents[1]
for p in (REPO, REPO / "tools"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import torch  # noqa: E402

from bench import data_coordinates, recipe  # noqa: E402
from edge_attr_extra_bench import gpu_info  # noqa: E402
from reduced_gaussian_bench import event_ms  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
EDGE_SETS = {"decoder": ("hidden", "to", "data"), "encoder": ("data", "to", "hidden")}


def build_graph():
    from anemoi_graphs_b200 import device
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.graph import HeteroData

    device.set_resident(True)
    graph = HeteroData()
    graph["data"].x = data_coordinates("o1280").cuda()
    graph = GraphCreator(recipe(7)).update_graph(graph)
    torch.cuda.synchronize()
    return graph


def alternate_ms(fns, reps: int, warmup: int) -> list[float]:
    """Median CUDA-event milliseconds of each function, the functions timed in turn within each repetition."""
    for _ in range(warmup):
        for fn in fns:
            fn()
    torch.cuda.synchronize()
    times = [[] for _ in fns]
    for _ in range(reps):
        for fn, t in zip(fns, times):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            t.append(a.elapsed_time(b))
    return [statistics.median(t) for t in times]


def run(name: str, graph, args) -> list[dict]:
    from anemoi_graphs_b200.export import EdgeSetOperator
    from anemoi_graphs_b200.export import edge_set_to_sparse

    key = EDGE_SETS[name]
    csr_build_ms = event_ms(lambda: EdgeSetOperator(graph, key), 5, 1)
    op = EdgeSetOperator(graph, key)
    m = edge_set_to_sparse(graph, key)
    n_dst, n_src = op.shape
    nnz = int(op._indices.numel())
    base = {"edge_set": name, "key": list(key), "shape": [n_dst, n_src], "nnz": nnz, "csr_build_ms": round(csr_build_ms, 4), **gpu_info()}
    rows = []
    gen = torch.Generator(device="cuda").manual_seed(0)
    for f in args.features:
        for dtype in (torch.float32, torch.bfloat16):
            x = torch.randn(n_src, f, device="cuda", generator=gen).to(dtype)
            elem = x.element_size()
            row = {**base, "features": f, "dtype": str(dtype).removeprefix("torch.")}
            if dtype == torch.float32:
                row["op_ms"], row["torch_sparse_mm_ms"] = alternate_ms([lambda: op(x), lambda: torch.sparse.mm(m, x)], args.reps, args.warmup)
                y, ref = op(x), torch.sparse.mm(m, x)
                row["max_diff_vs_torch_rel"] = float((y - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
                del y, ref
            else:
                row["op_ms"] = event_ms(lambda: op(x), args.reps, args.warmup)
            row["bytes"] = 8 * (n_dst + 1) + 8 * nnz + (n_src + n_dst) * f * elem
            row["gathered_bytes"] = 8 * (n_dst + 1) + 8 * nnz + (nnz + n_dst) * f * elem
            row["hbm_bound_ms"] = row["bytes"] / HBM_BYTES_PER_S * 1e3
            row["hbm_bound_share"] = row["hbm_bound_ms"] / row["op_ms"]
            row.update({"reps": args.reps, "warmup": args.warmup})
            rows.append({k: (round(v, 4) if isinstance(v, float) and k != "max_diff_vs_torch_rel" else v) for k, v in row.items()})
            del x
            torch.cuda.empty_cache()
    return rows


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--edge-sets", nargs="+", default=list(EDGE_SETS), choices=list(EDGE_SETS))
    ap.add_argument("--features", type=int, nargs="+", default=[1, 16, 64, 256])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    graph = build_graph()
    for name in args.edge_sets:
        for row in run(name, graph, args):
            line = json.dumps(row)
            print(line, flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(line + "\n")


if __name__ == "__main__":
    main()
