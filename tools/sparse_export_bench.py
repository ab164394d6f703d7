#!/usr/bin/env python
"""Edge sets as sparse matrices (``ops.edges_to_csr``, ``export.edge_set_to_sparse``) against scipy on the host.

    python tools/sparse_export_bench.py [--reps 20] [--warmup 3] [--host-reps 3] [--out profiles/sparse_export_bench.jsonl]

Workloads, each built once by ``GraphCreator`` on a device-resident graph:
* ``o96_to_o1280_knn4``: KNNEdges(k = 4) from the O96 nodes to the O1280 nodes (each O1280 node's 4 nearest O96 nodes,
  26.4 M entries, rows = O1280) with ``GaussianDistanceWeights()`` - an interpolation operator, rows sum to 1;
* ``o1280_res7_decoder``: the decoder of the ``bench.py`` O1280 -> TriNodes(7) graph (KNN-3, 19.8 M entries), no
  attribute (ones).
Per workload, one JSON line:
* ``ops.edges_to_csr`` (sort and CSR build) and ``ops.sort_permutation`` alone - CUDA events, median of --reps after
  --warmup;
* ``edge_set_to_sparse`` on the device-resident graph (CUDA events, as above) and on a host-resident copy of it
  (perf_counter, median of --host-reps: uploads, kernels, copies back, the scipy constructor);
* scipy's ``coo_matrix(...).tocsr()`` + ``sum_duplicates()`` on the same host arrays, and ``save_npz`` of the result,
  compressed (its default) and not - perf_counter, median of --host-reps, on the same box's host;
* whether the device CSR equals scipy's (indptr, indices, data bit for bit).
The card's name and power limit are read in the same run.
"""

from __future__ import annotations

import argparse
import json
import pathlib
import sys
import tempfile

REPO = pathlib.Path(__file__).resolve().parents[1]
for p in (REPO, REPO / "tools"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import data_coordinates, recipe  # noqa: E402
from edge_attr_extra_bench import gpu_info  # noqa: E402
from reduced_gaussian_bench import event_ms, host_ms  # noqa: E402

T = "anemoi.graphs."


def build(workload: str):
    """(device-resident graph, edge set key, attribute name or None)."""
    from anemoi_graphs_b200 import device
    from anemoi_graphs_b200 import grids
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.graph import HeteroData

    device.set_resident(True)
    graph = HeteroData()
    graph["data"].x = data_coordinates("o1280").cuda()
    if workload == "o96_to_o1280_knn4":
        lat, lon = grids.octahedral_grid(96)
        cfg = {
            "nodes": {"coarse": {"node_builder": {"_target_": T + "nodes.LatLonNodes", "latitudes": lat, "longitudes": lon}}},
            "edges": [{"source_name": "coarse", "target_name": "data",
                       "attributes": {"w": {"_target_": T + "edges.attributes.GaussianDistanceWeights"}},
                       "edge_builders": [{"_target_": T + "edges.KNNEdges", "num_nearest_neighbours": 4}]}],
        }  # fmt: skip
        key, attr = ("coarse", "to", "data"), "w"
    else:
        cfg = recipe(7)
        key, attr = ("hidden", "to", "data"), None
    graph = GraphCreator(cfg).update_graph(graph)
    torch.cuda.synchronize()
    return graph, key, attr


def host_copy(graph, key):
    """A host-resident graph holding the edge set ``key`` and its two node sets."""
    from anemoi_graphs_b200.graph import HeteroData

    g = HeteroData()
    for name in (key[0], key[2]):
        g[name].x = graph[name].x.cpu()
    for k, v in graph[key].items():
        if isinstance(v, torch.Tensor):
            g[key][k] = v.cpu()
    return g


def run(workload: str, args) -> dict:
    from scipy.sparse import coo_matrix
    from scipy.sparse import save_npz

    from anemoi_graphs_b200 import ops
    from anemoi_graphs_b200.export import edge_set_to_sparse

    graph, key, attr = build(workload)
    store = graph[key]
    ei = store.edge_index
    n_src, n_dst = int(graph[key[0]].num_nodes), int(graph[key[2]].num_nodes)
    values = None if attr is None else store[attr].reshape(-1).contiguous()
    e = int(ei.shape[1])
    row = {"workload": workload, "edges": e, "shape": [n_dst, n_src], "attribute": attr, **gpu_info()}

    row["edges_to_csr_ms"] = event_ms(lambda: ops.edges_to_csr(ei, n_dst, n_src, values), args.reps, args.warmup)
    row["sort_permutation_ms"] = event_ms(lambda: ops.sort_permutation(ei[1], ei[0], n_dst, n_src, False), args.reps, args.warmup)
    row["edge_set_to_sparse_device_ms"] = event_ms(lambda: edge_set_to_sparse(graph, key, attr), args.reps, args.warmup)
    dev = edge_set_to_sparse(graph, key, attr)
    got = [t.cpu().numpy() for t in (dev.crow_indices(), dev.col_indices(), dev.values())]

    host = host_copy(graph, key)
    edge_set_to_sparse(host, key, attr)  # warm-up
    row["edge_set_to_sparse_host_ms"], host_m = host_ms(lambda: edge_set_to_sparse(host, key, attr), args.host_reps)

    ei_h = host[key].edge_index.numpy()
    v_h = np.ones(e, dtype=np.float32) if attr is None else host[key][attr].numpy().reshape(-1)

    def scipy_route():
        m = coo_matrix((v_h, (ei_h[1], ei_h[0])), shape=(n_dst, n_src)).tocsr()
        m.sum_duplicates()
        return m

    row["scipy_tocsr_ms"], ref = host_ms(scipy_route, args.host_reps)
    row["equal_to_scipy"] = bool(
        np.array_equal(got[0], ref.indptr) and np.array_equal(got[1], ref.indices) and got[2].tobytes() == ref.data.tobytes()
    )
    row["host_equal_to_device"] = bool(
        np.array_equal(host_m.indptr, got[0]) and np.array_equal(host_m.indices, got[1]) and host_m.data.tobytes() == got[2].tobytes()
    )
    with tempfile.TemporaryDirectory() as tmp:
        path = pathlib.Path(tmp) / "m.npz"
        row["save_npz_compressed_ms"], _ = host_ms(lambda: save_npz(path, ref), args.host_reps)
        row["npz_compressed_bytes"] = path.stat().st_size
        row["save_npz_uncompressed_ms"], _ = host_ms(lambda: save_npz(path, ref, compressed=False), args.host_reps)
        row["npz_uncompressed_bytes"] = path.stat().st_size
    if attr is not None:
        sums = np.add.reduceat(got[2].astype(np.float64), got[0][:-1])
        row["max_abs_row_sum_minus_1"] = float(np.abs(sums - 1.0).max())
    row.update({"reps": args.reps, "warmup": args.warmup, "host_reps": args.host_reps})
    return {k: (round(v, 4) if isinstance(v, float) else v) for k, v in row.items()}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["o96_to_o1280_knn4", "o1280_res7_decoder"])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    for workload in args.workloads:
        line = json.dumps(run(workload, args))
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
