"""Edge sets as sparse matrices: ``ops.edges_to_csr``, ``export.edge_set_to_sparse``, ``GraphExporter`` and the
``export_to_sparse`` command, against scipy on the same host arrays.

The reference matrix is ``coo_matrix((v, (edge_index[1], edge_index[0])), shape).tocsr()`` + ``sum_duplicates()``:
``indptr`` and ``indices`` must be equal and the data bit-equal.  scipy sums a duplicated (target, source) pair in the
order its CSR row holds them after ``csr_sort_indices``, an unstable ``std::sort``: that order is the column order for
a pair that occurs at most twice (two float32 adds commute) and for a row of at most 16 entries (insertion sort), and
unspecified otherwise.  There the device's column order is checked against ``stable_reference`` instead.
"""

import numpy as np
import pytest
import torch

from anemoi_graphs_b200 import grids

T = "anemoi.graphs."
KEY = ("src", "to", "dst")


def scipy_csr(ei: np.ndarray, values: np.ndarray, shape):
    from scipy.sparse import coo_matrix

    m = coo_matrix((values, (ei[1], ei[0])), shape=shape).tocsr()
    m.sum_duplicates()
    return m


def stable_reference(ei: np.ndarray, values: np.ndarray, n_dst: int):
    """(indptr, indices, data) with duplicates summed in column order, float32 adds left to right (bool: OR)."""
    order = np.lexsort((ei[0], ei[1]))  # stable
    d, s, v = ei[1][order], ei[0][order], values[order]
    head = np.ones(len(order), dtype=bool)
    head[1:] = (d[1:] != d[:-1]) | (s[1:] != s[:-1])
    starts = np.flatnonzero(head)
    run = np.cumsum(head) - 1
    pos = np.arange(len(order)) - starts[run]
    data = v[starts].copy()
    for k in range(1, int(pos.max(initial=0)) + 1):
        sel = pos == k
        if values.dtype == np.bool_:
            data[run[sel]] |= v[sel]
        else:
            data[run[sel]] = (data[run[sel]] + v[sel]).astype(np.float32)
    indptr = np.searchsorted(d[starts], np.arange(n_dst + 1), side="left")
    return indptr, s[starts], data


def as_arrays(matrix):
    """(indptr, indices, data) numpy arrays of a CUDA sparse CSR tensor or a scipy CSR matrix."""
    if isinstance(matrix, torch.Tensor):
        assert matrix.layout == torch.sparse_csr and matrix.is_cuda
        return tuple(t.cpu().numpy() for t in (matrix.crow_indices(), matrix.col_indices(), matrix.values()))
    return matrix.indptr, matrix.indices, matrix.data


def assert_csr_equal(got, want) -> None:
    gi, gj, gv = got
    wi, wj, wv = want
    np.testing.assert_array_equal(gi, wi)
    np.testing.assert_array_equal(gj, wj)
    assert gv.dtype == wv.dtype and gv.shape == wv.shape
    assert gv.tobytes() == wv.tobytes()


def host_graph(src_x, dst_x, edge_index, attrs=None, key=KEY):
    from anemoi_graphs_b200.graph import HeteroData

    g = HeteroData()
    g[key[0]].x = torch.as_tensor(src_x)
    if key[2] != key[0]:
        g[key[2]].x = torch.as_tensor(dst_x)
    g[key].edge_index = torch.as_tensor(edge_index)
    for name, value in (attrs or {}).items():
        g[key][name] = torch.as_tensor(value)
    return g


def on_device(graph):
    """The same graph with every tensor on the GPU."""
    from anemoi_graphs_b200.graph import HeteroData

    g = HeteroData()
    for name in graph.node_types:
        for k, v in graph[name].items():
            g[name][k] = v.cuda() if isinstance(v, torch.Tensor) else v
    for name in graph.edge_types:
        for k, v in graph[name].items():
            g[name][k] = v.cuda() if isinstance(v, torch.Tensor) else v
    return g


def coords(n: int, seed: int) -> np.ndarray:
    lat, lon = grids.uniform_sphere(n, seed=seed)
    return grids.latlon_deg_to_x(np.asarray(lat, dtype=np.float64), np.asarray(lon, dtype=np.float64)).numpy()


def varied_float32(rng, n: int) -> np.ndarray:
    """Signed values over eight decades, so that the order of a sum shows in its bits."""
    return (rng.standard_normal(n) * 10.0 ** rng.integers(-4, 4, n)).astype(np.float32)


def with_duplicates(rng, n_src: int, n_dst: int, n_edges: int, n_dup: int, max_copies: int, dst_pool) -> np.ndarray:
    """int32 (2, n_edges + copies) edges into the targets of ``dst_pool`` only, ``n_dup`` columns copied 1 to
    ``max_copies - 1`` more times, shuffled."""
    ei = np.stack([rng.integers(0, n_src, n_edges), rng.choice(dst_pool, n_edges)])
    dup = rng.choice(n_edges, n_dup, replace=False)
    extra = np.repeat(dup, rng.integers(1, max_copies, n_dup))
    ei = np.concatenate([ei, ei[:, extra]], axis=1)
    return np.ascontiguousarray(ei[:, rng.permutation(ei.shape[1])]).astype(np.int32)


# ------------------------------------------------------------------------------------------------
# ops.edges_to_csr on hand-made edge lists
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "bool", "ones"])
@pytest.mark.parametrize("case", ["short_rows", "pairs_twice", "long_runs", "one_million"])
def test_edges_to_csr_duplicates_and_empty_rows(case, dtype):
    from anemoi_graphs_b200 import ops

    rng = np.random.default_rng(["short_rows", "pairs_twice", "long_runs", "one_million"].index(case))
    n_src, n_dst = (50, 40) if case != "one_million" else (30_000, 20_000)
    pool = rng.choice(n_dst, n_dst * 3 // 4, replace=False)  # a quarter of the target rows stay empty
    if case == "short_rows":  # <= 16 entries per row: scipy keeps column order, up to 5 copies of a pair
        ei = np.concatenate([with_duplicates(rng, 6, n_dst, 2, 1, 5, [t]) for t in pool], axis=1)
        ei = np.ascontiguousarray(ei[:, rng.permutation(ei.shape[1])])
    elif case == "pairs_twice":  # long rows, each pair at most twice
        ei = with_duplicates(rng, n_src, n_dst, 3000, 0, 2, pool)
        ei = np.unique(ei, axis=1)
        ei = np.concatenate([ei, ei[:, rng.choice(ei.shape[1], 600, replace=False)]], axis=1)
        ei = np.ascontiguousarray(ei[:, rng.permutation(ei.shape[1])]).astype(np.int32)
    elif case == "long_runs":  # long rows, pairs up to 40 times
        ei = with_duplicates(rng, 5, n_dst, 2000, 200, 40, pool)
    else:
        ei = with_duplicates(rng, n_src, n_dst, 1_000_000, 100_000, 6, pool)
    e = ei.shape[1]
    values = {"float32": varied_float32(rng, e), "bool": rng.random(e) < 0.3, "ones": np.ones(e, dtype=np.float32)}[dtype]
    dev_values = None if dtype == "ones" else torch.from_numpy(values).cuda()
    ei_dev = torch.from_numpy(ei).cuda()
    got = [tuple(t.cpu().numpy() for t in ops.edges_to_csr(ei_dev, n_dst, n_src, dev_values)) for _ in range(2)]
    assert got[0][0].dtype == np.int64 and got[0][1].dtype == np.int32 and got[0][2].dtype == values.dtype
    assert all(a.tobytes() == b.tobytes() for a, b in zip(*got))  # two calls, bit-identical
    ref = scipy_csr(ei, values, (n_dst, n_src))
    stable = stable_reference(ei, values, n_dst)
    assert_csr_equal(got[0], stable)
    assert np.setdiff1d(np.arange(n_dst), pool).size and (np.diff(got[0][0])[np.setdiff1d(np.arange(n_dst), pool)] == 0).all()
    np.testing.assert_array_equal(got[0][0], ref.indptr)
    np.testing.assert_array_equal(got[0][1], ref.indices)
    if case in ("short_rows", "pairs_twice") or dtype != "float32":
        assert got[0][2].tobytes() == ref.data.astype(values.dtype).tobytes()
    if case == "long_runs":
        assert np.bincount(np.unique(ei, axis=1, return_counts=True)[1]).size > 3  # runs of 3 and more were summed


@pytest.mark.gpu
@pytest.mark.parametrize("n_edges", [0, 1])
def test_edges_to_csr_empty_and_single_edge(n_edges):
    from anemoi_graphs_b200 import ops

    ei = torch.tensor([[2], [1]], dtype=torch.int32, device="cuda")[:, :n_edges]
    indptr, indices, data = ops.edges_to_csr(ei, 3, 4, None)
    assert indptr.tolist() == ([0, 0, 1, 1] if n_edges else [0, 0, 0, 0])
    assert indices.tolist() == [2][:n_edges] and data.tolist() == [1.0][:n_edges] and data.dtype == torch.float32


@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["source", "target", "negative"])
def test_out_of_range_endpoint_raises(bad):
    from anemoi_graphs_b200.export import edge_set_to_sparse

    rng = np.random.default_rng(3)
    ei = np.stack([rng.integers(0, 30, 500), rng.integers(0, 20, 500)]).astype(np.int32)
    ei[{"source": (0, 17), "target": (1, 499), "negative": (1, 0)}[bad]] = {"source": 30, "target": 20, "negative": -1}[bad]
    g = host_graph(coords(30, 1), coords(20, 2), ei)
    for graph in (g, on_device(g)):
        with pytest.raises(ValueError, match="outside"):
            edge_set_to_sparse(graph, KEY)


@pytest.mark.gpu
def test_attribute_shape_and_sharded_block_raise():
    from anemoi_graphs_b200.export import edge_set_to_sparse

    rng = np.random.default_rng(4)
    ei = np.stack([rng.integers(0, 30, 400), rng.integers(0, 20, 400)]).astype(np.int32)
    g = on_device(host_graph(coords(30, 1), coords(20, 2), ei, {"w2": np.ones((400, 2), np.float32), "w": np.ones((400, 1), np.float32)}))
    with pytest.raises(ValueError, match=r"'w2'.*\(400, 2\)"):
        edge_set_to_sparse(g, KEY, "w2")
    g[KEY]["edge_shard"] = {"rank": 0, "world": 2, "counts": [400, 400], "replicated": False}
    before = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in g[KEY].items()}
    for attr in (None, "w"):
        with pytest.raises(NotImplementedError, match="gather"):
            edge_set_to_sparse(g, KEY, attr)
    after = g[KEY]
    assert before.keys() == set(after.keys())
    for k, v in before.items():
        assert (v.cpu().numpy().tobytes() == after[k].cpu().numpy().tobytes()) if isinstance(v, torch.Tensor) else v == after[k]


# ------------------------------------------------------------------------------------------------
# graphs built by GraphCreator, device-resident and host-resident
# ------------------------------------------------------------------------------------------------
def _recipe() -> dict:
    lat, lon = grids.octahedral_grid(96)
    weights = {"w": {"_target_": T + "edges.attributes.GaussianDistanceWeights", "sigma": 0.02}}
    return {
        "nodes": {
            "data": {"node_builder": {"_target_": T + "nodes.LatLonNodes", "latitudes": lat, "longitudes": lon}},
            "hidden": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": 5}},
        },
        "edges": [
            {"source_name": "data", "target_name": "hidden", "attributes": weights,
             "edge_builders": [{"_target_": T + "edges.KNNEdges", "num_nearest_neighbours": 4}]},
            {"source_name": "hidden", "target_name": "data",
             "edge_builders": [{"_target_": T + "edges.CutOffEdges", "cutoff_factor": 0.6}]},
        ],
    }  # fmt: skip


def build(resident: bool):
    from anemoi_graphs_b200 import device
    from anemoi_graphs_b200.create import GraphCreator

    prev = device.set_resident(resident)
    try:
        return GraphCreator(_recipe()).create()
    finally:
        device.set_resident(prev)


@pytest.fixture(scope="module")
def graphs():
    return {"device": build(True), "host": build(False)}


@pytest.mark.gpu
def test_knn_gaussian_weights_matrix(graphs):
    from anemoi_graphs_b200.export import edge_set_to_sparse

    key = ("data", "to", "hidden")
    results = {}
    for where, g in graphs.items():
        assert g[key].edge_index.is_cuda == (where == "device")
        m = edge_set_to_sparse(g, key, "w")
        assert tuple(m.shape) == (g["hidden"].num_nodes, g["data"].num_nodes) == (10242, 40320)
        got = as_arrays(m)
        again = as_arrays(edge_set_to_sparse(g, key, "w"))
        assert all(a.tobytes() == b.tobytes() for a, b in zip(got, again))  # two calls, bit-identical
        ei = g[key].edge_index.cpu().numpy()
        w = g[key]["w"].cpu().numpy().reshape(-1)
        assert w.dtype == np.float32
        ref = scipy_csr(ei, w, tuple(m.shape))
        assert_csr_equal(got, (ref.indptr, ref.indices, ref.data))
        assert (np.diff(got[0]) == 4).all()
        row_sums = np.add.reduceat(got[2].astype(np.float64), got[0][:-1])
        np.testing.assert_allclose(row_sums, 1.0, rtol=0, atol=4 * 2.0**-24)
        results[where] = got
    assert all(a.tobytes() == b.tobytes() for a, b in zip(results["device"][1:], results["host"][1:]))
    np.testing.assert_array_equal(results["device"][0], results["host"][0])


@pytest.mark.gpu
def test_cutoff_matrix_of_ones_equals_adjacency_matrix(graphs):
    from anemoi_graphs_b200.edges import CutOffEdges
    from anemoi_graphs_b200.export import edge_set_to_sparse

    key = ("hidden", "to", "data")
    results = {}
    for where, g in graphs.items():
        got = as_arrays(edge_set_to_sparse(g, key))
        assert got[2].dtype == np.float32 and (got[2] == 1.0).all()
        ei = g[key].edge_index.cpu().numpy()
        ref = scipy_csr(ei, np.ones(ei.shape[1], dtype=np.float32), (g["data"].num_nodes, g["hidden"].num_nodes))
        assert_csr_equal(got, (ref.indptr, ref.indices, ref.data))
        builder = CutOffEdges("hidden", "data", cutoff_factor=0.6)
        adj = builder.get_adjacency_matrix(*builder.prepare_node_data(g)).tocsr()  # prepare_node_data sets the radius
        np.testing.assert_array_equal(got[0], adj.indptr)
        np.testing.assert_array_equal(got[1], adj.indices)
        np.testing.assert_array_equal(got[2], adj.data)
        results[where] = got
    for a, b in zip(results["device"], results["host"]):
        np.testing.assert_array_equal(a, b)


@pytest.mark.gpu
def test_export_to_sparse_command_round_trip(tmp_path):
    from scipy.sparse import load_npz

    from anemoi_graphs_b200.__main__ import main
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.describe import load_graph

    pt = tmp_path / "graph.pt"
    GraphCreator(_recipe()).create(save_path=pt)
    g = load_graph(pt)
    out = tmp_path / "out"
    with pytest.warns(UserWarning, match=r"without the attribute 'w'.*\('hidden', 'to', 'data'\)"):
        assert main(["export_to_sparse", str(pt), str(out), "--edges-attribute-name", "w"]) == 0
    assert sorted(p.name for p in out.iterdir()) == ["data_to_hidden.npz"]
    key = ("data", "to", "hidden")
    m = load_npz(out / "data_to_hidden.npz")
    ref = scipy_csr(g[key].edge_index.numpy(), g[key]["w"].numpy().reshape(-1), (10242, 40320))
    assert m.shape == ref.shape and m.dtype == np.float32
    assert_csr_equal((m.indptr, m.indices, m.data), (ref.indptr, ref.indices, ref.data))

    out2 = tmp_path / "ones"
    assert main(["export_to_sparse", str(pt), str(out2), "--edges-name", "hidden", "data", "--edges-name", "data", "hidden"]) == 0
    assert sorted(p.name for p in out2.iterdir()) == ["data_to_hidden.npz", "hidden_to_data.npz"]
    for key in (("data", "to", "hidden"), ("hidden", "to", "data")):
        m = load_npz(out2 / f"{key[0]}_to_{key[2]}.npz")
        ei = g[key].edge_index.numpy()
        ref = scipy_csr(ei, np.ones(ei.shape[1], dtype=np.float32), (g[key[2]].num_nodes, g[key[0]].num_nodes))
        assert_csr_equal((m.indptr, m.indices, m.data), (ref.indptr, ref.indices, ref.data))
    with pytest.raises(KeyError, match="nowhere"):
        main(["export_to_sparse", str(pt), str(tmp_path / "none"), "--edges-name", "data", "nowhere"])


@pytest.mark.gpu
def test_exporter_on_device_resident_graph(graphs, tmp_path):
    from scipy.sparse import load_npz

    from anemoi_graphs_b200.export import GraphExporter

    paths = GraphExporter(graphs["device"], tmp_path, edges_name=[("data", "hidden")], edge_attribute_name="w").export()
    assert paths == [tmp_path / "data_to_hidden.npz"]
    m = load_npz(paths[0])
    key = ("data", "to", "hidden")
    ref = scipy_csr(graphs["host"][key].edge_index.numpy(), graphs["host"][key]["w"].numpy().reshape(-1), (10242, 40320))
    assert_csr_equal((m.indptr, m.indices, m.data), (ref.indptr, ref.indices, ref.data))


@pytest.mark.gpu
def test_bool_attribute_matrix():
    from anemoi_graphs_b200.export import edge_set_to_sparse

    rng = np.random.default_rng(5)
    ei = with_duplicates(rng, 300, 200, 5000, 800, 4, np.arange(150))
    mask = (rng.random((ei.shape[1], 1)) < 0.5)
    g = host_graph(coords(300, 1), coords(200, 2), ei, {"m": mask})
    for graph in (g, on_device(g)):
        got = as_arrays(edge_set_to_sparse(graph, KEY, "m"))
        ref = scipy_csr(ei, mask.reshape(-1), (200, 300))
        assert got[2].dtype == np.bool_
        assert_csr_equal(got, (ref.indptr, ref.indices, ref.data))
