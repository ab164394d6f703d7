"""Edge post-processors: RestrictEdgeLength, SortEdgeIndexBySourceNodes, SortEdgeIndexByTargetNodes.

* RestrictEdgeLength keeps exactly the edges the cut-off search (``NeighbourIndex.radius``, CutOffEdges' kernel) finds
  at the same radius, in input order, and agrees with a numpy float64 haversine away from the threshold;
* the sorts equal numpy's (stable) ``lexsort`` on (possibly negated) keys, ``SortEdgeIndexByTargetNodes(False)``
  equals ``ref_path.canonical_sort``;
* every per-edge tensor comes back byte-identical to ``t[index]`` with its dtype, on the device it was on;
* invalid endpoints raise ``ValueError`` with the graph unchanged; sharded blocks raise ``NotImplementedError``;
* the three processors run from a recipe's ``post_processors`` through ``GraphCreator.create``.
"""

import math

import numpy as np
import pytest
import torch

from anemoi_graphs_b200 import EARTH_RADIUS, grids
from oracle import ref_path as R

T = "anemoi.graphs."
TAU = 2.0**-40


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def x_deg(lat, lon) -> np.ndarray:
    return grids.latlon_deg_to_x(np.asarray(lat, dtype=np.float64), np.asarray(lon, dtype=np.float64)).numpy()


def clustered(n_top: int, n_mid: int, n_leaf: int, seed: int) -> np.ndarray:
    """3-level clustered cloud (as in test_gpu_search_paths): centres, sub-centres within 0.2 rad, leaves within 3e-3."""
    rng = np.random.default_rng(seed)
    lat, lon = grids.uniform_sphere(n_top, seed=seed)
    c = R.latlon_rad_to_cartesian((np.deg2rad(lat), np.deg2rad(lon)), 1.0).astype(np.float64)
    pts = []
    for p in c:
        for _ in range(n_mid):
            s = p + rng.normal(scale=0.2, size=3)
            s /= np.linalg.norm(s)
            pts.append(s + rng.normal(scale=3e-3, size=(n_leaf, 3)))
    xyz = np.concatenate(pts)
    xyz /= np.linalg.norm(xyz, axis=1, keepdims=True)
    return np.stack([np.arcsin(np.clip(xyz[:, 2], -1, 1)), np.arctan2(xyz[:, 1], xyz[:, 0])], axis=1).astype(np.float32)


def make_graph(src_x, dst_x, edge_index, attrs=None, key=("src", "to", "dst")):
    from anemoi_graphs_b200.graph import HeteroData

    g = HeteroData()
    g[key[0]].x = torch.as_tensor(src_x)
    if key[2] != key[0]:
        g[key[2]].x = torch.as_tensor(dst_x)
    g[key].edge_index = torch.as_tensor(edge_index)
    g[key].edge_type = "Test"
    for name, value in (attrs or {}).items():
        g[key][name] = value
    return g


def snapshot(graph):
    """The public entries of every edge store (private ``_`` entries are caches)."""
    return {
        k: {n: (v.clone() if isinstance(v, torch.Tensor) else v) for n, v in graph[k].items() if not n.startswith("_")}
        for k in graph.edge_types
    }


def assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].keys() == b[k].keys()
        for n in a[k]:
            if isinstance(a[k][n], torch.Tensor):
                assert a[k][n].dtype == b[k][n].dtype and a[k][n].device == b[k][n].device
                assert a[k][n].cpu().numpy().tobytes() == b[k][n].cpu().numpy().tobytes(), (k, n)


def col_keys(ei, n_dst):
    ei = np.asarray(ei, dtype=np.int64)
    return ei[0] * n_dst + ei[1]


# ------------------------------------------------------------------------------------------------
# no GPU: constructors and recipe resolution
# ------------------------------------------------------------------------------------------------
def test_constructor_validation():
    from anemoi_graphs_b200.processors import RestrictEdgeLength, SortEdgeIndexBySourceNodes, SortEdgeIndexByTargetNodes

    for bad in (0, -1.0, "10", None):
        with pytest.raises(AssertionError):
            RestrictEdgeLength("a", "b", bad)
    p = RestrictEdgeLength("a", "b", 100, source_mask_attr_name="m")
    assert (p.max_length_km, p.source_mask_attr_name, p.target_mask_attr_name) == (100, "m", None)
    assert RestrictEdgeLength("a", "b", 2.5).max_length_km == 2.5
    for cls in (SortEdgeIndexBySourceNodes, SortEdgeIndexByTargetNodes):
        assert cls().descending is True
        assert cls(descending=False).descending is False
        with pytest.raises(AssertionError):
            cls(descending=1)


def test_recipe_resolves_the_processors():
    from anemoi_graphs_b200 import processors
    from anemoi_graphs_b200.config import resolve_target
    from anemoi_graphs_b200.create import GraphCreator

    names = ("RestrictEdgeLength", "SortEdgeIndexBySourceNodes", "SortEdgeIndexByTargetNodes")
    for name in names:
        assert resolve_target(T + "processors." + name) is getattr(processors, name)
    cfg = {
        "nodes": {},
        "edges": [],
        "post_processors": [
            {"_target_": T + "processors.RestrictEdgeLength", "source_name": "a", "target_name": "b", "max_length_km": 50},
            {"_target_": T + "processors.SortEdgeIndexBySourceNodes"},
            {"_target_": T + "processors.SortEdgeIndexByTargetNodes", "descending": False},
        ],
    }
    GraphCreator(cfg)  # _validate resolves every _target_


# ------------------------------------------------------------------------------------------------
# RestrictEdgeLength: parity with the cut-off search
# ------------------------------------------------------------------------------------------------
def _on_threshold_radius(lon0: float):
    """(r_km, radius): radius = r_km / EARTH_RADIUS is a float32 whose half has the same sin on the device and in the C
    library - references at longitude +-radius on the equator sit exactly on the threshold of a query at (0, 0)."""
    lon = np.float32(lon0)
    for _ in range(1000):
        r_km = float(lon) * EARTH_RADIUS
        radius = r_km / EARTH_RADIUS
        if radius == float(lon):
            half = 0.5 * radius
            if torch.sin(torch.tensor([half], dtype=torch.float64, device="cuda")).item() == math.sin(half):
                return r_km, radius
        lon = np.nextafter(lon, np.float32(1.0))
    pytest.skip("no representable threshold radius found")


@pytest.fixture(scope="module")
def clouds():
    base = x_deg(*grids.uniform_sphere(4000, seed=5))
    return {"uniform": base, "clustered": clustered(6, 8, 60, seed=9)}


@pytest.mark.gpu
@pytest.mark.parametrize("cloud", ["uniform", "clustered"])
def test_restrict_matches_cutoff_search(clouds, cloud):
    from anemoi_graphs_b200 import ops
    from anemoi_graphs_b200.processors import RestrictEdgeLength

    r_on, rad_on = _on_threshold_radius(0.02)
    ref = clouds[cloud]
    pairs = np.array([[0.0, rad_on], [0.0, -rad_on]], dtype=np.float32)
    src_x = np.concatenate([ref, pairs])
    dst_x = np.concatenate([ref[::3] + np.float32(1e-3), np.zeros((1, 2), dtype=np.float32)])  # no zero-length edges
    n_src, n_dst = src_x.shape[0], dst_x.shape[0]
    with ops.NeighbourIndex(dev(src_x), hint_k=16) as ix:
        knn = ix.knn(dev(dst_x), 16).cpu().numpy()
    rd = R.rdist64(dst_x[knn[1], 0], dst_x[knn[1], 1], src_x[knn[0], 0], src_x[knn[0], 1])
    below = 1e-3  # km: shorter than every edge of these clouds
    assert rd.min() > math.sin(0.5 * below / EARTH_RADIUS) ** 2
    for r_km in (below, r_on, 400.0, 3000.0, 30000.0):
        radius = r_km / EARTH_RADIUS
        with ops.NeighbourIndex(dev(src_x), hint_radius=radius) as ix:
            cut = ix.radius(dev(dst_x), radius).cpu().numpy()
        want = knn[:, np.isin(col_keys(knn, n_dst), col_keys(cut, n_dst))]
        g = make_graph(src_x, dst_x, knn.copy(), {"pos": torch.arange(knn.shape[1])})
        g = RestrictEdgeLength("src", "dst", r_km).update_graph(g)
        got = g[("src", "to", "dst")].edge_index
        assert got.dtype == torch.int32 and not got.is_cuda
        np.testing.assert_array_equal(got.numpy(), want)
        pos = g[("src", "to", "dst")]["pos"].numpy()
        np.testing.assert_array_equal(knn[:, pos], want)  # input order kept
        assert (np.diff(pos) > 0).all()
        # numpy float64 away from the threshold
        thr = math.sin(0.5 * min(radius, math.pi)) ** 2
        clear = np.abs(rd - thr) > TAU * thr
        kept = np.zeros(knn.shape[1], dtype=bool)
        kept[pos] = True
        np.testing.assert_array_equal(kept[clear], (rd <= thr)[clear])
        if r_km == below:
            assert pos.size == 0
        if r_km == r_on:
            on = (knn[1] == n_dst - 1) & (knn[0] >= n_src - 2)
            assert on.sum() == 2 and kept[on].all()  # exactly at the limit: kept
            assert (~kept).any()
        if r_km == 30000.0:
            assert kept.all()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["flat", "column"])
def test_restrict_masks(clouds, shape):
    from anemoi_graphs_b200 import ops
    from anemoi_graphs_b200.processors import RestrictEdgeLength

    src_x = clouds["uniform"]
    dst_x = src_x[1::2]
    with ops.NeighbourIndex(dev(src_x), hint_k=16) as ix:
        knn = ix.knn(dev(dst_x), 16).cpu().numpy()
    rng = np.random.default_rng(3)
    sm = rng.random(src_x.shape[0]) < 0.5
    tm = rng.random(dst_x.shape[0]) < 0.5
    r_km = 600.0
    thr = math.sin(0.5 * r_km / EARTH_RADIUS) ** 2
    rd = R.rdist64(dst_x[knn[1], 0], dst_x[knn[1], 1], src_x[knn[0], 0], src_x[knn[0], 1])
    assert (np.abs(rd - thr) > TAU * thr).all()
    long = rd > thr
    assert 0 < long.sum() < long.size
    as_attr = (lambda m: torch.from_numpy(m)) if shape == "flat" else (lambda m: torch.from_numpy(m[:, None]))
    for use_s, use_t in ((True, False), (False, True), (True, True)):
        g = make_graph(src_x, dst_x, knn.copy())
        g["src"]["sm"] = as_attr(sm)
        g["dst"]["tm"] = as_attr(tm)
        p = RestrictEdgeLength("src", "dst", r_km, "sm" if use_s else None, "tm" if use_t else None)
        g = p.update_graph(g)
        subject = (sm[knn[0]] if use_s else True) & (tm[knn[1]] if use_t else True)
        np.testing.assert_array_equal(g[("src", "to", "dst")].edge_index.numpy(), knn[:, ~(subject & long)])
    for bad in (torch.from_numpy(sm.astype(np.uint8)), torch.from_numpy(sm.astype(np.float32)),
                torch.from_numpy(np.stack([sm, sm], axis=1)), torch.from_numpy(sm[:-1])):  # fmt: skip
        g = make_graph(src_x, dst_x, knn.copy())
        g["src"]["sm"] = bad
        before = snapshot(g)
        with pytest.raises(ValueError, match="sm"):
            RestrictEdgeLength("src", "dst", r_km, source_mask_attr_name="sm").update_graph(g)
        assert_same(before, snapshot(g))


# ------------------------------------------------------------------------------------------------
# sorting
# ------------------------------------------------------------------------------------------------
def _random_edges(n_edges, n_src, n_dst, seed):
    """Endpoints over the whole node range and, for a third of the columns, from a small range (duplicates)."""
    rng = np.random.default_rng(seed)
    ei = np.stack([rng.integers(0, n_src, n_edges), rng.integers(0, n_dst, n_edges)]).astype(np.int32)
    dup = rng.random(n_edges) < 0.34
    ei[0, dup] = rng.integers(0, min(n_src, 3), int(dup.sum()))
    ei[1, dup] = rng.integers(0, min(n_dst, 3), int(dup.sum()))
    return ei


def _lexsort_order(ei, key_row, descending):
    k, o = ei[key_row].astype(np.int64), ei[1 - key_row].astype(np.int64)
    return np.lexsort((-o, -k)) if descending else np.lexsort((o, k))


SORT_CASES = [
    (0, 5, 7),
    (1, 1, 1),
    (1023, 1, 2**10),
    (1025, 2**10 + 1, 2**10),
    (5000, 2**16, 2**25 + 1),  # the other row leaves < 8 unused bits: one pass over every key bit
    (2**21 + 5, 2**20 + 1, 2**12),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n_edges,n_src,n_dst", SORT_CASES)
def test_sort_matches_lexsort(n_edges, n_src, n_dst):
    from anemoi_graphs_b200.processors import SortEdgeIndexBySourceNodes, SortEdgeIndexByTargetNodes

    ei = _random_edges(n_edges, n_src, n_dst, seed=n_edges)
    src_x, dst_x = torch.zeros((n_src, 2)), torch.zeros((n_dst, 2))
    for cls, key_row in ((SortEdgeIndexBySourceNodes, 0), (SortEdgeIndexByTargetNodes, 1)):
        for descending in (False, True):
            g = make_graph(src_x, dst_x, torch.from_numpy(ei), {"pos": torch.arange(n_edges, dtype=torch.int64)})
            g = cls(descending=descending).update_graph(g)
            order = _lexsort_order(ei, key_row, descending)
            store = g[("src", "to", "dst")]
            np.testing.assert_array_equal(store["pos"].numpy(), order)  # stable: duplicates keep their input order
            np.testing.assert_array_equal(store.edge_index.numpy(), ei[:, order])
            assert store.edge_type == "Test"


@pytest.mark.gpu
def test_sort_by_target_ascending_is_canonical(clouds):
    """``SortEdgeIndexByTargetNodes(False)`` = ``R.canonical_sort``; attributes as tests/test_gpu_builders.py's
    ``by_canonical_order`` (attribute[np.lexsort((ei[0], ei[1]))]) returns them."""
    from anemoi_graphs_b200 import ops
    from anemoi_graphs_b200.processors import SortEdgeIndexByTargetNodes

    src_x = clouds["clustered"]
    dst_x = clouds["uniform"][:1500]
    radius = 0.05
    with ops.NeighbourIndex(dev(src_x), hint_radius=radius) as ix:
        cut = ix.radius(dev(dst_x), radius).cpu().numpy()
    assert cut.shape[1] > 1000
    length = torch.from_numpy(np.random.default_rng(1).random((cut.shape[1], 1)).astype(np.float32))
    for on_gpu in (False, True):
        g = make_graph(src_x, dst_x, cut.copy(), {"edge_length": length.clone()})
        if on_gpu:
            for k in ("src", "dst"):
                g[k].x = g[k].x.cuda()
            store = g[("src", "to", "dst")]
            store.edge_index, store["edge_length"] = store.edge_index.cuda(), store["edge_length"].cuda()
        g = SortEdgeIndexByTargetNodes(descending=False).update_graph(g)
        store = g[("src", "to", "dst")]
        assert store.edge_index.is_cuda == on_gpu and store["edge_length"].is_cuda == on_gpu
        np.testing.assert_array_equal(store.edge_index.cpu().numpy(), R.canonical_sort(cut))
        np.testing.assert_array_equal(store["edge_length"].cpu().numpy(), length.numpy()[np.lexsort((cut[0], cut[1]))])


# ------------------------------------------------------------------------------------------------
# the gather: every width, both index dtypes, CPU and CUDA graphs
# ------------------------------------------------------------------------------------------------
def _attr_zoo(n_edges, seed):
    rng = np.random.default_rng(seed)
    f = lambda *s: rng.normal(size=(n_edges, *s))  # noqa: E731
    wide = torch.from_numpy(f(4).astype(np.float32))
    h = f(3).astype(np.float16)
    h[::7, 1] = np.nan
    return {
        "f16_3": torch.from_numpy(h),
        "f32_1": torch.from_numpy(f(1).astype(np.float32)),
        "f32_2": torch.from_numpy(f(2).astype(np.float32)),
        "f64_1": torch.from_numpy(f(1)),
        "f64_flat": torch.from_numpy(f()),
        "bool_1": torch.from_numpy(rng.random((n_edges, 1)) < 0.5),
        "bool_3": torch.from_numpy(rng.random((n_edges, 3)) < 0.5),
        "i64_3": torch.from_numpy(rng.integers(-(2**62), 2**62, size=(n_edges, 3))),
        "u8_5": torch.from_numpy(rng.integers(0, 256, size=(n_edges, 5)).astype(np.uint8)),
        "i16_1": torch.from_numpy(rng.integers(-(2**15), 2**15, size=(n_edges, 1)).astype(np.int16)),
        "view": wide[:, ::2],  # non-contiguous
    }


@pytest.mark.gpu
@pytest.mark.parametrize("on_gpu", [False, True])
@pytest.mark.parametrize("index_dtype", [torch.int32, torch.int64])
def test_gather_widths(clouds, on_gpu, index_dtype):
    from anemoi_graphs_b200 import ops
    from anemoi_graphs_b200.processors import RestrictEdgeLength, SortEdgeIndexBySourceNodes

    src_x = clouds["uniform"]
    dst_x = src_x[::2]
    with ops.NeighbourIndex(dev(src_x), hint_k=7) as ix:
        knn = ix.knn(dev(dst_x), 7).cpu().numpy()
    n_edges = knn.shape[1]
    zoo = _attr_zoo(n_edges, seed=4)
    assert not zoo["view"].is_contiguous()
    rd = R.rdist64(dst_x[knn[1], 0], dst_x[knn[1], 1], src_x[knn[0], 0], src_x[knn[0], 1])
    r_km = 500.0
    thr = math.sin(0.5 * r_km / EARTH_RADIUS) ** 2
    assert (np.abs(rd - thr) > TAU * thr).all()
    cases = (
        (SortEdgeIndexBySourceNodes(descending=True), _lexsort_order(knn, 0, True)),
        (RestrictEdgeLength("src", "dst", r_km), np.nonzero(rd <= thr)[0]),
    )
    for proc, index in cases:
        assert 0 < index.size
        move = (lambda t: t.cuda()) if on_gpu else (lambda t: t)
        attrs = {k: move(v) for k, v in zoo.items()}
        g = make_graph(move(torch.from_numpy(src_x)), move(torch.from_numpy(dst_x)), move(torch.from_numpy(knn).to(index_dtype)), attrs)
        g = proc.update_graph(g)
        store = g[("src", "to", "dst")]
        assert store.edge_index.dtype == index_dtype and store.edge_index.is_cuda == on_gpu
        np.testing.assert_array_equal(store.edge_index.cpu().numpy(), knn[:, index])
        for name, t in zoo.items():
            got = store[name]
            assert got.dtype == t.dtype and got.shape == (index.size, *t.shape[1:]) and got.is_cuda == on_gpu, name
            assert got.cpu().numpy().tobytes() == t[torch.from_numpy(index)].numpy().tobytes(), name
        assert store.edge_type == "Test"


# ------------------------------------------------------------------------------------------------
# errors
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["source", "target", "negative"])
def test_out_of_range_endpoint_leaves_the_graph_unchanged(bad):
    from anemoi_graphs_b200.processors import RestrictEdgeLength, SortEdgeIndexBySourceNodes, SortEdgeIndexByTargetNodes

    src_x = x_deg(*grids.uniform_sphere(300, seed=1))
    dst_x = x_deg(*grids.uniform_sphere(200, seed=2))
    good = _random_edges(2000, 300, 200, seed=7)
    wrong = _random_edges(3000, 300, 200, seed=8)
    if bad == "source":
        wrong[0, 1777] = 300
    elif bad == "target":
        wrong[1, 5] = 200
    else:
        wrong[1, 2999] = -1
    g = make_graph(src_x, dst_x, good, {"a": torch.arange(2000.0)}, key=("src", "to", "dst"))
    g[("dst", "to", "src")].edge_index = torch.from_numpy(np.ascontiguousarray(wrong[::-1]))
    g[("dst", "to", "src")]["a"] = torch.arange(3000.0)
    g[("src", "to", "src")].edge_index = torch.from_numpy(np.ascontiguousarray(wrong) if bad == "source" else good[:, :0])
    before = snapshot(g)
    for proc in (SortEdgeIndexBySourceNodes(), SortEdgeIndexByTargetNodes(descending=False),
                 RestrictEdgeLength("dst", "src", 100.0)):  # fmt: skip
        with pytest.raises(ValueError, match="outside"):
            proc.update_graph(g)
        assert_same(before, snapshot(g))
    with pytest.raises(ValueError, match="no edge set"):
        RestrictEdgeLength("src", "nowhere", 100.0).update_graph(g)
    assert ("src", "to", "nowhere") not in g.edge_types


@pytest.mark.gpu
def test_sharded_store_is_refused():
    from anemoi_graphs_b200.processors import RestrictEdgeLength, SortEdgeIndexByTargetNodes

    x = x_deg(*grids.uniform_sphere(100, seed=3))
    g = make_graph(x, x, _random_edges(500, 100, 100, seed=1), key=("n", "to", "n"))
    g[("n", "to", "n")]["edge_shard"] = {"rank": 0, "world": 2, "counts": [500, 500], "replicated": False}
    before = snapshot(g)
    for proc in (RestrictEdgeLength("n", "n", 100.0), SortEdgeIndexByTargetNodes()):
        with pytest.raises(NotImplementedError, match="gather"):
            proc.update_graph(g)
    assert_same(before, snapshot(g))


@pytest.mark.gpu
@pytest.mark.parametrize("n_edges", [0, 1])
def test_empty_and_tiny_edge_sets(n_edges):
    from anemoi_graphs_b200.processors import RestrictEdgeLength, SortEdgeIndexBySourceNodes

    x = np.array([[0.0, 0.0], [0.0, 0.1]], dtype=np.float32)
    ei = np.array([[1], [0]], dtype=np.int32)[:, :n_edges]
    for proc in (RestrictEdgeLength("n", "n", 1.0), RestrictEdgeLength("n", "n", 1e4), SortEdgeIndexBySourceNodes()):
        g = make_graph(x, x, ei.copy(), {"w": torch.ones((n_edges, 2), dtype=torch.float16)}, key=("n", "to", "n"))
        g = proc.update_graph(g)
        store = g[("n", "to", "n")]
        keep_all = not (isinstance(proc, RestrictEdgeLength) and proc.max_length_km == 1.0)
        m = n_edges if keep_all else 0
        assert store.edge_index.shape == (2, m) and store["w"].shape == (m, 2) and store["w"].dtype == torch.float16


# ------------------------------------------------------------------------------------------------
# recipe route: a reduced limited-area (config 4) recipe through GraphCreator.create
# ------------------------------------------------------------------------------------------------
class _CutoutDataset:
    def __init__(self, lat, lon, grids_):
        self.latitudes, self.longitudes, self.grids = lat, lon, grids_


MAX_KM = 150.0


def _recipe(post: bool) -> dict:
    attrs = {
        "edge_length": {"_target_": T + "edges.attributes.EdgeLength", "norm": "unit-max"},
        "edge_dirs": {"_target_": T + "edges.attributes.EdgeDirection", "norm": "unit-std"},
    }
    cfg = {
        "nodes": {
            "data": {"node_builder": {"_target_": T + "nodes.ZarrDatasetNodes", "dataset": {"cutout": ["lam", "global"]}},
                     "attributes": {"cutout": {"_target_": T + "nodes.attributes.CutOutMask"},
                                    "global": {"_target_": T + "nodes.attributes.BooleanNot", "masks": "cutout"}}},
            "tri": {"node_builder": {"_target_": T + "nodes.StretchedTriNodes", "global_resolution": 3, "lam_resolution": 6,
                                     "reference_node_name": "data", "mask_attr_name": "cutout", "margin_radius_km": 100.0}},
        },
        "edges": [
            {"source_name": "data", "target_name": "tri", "attributes": attrs,
             "edge_builders": [{"_target_": T + "edges.CutOffEdges", "cutoff_factor": 0.05}]},
            {"source_name": "tri", "target_name": "tri", "attributes": attrs,
             "edge_builders": [{"_target_": T + "edges.MultiScaleEdges", "x_hops": 1}]},
            {"source_name": "tri", "target_name": "data", "attributes": attrs,
             "edge_builders": [{"_target_": T + "edges.KNNEdges", "num_nearest_neighbours": 3, "target_mask_attr_name": "cutout"},
                               {"_target_": T + "edges.KNNEdges", "num_nearest_neighbours": 1}]},
        ],
    }  # fmt: skip
    if post:
        cfg["post_processors"] = [
            {"_target_": T + "processors.RestrictEdgeLength", "source_name": "tri", "target_name": "data",
             "max_length_km": MAX_KM, "target_mask_attr_name": "global"},
            {"_target_": T + "processors.RemoveUnconnectedNodes", "nodes_name": "data"},
            {"_target_": T + "processors.SortEdgeIndexByTargetNodes"},
        ]  # fmt: skip
    return cfg


@pytest.mark.gpu
def test_recipe_route_matches_numpy(monkeypatch):
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.nodes.builders import from_file

    lam_lat, lam_lon = grids.lam_patch(96, 96, 5.0)
    glob_lat, glob_lon = grids.octahedral_grid(24)
    ds = _CutoutDataset(np.concatenate([lam_lat, glob_lat]), np.concatenate([lam_lon, glob_lon]), (lam_lat.size, glob_lat.size))
    monkeypatch.setattr(from_file, "open_dataset", lambda *a, **k: ds)

    plain = GraphCreator(_recipe(False)).create()
    got = GraphCreator(_recipe(True)).create()

    # 1. RestrictEdgeLength on tri -> data, only edges into global points
    dx, tx = plain["data"].x.numpy(), plain["tri"].x.numpy()
    glob = plain["data"]["global"].numpy()[:, 0]
    want = {k: {n: plain[k][n].numpy() for n in plain[k].edge_attrs()} for k in plain.edge_types}
    dec = want[("tri", "to", "data")]
    ei = dec["edge_index"]
    rd = R.rdist64(dx[ei[1], 0], dx[ei[1], 1], tx[ei[0], 0], tx[ei[0], 1])
    thr = math.sin(0.5 * MAX_KM / EARTH_RADIUS) ** 2
    assert (np.abs(rd - thr) > TAU * thr).all()
    keep = ~glob[ei[1]] | (rd <= thr)
    assert 0 < (~keep).sum() and keep.sum() > 0
    for n in dec:
        dec[n] = dec[n][:, keep] if n == "edge_index" else dec[n][keep]
    # 2. RemoveUnconnectedNodes on data
    mask = np.zeros(dx.shape[0], dtype=bool)
    for (s, _, t), arrays in want.items():
        if s == "data":
            mask[arrays["edge_index"][0]] = True
        if t == "data":
            mask[arrays["edge_index"][1]] = True
    assert (~mask).any()
    new_index = np.cumsum(mask) - 1
    for (s, _, t), arrays in want.items():
        if s == "data":
            arrays["edge_index"][0] = new_index[arrays["edge_index"][0]]
        if t == "data":
            arrays["edge_index"][1] = new_index[arrays["edge_index"][1]]
    # 3. SortEdgeIndexByTargetNodes (descending by default)
    for arrays in want.values():
        order = _lexsort_order(arrays["edge_index"], 1, True)
        for n in arrays:
            arrays[n] = arrays[n][:, order] if n == "edge_index" else arrays[n][order]

    np.testing.assert_array_equal(got["data"].x.numpy().view(np.int32), dx[mask].view(np.int32))
    np.testing.assert_array_equal(got["data"]["global"].numpy()[:, 0], glob[mask])
    assert sorted(got.edge_types) == sorted(want)
    for key, arrays in want.items():
        assert sorted(got[key].edge_attrs()) == sorted(arrays)
        for n, value in arrays.items():
            assert got[key][n].dtype == plain[key][n].dtype
            np.testing.assert_array_equal(got[key][n].numpy(), value, err_msg=f"{key} {n}")
