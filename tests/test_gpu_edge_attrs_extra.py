"""Edge attributes of newer anemoi-graphs releases: Azimuth, GaussianDistanceWeights, AttributeFromSourceNode and
AttributeFromTargetNode.

* Azimuth agrees with the float64 numpy formula on adversarial edges (1e-6 rad modulo 2 pi; every norm);
* GaussianDistanceWeights(norm=None) is float32(exp(-L^2 / (2 sigma^2))) of the graph's own EdgeLength L (1 ulp); every
  norm agrees per target group with numpy (2 ulp) on KNN, cut-off, merged, sorted, huge-group and tiny edge lists and
  on each degenerate group; a permutation of the columns permutes the output, bytes equal;
* AttributeFrom*Node equals ``attr[edge_index[row]].bool()`` on host- and device-resident graphs;
* invalid endpoints raise ValueError, sharded blocks NotImplementedError, with the graph unchanged;
* a recipe through GraphCreator.create gives the same bits with and without the lazy node order, and leaves
  EdgeLength / EdgeDirection as they are without the new attributes.
"""

import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from anemoi_graphs_b200 import grids

T = "anemoi.graphs."
REPO = Path(__file__).resolve().parents[1]
NORMS = [None, "l1", "l2", "unit-max", "unit-range", "unit-std"]
KEY = ("src", "to", "dst")


# ------------------------------------------------------------------------------------------------
# float64 numpy references
# ------------------------------------------------------------------------------------------------
def ref_azimuth(src: np.ndarray, dst: np.ndarray) -> np.ndarray:
    """Bearing at the target (dst rows) towards the source (src rows), float64 from the float32 (lat, lon)."""
    ls, os_ = src[:, 0].astype(np.float64), src[:, 1].astype(np.float64)
    lt, ot = dst[:, 0].astype(np.float64), dst[:, 1].astype(np.float64)
    dl = os_ - ot
    return np.arctan2(np.sin(dl) * np.cos(ls), np.cos(lt) * np.sin(ls) - np.sin(lt) * np.cos(ls) * np.cos(dl))


def ref_norm(v: np.ndarray, norm):
    """normalise.py on a whole array (NaN propagates through sum / amax / amin / std)."""
    with np.errstate(all="ignore"):
        if norm is None:
            return v
        if norm == "l1":
            return v / np.sum(v)
        if norm == "l2":
            return v / np.linalg.norm(v)
        if norm == "unit-max":
            return v / np.amax(v)
        if norm == "unit-range":
            return (v - np.amin(v)) / (np.amax(v) - np.amin(v))
        std = np.std(v)
        return v if std == 0 else v / std


def ref_gaussian(lengths: np.ndarray, dst_row: np.ndarray, sigma: float, norm) -> np.ndarray:
    """float32 (E,) weights normalised per target group; bit-equal groups are left unnormalised under unit-std."""
    w = np.exp(-(lengths.astype(np.float64) ** 2) / (2 * sigma**2))
    out = np.empty_like(w)
    order = np.argsort(dst_row, kind="stable")
    ts = dst_row[order]
    starts = np.flatnonzero(np.r_[True, ts[1:] != ts[:-1]]) if ts.size else np.zeros(0, dtype=np.int64)
    ends = np.r_[starts[1:], ts.size]
    for a, b in zip(starts, ends):
        idx = order[a:b]
        g = w[idx]
        if norm == "unit-std" and np.all(g.view(np.int64) == g[0].view(np.int64)):
            out[idx] = g
        else:
            out[idx] = ref_norm(g, norm)
    return out.astype(np.float32)


def assert_ulp(got, want, ulps, msg=""):
    got, want = np.asarray(got, dtype=np.float32).ravel(), np.asarray(want, dtype=np.float32).ravel()
    assert got.shape == want.shape, msg
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=f"{msg}: NaN positions")
    g, w = got[~nan], want[~nan]
    np.testing.assert_array_equal(np.isposinf(g), np.isposinf(w), err_msg=f"{msg}: inf positions")
    np.testing.assert_array_equal(np.isneginf(g), np.isneginf(w), err_msg=f"{msg}: inf positions")
    g, w = np.where(np.isinf(w), 0, g), np.where(np.isinf(w), 0, w)
    tol = ulps * np.spacing(np.maximum(np.abs(g), np.abs(w)))
    bad = np.abs(g.astype(np.float64) - w.astype(np.float64)) > tol
    assert not bad.any(), f"{msg}: {bad.sum()} values off by more than {ulps} ulp, e.g. {g[bad][:4]} vs {w[bad][:4]}"


# ------------------------------------------------------------------------------------------------
# no GPU
# ------------------------------------------------------------------------------------------------
def test_constructor_validation():
    from anemoi_graphs_b200.edges.attributes import (
        AttributeFromSourceNode,
        AttributeFromTargetNode,
        Azimuth,
        GaussianDistanceWeights,
    )

    for bad in (0, -1, "1", None):
        with pytest.raises(AssertionError):
            GaussianDistanceWeights(sigma=bad)
    g = GaussianDistanceWeights()
    assert (g.sigma, g.norm) == (1.0, "l1")
    assert GaussianDistanceWeights(sigma=0.05, norm=None).norm is None
    for cls in (AttributeFromSourceNode, AttributeFromTargetNode):
        assert cls("mask").node_attr_name == "mask"
        with pytest.raises(AssertionError):
            cls(3)
    for make in (lambda n: Azimuth(norm=n), lambda n: GaussianDistanceWeights(norm=n)):
        with pytest.raises(ValueError, match="is not valid"):
            make("l3")
    assert Azimuth().norm is None


def test_recipe_resolves_the_attributes():
    from anemoi_graphs_b200.config import resolve_target
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.edges import attributes

    names = ("Azimuth", "GaussianDistanceWeights", "AttributeFromSourceNode", "AttributeFromTargetNode")
    for name in names:
        assert resolve_target(T + "edges.attributes." + name) is getattr(attributes, name)
    cfg = {"nodes": {}, "edges": [{"source_name": "a", "target_name": "b", "edge_builders": [],
                                   "attributes": {"az": {"_target_": T + "edges.attributes.Azimuth"},
                                                  "w": {"_target_": T + "edges.attributes.GaussianDistanceWeights"},
                                                  "m": {"_target_": T + "edges.attributes.AttributeFromSourceNode",
                                                        "node_attr_name": "cutout"}}}]}  # fmt: skip
    GraphCreator(cfg)  # _validate resolves every _target_


def test_reference_helpers_on_hand_cases():
    d = 1e-3
    dst = np.zeros((4, 2), dtype=np.float32)
    src = np.array([[d, 0.0], [0.0, d], [-d, 0.0], [0.0, -d]], dtype=np.float32)
    az = ref_azimuth(src, dst)
    np.testing.assert_allclose(az[[0, 1, 3]], [0.0, np.pi / 2, -np.pi / 2], atol=1e-12)
    assert abs(abs(az[2]) - np.pi) < 1e-12
    rng = np.random.default_rng(0)
    lengths = rng.random(500).astype(np.float32)
    dst_row = rng.integers(0, 40, 500)
    w = ref_gaussian(lengths, dst_row, 0.5, "l1").astype(np.float64)
    np.testing.assert_allclose(np.bincount(dst_row, weights=w, minlength=40)[np.unique(dst_row)], 1.0, rtol=1e-6)


def test_endpoint_check_on_hand_cases():
    from anemoi_graphs_b200.edges.attributes import _check_endpoints

    ei = torch.tensor([[0, 4, 2], [1, 0, 6]], dtype=torch.int32)
    _check_endpoints(ei, 5, 7)
    _check_endpoints(ei[:, :0], 0, 0)
    for n_src, n_dst, row, col, v in ((4, 7, 0, 0, 0), (5, 6, 0, 0, 0), (5, 7, 1, 2, -1), (5, 7, 0, 1, -3)):
        bad = ei.clone()
        bad[row, col] = v if v < 0 else bad[row, col]
        with pytest.raises(ValueError, match="outside"):
            _check_endpoints(bad, n_src, n_dst)


# ------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------
def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def f32(lat, lon) -> np.ndarray:
    return np.stack([np.asarray(lat, dtype=np.float64), np.asarray(lon, dtype=np.float64)], axis=1).astype(np.float32)


def wrap_pi(lon):
    return (np.asarray(lon) + np.pi) % (2 * np.pi) - np.pi


def destination(lat, lon, d, bearing):
    s = np.clip(np.sin(lat) * np.cos(d) + np.cos(lat) * np.sin(d) * np.cos(bearing), -1.0, 1.0)
    lat2 = np.arcsin(s)
    return lat2, lon + np.arctan2(np.sin(bearing) * np.sin(d) * np.cos(lat), np.cos(d) - np.sin(lat) * s)


def make_graph(src_x, dst_x, edge_index, on_gpu=False):
    from anemoi_graphs_b200.graph import HeteroData

    move = (lambda t: torch.as_tensor(t).cuda()) if on_gpu else torch.as_tensor
    g = HeteroData()
    g["src"].x = move(src_x)
    g["dst"].x = move(dst_x)
    g[KEY].edge_index = move(np.ascontiguousarray(edge_index))
    g[KEY].edge_type = "Test"
    return g


def snapshot(graph):
    return {k: {n: (v.clone() if isinstance(v, torch.Tensor) else v) for n, v in graph[k].items() if not n.startswith("_")}
            for k in (*graph.node_types, *graph.edge_types)}  # fmt: skip


def assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].keys() == b[k].keys(), k
        for n in a[k]:
            if isinstance(a[k][n], torch.Tensor):
                assert a[k][n].cpu().numpy().tobytes() == b[k][n].cpu().numpy().tobytes(), (k, n)


def compute(attr, g):
    out = attr.compute(g, KEY)
    return out.cpu().numpy()


def length_of(g):
    from anemoi_graphs_b200.edges.attributes import EdgeLength

    return compute(EdgeLength(), g)[:, 0]


# ------------------------------------------------------------------------------------------------
# Azimuth
# ------------------------------------------------------------------------------------------------
def azimuth_pairs(seed=21):
    rng = np.random.default_rng(seed)
    pairs = []

    def add(lat, lon, d, bearing):
        lat2, lon2 = destination(lat, lon, d, bearing)
        pairs.append((f32(lat2, wrap_pi(lon2)), f32(lat, lon)))  # (source, target)

    d = np.logspace(-7, np.log10(np.pi), 300)
    add(np.arcsin(rng.uniform(-1, 1, d.size)), rng.uniform(-np.pi, np.pi, d.size), d, rng.uniform(0, 2 * np.pi, d.size))
    for pole in (1.0, -1.0):  # targets at and near both poles
        for off in (0.0, 3e-6, 1e-3):
            m = 24
            add(np.full(m, pole * (np.pi / 2 - off)), rng.uniform(-np.pi, np.pi, m), np.logspace(-6, 0, m),
                rng.uniform(0, 2 * np.pi, m))  # fmt: skip
    m = 16  # the date line in both conventions, |dlon| > pi
    lat = rng.uniform(-1.2, 1.2, m)
    dl = np.logspace(-5, -0.5, m)
    pairs.append((f32(lat, np.pi - dl / 2), f32(lat + 1e-3, -np.pi + dl / 2)))
    pairs.append((f32(lat, dl / 2), f32(lat + 2e-3, 2 * np.pi - dl / 2)))
    pairs.append((f32(lat, -np.pi + dl), f32(lat, 2 * np.pi - dl)))
    m = 16  # near-antipodal
    add(np.arcsin(rng.uniform(-0.9, 0.9, m)), rng.uniform(-np.pi, np.pi, m), np.pi - np.logspace(-4, -1, m),
        rng.uniform(0, 2 * np.pi, m))  # fmt: skip
    src = np.concatenate([p[0] for p in pairs])
    dst = np.concatenate([p[1] for p in pairs])
    return src, dst


@pytest.mark.gpu
@pytest.mark.parametrize("on_gpu", [False, True])
def test_azimuth_matches_numpy(on_gpu):
    from anemoi_graphs_b200.edges.attributes import Azimuth

    src, dst = azimuth_pairs()
    coincident = f32(np.arcsin(np.linspace(-1, 1, 9)), np.linspace(-3, 3, 9))
    src, dst = np.concatenate([src, coincident]), np.concatenate([dst, coincident])
    n = src.shape[0]
    ei = np.stack([np.arange(n), np.arange(n)]).astype(np.int32)
    g = make_graph(src, dst, ei, on_gpu)
    raw = compute(Azimuth(), g)
    assert raw.dtype == np.float32 and raw.shape == (n, 1)
    raw = raw[:, 0].astype(np.float64)
    assert np.isfinite(raw).all() and (np.abs(raw) <= np.float32(np.pi)).all()
    ref = ref_azimuth(src, dst)
    moved = np.abs(wrap_pi(raw - ref))
    assert moved[:-9].max() <= 1e-6, moved[:-9].max()
    stored = raw.astype(np.float32).astype(np.float64)
    for norm in NORMS[1:]:
        got = compute(Azimuth(norm=norm), g)[:, 0].astype(np.float64)
        want = ref_norm(stored, norm)  # float64 statistics of the stored values, as for EdgeLength
        assert np.all(np.abs(got - want) <= 1e-6 * np.maximum(1.0, np.abs(want))), norm


# ------------------------------------------------------------------------------------------------
# GaussianDistanceWeights
# ------------------------------------------------------------------------------------------------
def _knn(src_x, dst_x, k):
    from anemoi_graphs_b200 import ops

    with ops.NeighbourIndex(dev(src_x), hint_k=k) as ix:
        return ix.knn(dev(dst_x), k).cpu().numpy()


def _cutoff(src_x, dst_x, radius):
    from anemoi_graphs_b200 import ops

    with ops.NeighbourIndex(dev(src_x), hint_radius=radius) as ix:
        return ix.radius(dev(dst_x), radius).cpu().numpy()


@pytest.fixture(scope="module")
def clouds():
    src = grids.latlon_deg_to_x(*grids.uniform_sphere(6000, seed=5)).numpy()
    dst = grids.latlon_deg_to_x(*grids.uniform_sphere(1500, seed=6)).numpy()
    return src, dst


def _edge_lists(clouds):
    """name -> (src_x, dst_x, edge_index)."""
    from anemoi_graphs_b200.processors import SortEdgeIndexBySourceNodes

    src, dst = clouds
    out = {f"knn{k}": (src, dst, _knn(src, dst, k)) for k in (1, 3, 7, 33, 64)}
    cut = _cutoff(src, dst, 0.06)
    dense = _cutoff(src, dst[:50], 0.5)
    assert np.bincount(dense[1]).max() > 320
    out["cutoff"] = (src, dst, cut)
    out["cutoff_dense"] = (src, dst[:50], dense)
    knn = out["knn3"][2]
    out["some_targets_empty"] = (src, dst, knn[:, knn[1] % 3 != 0])
    out["merged"] = (src, dst, np.unique(np.concatenate([knn, cut], axis=1), axis=1))
    g = make_graph(src, dst, cut.copy())
    g = SortEdgeIndexBySourceNodes().update_graph(g)
    out["source_sorted"] = (src, dst, g[KEY].edge_index.numpy())
    out["empty"] = (src, dst, np.zeros((2, 0), dtype=np.int32))
    out["single"] = (src, dst, np.array([[5], [7]], dtype=np.int32))
    return out


@pytest.fixture(scope="module")
def edge_lists(clouds):
    return _edge_lists(clouds)


@pytest.fixture(scope="module")
def huge_group():
    """Target 0 holds 2^21 edges, targets 1 and 2 a few, target 3 none."""
    rng = np.random.default_rng(8)
    n = 2**21
    src = grids.latlon_deg_to_x(*grids.uniform_sphere(n, seed=9)).numpy()
    dst = np.array([[0.3, 0.2], [-1.0, 2.0], [1.2, -2.5], [0.0, 0.0]], dtype=np.float32)
    ei = np.concatenate([np.stack([np.arange(n), np.zeros(n, dtype=np.int64)]),
                         np.stack([rng.integers(0, n, 40), rng.integers(1, 3, 40)])], axis=1).astype(np.int32)  # fmt: skip
    return src, dst, ei[:, rng.permutation(ei.shape[1])]


def _check_gaussian(src, dst, ei, sigmas=(1e-3, 0.05, 1.0), on_gpu=False, msg=""):
    from anemoi_graphs_b200.edges.attributes import GaussianDistanceWeights

    g = make_graph(src, dst, ei, on_gpu)
    L = length_of(g)
    for sigma in sigmas:
        raw = compute(GaussianDistanceWeights(sigma=sigma, norm=None), g)
        assert raw.shape == (ei.shape[1], 1) and raw.dtype == np.float32
        assert_ulp(raw, np.exp(-(L.astype(np.float64) ** 2) / (2 * sigma**2)), 1, f"{msg} sigma={sigma} raw")
        for norm in NORMS[1:]:
            got = compute(GaussianDistanceWeights(sigma=sigma, norm=norm), g)
            assert_ulp(got, ref_gaussian(L, ei[1], sigma, norm), 2, f"{msg} sigma={sigma} {norm}")


@pytest.mark.gpu
@pytest.mark.parametrize(
    "case",
    ["knn1", "knn3", "knn7", "knn33", "knn64", "cutoff", "cutoff_dense", "some_targets_empty", "merged",
     "source_sorted", "empty", "single"],
)  # fmt: skip
def test_gaussian_weights_match_numpy(edge_lists, case):
    src, dst, ei = edge_lists[case]
    _check_gaussian(src, dst, ei, msg=case)


@pytest.mark.gpu
def test_gaussian_weights_huge_group(huge_group):
    src, dst, ei = huge_group
    _check_gaussian(src, dst, ei, sigmas=(0.05, 1.0), on_gpu=True, msg="2^21")


@pytest.mark.gpu
def test_gaussian_degenerate_groups():
    from anemoi_graphs_b200.edges.attributes import GaussianDistanceWeights

    # target 0: one edge; 1: three duplicate columns (bit-equal weights); 2: one NaN (antipodal) among finite edges;
    # 3: long edges only (underflow at sigma = 1e-3); 4: ordinary
    rng = np.random.default_rng(3)
    lat = rng.uniform(-1.4, 1.4, 256)
    lon = rng.uniform(-np.pi, np.pi, 256)
    anti_s, anti_t = f32(lat, lon), f32(-lat, wrap_pi(lon + np.pi))
    from oracle import ref_path as R

    nan_at = np.flatnonzero(np.isnan(R.haversine_distance(anti_s, anti_t)))
    assert nan_at.size
    t_x = np.concatenate([f32([0.1, -0.4, 0.0, 0.7, -1.0], [0.2, 1.0, 0.0, -2.0, 0.5]), anti_t[nan_at[:1]]])
    s_x = f32([0.1, -0.4 + 1e-3, 0.0, 0.002, 0.7 + 0.3, -1.0 + 1e-3, -1.0 + 2e-3, -1.0 + 3e-3],
              [0.2 + 1e-3, 1.0, 0.003, 0.0, -2.0, 0.5, 0.5, 0.5])  # fmt: skip
    s_x = np.concatenate([s_x, anti_s[nan_at[:1]]])
    nan_target = 5
    ei = np.array([[0, 1, 1, 1, 8, 2, 3, 4, 5, 6, 7], [0, 1, 1, 1, nan_target, nan_target, nan_target, 3, 4, 4, 4]],
                  dtype=np.int32)  # fmt: skip
    g = make_graph(s_x, t_x, ei)
    L = length_of(g)
    assert np.isnan(L[4]) and np.isfinite(np.delete(L, 4)).all()
    for sigma in (1e-3, 0.05, 1.0):
        w = {n: compute(GaussianDistanceWeights(sigma=sigma, norm=n), g)[:, 0] for n in NORMS}
        for n in NORMS[1:]:
            assert_ulp(w[n], ref_gaussian(L, ei[1], sigma, n), 2, f"sigma={sigma} {n}")
            assert np.isnan(w[n][ei[1] == nan_target]).all()  # the NaN stays inside its own group ...
        assert np.isfinite(w["unit-max"][ei[1] != nan_target]).all() or sigma == 1e-3  # ... and no other
        assert w["l1"][0] == 1.0 and w["unit-max"][0] == 1.0 and np.isnan(w["unit-range"][0])  # degree 1
        np.testing.assert_array_equal(w["unit-std"][1:4], w[None][1:4])  # bit-equal weights: unnormalised
        if sigma == 1e-3:
            assert (w[None][ei[1] == 3] == 0).all() and np.isnan(w["l1"][ei[1] == 3]).all()  # all underflowed
        else:
            assert np.isfinite(w["l1"][ei[1] == 3]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["knn7", "cutoff", "huge"])
def test_gaussian_weights_are_permutation_invariant(edge_lists, huge_group, case):
    """The 2^21-edge group makes the float64 reduction order visible in the float32 output: a sum in another order
    differs by ~1e-13 relative, which moves a few of its two million float32 roundings."""
    from anemoi_graphs_b200.edges.attributes import GaussianDistanceWeights

    src, dst, ei = huge_group if case == "huge" else edge_lists[case]
    sigma = 1.0 if case == "huge" else 0.05  # every weight of the huge group counts
    perm = np.random.default_rng(1).permutation(ei.shape[1])
    g0, g1 = make_graph(src, dst, ei), make_graph(src, dst, ei[:, perm])
    for norm in NORMS:
        a = compute(GaussianDistanceWeights(sigma=sigma, norm=norm), g0)
        b = compute(GaussianDistanceWeights(sigma=sigma, norm=norm), g1)
        assert a[perm].tobytes() == b.tobytes(), norm


# ------------------------------------------------------------------------------------------------
# AttributeFromSourceNode / AttributeFromTargetNode
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("on_gpu", [False, True])
def test_attribute_from_node(edge_lists, on_gpu):
    from anemoi_graphs_b200.edges.attributes import AttributeFromSourceNode, AttributeFromTargetNode

    src, dst, ei = edge_lists["cutoff"]
    rng = np.random.default_rng(2)
    for nodes_name, row, cls in (("src", 0, AttributeFromSourceNode), ("dst", 1, AttributeFromTargetNode)):
        n = (src if row == 0 else dst).shape[0]
        values = {"flat": torch.from_numpy(rng.random(n) < 0.5), "column": torch.from_numpy(rng.random((n, 1)) < 0.5),
                  "f32_3": torch.from_numpy(rng.normal(size=(n, 3)).astype(np.float32) * (rng.random((n, 3)) < 0.5))}  # fmt: skip
        for name, value in values.items():
            g = make_graph(src, dst, ei, on_gpu)
            g[nodes_name][name] = value.cuda() if on_gpu else value
            got = cls(name).compute(g, KEY)
            assert got.is_cuda == on_gpu and got.dtype == torch.bool
            want = value.reshape(n, -1)[torch.from_numpy(ei[row]).long()].bool()
            assert tuple(got.shape) == tuple(want.shape)
            np.testing.assert_array_equal(got.cpu().numpy(), want.numpy(), err_msg=f"{cls.__name__} {name}")
        g = make_graph(src, dst, ei, on_gpu)
        g[nodes_name]["short"] = torch.ones(n - 1, dtype=torch.bool)
        for missing in ("nowhere", "short"):
            with pytest.raises(ValueError, match=f"{missing}.*{nodes_name}"):
                cls(missing).compute(g, KEY)


# ------------------------------------------------------------------------------------------------
# errors
# ------------------------------------------------------------------------------------------------
def _all_four():
    from anemoi_graphs_b200.edges.attributes import (
        AttributeFromSourceNode,
        AttributeFromTargetNode,
        Azimuth,
        GaussianDistanceWeights,
    )

    return [Azimuth(), Azimuth(norm="l1"), GaussianDistanceWeights(norm=None), GaussianDistanceWeights(),
            AttributeFromSourceNode("m"), AttributeFromTargetNode("m")]  # fmt: skip


@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["source", "target", "negative"])
def test_out_of_range_endpoint_raises(bad):
    src = grids.latlon_deg_to_x(*grids.uniform_sphere(300, seed=1)).numpy()
    dst = grids.latlon_deg_to_x(*grids.uniform_sphere(200, seed=2)).numpy()
    rng = np.random.default_rng(4)
    ei = np.stack([rng.integers(0, 300, 3000), rng.integers(0, 200, 3000)]).astype(np.int32)
    if bad == "source":
        ei[0, 1777] = 300
    elif bad == "target":
        ei[1, 5] = 200
    else:
        ei[1, 2999] = -1
    for on_gpu in (False, True):
        g = make_graph(src, dst, ei, on_gpu)
        g["src"]["m"] = torch.ones(300, dtype=torch.bool)
        g["dst"]["m"] = torch.ones(200, dtype=torch.bool)
        before = snapshot(g)
        for attr in _all_four():
            with pytest.raises(ValueError, match="outside"):
                attr.compute(g, KEY)
            assert_same(before, snapshot(g))


@pytest.mark.gpu
def test_sharded_store_is_refused():
    x = grids.latlon_deg_to_x(*grids.uniform_sphere(100, seed=3)).numpy()
    ei = np.random.default_rng(1).integers(0, 100, (2, 500)).astype(np.int32)
    g = make_graph(x, x, ei)
    g[KEY]["edge_shard"] = {"rank": 0, "world": 2, "counts": [500, 500], "replicated": False}
    g["src"]["m"] = torch.ones(100, dtype=torch.bool)
    g["dst"]["m"] = torch.ones(100, dtype=torch.bool)
    before = snapshot(g)
    for attr in _all_four():
        with pytest.raises(NotImplementedError, match="gather"):
            attr.compute(g, KEY)
    assert_same(before, snapshot(g))


# ------------------------------------------------------------------------------------------------
# end to end: a recipe through GraphCreator.create
# ------------------------------------------------------------------------------------------------
DEC = ("hidden", "to", "data")


def _recipe(grid_dir: str, extra: bool) -> dict:
    attrs = {
        "edge_length": {"_target_": T + "edges.attributes.EdgeLength", "norm": "unit-max"},
        "edge_dirs": {"_target_": T + "edges.attributes.EdgeDirection", "norm": "unit-std"},
    }
    if extra:
        attrs = {
            "azimuth": {"_target_": T + "edges.attributes.Azimuth", "norm": "unit-max"},
            **attrs,
            "weights": {"_target_": T + "edges.attributes.GaussianDistanceWeights", "sigma": 0.02, "norm": "l1"},
            "from_src": {"_target_": T + "edges.attributes.AttributeFromSourceNode", "node_attr_name": "area"},
            "from_dst": {"_target_": T + "edges.attributes.AttributeFromTargetNode", "node_attr_name": "area"},
        }
    area = {"area": {"_target_": T + "nodes.attributes.SphericalAreaWeights"}}
    return {
        "nodes": {
            "data": {"node_builder": {"_target_": T + "nodes.NPZFileNodes", "resolution": "t", "grid_definition_path": grid_dir},
                     "attributes": area},
            "hidden": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": 4}, "attributes": area},
        },
        "edges": [{"source_name": "hidden", "target_name": "data", "attributes": attrs,
                   "edge_builders": [{"_target_": T + "edges.KNNEdges", "num_nearest_neighbours": 3}]}],
    }  # fmt: skip


def build_recipe(grid_dir: str, extra: bool, resident: bool) -> dict:
    """name -> numpy array of every per-edge tensor of the decoder, and the node attributes it reads."""
    from anemoi_graphs_b200 import device
    from anemoi_graphs_b200.create import GraphCreator

    prev = device.set_resident(resident)
    try:
        g = GraphCreator(_recipe(grid_dir, extra)).create()
    finally:
        device.set_resident(prev)
    out = {n: g[DEC][n].cpu().numpy() for n in g[DEC].edge_attrs()}
    out["is_cuda"] = np.array([g[DEC].edge_index.is_cuda])
    for k in ("hidden", "data"):
        out[f"{k}/area"] = g[k]["area"].cpu().numpy()
    return out


_CHILD = """
import sys
sys.path[:0] = [{repo!r}, {tests!r}]
import numpy as np
from test_gpu_edge_attrs_extra import build_recipe
out = {{}}
for resident in (False, True):
    for n, v in build_recipe({grid_dir!r}, True, resident).items():
        out[f"{{resident}}:{{n}}"] = v
np.savez({out!r}, **out)
"""


@pytest.mark.gpu
def test_recipe_end_to_end(tmp_path):
    lat, lon = grids.octahedral_grid(48)
    np.savez(tmp_path / "grid-t.npz", latitudes=lat, longitudes=lon)
    grid_dir = str(tmp_path)
    out = tmp_path / "serial.npz"
    code = _CHILD.format(repo=str(REPO), tests=str(REPO / "tests"), grid_dir=grid_dir, out=str(out))
    run = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, AGX_LAZY_ORDER="0"), capture_output=True,
                         text=True, timeout=600)  # fmt: skip
    assert run.returncode == 0, run.stderr[-3000:]
    serial = np.load(out)
    for resident in (False, True):
        got = build_recipe(grid_dir, True, resident)
        plain = build_recipe(grid_dir, False, resident)
        assert bool(got["is_cuda"][0]) == resident
        for n, v in got.items():
            assert v.tobytes() == serial[f"{resident}:{n}"].tobytes(), f"lazy vs serial order: {n}"
        for n in ("edge_index", "edge_length", "edge_dirs"):
            assert got[n].tobytes() == plain[n].tobytes(), f"{n} changed by the new attributes"
        ei = got["edge_index"]
        assert got["azimuth"].shape == (ei.shape[1], 1) and got["weights"].dtype == np.float32
        sums = np.bincount(ei[1], weights=got["weights"][:, 0].astype(np.float64))
        np.testing.assert_allclose(sums[np.unique(ei[1])], 1.0, rtol=1e-6)
        np.testing.assert_array_equal(got["from_src"], got["hidden/area"].reshape(-1, 1)[ei[0]].astype(bool))
        np.testing.assert_array_equal(got["from_dst"], got["data/area"].reshape(-1, 1)[ei[1]].astype(bool))
