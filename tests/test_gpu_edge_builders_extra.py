"""Edge builders of newer anemoi-graphs releases: ``ReversedKNNEdges``, ``ReversedCutOffEdges`` and
``MultiScaleEdges(scale_resolutions=...)``.

The reversed builders are checked against the forward builders with their rows swapped (column for column), against
the canonical oracle (``ref_path.knn_edges_canonical``: float64 ``rdist``, ties to the lower index of the indexed side)
and against sklearn.  The level subsets of ``MultiScaleEdges`` are checked against the oracles of every node type.
Constructor and recipe validation run without a GPU."""

import numpy as np
import pytest
import torch

from anemoi_graphs_b200 import grids
from oracle import h3_restated as H
from oracle import ref_path as R

T = "anemoi.graphs."
ATTR_RTOL = 1e-6  # DESIGN.md section 4


def swap(ei: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(ei[::-1])


def by_source(ei) -> np.ndarray:
    """Columns sorted by (source, target)."""
    ei = ei.cpu().numpy() if isinstance(ei, torch.Tensor) else np.asarray(ei)
    return ei[:, np.lexsort((ei[1], ei[0]))]


def canon(ei) -> np.ndarray:
    ei = ei.cpu().numpy() if isinstance(ei, torch.Tensor) else np.asarray(ei)
    return R.canonical_sort(ei)


# ------------------------------------------------------------------------------------------------
# constructors and recipe validation (CPU)
# ------------------------------------------------------------------------------------------------
def test_constructor_validation():
    from anemoi_graphs_b200.edges import MultiScaleEdges, ReversedCutOffEdges, ReversedKNNEdges

    assert ReversedKNNEdges("a", "b", 3).num_nearest_neighbours == 3
    with pytest.raises(AssertionError, match="Number of nearest neighbours must be an integer"):
        ReversedKNNEdges("a", "b", 3.0)
    with pytest.raises(AssertionError, match="Number of nearest neighbours must be positive"):
        ReversedKNNEdges("a", "b", 0)
    assert ReversedCutOffEdges("a", "b", 0.6, source_mask_attr_name="m").source_mask_attr_name == "m"
    with pytest.raises(AssertionError, match="Cutoff factor must be a float"):
        ReversedCutOffEdges("a", "b", "0.6")
    with pytest.raises(AssertionError, match="Cutoff factor must be positive"):
        ReversedCutOffEdges("a", "b", -1.0)

    def levels(v):
        return MultiScaleEdges("h", "h", 1, scale_resolutions=v).scale_resolutions

    assert levels(None) is None
    assert levels(3) == [1, 2, 3]
    assert levels([4, 2, 4]) == [2, 4]
    assert levels((1,)) == [1]
    for bad in (0, -2, [0, 1], [1, -1], [1, 2.0], [True]):
        with pytest.raises(AssertionError, match="The scale_resolutions argument only supports positive integers."):
            levels(bad)
    for bad in ("3", "[1, 2]", [], 2.0, {1: 2}):
        with pytest.raises(AssertionError, match="The scale_resolutions argument is not valid."):
            levels(bad)


def test_multiscale_levels_are_checked_against_the_node_set():
    """Before any kernel: a level finer than the nodes, more levels than the kernel takes."""
    from anemoi_graphs_b200.edges import MultiScaleEdges

    nodes = {"_resolutions": list(range(6))}
    assert MultiScaleEdges("h", "h", 1).levels(nodes) == list(range(6))  # None: every level, level 0 included
    assert MultiScaleEdges("h", "h", 1, scale_resolutions=5).levels(nodes) == [1, 2, 3, 4, 5]
    assert MultiScaleEdges("h", "h", 1, scale_resolutions=[5, 3]).levels(nodes) == [3, 5]
    with pytest.raises(ValueError, match="finest level 5"):
        MultiScaleEdges("h", "h", 1, scale_resolutions=[2, 6]).levels(nodes)
    with pytest.raises(NotImplementedError, match="17 scale_resolutions > 16"):
        MultiScaleEdges("h", "h", 1, scale_resolutions=17).levels({"_resolutions": list(range(20))})


def _recipe(builder: dict, hidden: dict | None = None) -> dict:
    hidden = hidden or {"_target_": T + "nodes.TriNodes", "resolution": 5}
    return {
        "nodes": {"hidden": {"node_builder": hidden}},
        "edges": [{"source_name": "hidden", "target_name": "hidden", "edge_builders": [builder]}],
    }


def test_recipe_validation():
    from anemoi_graphs_b200.config import resolve_target
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.edges import ReversedCutOffEdges, ReversedKNNEdges

    assert resolve_target(T + "edges.ReversedKNNEdges") is ReversedKNNEdges
    assert resolve_target(T + "edges.ReversedCutOffEdges") is ReversedCutOffEdges
    GraphCreator(_recipe({"_target_": T + "edges.ReversedKNNEdges", "num_nearest_neighbours": 64}))
    GraphCreator(_recipe({"_target_": T + "edges.ReversedCutOffEdges", "cutoff_factor": 0.6}))
    for name in ("KNNEdges", "ReversedKNNEdges"):
        with pytest.raises(NotImplementedError, match=f"{name}: num_nearest_neighbours = 65 > 64"):
            GraphCreator(_recipe({"_target_": T + f"edges.{name}", "num_nearest_neighbours": 65}))

    def ms(levels, hidden=None):
        return GraphCreator(_recipe({"_target_": T + "edges.MultiScaleEdges", "x_hops": 1, "scale_resolutions": levels},
                                    hidden))  # fmt: skip

    ms(5)
    ms([1, 3, 5])
    ms([7], {"_target_": T + "nodes.StretchedTriNodes", "global_resolution": 3, "lam_resolution": 7,
             "reference_node_name": "data", "mask_attr_name": "m"})  # fmt: skip
    ms([9], {"_target_": T + "nodes.NPZFileNodes", "resolution": "o96", "grid_definition_path": "."})  # not known yet
    with pytest.raises(AssertionError, match="not valid"):
        ms("5")
    with pytest.raises(AssertionError, match="positive integers"):
        ms([0, 2])
    with pytest.raises(ValueError, match="finest level 5"):
        ms(6)
    with pytest.raises(ValueError, match="finest level 4"):
        ms([2, 5], {"_target_": T + "nodes.HexNodes", "resolution": [0, 2, 4]})
    with pytest.raises(NotImplementedError, match="17 scale_resolutions > 16"):
        ms(17, {"_target_": T + "nodes.TriNodes", "resolution": 17})


# ------------------------------------------------------------------------------------------------
# ReversedKNNEdges / ReversedCutOffEdges on O96 -> TriNodes(5)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def o96():
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.graph import HeteroData

    lat, lon = grids.octahedral_grid(96)
    recipe = {
        "nodes": {
            "data": {"node_builder": {"_target_": T + "nodes.LatLonNodes", "latitudes": lat, "longitudes": lon}},
            "hidden": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": 5}},
        }
    }
    g = GraphCreator(recipe).update_graph(HeteroData())
    dx, hx = g["data"].x.numpy().copy(), g["hidden"].x.numpy().copy()
    masks = {"data": dx[:, 0] > -0.5, "hidden": (hx[:, 1] < 1.0) | (hx[:, 0] > 0.3)}
    return dx, hx, masks


def _graph(o96):
    from anemoi_graphs_b200.graph import HeteroData

    dx, hx, masks = o96
    g = HeteroData()
    for name, x in (("data", dx), ("hidden", hx)):
        g[name].x = torch.from_numpy(x)
        g[name]["m"] = torch.from_numpy(masks[name].reshape(-1, 1))
    return g


def _sel(o96, name, masked):
    n = o96[0 if name == "data" else 1].shape[0]
    return np.nonzero(o96[2][name])[0] if masked else np.arange(n)


MASKS = [(False, False), (True, False), (False, True), (True, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 16, 64])
@pytest.mark.parametrize("smask,tmask", MASKS)
def test_reversed_knn_is_the_swapped_forward_search(o96, k, smask, tmask):
    from anemoi_graphs_b200.edges import KNNEdges, ReversedKNNEdges

    dx, hx, _ = o96
    g = _graph(o96)
    sm, tm = ("m" if smask else None), ("m" if tmask else None)
    ReversedKNNEdges("data", "hidden", k, source_mask_attr_name=sm, target_mask_attr_name=tm).update_graph(g)
    KNNEdges("hidden", "data", k, source_mask_attr_name=tm, target_mask_attr_name=sm).update_graph(g)
    rev = g[("data", "to", "hidden")]
    assert rev.edge_type == "ReversedKNNEdges" and rev.edge_index.dtype == torch.int32
    got = rev.edge_index.numpy()
    np.testing.assert_array_equal(got, swap(g[("hidden", "to", "data")].edge_index.numpy()))  # column for column
    s_sel, t_sel = _sel(o96, "data", smask), _sel(o96, "hidden", tmask)
    np.testing.assert_array_equal(got[0], np.repeat(s_sel, k))  # grouped by source, k per source

    # the oracle: the sources are the queries of an index over the targets
    want, info = R.knn_edges_canonical(hx[t_sel], dx[s_sel], k)
    assert info["untied_mismatch"].size == 0
    want = np.stack([s_sel[want[1]], t_sel[want[0]]])
    np.testing.assert_array_equal(by_source(got), by_source(want))
    # sklearn NearestNeighbors.fit(target).kneighbors(source): the same set wherever no tie decides it
    ref = R.knn_edges(hx[t_sel], dx[s_sel], k)
    ref = by_source(np.stack([s_sel[ref[1]], t_sel[ref[0]]]))
    tied = s_sel[info["tied_queries"]]
    got_s = by_source(got)
    np.testing.assert_array_equal(got_s[:, ~np.isin(got_s[0], tied)], ref[:, ~np.isin(ref[0], tied)])


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 5])
def test_reversed_knn_ties_go_to_the_lower_target_index(k):
    """Queries on the mirror plane lon = 0 of a target set made of mirror pairs (lat, +-lon): every pair is bit-equally
    far, so with odd k every query's k-th boundary is a tie.  Pairs are shuffled, so the lower index is on either side."""
    from anemoi_graphs_b200.edges import KNNEdges, ReversedKNNEdges
    from anemoi_graphs_b200.graph import HeteroData

    rng = np.random.default_rng(11)
    lat = rng.uniform(-1.2, 1.2, 400).astype(np.float32)
    lon = rng.uniform(0.02, 0.8, 400).astype(np.float32)
    tx = np.concatenate([np.stack([lat, lon], 1), np.stack([lat, -lon], 1)])[rng.permutation(800)]
    sx = np.stack([rng.uniform(-1.1, 1.1, 300), np.zeros(300)], 1).astype(np.float32)
    g = HeteroData()
    g["s"].x = torch.from_numpy(sx)
    g["t"].x = torch.from_numpy(tx)
    ReversedKNNEdges("s", "t", k).update_graph(g)
    KNNEdges("t", "s", k).update_graph(g)
    got = g[("s", "to", "t")].edge_index.numpy()
    np.testing.assert_array_equal(got, swap(g[("t", "to", "s")].edge_index.numpy()))
    want, info = R.knn_edges_canonical(tx, sx, k)
    assert info["tied_queries"].size == sx.shape[0]
    np.testing.assert_array_equal(by_source(got), by_source(swap(want)))


@pytest.mark.gpu
def test_reversed_knn_needs_k_targets():
    from anemoi_graphs_b200.edges import ReversedKNNEdges
    from anemoi_graphs_b200.graph import HeteroData

    g = HeteroData()
    g["s"].x = torch.from_numpy(np.zeros((50, 2), dtype=np.float32))
    g["t"].x = torch.from_numpy(np.stack([np.linspace(-1, 1, 12), np.zeros(12)], 1).astype(np.float32))
    with pytest.raises(ValueError, match="Expected n_neighbors <= n_samples_fit, but n_neighbors = 13, n_samples_fit = 12"):
        ReversedKNNEdges("s", "t", 13).update_graph(g)


@pytest.mark.gpu
@pytest.mark.parametrize("resident", [False, True])
def test_reversed_knn_list_is_not_walked_by_target(o96, resident):
    """A reversed KNN list is k edges per SOURCE: the metadata that lets the attribute kernel walk a list target by target
    (and the a-priori target row) must not be set, and its attributes are the per-edge values."""
    from anemoi_graphs_b200 import device
    from anemoi_graphs_b200.edges import KNNEdges, ReversedKNNEdges
    from anemoi_graphs_b200.edges.attributes import EdgeDirection, EdgeLength

    dx, hx, _ = o96
    g = _graph(o96)
    if resident:
        for name in ("data", "hidden"):
            g[name].x = g[name].x.cuda()
    prev = device.set_resident(resident)
    try:
        ReversedKNNEdges("data", "hidden", 3).update_graph(g)
        KNNEdges("hidden", "data", 3).update_graph(g)
        for key, k in ((("data", "to", "hidden"), 0), (("hidden", "to", "data"), 3)):
            meta = device.edge_meta(device.device_edge_index(g[key]))
            assert (meta.regular_k if meta is not None else 0) == k
            assert bool(meta is not None and meta.regular_targets) == (k > 0)
        key = ("data", "to", "hidden")
        length = EdgeLength(norm=None).compute(g, key)
        dirs = EdgeDirection(norm=None).compute(g, key)
    finally:
        device.set_resident(prev)
    ei = g[key].edge_index.cpu().numpy()
    np.testing.assert_allclose(length.cpu().numpy(), R.edge_length(dx, hx, ei), rtol=ATTR_RTOL, atol=0)
    want = R.edge_direction(dx, hx, ei)
    np.testing.assert_allclose(dirs.cpu().numpy(), want, rtol=ATTR_RTOL, atol=ATTR_RTOL * np.abs(want).max())


@pytest.mark.gpu
@pytest.mark.parametrize("src,dst,factor,masked", [("data", "hidden", 2.0, False), ("hidden", "data", 0.6, False),
                                                   ("hidden", "data", 0.9, True)])  # fmt: skip
def test_reversed_cutoff_is_the_swapped_forward_search(o96, src, dst, factor, masked):
    from anemoi_graphs_b200.edges import CutOffEdges, ReversedCutOffEdges

    x = {"data": o96[0], "hidden": o96[1]}
    g = _graph(o96)
    sm = tm = "m" if masked else None
    rev = ReversedCutOffEdges(src, dst, factor, source_mask_attr_name=sm, target_mask_attr_name=tm)
    rev.update_graph(g)
    CutOffEdges(dst, src, factor, source_mask_attr_name=tm, target_mask_attr_name=sm).update_graph(g)
    radius = R.cutoff_radius(x[src], factor)
    assert rev.radius == radius  # sklearn's float64 bits, of the SOURCE (query) set
    got = g[(src, "to", dst)].edge_index.numpy()
    assert got.shape[1] > 0
    np.testing.assert_array_equal(got, swap(g[(dst, "to", src)].edge_index.numpy()))
    s_sel, t_sel = _sel(o96, src, masked), _sel(o96, dst, masked)
    assert np.all(np.diff(got[0]) >= 0)  # grouped by source
    want = R.cutoff_edges(x[dst][t_sel], x[src][s_sel], factor, radius=radius)
    want = np.stack([s_sel[want[1]], t_sel[want[0]]])
    np.testing.assert_array_equal(by_source(got), by_source(want))


# ------------------------------------------------------------------------------------------------
# through GraphCreator: a TriNodes target in provisional numbering
# ------------------------------------------------------------------------------------------------
def _attrs(norm):
    return {
        "edge_length": {"_target_": T + "edges.attributes.EdgeLength", "norm": norm},
        "edge_dirs": {"_target_": T + "edges.attributes.EdgeDirection", "norm": norm},
    }


def _creator_recipe():
    return {
        "nodes": {"hidden": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": 5}}},
        "edges": [
            # every data point gets its 3 nearest mesh nodes: the index is over the provisionally numbered mesh
            {"source_name": "data", "target_name": "hidden", "attributes": _attrs("unit-std"),
             "edge_builders": [{"_target_": T + "edges.ReversedKNNEdges", "num_nearest_neighbours": 3}]},
            # mesh nodes as queries, merged with a second builder on the same pair
            {"source_name": "hidden", "target_name": "data", "attributes": _attrs(None),
             "edge_builders": [{"_target_": T + "edges.ReversedCutOffEdges", "cutoff_factor": 0.4},
                               {"_target_": T + "edges.ReversedKNNEdges", "num_nearest_neighbours": 2}]},
        ],
    }  # fmt: skip


@pytest.mark.gpu
@pytest.mark.parametrize("resident", [False, True])
def test_reversed_builders_under_provisional_numbering(o96, resident, monkeypatch):
    from anemoi_graphs_b200 import device as agx_device
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.edges import KNNEdges
    from anemoi_graphs_b200.graph import HeteroData

    dx = o96[0]
    redecided = []
    real = KNNEdges._redecide_ties

    def spy(prov, index, out, tie_list, queries, k, swap_rows):
        redecided.append((k, swap_rows))
        return real(prov, index, out, tie_list, queries, k, swap_rows)

    monkeypatch.setattr(KNNEdges, "_redecide_ties", staticmethod(spy))

    def run(lazy):
        monkeypatch.setattr(agx_device, "LAZY_NODE_ORDER", lazy)
        prev = agx_device.set_resident(resident)
        try:
            g = HeteroData()
            x = torch.from_numpy(dx)
            g["data"].x = x.cuda() if resident else x
            g["data"].node_type = "LatLonNodes"
            g = GraphCreator(_creator_recipe()).update_graph(g)
            torch.cuda.synchronize()
            return g
        finally:
            agx_device.set_resident(prev)

    a = run(True)
    assert redecided == [(3, True)]  # searched before the mesh order was known, ties re-decided on the final order
    b = run(False)
    assert len(redecided) == 1
    hx = a["hidden"].x.cpu().numpy()
    np.testing.assert_array_equal(hx.view(np.int32), b["hidden"].x.cpu().numpy().view(np.int32))
    for key in (("data", "to", "hidden"), ("hidden", "to", "data")):
        assert a[key].edge_index.is_cuda == resident
        ea, eb = a[key].edge_index.cpu().numpy(), b[key].edge_index.cpu().numpy()
        oa, ob = np.lexsort((ea[1], ea[0])), np.lexsort((eb[1], eb[0]))
        np.testing.assert_array_equal(ea[:, oa], eb[:, ob])
        assert a[key].edge_type == b[key].edge_type
        for name in ("edge_length", "edge_dirs"):
            va, vb = a[key][name].cpu().numpy()[oa], b[key][name].cpu().numpy()[ob]
            np.testing.assert_allclose(va, vb, rtol=3e-7, atol=1e-7 * np.abs(vb).max())

    # the encoder against the oracle, attributes included
    key = ("data", "to", "hidden")
    ei = a[key].edge_index.cpu().numpy()
    np.testing.assert_array_equal(ei[0], np.repeat(np.arange(dx.shape[0]), 3))
    want, _ = R.knn_edges_canonical(hx, dx, 3)
    np.testing.assert_array_equal(by_source(ei), by_source(swap(want)))
    np.testing.assert_allclose(a[key]["edge_length"].cpu().numpy(), R.edge_length(dx, hx, ei, "unit-std"),
                               rtol=ATTR_RTOL, atol=0)  # fmt: skip
    want_d = R.edge_direction(dx, hx, ei, "unit-std")
    np.testing.assert_allclose(a[key]["edge_dirs"].cpu().numpy(), want_d, rtol=ATTR_RTOL,
                               atol=ATTR_RTOL * np.abs(want_d).max())  # fmt: skip
    # the merged pair: the union of both builders' edges, sorted and de-duplicated
    key = ("hidden", "to", "data")
    assert a[key].edge_type == "ReversedCutOffEdges,ReversedKNNEdges"
    ei = a[key].edge_index.cpu().numpy()
    cut = swap(R.cutoff_edges(dx, hx, 0.4, radius=R.cutoff_radius(hx, 0.4)))
    knn = swap(R.knn_edges_canonical(dx, hx, 2)[0])
    union = np.unique(np.concatenate([cut, knn], axis=1), axis=1)
    assert union.shape[1] > max(cut.shape[1], knn.shape[1])  # both builders contribute edges
    np.testing.assert_array_equal(by_source(ei), by_source(union))
    assert np.unique(ei, axis=1).shape == ei.shape
    np.testing.assert_allclose(a[key]["edge_length"].cpu().numpy(), R.edge_length(hx, dx, ei), rtol=ATTR_RTOL, atol=0)
    want_d = R.edge_direction(hx, dx, ei)
    np.testing.assert_allclose(a[key]["edge_dirs"].cpu().numpy(), want_d, rtol=ATTR_RTOL,
                               atol=ATTR_RTOL * np.abs(want_d).max())  # fmt: skip


# ------------------------------------------------------------------------------------------------
# MultiScaleEdges(scale_resolutions=...) on every node type
# ------------------------------------------------------------------------------------------------
SPECS = [(None, None), (3, [1, 2, 3]), ([2, 3], [2, 3]), ([1, 3], [1, 3]), ([2], [2])]


@pytest.mark.gpu
@pytest.mark.parametrize("spec,levels", SPECS + [(4, [1, 2, 3, 4]), ([4, 1], [1, 4])])
@pytest.mark.parametrize("hops", [1, 2])
def test_scale_resolutions_on_global_tri_nodes(spec, levels, hops, monkeypatch):
    """Through GraphCreator, with the mesh in provisional numbering: the edges are built before its order is known."""
    from anemoi_graphs_b200 import device as agx_device
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.generate import tri_icosahedron
    from anemoi_graphs_b200.graph import HeteroData

    monkeypatch.setattr(agx_device, "LAZY_NODE_ORDER", True)
    provisional = []
    real = tri_icosahedron.multiscale_edges

    def spy(*args, **kwargs):
        out = real(*args, **kwargs)
        provisional.append(agx_device.row_tags(out) != (None, None))
        return out

    monkeypatch.setattr(tri_icosahedron, "multiscale_edges", spy)
    builder = {"_target_": T + "edges.MultiScaleEdges", "x_hops": hops, "scale_resolutions": spec}
    g = GraphCreator(_recipe(builder, {"_target_": T + "nodes.TriNodes", "resolution": 4})).update_graph(HeteroData())
    assert provisional == [True]
    order = np.asarray(g["hidden"]["_node_ordering"])
    want = R.multiscale_edges_tri(levels if levels is not None else range(5), hops, order)
    np.testing.assert_array_equal(canon(g[("hidden", "to", "hidden")].edge_index), R.canonical_sort(want))


def _lam_graph(g):
    from anemoi_graphs_b200.graph import HeteroData

    graph = HeteroData()
    graph["data"].x = torch.from_numpy(g["data_x"])
    graph["data"].node_type = "LatLonNodes"
    graph["data"]["cutout"] = torch.from_numpy(g["cutout"])
    return graph


TRI_SPECS = [(None, list(range(7))), (6, [1, 2, 3, 4, 5, 6]), ([5, 6], [5, 6]), ([2, 6], [2, 6]), ([4], [4])]


@pytest.mark.gpu
@pytest.mark.parametrize("spec,levels", TRI_SPECS)
@pytest.mark.parametrize("kind", ["LimitedAreaTriNodes", "StretchedTriNodes"])
def test_scale_resolutions_on_limited_area_and_stretched_tri_nodes(golden, kind, spec, levels):
    from anemoi_graphs_b200.edges import MultiScaleEdges
    from anemoi_graphs_b200.nodes import LimitedAreaTriNodes, StretchedTriNodes

    g = golden("lam")
    graph = _lam_graph(g)
    if kind == "LimitedAreaTriNodes":
        graph = LimitedAreaTriNodes(6, "data", "n", mask_attr_name="cutout", margin_radius_km=100.0).update_graph(graph, {})
    else:
        graph = StretchedTriNodes(2, 6, "n", "data", "cutout", margin_radius_km=100.0).update_graph(graph, {})
    MultiScaleEdges("n", "n", 1, scale_resolutions=spec).update_graph(graph)
    x = graph["n"].x.numpy()
    dx, cut = g["data_x"], g["cutout"].squeeze()
    ref_x, margin = (dx[cut], 100.0) if kind == "LimitedAreaTriNodes" else (x, 1.0)
    want = R.multiscale_edges_tri_masked(levels, 1, x, ref_x, margin)
    assert want.shape[1] > 0
    np.testing.assert_array_equal(canon(graph[("n", "to", "n")].edge_index), R.canonical_sort(want))


def _hex_graph(kind):
    from anemoi_graphs_b200.graph import HeteroData
    from anemoi_graphs_b200.nodes import HexNodes, LimitedAreaHexNodes

    if kind == "HexNodes":
        return HexNodes(3, "n").update_graph(HeteroData(), {}), None
    lat, lon = np.meshgrid(np.linspace(35.0, 65.0, 61), np.linspace(-10.0, 30.0, 81), indexing="ij")
    x = np.deg2rad(np.stack([lat.reshape(-1), lon.reshape(-1)], axis=1)).astype(np.float32)
    graph = HeteroData()
    graph["data"].x = torch.from_numpy(x)
    graph["data"].node_type = "LatLonNodes"
    graph = LimitedAreaHexNodes(3, "data", "n", margin_radius_km=150.0).update_graph(graph, {})
    return graph, R.knn_area_mask(x, H.hex_nodes_latlon(3), 150.0)


def _hex_edges(graph, spec, hops):
    from anemoi_graphs_b200.edges import MultiScaleEdges

    return canon(MultiScaleEdges("n", "n", hops, scale_resolutions=spec).get_edge_index(graph))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["HexNodes", "LimitedAreaHexNodes"])
def test_scale_resolutions_on_hex_nodes(kind):
    graph, in_graph = _hex_graph(kind)
    order = np.asarray(graph["n"]["_node_ordering"])
    # the oracle takes the graph's level to be the finest one it is given: level lists that reach level 3
    for spec, levels in [(None, [0, 1, 2, 3])] + SPECS[1:4] + [([3], [3])]:
        for hops in (1, 2):
            want = H.multiscale_edges_hex(levels, hops, order, in_graph=in_graph)
            assert want.shape[1] > 0
            np.testing.assert_array_equal(_hex_edges(graph, spec, hops), want, err_msg=f"{spec} {hops}")
    # levels that stop short of the nodes' level: joined with the finest level's edges they give the oracle's
    finest = _hex_edges(graph, [3], 1)
    for levels in ([2], [1, 2]):
        part = _hex_edges(graph, levels, 1)
        want = H.multiscale_edges_hex(levels + [3], 1, order, in_graph=in_graph)
        assert part.shape[1] > 0
        np.testing.assert_array_equal(R.canonical_sort(np.unique(np.concatenate([part, finest], 1), axis=1)), want)
        assert {tuple(c) for c in part.T} <= {tuple(c) for c in want.T}
