"""Pins ``oracle/ref_path.py`` (the CPU restatement) to outputs of the UNMODIFIED reference
(``tests/golden/*.npz``, produced by ``oracle/make_golden.py``) and to the reference's published
counts.  CPU only."""

import numpy as np
import pytest

from anemoi_graphs_b200 import grids
from oracle import ref_path as R

NORMS = [None, "l1", "l2", "unit-max", "unit-range", "unit-std"]


def _n(norm):
    return "none" if norm is None else norm.replace("-", "_")


def test_tri_nodes_match_reference(golden):
    g = golden("tri_nodes")
    for res in range(5):
        x, order = R.tri_nodes(res)
        assert x.dtype == np.float32
        np.testing.assert_array_equal(order, g[f"res{res}_node_ordering"])
        np.testing.assert_array_equal(x.view(np.int32), g[f"res{res}_x"].view(np.int32))
    # reference's own pin: tests/nodes/test_tri_nodes.py:32
    assert R.tri_nodes(2)[0].shape == (162, 2)


@pytest.mark.parametrize("hops", [1, 2, 3])
def test_multiscale_matches_reference(golden, hops):
    g = golden("tri_nodes")
    ei = R.multiscale_edges_tri(range(4), hops, g["res3_node_ordering"])
    np.testing.assert_array_equal(ei, g[f"res3_hops{hops}_edge_index"])


def test_multiscale_resolution_list_and_networkx_variant(golden):
    g = golden("tri_nodes")
    ei = R.multiscale_edges_tri([1, 3], 1, g["res3_node_ordering"])
    np.testing.assert_array_equal(ei, g["res_1_3_hops1_edge_index"])
    slow = R.multiscale_edges_tri_networkx(range(3), 2, g["res2_node_ordering"], g["res2_x"])
    fast = R.multiscale_edges_tri(range(3), 2, g["res2_node_ordering"])
    np.testing.assert_array_equal(R.canonical_sort(slow), fast)


def test_multiscale_published_counts():
    # docs/graphs/edges/tri_refined_edges.csv: multilevel edge counts for levels 0..4
    expect = [60, 300, 1260, 5100, 20460]
    for res, e in enumerate(expect):
        _, order = R.tri_nodes(res)
        assert R.multiscale_edges_tri(range(res + 1), 1, order).shape[1] == e


def test_toy_edges_match_reference(golden):
    g = golden("toy")
    dx, hx = g["data_x"], g["hidden_x"]
    np.testing.assert_array_equal(
        grids.latlon_deg_to_x(g["data_lat_deg"], g["data_lon_deg"]).numpy().view(np.int32), dx.view(np.int32)
    )
    np.testing.assert_array_equal(R.cutoff_edges(dx, hx, 0.6), g["cutoff_edge_index"])
    np.testing.assert_array_equal(R.knn_edges(hx, dx, 3), g["knn3_edge_index"])
    np.testing.assert_array_equal(R.knn_edges(hx, hx, 4), g["hidden_self_knn4_edge_index"])
    ms1 = R.multiscale_edges_tri(range(3), 1, g["hidden_node_ordering"])
    np.testing.assert_array_equal(ms1, R.canonical_sort(g["multiscale1_edge_index"]))
    ms2 = R.multiscale_edges_tri(range(3), 2, g["hidden_node_ordering"])
    np.testing.assert_array_equal(ms2, R.canonical_sort(g["multiscale2_edge_index"]))
    both = R.concat_edges(R.cutoff_edges(dx, hx, 0.6), R.knn_edges(dx, hx, 5))
    np.testing.assert_array_equal(both, g["cutoff_plus_knn5_edge_index"])
    np.testing.assert_array_equal(
        R.masked_edges("knn", hx, dx, g["hidden_mask"], g["data_mask"], 3), g["masked_knn3_edge_index"]
    )
    np.testing.assert_array_equal(
        R.masked_edges("cutoff", dx, hx, g["data_mask"], g["hidden_mask"], 0.6), g["masked_cutoff_edge_index"]
    )


def test_toy_canonical_knn_has_no_untied_mismatch(golden):
    g = golden("toy")
    ei, info = R.knn_edges_canonical(g["hidden_x"], g["data_x"], 3)
    assert info["untied_mismatch"].size == 0
    assert info["tied_queries"].size == 0  # random points: no exact ties
    np.testing.assert_array_equal(ei, R.canonical_sort(g["knn3_edge_index"]))


def test_toy_attributes_match_reference(golden):
    g = golden("toy")
    dx, hx = g["data_x"], g["hidden_x"]
    cases = (
        ("cutoff", dx, hx, g["cutoff_edge_index"]),
        ("ms1", hx, hx, g["multiscale1_edge_index"]),
        ("knn3", hx, dx, g["knn3_edge_index"]),
    )
    for tag, sx, tx, ei in cases:
        for norm in NORMS:
            np.testing.assert_array_equal(R.edge_length(sx, tx, ei, norm), g[f"{tag}_len_{_n(norm)}"])
            np.testing.assert_array_equal(R.edge_direction(sx, tx, ei, norm), g[f"{tag}_dir_rot_{_n(norm)}"])
        np.testing.assert_array_equal(R.edge_length(sx, tx, ei, "unit-max", invert=True), g[f"{tag}_len_inv_unit_max"])
        np.testing.assert_array_equal(
            R.edge_direction(sx, tx, ei, "unit-std", rotated=False), g[f"{tag}_dir_norot_unit_std"]
        )


def test_attr_vectors(golden):
    g = golden("attr_vectors")
    src, dst = g["src"], g["dst"]
    with np.errstate(all="ignore"):
        rot = R.edge_directions_raw(src.T.copy(), dst.T.copy(), True).T
        length = R.haversine_distance(src, dst)
    np.testing.assert_array_equal(rot, g["dir_rotated"])
    np.testing.assert_array_equal(length, g["length"])
    np.testing.assert_array_equal(R.edge_directions_raw(src.T.copy(), dst.T.copy(), False).T, g["dir_nonrotated"])
    # SURVEY appendix B known answers
    np.testing.assert_allclose(rot[0], (-0.808158205, -0.588965463), rtol=0, atol=1e-9)
    np.testing.assert_allclose(length[0], 0.053570323, rtol=1e-7)


def test_reference_normalise_propagates_nan(golden):
    """The reference's normalisation turns one NaN value (the antipodal pair of the golden vectors, row 9) into NaN
    everywhere, for every norm - the behaviour the attribute kernel reproduces (tests/test_gpu_attr_paths.py)."""
    g = golden("attr_vectors")
    n = g["src"].shape[0]
    ei = np.stack([np.arange(n), np.arange(n)])
    values = np.array([[0.5, 1.0], [np.nan, 2.0], [3.0, 4.0]], dtype=np.float32)
    with np.errstate(all="ignore"):
        for norm in ("l1", "l2", "unit-max", "unit-range", "unit-std"):
            assert np.isnan(R.edge_length(g["src"], g["dst"], ei, norm)).all(), norm
            assert np.isnan(R.edge_length(g["src"], g["dst"], ei, norm, invert=True)).all(), norm
            for v in (values, values.astype(np.float64)):
                assert np.isnan(R.normalise(v, norm)).all(), norm
        length = R.edge_length(g["src"], g["dst"], ei, None)
    assert np.isnan(length[9]).all() and np.isfinite(np.delete(length, 9)).all()
def test_o96_res5_matches_reference_and_published_counts(golden):
    g = golden("o96_res5")
    lat, lon = grids.octahedral_grid(96)
    dx = grids.latlon_deg_to_x(lat, lon).numpy()
    assert dx.shape == (40320, 2)
    hx, order = R.tri_nodes(5)
    np.testing.assert_array_equal(hx.view(np.int32), g["hidden_x"].view(np.int32))
    np.testing.assert_array_equal(order, g["hidden_node_ordering"])
    assert R.grid_reference_distance(hx) == float(g["reference_distance"])
    cut = R.canonical_sort(R.cutoff_edges(dx, hx, 0.6))
    knn = R.canonical_sort(R.knn_edges(hx, dx, 3))
    ms = R.multiscale_edges_tri(range(6), 1, order)
    # docs/_static/hetero_data_graph.txt:13,19,25
    assert (cut.shape[1], ms.shape[1], knn.shape[1]) == (62980, 81900, 120960)
    np.testing.assert_array_equal(cut, g["cutoff_edge_index"])
    np.testing.assert_array_equal(ms, g["multiscale_edge_index"])
    np.testing.assert_array_equal(knn, g["knn3_edge_index"])
    stride = int(g["attr_sample_stride"])
    for tag, sx, tx, ei in (("cutoff", dx, hx, cut), ("multiscale", hx, hx, ms), ("knn3", hx, dx, knn)):
        np.testing.assert_array_equal(R.edge_length(sx, tx, ei, "unit-std")[::stride], g[f"{tag}_edge_length_sample"])
        np.testing.assert_array_equal(R.edge_direction(sx, tx, ei, "unit-std")[::stride], g[f"{tag}_edge_dirs_sample"])


def test_o96_res5_tie_enumeration(golden):
    """SURVEY appendix B: 88 queries have an exact k/k+1 tie, 46 of them resolved differently by sklearn."""
    g = golden("o96_res5")
    lat, lon = grids.octahedral_grid(96)
    dx = grids.latlon_deg_to_x(lat, lon).numpy()
    ei, info = R.knn_edges_canonical(g["hidden_x"], dx, 3)
    assert info["untied_mismatch"].size == 0
    assert info["tied_queries"].size == 88
    assert info["differs_from_reference"].size == 46
    ref = g["knn3_edge_index"]
    untied = ~np.isin(ref[1], info["tied_queries"])
    np.testing.assert_array_equal(ei[:, ~np.isin(ei[1], info["tied_queries"])], ref[:, untied])


def test_lam_and_stretched_match_reference(golden):
    """Config 4 in miniature (tests/golden/lam.npz): LimitedAreaTriNodes / StretchedTriNodes and their
    MultiScaleEdges, masked KNN / CutOff, from the unmodified reference."""
    g = golden("lam")
    dx, cut = g["data_x"], g["cutout"].squeeze()
    lam_x, lam_order, _ = R.lam_tri_nodes(6, dx[cut], 100.0)
    np.testing.assert_array_equal(lam_order, g["lam_node_ordering"])
    np.testing.assert_array_equal(lam_x.view(np.int32), g["lam_x"].view(np.int32))
    str_x, str_order, _ = R.stretched_tri_nodes(2, 6, dx[cut], 100.0)
    np.testing.assert_array_equal(str_order, g["str_node_ordering"])
    np.testing.assert_array_equal(str_x.view(np.int32), g["str_x"].view(np.int32))
    for hops in (1, 2):
        ei = R.multiscale_edges_tri_masked(range(7), hops, lam_x, dx[cut], 100.0)
        np.testing.assert_array_equal(ei, g[f"lam_hops{hops}_edge_index"])
        ei = R.multiscale_edges_tri_masked(range(7), hops, str_x, str_x, 1.0)
        np.testing.assert_array_equal(ei, g[f"str_hops{hops}_edge_index"])
    np.testing.assert_array_equal(R.masked_edges("knn", lam_x, dx, None, g["cutout"], 4), g["lam_knn4_edge_index"])
    np.testing.assert_array_equal(R.masked_edges("cutoff", dx, lam_x, g["cutout"], None, 0.6), g["lam_cutoff_edge_index"])
    np.testing.assert_array_equal(R.knn_edges(str_x, dx, 4), g["str_knn4_edge_index"])
    np.testing.assert_array_equal(R.cutoff_edges(dx, str_x, 0.6), g["str_cutoff_edge_index"])
    assert R.grid_reference_distance(str_x) == float(g["str_reference_distance"])


def test_oracle_area_weights_match_reference(golden):
    """SphericalAreaWeights: the oracle's scipy call against the unmodified reference class, every norm."""
    g = golden("area_weights")
    for name in ("o24", "tri3", "random"):
        x = g[f"{name}_x"]
        np.testing.assert_array_equal(R.spherical_area_weights(x, None, "float64"), g[f"{name}_raw64"])
        for norm in [None, "l1", "l2", "unit-max", "unit-range", "unit-std"]:
            np.testing.assert_array_equal(R.spherical_area_weights(x, norm), g[f"{name}_{norm}"])
        # the areas tile the sphere (up to the float32 rounding of the generators)
        np.testing.assert_allclose(g[f"{name}_raw64"].sum(), 4 * np.pi, rtol=1e-7)
