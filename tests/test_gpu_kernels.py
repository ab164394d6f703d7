"""GPU parity of the device-level ops (through the C ABI) against the oracle and the golden fixtures
produced by the unmodified reference.  Index work is bit-exact; attribute tolerances are stated
where used (north star: 1e-6 relative in fp32)."""

import numpy as np
import pytest
import torch

from anemoi_graphs_b200 import grids
from oracle import ref_path as R
from oracle import trimesh_icosphere as TM

pytestmark = pytest.mark.gpu

ATTR_RTOL = 1e-6


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def canon(ei):
    ei = ei.cpu().numpy() if isinstance(ei, torch.Tensor) else np.asarray(ei)
    return R.canonical_sort(ei)


@pytest.fixture(scope="module")
def ops():
    from anemoi_graphs_b200 import ops as _ops

    return _ops


# ------------------------------------------------------------------------------------------------
# search vectors: the error bound the FP32 filter margin (DESIGN.md section 3) is derived from
# ------------------------------------------------------------------------------------------------
def test_search_vectors_within_half_ulp_of_exact(ops):
    lat, lon = grids.uniform_sphere(300000, seed=3)
    x = grids.latlon_deg_to_x(lat, lon).numpy()
    x[:6] = np.array(
        [[np.pi / 2, 0], [-np.pi / 2, 3], [0, 0], [1.0, 2 * np.pi], [0.5, -np.pi], [-0.25, 700.0]], dtype=np.float32
    )
    got = ops.search_vectors(dev(x)).cpu().numpy().astype(np.float64)
    la, lo = x[:, 0].astype(np.float64), x[:, 1].astype(np.float64)
    want = np.stack([np.cos(la) * np.cos(lo), np.cos(la) * np.sin(lo), np.sin(la)], axis=1)
    err = np.abs(got - want)
    # float32 rounding of a value in [-1, 1] is at most 2^-25; the float64 trig adds < 3e-11
    assert err.max() <= 2.0**-25 + 3e-11, err.max()


def test_node_records_layout(ops):
    """Source record = (x, y, z, cos lat, lat, lon, 0, 0); target record's 4th double carries the (lat, lon) bits."""
    lat, lon = grids.uniform_sphere(5000, seed=4)
    x = grids.latlon_deg_to_x(lat, lon).numpy()
    t = ops.NodeTables(dev(x))
    src, dst = t.src_rec.cpu().numpy(), t.dst_rec.cpu().numpy()
    assert src.shape == (5000, 8) and dst.shape == (5000, 4)
    np.testing.assert_array_equal(src[:, 4:6].view(np.int32), x.view(np.int32))
    np.testing.assert_array_equal(src[:, 6:], 0)
    packed = np.ascontiguousarray(dst[:, 3]).view(np.int32).reshape(-1, 2)
    np.testing.assert_array_equal(packed, x.view(np.int32))
    q = dst[:, :3]
    np.testing.assert_allclose((q**2).sum(axis=1), 1.0, rtol=0, atol=1e-12)  # unit quaternion with z = 0
    # the quaternion is evaluated without trigonometry (half-angle square roots): it is scipy's
    # Rotation.from_rotvec(direction_vec(p, z) * arccos(p_z)) (edges/directional.py:19-37) to 1e-15
    from scipy.spatial.transform import Rotation

    xyz = R.latlon_rad_to_cartesian((x[:, 0], x[:, 1]), 1.0).astype(np.float64)
    v = R.direction_vec(xyz.copy(), np.array([0, 0, 1]))
    theta = np.arccos(xyz[:, 2])
    want = Rotation.from_rotvec(np.transpose(v * theta)).as_quat()  # (x, y, z, w)
    sign = np.where(want[:, 3] < 0, -1.0, 1.0)[:, None]
    np.testing.assert_allclose(q, (want * sign)[:, [0, 1, 3]], rtol=0, atol=2e-15)


# ------------------------------------------------------------------------------------------------
# KNN
# ------------------------------------------------------------------------------------------------
def test_knn_toy_matches_reference(ops, golden):
    g = golden("toy")
    with ops.NeighbourIndex(dev(g["hidden_x"]), hint_k=3) as ix:
        ei = ix.knn(dev(g["data_x"]), 3)
    np.testing.assert_array_equal(canon(ei), canon(g["knn3_edge_index"]))
    with ops.NeighbourIndex(dev(g["hidden_x"]), hint_k=4) as ix:
        ei = ix.knn(dev(g["hidden_x"]), 4)  # self query: the node itself is neighbour 0
    # a symmetric mesh queried against itself is all ties at the 4th neighbour: compare with the oracle under
    # the lower-index rule, and with the unmodified reference on the untied queries only
    want, info = R.knn_edges_canonical(g["hidden_x"], g["hidden_x"], 4)
    got = canon(ei)
    np.testing.assert_array_equal(got, want)
    ref = canon(g["hidden_self_knn4_edge_index"])
    tied = info["tied_queries"]
    assert tied.size > 0 and info["untied_mismatch"].size == 0
    np.testing.assert_array_equal(got[:, ~np.isin(got[1], tied)], ref[:, ~np.isin(ref[1], tied)])


def test_knn_o96_res5_bit_exact_modulo_enumerated_ties(ops, golden):
    g = golden("o96_res5")
    lat, lon = grids.octahedral_grid(96)
    dx = grids.latlon_deg_to_x(lat, lon)
    stats = ops.new_stats("cuda")
    with ops.NeighbourIndex(dev(g["hidden_x"]), hint_k=3) as ix:
        ei = ix.knn(dx.cuda(), 3, stats=stats)
    got = canon(ei)
    want, info = R.knn_edges_canonical(g["hidden_x"], dx.numpy(), 3)
    # bit-exact against the oracle under the north-star tie rule (lower source index)
    np.testing.assert_array_equal(got, want)
    # and identical to the unmodified reference on every query without an exact tie
    ref = g["knn3_edge_index"]
    tied = info["tied_queries"]
    np.testing.assert_array_equal(got[:, ~np.isin(got[1], tied)], ref[:, ~np.isin(ref[1], tied)])
    st = stats.cpu().numpy()
    assert st[1] == tied.size == 88  # the kernel's own tie enumeration agrees with the oracle's


@pytest.mark.parametrize("k", [1, 2, 3, 5, 8, 16, 32])
def test_knn_random_sphere_all_k(ops, k):
    lat, lon = grids.uniform_sphere(3000, seed=k)
    ref = grids.latlon_deg_to_x(lat, lon).numpy()
    lat, lon = grids.uniform_sphere(5000, seed=100 + k)
    q = grids.latlon_deg_to_x(lat, lon).numpy()
    with ops.NeighbourIndex(dev(ref), hint_k=k) as ix:
        ei, rd = ix.knn(dev(q), k, return_rdist=True)
    want, info = R.knn_edges_canonical(ref, q, k)
    assert info["tied_queries"].size == 0
    np.testing.assert_array_equal(canon(ei), want)
    # float64 rdist matches the formula to a few ulp
    e = ei.cpu().numpy()
    rd_want = R.rdist64(q[e[1], 0], q[e[1], 1], ref[e[0], 0], ref[e[0], 1])
    np.testing.assert_allclose(rd.cpu().numpy().reshape(-1), rd_want, rtol=1e-13, atol=0)


@pytest.mark.parametrize("k", [3, 16])
def test_knn_incoherent_query_order_is_binned(ops, k, monkeypatch):
    """A shuffled point cloud: large inputs are sampled, found incoherent and searched in spatially binned order.
    The result must not depend on the processing order (forced on / off) and must match the oracle on a subsample."""
    lat, lon = grids.uniform_sphere(40000, seed=11)
    ref = grids.latlon_deg_to_x(lat, lon).numpy()
    lat, lon = grids.uniform_sphere(300000, seed=12)
    q = grids.latlon_deg_to_x(lat, lon).numpy()
    outs = {}
    for mode in ("auto", "0", "1"):
        if mode == "auto":
            monkeypatch.delenv("AGX_KNN_BIN", raising=False)
        else:
            monkeypatch.setenv("AGX_KNN_BIN", mode)
        st = ops.new_stats("cuda")
        with ops.NeighbourIndex(dev(ref), hint_k=k) as ix:
            outs[mode] = (ix.knn(dev(q), k, stats=st).cpu().numpy(), st.cpu().tolist())
    # the same edge SET whatever the processing order (within a query, sources closer than 2^-14 relative may swap:
    # the staged scan orders them by truncated FP32 chord, the per-thread search by exact FP32 chord)
    np.testing.assert_array_equal(canon(outs["0"][0]), canon(outs["1"][0]))
    np.testing.assert_array_equal(outs["auto"][0], outs["1"][0])  # auto = binned here, bit for bit reproducible
    assert outs["0"][1][3] == 0 and outs["auto"][1][3] > 0  # unbinned: no tile could be staged; auto: staged
    sub = np.arange(0, q.shape[0], 37)
    want, info = R.knn_edges_canonical(ref, q[sub], k)
    got = outs["auto"][0].reshape(2, -1, k)[:, sub, :]
    got[1] = np.arange(sub.size)[:, None]
    np.testing.assert_array_equal(canon(got.reshape(2, -1)), want)


def test_knn_sparse_clustered_and_polar(ops):
    """Queries far from every reference point (cap growth), references clustered in one cell, both poles."""
    rng = np.random.default_rng(3)
    ref = np.stack([np.deg2rad(50 + rng.random(400)), np.deg2rad(10 + rng.random(400))], axis=1).astype(np.float32)
    ref = np.concatenate([ref, np.array([[np.pi / 2, 0.0], [-np.pi / 2, 1.0]], dtype=np.float32)])
    lat, lon = grids.uniform_sphere(2000, seed=5)
    q = grids.latlon_deg_to_x(lat, lon).numpy()
    q = np.concatenate([q, np.array([[np.pi / 2, 2.0], [-np.pi / 2, 0.0], [0.0, 0.0], [0.0, 2 * np.pi]], dtype=np.float32)])
    for k in (1, 4):
        for cells in (0, 1, 64):
            with ops.NeighbourIndex(dev(ref), cells_per_face=cells, hint_k=k) as ix:
                ei = ix.knn(dev(q), k)
            want, _ = R.knn_edges_canonical(ref, q, k)
            np.testing.assert_array_equal(canon(ei), want)


def test_knn_search_limit_on_clustered_references(ops):
    """max_radius: exact for queries whose nearest reference point lies within it, -1 / +inf (or a point beyond it)
    for the others - the contract KNNAreaMaskBuilder relies on for limited-area patches (SURVEY.md H5)."""
    ref = grids.latlon_deg_to_x(*grids.lam_patch(150, 150, 10.0)).numpy()  # 22 500 points in a 1500 km patch
    q = grids.latlon_deg_to_x(*grids.uniform_sphere(60000, seed=8)).numpy()
    q = np.concatenate([q, ref[::50] + np.float32(1e-3)])  # and some queries inside the patch
    limit = 300.0 / 6371.0
    with ops.NeighbourIndex(dev(ref), hint_k=1) as ix:
        full, rd_full = ix.knn(dev(q), 1, return_rdist=True)
        lim, rd_lim = ix.knn(dev(q), 1, return_rdist=True, max_radius=limit)
    full, lim = full.cpu().numpy()[0], lim.cpu().numpy()[0]
    d_full = 2.0 * np.arcsin(np.sqrt(rd_full.cpu().numpy()[:, 0]))
    d_lim = 2.0 * np.arcsin(np.sqrt(np.minimum(rd_lim.cpu().numpy()[:, 0], 1.0)))
    near = d_full <= limit
    assert near.sum() > 500 and (~near).sum() > 10000
    np.testing.assert_array_equal(lim[near], full[near])
    np.testing.assert_array_equal(rd_lim.cpu().numpy()[near, 0], rd_full.cpu().numpy()[near, 0])
    assert ((lim[~near] == -1) | (d_lim[~near] > limit)).all()
    assert np.isinf(rd_lim.cpu().numpy()[~near, 0][lim[~near] == -1]).all()
    # the mask the reference computes (generate/masks.py:94-99) from a bounded search
    want = R.knn_area_mask(ref, q, 250.0)
    np.testing.assert_array_equal(d_lim * 6371.0 <= 250.0, want)


def test_knn_argument_errors(ops):
    ref = np.zeros((3, 2), dtype=np.float32)
    with ops.NeighbourIndex(dev(ref)) as ix:
        with pytest.raises(ValueError, match="n_neighbors <= n_samples_fit"):
            ix.knn(dev(ref), 4)
        with pytest.raises(ValueError):
            ix.knn(dev(ref), 0)
        assert ix.knn(dev(np.zeros((0, 2), dtype=np.float32)), 2).shape == (2, 0)
    with pytest.raises(ValueError):
        ops.NeighbourIndex(dev(np.zeros((0, 2), dtype=np.float32)))


# ------------------------------------------------------------------------------------------------
# cut-off
# ------------------------------------------------------------------------------------------------
def test_reference_distance_bits(ops, golden):
    g = golden("o96_res5")
    assert ops.grid_reference_distance(dev(g["hidden_x"])) == float(g["reference_distance"])
    t = golden("toy")
    assert ops.grid_reference_distance(dev(t["hidden_x"])) == R.grid_reference_distance(t["hidden_x"])


def test_cutoff_toy_and_o96(ops, golden):
    t = golden("toy")
    radius = R.cutoff_radius(t["hidden_x"], 0.6)
    with ops.NeighbourIndex(dev(t["data_x"]), hint_radius=radius) as ix:
        ei = ix.radius(dev(t["hidden_x"]), radius)
    np.testing.assert_array_equal(canon(ei), canon(t["cutoff_edge_index"]))

    g = golden("o96_res5")
    lat, lon = grids.octahedral_grid(96)
    dx = grids.latlon_deg_to_x(lat, lon)
    radius = float(g["reference_distance"]) * 0.6
    stats = ops.new_stats("cuda")
    with ops.NeighbourIndex(dx.cuda(), hint_radius=radius) as ix:
        ei = ix.radius(dev(g["hidden_x"]), radius, stats=stats)
    assert ei.shape[1] == 62980  # docs/_static/hetero_data_graph.txt:13
    np.testing.assert_array_equal(canon(ei), g["cutoff_edge_index"])
    assert stats.cpu().numpy()[1] == 0  # no pair within 2^-40 of the threshold
    # output is grouped by query (target) in ascending order
    assert (np.diff(ei[1].cpu().numpy()) >= 0).all()


@pytest.mark.parametrize("radius", [0.0, 1e-4, 0.02, 0.3, 2.0, 3.1])
def test_cutoff_random_radii(ops, radius):
    lat, lon = grids.uniform_sphere(4000, seed=21)
    ref = grids.latlon_deg_to_x(lat, lon).numpy()
    q = ref[:300].copy()  # includes coincident pairs (distance 0, inclusive test)
    with ops.NeighbourIndex(dev(ref), hint_radius=radius) as ix:
        ei = ix.radius(dev(q), radius, dst_base=7)
    want = R.cutoff_edges(ref, q, 1.0, radius=radius)
    want[1] += 7
    np.testing.assert_array_equal(canon(ei), canon(want))


@pytest.mark.parametrize("degree", [6, 40])
def test_cutoff_tile_and_warp_forms_agree_bit_for_bit(ops, degree, monkeypatch):
    """The low-degree tile kernel and the warp-per-query kernel emit the same pairs in the same order, for coherent
    and for shuffled (binned) query orders; checked against the oracle on a subsample."""
    n_ref = 200000
    ref = grids.latlon_deg_to_x(*grids.uniform_sphere(n_ref, seed=21)).numpy()
    q = grids.latlon_deg_to_x(*grids.uniform_sphere(300000, seed=22)).numpy()
    radius = float(np.arccos(1.0 - 2.0 * degree / n_ref))
    outs = {}
    for tile, binned in (("0", "0"), ("1", "0"), ("1", "1"), ("1", None)):
        monkeypatch.setenv("AGX_RADIUS_TILE", tile)
        if binned is None:
            monkeypatch.delenv("AGX_RADIUS_BIN", raising=False)
        else:
            monkeypatch.setenv("AGX_RADIUS_BIN", binned)
        with ops.NeighbourIndex(dev(ref), hint_radius=radius) as ix:
            outs[(tile, binned)] = ix.radius(dev(q), radius).cpu().numpy()
    for key, val in outs.items():
        np.testing.assert_array_equal(val, outs[("0", "0")], err_msg=str(key))
    sub = np.arange(0, q.shape[0], 61)
    want = R.canonical_sort(R.cutoff_edges(ref, q[sub], 1.0, radius=radius))
    got = outs[("1", None)]
    pick = np.isin(got[1], sub)
    got = got[:, pick]
    got[1] = np.searchsorted(sub, got[1])
    np.testing.assert_array_equal(canon(got), want)


def test_cutoff_radius_beyond_pi_connects_everything(ops):
    """For r >= pi every point is within reach.  (sklearn itself is not monotone there: its leaf test uses
    sin^2(r/2), which DEcreases past pi, while whole-node acceptance uses r - the result depends on the tree
    layout; the great-circle answer is 'all pairs'.)"""
    lat, lon = grids.uniform_sphere(500, seed=2)
    ref = grids.latlon_deg_to_x(lat, lon)
    with ops.NeighbourIndex(ref.cuda()) as ix:
        assert ix.radius(ref[:40].cuda(), 3.2).shape[1] == 40 * 500
        assert ix.radius(ref[:40].cuda(), float(np.pi)).shape[1] == 40 * 500


# ------------------------------------------------------------------------------------------------
# icosphere + multi-scale
# ------------------------------------------------------------------------------------------------
def test_icosphere_bit_exact(ops, golden):
    ico = ops.Icosphere(5)
    v, f = TM.icosphere(5)
    np.testing.assert_array_equal(ico.vertices.cpu().numpy().view(np.int64), v.view(np.int64))
    np.testing.assert_array_equal(ico.faces(5).cpu().numpy(), f)
    for lvl in range(5):
        np.testing.assert_array_equal(ico.faces(lvl).cpu().numpy(), TM.icosphere(lvl)[1])
    g = golden("o96_res5")
    ll = ico.latlon.cpu().numpy()
    np.testing.assert_array_equal(ll[g["hidden_node_ordering"]].view(np.int32), g["hidden_x"].view(np.int32))


@pytest.mark.parametrize("hops", [1, 2, 3])
def test_multiscale_res3(ops, golden, hops):
    g = golden("tri_nodes")
    ico = ops.Icosphere(3)
    ei = ops.multiscale_tri_edges(ico, [0, 1, 2, 3], hops, dev(g["res3_node_ordering"]))
    np.testing.assert_array_equal(ei.cpu().numpy(), g[f"res3_hops{hops}_edge_index"])  # already canonical


def test_multiscale_level_list_and_o96(ops, golden):
    g = golden("tri_nodes")
    ico = ops.Icosphere(3)
    ei = ops.multiscale_tri_edges(ico, [1, 3], 1, dev(g["res3_node_ordering"]))
    np.testing.assert_array_equal(ei.cpu().numpy(), g["res_1_3_hops1_edge_index"])
    o = golden("o96_res5")
    ico = ops.Icosphere(5)
    ei = ops.multiscale_tri_edges(ico, list(range(6)), 1, dev(o["hidden_node_ordering"]))
    assert ei.shape[1] == 81900  # docs/_static/hetero_data_graph.txt:19
    np.testing.assert_array_equal(ei.cpu().numpy(), o["multiscale_edge_index"])


# ------------------------------------------------------------------------------------------------
# attributes
# ------------------------------------------------------------------------------------------------
NORMS = [None, "l1", "l2", "unit-max", "unit-range", "unit-std"]


def _n(norm):
    return "none" if norm is None else norm.replace("-", "_")


def test_node_tables_match_numpy_float32(ops):
    lat, lon = grids.uniform_sphere(200000, seed=9)
    x = grids.latlon_deg_to_x(lat, lon).numpy()
    x[:4] = np.array([[np.pi / 2, 0], [-np.pi / 2, 3], [0, 0], [1.0, 2 * np.pi]], dtype=np.float32)
    t = ops.NodeTables(dev(x), with_rotation=True)
    want = R.latlon_rad_to_cartesian((x[:, 0], x[:, 1]), 1.0)
    assert want.dtype == np.float32
    got = t.xyzc.cpu().numpy()
    np.testing.assert_array_equal(got[:, :3].view(np.int32), want.view(np.int32))  # numpy's float32 bits
    np.testing.assert_array_equal(got[:, 3].view(np.int32), np.cos(x[:, 0]).view(np.int32))


def test_attributes_toy_all_norms(ops, golden):
    g = golden("toy")
    dx, hx = g["data_x"], g["hidden_x"]
    cases = (
        ("cutoff", dx, hx, g["cutoff_edge_index"]),
        ("ms1", hx, hx, g["multiscale1_edge_index"]),
        ("knn3", hx, dx, g["knn3_edge_index"]),
    )
    for tag, sx, tx, ei in cases:
        src = ops.NodeTables(dev(sx), with_rotation=False)
        dst = ops.NodeTables(dev(tx), with_rotation=True)
        e = dev(ei)
        for norm in NORMS:
            ln, dr = ops.edge_attributes(e, src, dst, length_norm=norm, direction_norm=norm)
            want = g[f"{tag}_len_{_n(norm)}"]
            # unit-range subtracts the minimum: values next to it are differences of nearly equal float32
            # numbers, so the tolerance there is absolute (1e-6 of the attribute's range)
            atol = ATTR_RTOL * np.abs(want).max() if norm == "unit-range" else 0
            np.testing.assert_allclose(ln.cpu().numpy(), want, rtol=ATTR_RTOL, atol=atol, err_msg=f"{tag} len {norm}")
            want = g[f"{tag}_dir_rot_{_n(norm)}"]
            np.testing.assert_allclose(dr.cpu().numpy(), want, rtol=ATTR_RTOL, atol=ATTR_RTOL * np.abs(want).max())
        ln, dr = ops.edge_attributes(
            e, src, dst, length_norm="unit-max", length_invert=True, direction_norm="unit-std", direction_rotated=False
        )
        np.testing.assert_allclose(ln.cpu().numpy(), g[f"{tag}_len_inv_unit_max"], rtol=0, atol=ATTR_RTOL)
        want = g[f"{tag}_dir_norot_unit_std"]
        np.testing.assert_allclose(dr.cpu().numpy(), want, rtol=ATTR_RTOL, atol=ATTR_RTOL * np.abs(want).max())


def test_attribute_edge_cases(ops, golden):
    g = golden("attr_vectors")
    src, dst = g["src"], g["dst"]
    n = src.shape[0]
    ei = dev(np.stack([np.arange(n), np.arange(n)]).astype(np.int32))
    s = ops.NodeTables(dev(src), with_rotation=False)
    d = ops.NodeTables(dev(dst), with_rotation=True)
    ln, dr = ops.edge_attributes(ei, s, d)
    ln, dr = ln.cpu().numpy()[:, 0], dr.cpu().numpy()
    want_len, want_dir = g["length"], g["dir_rotated"]
    finite = np.isfinite(want_len)
    np.testing.assert_allclose(ln[finite], want_len[finite], rtol=ATTR_RTOL, atol=0)
    assert np.isnan(ln[~finite]).all()  # antipodal pair: a > 1 in float32, NaN in the reference too
    # coincident endpoints (rows 7, 8) have no defined direction: the reference returns amplified rounding noise
    defined = np.ones(n, dtype=bool)
    defined[[7, 8]] = False
    np.testing.assert_allclose(dr[defined], want_dir[defined], rtol=0, atol=2e-6)
    _, nr = ops.edge_attributes(ei, s, d, length=False, direction_rotated=False)
    np.testing.assert_array_equal(nr.cpu().numpy(), g["dir_nonrotated"])


def test_attributes_o96_samples(ops, golden):
    g = golden("o96_res5")
    lat, lon = grids.octahedral_grid(96)
    dx = grids.latlon_deg_to_x(lat, lon).numpy()
    hx = g["hidden_x"]
    stride = int(g["attr_sample_stride"])
    for tag, sx, tx in (("cutoff", dx, hx), ("multiscale", hx, hx), ("knn3", hx, dx)):
        ei = g[f"{tag}_edge_index"]
        src = ops.NodeTables(dev(sx), with_rotation=False)
        dst = ops.NodeTables(dev(tx), with_rotation=True)
        ln, dr = ops.edge_attributes(dev(ei), src, dst, length_norm="unit-std", direction_norm="unit-std")
        np.testing.assert_allclose(ln.cpu().numpy()[::stride], g[f"{tag}_edge_length_sample"], rtol=ATTR_RTOL, atol=0)
        want = g[f"{tag}_edge_dirs_sample"]
        np.testing.assert_allclose(dr.cpu().numpy()[::stride], want, rtol=ATTR_RTOL, atol=ATTR_RTOL * np.abs(want).max())
        np.testing.assert_allclose(ln.double().sum().item(), float(g[f"{tag}_edge_length_sum64"]), rtol=1e-6)
        np.testing.assert_allclose(dr.double().abs().sum().item(), float(g[f"{tag}_edge_dirs_abs_sum64"]), rtol=1e-6)


# ------------------------------------------------------------------------------------------------
# small entry points used by the provisional-numbering path, exercised directly through the C ABI
# ------------------------------------------------------------------------------------------------
def test_max_positive_entry_point():
    """agx_max_positive: `dists[dists > 0].max()` (utils.py:62-63) + its first flat position; the result comes back
    through agx_readback (mapped pinned memory, not the copy engine)."""
    from ctypes import byref, c_double, c_int64

    from anemoi_graphs_b200 import _cabi

    lib = _cabi.load_library()
    rng = np.random.default_rng(3)
    v = rng.normal(size=100001)
    v[::7] = 0.0
    v[12345] = v[54321] = 9.5  # the maximum twice: the lower position is reported
    value, index = c_double(), c_int64()
    _cabi.check(lib.agx_max_positive(dev(v).data_ptr(), v.size, byref(value), byref(index), _cabi.current_stream()))
    assert value.value == 9.5 and index.value == 12345
    neg = dev(-np.abs(v))
    _cabi.check(lib.agx_max_positive(neg.data_ptr(), v.size, byref(value), byref(index), _cabi.current_stream()))
    assert index.value == -1  # nothing strictly positive


def test_order_resolve_entry_point():
    """agx_order_resolve == arange(n)[index_latitude][index_longitude[::-1]] (generate/utils.py:30-33), its inverse and
    coords[node_ordering] (nodes/builders/from_refined_icosahedron.py:66)."""
    from anemoi_graphs_b200 import _cabi

    lib = _cabi.load_library()
    rng = np.random.default_rng(4)
    n = 50003
    x = rng.normal(size=(n, 2)).astype(np.float32)
    il = np.argsort(x[:, 1])
    ilon = np.argsort(x[il][:, 0])
    want = np.arange(n)[il][ilon[::-1]]
    x_out = torch.empty((n, 2), dtype=torch.float32, device="cuda")
    order = torch.empty(n, dtype=torch.int64, device="cuda")
    rank = torch.empty(n, dtype=torch.int64, device="cuda")
    xd, ild, ilond = dev(x), dev(il.astype(np.int64)), dev(ilon.astype(np.int64))
    _cabi.check(
        lib.agx_order_resolve(ild.data_ptr(), ilond.data_ptr(), n, xd.data_ptr(), x_out.data_ptr(), order.data_ptr(),
                              rank.data_ptr(), _cabi.current_stream())
    )  # fmt: skip
    np.testing.assert_array_equal(order.cpu().numpy(), want)
    np.testing.assert_array_equal(rank.cpu().numpy()[want], np.arange(n))
    np.testing.assert_array_equal(x_out.cpu().numpy(), x[want])


def test_knn_flag_and_redecide_equals_final_numbering(ops, golden):
    """Search with permuted source labels + flags, relabel, re-decide the flagged queries: identical (as a set per
    query) to searching with the final labels - including the tied queries of the O96 -> res 5 decoder."""
    g = golden("o96_res5")
    hx = g["hidden_x"]
    lat, lon = grids.octahedral_grid(96)
    dx = grids.latlon_deg_to_x(lat, lon).numpy()
    k, nq, n = 3, dx.shape[0], hx.shape[0]
    rng = np.random.default_rng(5)
    perm = rng.permutation(n)  # provisional label p is final node perm[p]
    hx_prov = hx[perm]
    flags = torch.zeros(nq, dtype=torch.uint8, device="cuda")
    with ops.NeighbourIndex(dev(hx_prov), hint_k=k) as index:
        out = index.knn(dev(dx), k, tie_flags=flags)
    assert int(flags.sum().item()) > 0  # the mirror-plane ties of this configuration (DESIGN.md section 4)
    out[0] = dev(perm.astype(np.int32))[out[0].long()]  # provisional -> final labels
    with ops.NeighbourIndex(dev(hx), hint_k=k) as index:
        index.knn_redecide(dev(dx), k, out, flags)
        want = index.knn(dev(dx), k)
    np.testing.assert_array_equal(canon(out), canon(want))
    oracle, info = R.knn_edges_canonical(hx, dx, k)  # the lower-index tie rule on the final labels
    assert info["tied_queries"].size == int(flags.sum().item()) == 88
    np.testing.assert_array_equal(canon(out), oracle)


def test_knn_ranked_redecide_needs_no_second_index(ops, golden):
    """``agx_knn_redecide_ranked``: the flagged queries are re-decided against the SAME provisionally labelled index
    (ties by ``rank[label]``, provisional labels written), then ONE ``agx_relabel_rows`` launch gives the final row -
    identical to searching the finally labelled points."""
    g = golden("o96_res5")
    hx = g["hidden_x"]
    dx = grids.latlon_deg_to_x(*grids.octahedral_grid(96)).numpy()
    k, nq, n = 3, dx.shape[0], hx.shape[0]
    rng = np.random.default_rng(6)
    perm = rng.permutation(n)  # provisional label p is final node perm[p]  => rank = perm, order = its inverse
    rank = dev(perm.astype(np.int64))
    order = torch.empty_like(rank)
    order[rank] = torch.arange(n, dtype=torch.int64, device="cuda")
    flags = torch.zeros(nq, dtype=torch.uint8, device="cuda")
    with ops.NeighbourIndex(dev(_prov_coords(hx, perm)), hint_k=k) as index:
        out = index.knn(dev(dx), k, tie_flags=flags)
        before = out.clone()
        index.knn_redecide(dev(dx), k, out, flags, rank=rank, order=order)
    assert int(flags.sum().item()) == 88
    changed = (before[0] != out[0]).view(nq, k).any(dim=1)
    assert int(changed.sum().item()) > 0 and bool((flags[changed] == 1).all())  # only flagged queries are touched
    other = torch.arange(7, dtype=torch.int32, device="cuda")  # a second row rides along in the same launch
    want_other = rank[other.long()].to(torch.int32)
    ops.relabel_rows([out[0], other], rank)
    np.testing.assert_array_equal(other.cpu().numpy(), want_other.cpu().numpy())
    oracle, info = R.knn_edges_canonical(hx, dx, k)  # the lower-index tie rule on the final labels
    np.testing.assert_array_equal(canon(out), oracle)


def _prov_coords(hx: np.ndarray, perm: np.ndarray) -> np.ndarray:
    """Coordinates in provisional numbering when provisional label p is final node perm[p]."""
    return hx[perm]


def test_attribute_flag_modes_of_the_stats_entry_point_split_the_statistics(ops, golden):
    """``agx_edge_attrs_stats`` flag modes: "skip" + "only" partition the statistics of an edge set by target flag, and
    the deferred three-step evaluation (raw / patch / apply) equals the one-call result."""
    g = golden("toy")
    dx, hx = g["data_x"], g["hidden_x"]
    ei = dev(g["knn3_edge_index"].astype(np.int32))
    src, dst = ops.NodeTables(dev(hx)), ops.NodeTables(dev(dx))
    flags = torch.zeros(dx.shape[0], dtype=torch.uint8, device="cuda")
    flags[::7] = 1
    for norm in ("unit-std", "unit-range", "l1"):
        want_len, want_dir = ops.edge_attributes(ei, src, dst, length_norm=norm, direction_norm=norm)
        job = ops.DeferredEdgeAttributes(ei, src, dst, flags, length_norm=norm, direction_norm=norm)
        job.raw()
        job.out_len[(flags[ei[1].long()] == 1)] = float("nan")  # what "patch" must overwrite
        job.patch()
        job.apply()
        np.testing.assert_allclose(job.out_len.cpu().numpy(), want_len.cpu().numpy(), rtol=3e-7)
        np.testing.assert_allclose(job.out_dir.cpu().numpy(), want_dir.cpu().numpy(), rtol=3e-7, atol=1e-7)
        # the two statistics sets add up to the whole set's
        whole = torch.empty(8, dtype=torch.float64, device="cuda")
        raw_len, raw_dir = torch.empty_like(want_len), torch.empty_like(want_dir)
        check = __import__("anemoi_graphs_b200._cabi", fromlist=["check"]).check
        check(ops.load_library().agx_edge_attrs_stats(ei[0].data_ptr(), ei[1].data_ptr(), int(ei.shape[1]), src.src_rec.data_ptr(),
              None, dst.dst_rec.data_ptr(), None, 1, 1, 1, raw_len.data_ptr(), raw_dir.data_ptr(), whole.data_ptr(),
              ops._attr_workspace(ei.device).data_ptr(), None, 0, None, None, 0,
              torch.cuda.current_stream().cuda_stream))  # fmt: skip
        st = job.stats.cpu().numpy()
        w = whole.cpu().numpy()
        np.testing.assert_allclose(st[0, [0, 1, 4, 5]] + st[1, [0, 1, 4, 5]], w[[0, 1, 4, 5]], rtol=1e-12)
        np.testing.assert_array_equal(np.minimum(st[0, [2, 6]], st[1, [2, 6]]), w[[2, 6]])
        np.testing.assert_array_equal(np.maximum(st[0, [3, 7]], st[1, [3, 7]]), w[[3, 7]])


def test_attributes_from_coordinates_equal_tabulated_records(ops, golden):
    """The attribute kernel evaluates per-node quantities from the 8-byte coordinates for large node sets and gathers
    tabulated records for small ones: all four combinations give BIT-identical attributes - also for edge lists whose
    rows are not 8-byte aligned (odd edge counts: scalar lanes instead of adjacent pairs) and at the poles."""
    g = golden("toy")
    dx, hx = g["data_x"].copy(), g["hidden_x"]
    dx[:3] = np.array([[np.pi / 2, 0.0], [-np.pi / 2, 1.0], [0.0, 0.0]], dtype=np.float32)
    for name, sx, tx in (("knn3", hx, dx), ("cutoff", dx, hx)):
        ei_np = g[f"{name}_edge_index"].astype(np.int32)
        for cut in (0, 1):  # odd / even number of edges: row 1 of the (2, E) list is / is not 8-byte aligned
            ei = dev(np.ascontiguousarray(ei_np[:, : ei_np.shape[1] - cut]))
            outs = []
            for ts, tt in ((True, True), (False, True), (True, False), (False, False)):
                src, dst = ops.NodeTables(dev(sx), tabulate=ts), ops.NodeTables(dev(tx), tabulate=tt)
                ln, dr = ops.edge_attributes(ei, src, dst, length_norm="unit-max", direction_norm="unit-max")
                outs.append((ln.cpu().numpy(), dr.cpu().numpy()))
            if name == "knn3" and cut == 0:  # the same list walked by TARGET (k edges per target), both target forms
                for tt in (True, False):
                    src, dst = ops.NodeTables(dev(sx), tabulate=True), ops.NodeTables(dev(tx), tabulate=tt)
                    ln, dr = ops.edge_attributes(ei, src, dst, length_norm="unit-max", direction_norm="unit-max", regular_k=3)
                    outs.append((ln.cpu().numpy(), dr.cpu().numpy()))
            for ln, dr in outs[1:]:
                np.testing.assert_array_equal(ln.view(np.int32), outs[0][0].view(np.int32))
                np.testing.assert_array_equal(dr.view(np.int32), outs[0][1].view(np.int32))
            e = ei.cpu().numpy()
            want_dir = R.edge_direction(sx, tx, e, "unit-max")
            np.testing.assert_allclose(outs[0][1], want_dir, rtol=1e-6, atol=1e-6 * np.abs(want_dir).max())
            np.testing.assert_allclose(outs[0][0], R.edge_length(sx, tx, e, "unit-max"), rtol=1e-6)


def _pool_high_water(reset: bool = False) -> int:
    """High-water mark of the device's default stream-ordered memory pool (what libagx_b200's scratch comes from)."""
    from cuda.bindings import driver as dr
    from cuda.bindings import runtime as rt

    err, pool = rt.cudaDeviceGetDefaultMemPool(torch.cuda.current_device())
    assert int(err) == 0
    if reset:
        (err,) = rt.cudaMemPoolSetAttribute(pool, rt.cudaMemPoolAttr.cudaMemPoolAttrUsedMemHigh, dr.cuuint64_t(0))
        assert int(err) == 0
    err, value = rt.cudaMemPoolGetAttribute(pool, rt.cudaMemPoolAttr.cudaMemPoolAttrUsedMemHigh)
    assert int(err) == 0
    return int(value)


def test_concat_edges_kernel_matches_torch_unique_and_reference_order():
    """utils.concat_edges (utils.py:66-81): sorted unique columns of two edge lists - small case against the reference's
    own expression, with duplicates inside and across the lists and an empty list."""
    from anemoi_graphs_b200.utils import concat_edges_device

    rng = np.random.default_rng(3)
    e1 = rng.integers(0, 50, size=(2, 4000)).astype(np.int32)
    e2 = rng.integers(0, 50, size=(2, 3001)).astype(np.int32)
    got = concat_edges_device(dev(e1), dev(e2), 50, 50).cpu()
    want = torch.unique(torch.cat([torch.from_numpy(e1), torch.from_numpy(e2)], dim=1), dim=1)  # the reference's line
    assert got.dtype == torch.int32 and torch.equal(got, want)
    assert torch.equal(concat_edges_device(dev(e1), dev(e2)).cpu(), want)  # node counts unknown: all key bits sorted
    empty = torch.empty((2, 0), dtype=torch.int32, device="cuda")
    assert torch.equal(concat_edges_device(dev(e1), empty, 50, 50).cpu(), torch.unique(torch.from_numpy(e1), dim=1))
    assert concat_edges_device(empty, empty, 50, 50).shape == (2, 0)


def test_concat_edges_120m_edges_within_twice_the_output():
    """>= 100 M edges (VERDICT r01 item 8): two 60 M-edge lists over 6.6 M x 164 k nodes, 25 % of the second duplicating
    the first.  Sorted, unique, the right count - and the memory beyond the result (the kernel's scratch high-water mark
    + the worst-case slack of the result allocation, which doubles as the sort's second buffer) stays well within 2 x the
    result, where cat -> int64 -> torch.unique needs > 5 x."""
    from anemoi_graphs_b200.utils import concat_edges_device

    n_src, n_dst, m = 6_599_680, 163_842, 60_000_000
    g = torch.Generator(device="cuda").manual_seed(1)
    e1 = torch.stack([torch.randint(0, n_src, (m,), device="cuda", generator=g, dtype=torch.int32),
                      torch.randint(0, n_dst, (m,), device="cuda", generator=g, dtype=torch.int32)])  # fmt: skip
    e2 = torch.stack([torch.randint(0, n_src, (m,), device="cuda", generator=g, dtype=torch.int32),
                      torch.randint(0, n_dst, (m,), device="cuda", generator=g, dtype=torch.int32)])  # fmt: skip
    e2[:, : m // 4] = e1[:, : m // 4]
    torch.cuda.synchronize()
    _pool_high_water(reset=True)
    out = concat_edges_device(e1, e2, n_src, n_dst)
    torch.cuda.synchronize()
    peak = _pool_high_water()
    out_bytes = out.numel() * 4
    slack = out.untyped_storage().nbytes() - out_bytes  # the allocation is sized for "no duplicates"
    assert peak + slack <= 1.5 * out_bytes + (64 << 20), (peak, slack, out_bytes)
    key = (out[0].to(torch.int64) << 32) | out[1].to(torch.int64)
    assert bool((key[1:] > key[:-1]).all())  # strictly ascending (src, dst): sorted and unique
    del key
    # the right set: the distinct keys of the inputs, counted independently in two halves of the key space
    k1 = (e1[0].to(torch.int64) << 32) | e1[1].to(torch.int64)
    k2 = (e2[0].to(torch.int64) << 32) | e2[1].to(torch.int64)
    want = torch.unique(torch.cat([k1, k2]))
    assert want.numel() == out.shape[1]
    assert torch.equal(want, (out[0].to(torch.int64) << 32) | out[1].to(torch.int64))


def test_masked_searches_write_original_node_indices(ops, golden):
    """``ops.output_maps``: undo_masking fused into the KNN / cut-off writes equals searching the masked coordinates and
    mapping the compact indices back afterwards (edges/builder.py:176-193)."""
    g = golden("toy")
    dx, hx = g["data_x"], g["hidden_x"]
    rng = np.random.default_rng(11)
    src_sel = np.sort(rng.choice(hx.shape[0], size=hx.shape[0] // 2, replace=False)).astype(np.int64)
    dst_sel = np.sort(rng.choice(dx.shape[0], size=dx.shape[0] // 3, replace=False)).astype(np.int64)
    with ops.NeighbourIndex(dev(hx[src_sel]), hint_k=3) as ix:
        plain = ix.knn(dev(dx[dst_sel]), 3).cpu().numpy()
        with ops.output_maps(dev(src_sel), dev(dst_sel)):
            fused = ix.knn(dev(dx[dst_sel]), 3).cpu().numpy()
        again = ix.knn(dev(dx[dst_sel]), 3).cpu().numpy()  # the maps are gone after the block
    np.testing.assert_array_equal(fused, np.stack([src_sel[plain[0]], dst_sel[plain[1]]]).astype(np.int32))
    np.testing.assert_array_equal(again, plain)
    with ops.NeighbourIndex(dev(dx[dst_sel]), hint_radius=0.3) as ix:
        plain = ix.radius(dev(hx[src_sel]), 0.3).cpu().numpy()
        with ops.output_maps(dev(dst_sel), dev(src_sel)):
            fused = ix.radius(dev(hx[src_sel]), 0.3).cpu().numpy()
    np.testing.assert_array_equal(fused, np.stack([dst_sel[plain[0]], src_sel[plain[1]]]).astype(np.int32))
