"""Adversarial parity of the neighbour searches: every KNN template instantiation (CAP = 4 / 8 / 17 / 33 / 65) and
every branch of the KNN kernel (staged, stage overflow, cap growth, whole sphere, float64 re-decision, search limit),
exact-duplicate tie groups wider than the list and the stage, cube edges / corners / cell borders, the cut-off
threshold, and the counting backbone (exclusive scan, flag compaction).  Every result is compared with a float64
reference of the same operation: a brute-force all-pairs search here, or ``oracle/exact_search``."""

import math
from ctypes import byref, c_int64

import numpy as np
import pytest
import torch

from anemoi_graphs_b200 import grids
from oracle import exact_search as X
from oracle import ref_path as R

TAU = 2.0**-40
INT32_MAX = 2**31 - 1
SCAN_TILE = 512 * 8  # agx_util.cu: SCAN_THREADS * SCAN_ITEMS
CAP_K = (3, 7, 16, 32, 64)  # one k per KNN template instantiation: CAP = 4, 8, 17, 33, 65


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def canon(ei):
    ei = ei.cpu().numpy() if isinstance(ei, torch.Tensor) else np.asarray(ei)
    return R.canonical_sort(ei)


def x_deg(lat, lon) -> np.ndarray:
    return grids.latlon_deg_to_x(np.asarray(lat, dtype=np.float64), np.asarray(lon, dtype=np.float64)).numpy()


def xyz_to_x(xyz) -> np.ndarray:
    """float32 (lat, lon) radians of unit vectors (rows of xyz, any length)."""
    xyz = np.asarray(xyz, dtype=np.float64)
    xyz = xyz / np.linalg.norm(xyz, axis=1, keepdims=True)
    return np.stack([np.arcsin(np.clip(xyz[:, 2], -1, 1)), np.arctan2(xyz[:, 1], xyz[:, 0])], axis=1).astype(np.float32)


def ulp_neighbours(x: np.ndarray) -> np.ndarray:
    """x and every point one float32 ulp away in lat or lon."""
    x = np.asarray(x, dtype=np.float32)
    out = [x]
    for col in (0, 1):
        for to in (np.inf, -np.inf):
            y = x.copy()
            y[:, col] = np.nextafter(y[:, col], np.float32(to))
            out.append(y)
    return np.concatenate(out)


def clustered(n_top: int, n_mid: int, n_leaf: int, seed: int) -> np.ndarray:
    """3-level clustered cloud: n_top centres on the sphere, n_mid sub-centres within 0.2 rad of each, n_leaf points
    within 3e-3 rad of each sub-centre."""
    rng = np.random.default_rng(seed)
    lat, lon = grids.uniform_sphere(n_top, seed=seed)
    c = R.latlon_rad_to_cartesian((np.deg2rad(lat), np.deg2rad(lon)), 1.0).astype(np.float64)
    pts = []
    for p in c:
        for _ in range(n_mid):
            s = p + rng.normal(scale=0.2, size=3)
            s /= np.linalg.norm(s)
            pts.append(s + rng.normal(scale=3e-3, size=(n_leaf, 3)))
    return xyz_to_x(np.concatenate(pts))


# ------------------------------------------------------------------------------------------------
# brute-force reference: all pairs, float64 rdist on the float32 inputs, lower-index rule for ties of any width
# ------------------------------------------------------------------------------------------------
def all_rdist(ref: np.ndarray, q: np.ndarray) -> np.ndarray:
    """(nq, n_ref) float64 sklearn rdist (``ref_path.rdist64``, x1 = query)."""
    return R.rdist64(q[:, 0:1], q[:, 1:2], ref[None, :, 0], ref[None, :, 1])


def brute_knn(ref: np.ndarray, q: np.ndarray, k: int, rd: np.ndarray | None = None, tau: float = TAU):
    """``(edge_index sorted by (dst, src), tied (nq,) bool)``: per query the k nearest reference points; a tie group
    is every point within ``tau`` (relative) of the k-th smallest rdist and its LOWER indices are kept (the rule of
    ``ref_path.knn_edges_canonical``, without a limit on the group's width).  A query is tied when the group reaches
    past position k."""
    if rd is None:
        rd = all_rdist(ref, q)
    nq = rd.shape[0]
    r_k = np.partition(rd, k - 1, axis=1)[:, k - 1]
    group = np.abs(rd - r_k[:, None]) <= tau * r_k[:, None]
    below = (rd < r_k[:, None]) & ~group
    tied = (below | group).sum(axis=1) > k
    chosen = np.empty((nq, k), dtype=np.int64)
    for i in range(nq):
        b = np.nonzero(below[i])[0]
        g = np.nonzero(group[i])[0]  # ascending index
        chosen[i] = np.sort(np.concatenate([b, g[: k - b.size]]))
    dst = np.repeat(np.arange(nq), k)
    return np.stack([chosen.reshape(-1), dst]).astype(np.int32), tied


def oracle_knn(ref, q, k, extra: int = 8):
    want, info = X.knn_edges_canonical(ref, q, k, extra=extra)
    tied = np.zeros(q.shape[0], dtype=bool)
    tied[info["tied_queries"]] = True
    return want, tied


def assert_rows_ascending(src: np.ndarray, rd: np.ndarray) -> None:
    """Each row ascending (rdist, index) under the 2^-40 tie rule; missing slots (-1, +inf) last."""
    r0, r1, i0, i1 = rd[:, :-1], rd[:, 1:], src[:, :-1], src[:, 1:]
    both_inf = np.isinf(r0) & np.isinf(r1)
    with np.errstate(invalid="ignore"):
        tie = np.isfinite(r0) & np.isfinite(r1) & (np.abs(r0 - r1) <= TAU * np.maximum(r0, r1))
    ok = both_inf | np.where(tie, i0 < i1, r0 < r1)
    assert ok.all(), np.argwhere(~ok)[:5]
    assert ((src == -1) == np.isinf(rd)).all()


def assert_rdist_exact(ref, q, src, rd) -> None:
    have = src >= 0
    qi = np.nonzero(have)[0]
    want = R.rdist64(q[qi, 0], q[qi, 1], ref[src[have], 0], ref[src[have], 1])
    np.testing.assert_allclose(rd[have], want, rtol=1e-13, atol=0)


@pytest.fixture(scope="module")
def ops():
    from anemoi_graphs_b200 import ops as _ops

    return _ops


def run_knn(ops, ref, q, k, cells=0, **kw):
    stats = ops.new_stats("cuda")
    with ops.NeighbourIndex(dev(ref), cells_per_face=cells, hint_k=k) as ix:
        out = ix.knn(dev(q), k, stats=stats, **kw)
    if isinstance(out, tuple):
        return out[0].cpu().numpy(), out[1].cpu().numpy(), stats.cpu().numpy()
    return out.cpu().numpy(), None, stats.cpu().numpy()


# ------------------------------------------------------------------------------------------------
# the reference itself (no GPU)
# ------------------------------------------------------------------------------------------------
def test_brute_force_reference_matches_exact_search():
    """The brute-force helper agrees with ``exact_search`` (edge sets and tied queries) on a cloud with exact
    duplicates, mirror-image points and queries on both."""
    base = x_deg(*grids.uniform_sphere(600, seed=41))
    dup = np.repeat(base[:30], 3, axis=0)  # groups of 3 identical points (plus the original: 4)
    mirror = np.array([[0.3, 0.01], [0.3, -0.01], [-0.7, 2.0], [-0.7, 2.02]], dtype=np.float32)
    ref = np.concatenate([base, dup, mirror])
    ref = ref[np.random.default_rng(2).permutation(ref.shape[0])]
    q = np.concatenate([base[:60], np.array([[0.3, 0.0], [-0.7, 2.01]], dtype=np.float32), x_deg(*grids.uniform_sphere(200, seed=42))])
    n_tied = 0
    for k in (1, 2, 3, 4, 5, 9):
        got, tied = brute_knn(ref, q, k)
        want, want_tied = oracle_knn(ref, q, k, extra=ref.shape[0])
        np.testing.assert_array_equal(got, want)
        np.testing.assert_array_equal(tied, want_tied)
        n_tied += int(tied.sum())
    assert n_tied > 100


# ------------------------------------------------------------------------------------------------
# 1. k ladder
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ladder_sets():
    uni_ref = x_deg(*grids.uniform_sphere(4000, seed=51))
    uni_q = x_deg(*grids.uniform_sphere(3000, seed=52))
    cl_ref = clustered(4, 6, 150, seed=53)  # 3600 points
    cl_q = np.concatenate([clustered(4, 6, 40, seed=53), x_deg(*grids.uniform_sphere(1000, seed=54))])
    return {"uniform": (uni_ref, uni_q), "clustered": (cl_ref, cl_q)}


@pytest.mark.gpu
@pytest.mark.parametrize("cloud", ["uniform", "clustered"])
@pytest.mark.parametrize("k", [1, 3, 4, 7, 8, 16, 17, 32, 33, 48, 64])
def test_knn_k_ladder(ops, ladder_sets, cloud, k):
    ref, q = ladder_sets[cloud]
    ei, rd, _ = run_knn(ops, ref, q, k, return_rdist=True)
    want, _ = oracle_knn(ref, q, k)
    np.testing.assert_array_equal(canon(ei), want)
    src = ei[0].reshape(-1, k)
    assert_rdist_exact(ref, q, src, rd)
    assert_rows_ascending(src, rd)
    assert (np.diff(rd, axis=1) >= 0).all()
    # without rdist: the same set (the order inside a row is not defined)
    ei2, _, _ = run_knn(ops, ref, q, k)
    np.testing.assert_array_equal(canon(ei2), want)


# ------------------------------------------------------------------------------------------------
# 2. every branch of the KNN kernel, proven taken by the stats counters
# ------------------------------------------------------------------------------------------------
def _both_orders(ops, monkeypatch, ref, q, k, **kw):
    """Runs with the queries walked as given and spatially binned: the same sets.  Returns the as-given run."""
    outs = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("AGX_KNN_BIN", mode)
        outs[mode] = run_knn(ops, ref, q, k, **kw)
    monkeypatch.delenv("AGX_KNN_BIN")
    np.testing.assert_array_equal(canon(outs["0"][0]), canon(outs["1"][0]))
    return outs["0"], outs["1"]


def _coherent_queries(n: int) -> np.ndarray:
    return x_deg(*grids.octahedral_grid(n))  # grid order: consecutive points are neighbours


@pytest.mark.gpu
@pytest.mark.parametrize("k", CAP_K)
def test_knn_path_staged(ops, monkeypatch, k):
    """A tight query patch (32 queries span 32 km) over 0.0245 rad cells: the union window of a tile holds fewer than
    320 records even for k = 64."""
    ref = x_deg(*grids.uniform_sphere(20000, seed=61))
    q = x_deg(*grids.lam_patch(16, 64, 1.0))
    (ei, _, st), (_, _, st_bin) = _both_orders(ops, monkeypatch, ref, q, k, cells=64)
    assert st[3] > 0 and st_bin[3] > 0
    np.testing.assert_array_equal(canon(ei), oracle_knn(ref, q, k)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("k", CAP_K)
def test_knn_path_stage_overflow(ops, monkeypatch, k):
    """A cluster of 2000 points in a 1e-4 rad spot: every tile of the queries around it has more than 320 records
    in its window and is searched per thread (nothing staged)."""
    rng = np.random.default_rng(62)
    background = x_deg(*grids.uniform_sphere(20000, seed=62))
    centre = np.array([0.4, 1.1])
    cluster = (centre + rng.normal(scale=1e-4, size=(2000, 2))).astype(np.float32)
    q = (centre + rng.normal(scale=1e-4, size=(64, 2))).astype(np.float32)
    ref = np.concatenate([background, cluster])
    (ei, _, st), (_, _, st_bin) = _both_orders(ops, monkeypatch, ref, q, k)
    assert st[3] == 0 and st_bin[3] == 0
    np.testing.assert_array_equal(canon(ei), brute_knn(ref, q, k)[0])
    if k <= 16:  # control: without the cluster the same tiles are staged
        _, _, st = run_knn(ops, background, q, k)
        assert st[3] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("k", CAP_K)
def test_knn_path_cap_growth(ops, monkeypatch, k):
    """References only in a northern patch, queries in the south: the first cap holds nothing and every lane widens
    its own search."""
    lat, lon = grids.uniform_sphere(80000, seed=63)
    sel = (lat > 30) & (lat < 60) & (lon > 0) & (lon < 60)
    ref = x_deg(lat[sel], lon[sel])
    glat, glon = grids.octahedral_grid(24)
    south = glat < -30
    q = x_deg(glat[south], glon[south])
    (ei, _, st), (_, _, st_bin) = _both_orders(ops, monkeypatch, ref, q, k)
    assert st[2] > 0 and st_bin[2] > 0
    np.testing.assert_array_equal(canon(ei), oracle_knn(ref, q, k)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("k", CAP_K)
@pytest.mark.parametrize("extra", [0, 1, 2])
def test_knn_path_whole_sphere(ops, monkeypatch, k, extra):
    """n_ref = k + extra: the first cap already exceeds chord^2 1.9, every cell is scanned, nothing is staged or
    widened."""
    ref = x_deg(*grids.uniform_sphere(k + extra, seed=64 + extra))
    q = _coherent_queries(4)
    (ei, _, st), (_, _, st_bin) = _both_orders(ops, monkeypatch, ref, q, k)
    assert st[3] == 0 and st[2] == 0 and st_bin[3] == 0
    np.testing.assert_array_equal(canon(ei), brute_knn(ref, q, k)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("k", CAP_K)
def test_knn_path_float64_redecision(ops, monkeypatch, k):
    """Every reference point duplicated (twice for odd k, three times otherwise), so that the k-th and (k+1)-th
    candidates of EVERY query are identical points: all queries are re-decided in float64, all are tied."""
    base = x_deg(*grids.uniform_sphere(3000, seed=65))
    reps = 2 if k % 2 else 3
    ref = np.concatenate([base] * reps)
    ref = ref[np.random.default_rng(65).permutation(ref.shape[0])]
    q = _coherent_queries(6)
    (ei, _, st), (_, _, st_bin) = _both_orders(ops, monkeypatch, ref, q, k)
    want, tied = brute_knn(ref, q, k)
    assert tied.all()
    assert st[0] >= q.shape[0] and st[1] == q.shape[0] and st_bin[1] == q.shape[0]
    np.testing.assert_array_equal(canon(ei), want)


# ------------------------------------------------------------------------------------------------
# 3. exact-duplicate tie groups of width 2, k, k + 1, 40 and 400 (one cell, wider than the stage)
# ------------------------------------------------------------------------------------------------
def _tie_group_cloud(k: int):
    rng = np.random.default_rng(70 + k)
    background = x_deg(*grids.uniform_sphere(2000, seed=71))
    sizes = [2, k, k + 1, 40, 400]
    # groups in mirror pairs about a meridian (lon -> -lon relative to lon0 keeps rdist bit-equal), the last one alone
    # (offsets of 2^-8 and 3 * 2^-10 rad: lon0 +- d is exact in float32, so the two distances are bit-equal)
    spots = [(0.5, 1.0 - 2**-8), (0.5, 1.0 + 2**-8), (-0.3, -2.0 - 3 * 2**-10), (-0.3, -2.0 + 3 * 2**-10), (1.2, 0.3)]
    groups = [np.tile(np.array(s, dtype=np.float32), (m, 1)) for s, m in zip(spots, sizes)]
    ref = np.concatenate([background, *groups])
    ref = ref[rng.permutation(ref.shape[0])]  # group members at scattered indices
    on = np.array(spots, dtype=np.float32)
    near = (on[:, None, :] + rng.normal(scale=2e-4, size=(5, 6, 2))).reshape(-1, 2).astype(np.float32)
    mirror = np.array([[0.5, 1.0], [-0.3, -2.0]], dtype=np.float32)
    q = np.concatenate([on, near, mirror, x_deg(*grids.uniform_sphere(300, seed=72))])
    return ref, q


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 7, 16, 64])
def test_knn_duplicate_tie_groups(ops, k):
    ref, q = _tie_group_cloud(k)
    nq, n = q.shape[0], ref.shape[0]
    want, tied = brute_knn(ref, q, k)
    assert tied[:5].sum() >= 4 and tied[-302:-300].all()  # on the groups of width > k, and at the mirror points
    flags = torch.zeros(nq, dtype=torch.uint8, device="cuda")
    ei, _, st = run_knn(ops, ref, q, k, tie_flags=flags)
    np.testing.assert_array_equal(canon(ei), want)
    np.testing.assert_array_equal(flags.cpu().numpy().astype(bool), tied)
    assert st[1] == tied.sum() and st[0] >= tied.sum()

    # the provisional-numbering path: search with permuted labels, then re-decide the flagged queries three ways
    perm = np.random.default_rng(73 + k).permutation(n)  # provisional label p is final point perm[p]
    rank = dev(perm.astype(np.int64))
    order = torch.empty_like(rank)
    order[rank] = torch.arange(n, dtype=torch.int64, device="cuda")
    qd = dev(q)
    flags = torch.zeros(nq, dtype=torch.uint8, device="cuda")
    with ops.NeighbourIndex(dev(ref[perm]), hint_k=k) as prov:
        first = prov.knn(qd, k, tie_flags=flags)
        np.testing.assert_array_equal(flags.cpu().numpy().astype(bool), tied)
        ranked = first.clone()
        prov.knn_redecide(qd, k, ranked, flags, rank=rank, order=order)
        listed = first.clone()
        flag_list, count = ops.compact_flags(flags)
        assert int(count.item()) == tied.sum()
        prov.knn_redecide_list(qd, k, listed, flag_list, count, rank=rank, order=order)
    final = first.clone()
    final[0] = rank[final[0].long()].to(torch.int32)
    with ops.NeighbourIndex(dev(ref), hint_k=k) as ix:
        ix.knn_redecide(qd, k, final, flags)
    for out in (ranked, listed):
        out[0] = rank[out[0].long()].to(torch.int32)
    for name, out in (("redecide", final), ("ranked", ranked), ("list", listed)):
        np.testing.assert_array_equal(canon(out), want, err_msg=name)


# ------------------------------------------------------------------------------------------------
# tie flags: the vectorised tile scan needs a 16-byte aligned array
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_knn_redecide_rejects_unaligned_tie_flags(ops):
    """A flag view at byte offset 1 or 8 of a larger array is refused on the host (ValueError, nothing launched);
    at offset 16 it works and gives the result of a fresh array."""
    ref, q = _tie_group_cloud(3)
    k, nq = 3, q.shape[0]
    qd = dev(q)
    fresh = torch.zeros(nq, dtype=torch.uint8, device="cuda")
    with ops.NeighbourIndex(dev(ref), hint_k=k) as ix:
        base = ix.knn(qd, k, tie_flags=fresh)
        assert int(fresh.sum().item()) > 0
        big = torch.zeros(nq + 64, dtype=torch.uint8, device="cuda")
        assert big.data_ptr() % 16 == 0
        for off in (1, 8):
            view = big[off : off + nq]
            view.copy_(fresh)
            out = base.clone()
            with pytest.raises(ValueError, match="16-byte aligned"):
                ix.knn_redecide(qd, k, out, view)
            with pytest.raises(ValueError, match="16-byte aligned"):
                ix.knn_redecide(qd, k, out, view, rank=torch.arange(ref.shape[0], device="cuda"),
                                order=torch.arange(ref.shape[0], device="cuda"))  # fmt: skip
            assert torch.equal(out, base)
        want = base.clone()
        ix.knn_redecide(qd, k, want, fresh)
        view = big[16 : 16 + nq]
        view.copy_(fresh)
        got = base.clone()
        ix.knn_redecide(qd, k, got, view)
        assert torch.equal(got, want)
        with pytest.raises(AssertionError):
            ix.knn_redecide(qd, k, base.clone(), big[: 2 * nq : 2])  # not contiguous


# ------------------------------------------------------------------------------------------------
# 4. cube-sphere geometry: cube edges and corners, cell borders, poles, wrapped longitudes
# ------------------------------------------------------------------------------------------------
def _cube_edges_and_corners(m: int) -> np.ndarray:
    pts = []
    t = np.linspace(-1.0, 1.0, m)
    for i, j in ((0, 1), (0, 2), (1, 2)):
        free = 3 - i - j
        for si in (-1.0, 1.0):
            for sj in (-1.0, 1.0):
                p = np.zeros((m, 3))
                p[:, i], p[:, j], p[:, free] = si, sj, t
                pts.append(p)
    corners = np.array([[a, b, c] for a in (-1, 1) for b in (-1, 1) for c in (-1, 1)], dtype=np.float64)
    return xyz_to_x(np.concatenate(pts + [corners]))


def _cell_borders(cells: int, n_border: int, n_along: int, seed: int) -> np.ndarray:
    """Points whose in-face angle is a cell border -pi/4 + m pi / (2 C), evaluated in float64, on every face."""
    rng = np.random.default_rng(seed)
    m = rng.choice(cells + 1, size=min(n_border, cells + 1), replace=False)
    alpha = -np.pi / 4 + m * (np.pi / 2) / cells
    beta = rng.uniform(-np.pi / 4, np.pi / 4, size=n_along)
    a, b = np.meshgrid(np.tan(alpha), np.tan(beta))
    a, b = a.reshape(-1), b.reshape(-1)
    face = np.stack([a, b, np.ones_like(a)], axis=1)
    pts = []
    for perm in ((0, 1, 2), (1, 2, 0), (2, 0, 1)):  # the border on each axis of each face pair
        for sign in (1.0, -1.0):
            p = face[:, perm].copy()
            p[:, perm.index(2)] *= sign
            pts.append(p)
            p2 = p.copy()
            p2[:, [perm.index(0), perm.index(1)]] = p2[:, [perm.index(1), perm.index(0)]]
            pts.append(p2)
    return xyz_to_x(np.concatenate(pts))


def _special_longitudes() -> np.ndarray:
    lats = np.array([np.pi / 2, -np.pi / 2, 0.0, 0.7, -1.2, 1.5707, -1.5707])
    lons = np.array([0.0, np.pi, -np.pi, 2 * np.pi, -3 * np.pi, 700.0, 1e-7, -1e-7])
    la, lo = np.meshgrid(lats, lons)
    return np.stack([la.reshape(-1), lo.reshape(-1)], axis=1).astype(np.float32)


@pytest.fixture(scope="module")
def geometry_sets():
    sets = {}
    special = np.concatenate([_cube_edges_and_corners(9), _special_longitudes()])
    background = x_deg(*grids.uniform_sphere(3000, seed=81))
    for cells in (1, 2, 7, 64, 1024, 2048):
        border = _cell_borders(cells, 12, 4, seed=cells)
        pts = ulp_neighbours(np.concatenate([special, border]))
        rng = np.random.default_rng(cells)
        ref = np.concatenate([background, pts[rng.permutation(pts.shape[0])[: pts.shape[0] // 2]]])
        sets[cells] = (ref, pts)
    return sets


@pytest.mark.gpu
@pytest.mark.parametrize("cells", [1, 2, 7, 64, 1024, 2048])
def test_knn_cube_geometry(ops, geometry_sets, cells):
    """References and queries on the 12 cube edges, the 8 corners, within 1 float32 ulp of cell borders, at the poles
    and at longitudes 0, +-pi, 2 pi, -3 pi, 700 rad - with the index built explicitly at each C."""
    ref, q = geometry_sets[cells]
    rd = all_rdist(ref, q)
    for k in (1, 4, 17):
        ei, rdist, _ = run_knn(ops, ref, q, k, cells=cells, return_rdist=True)
        np.testing.assert_array_equal(canon(ei), brute_knn(ref, q, k, rd=rd)[0], err_msg=f"k={k}")
        assert_rows_ascending(ei[0].reshape(-1, k), rdist)


def _window_edge_case(cells: int, variant: int):
    """The tightest inputs for the cap -> cell window: on the equator (where the in-face angle of faces +-x / +-y IS
    the longitude offset, and a distance IS a longitude difference) a reference point ("partner") sits on a cell
    border; its query lies inward at the largest distance the first cap accepts, so that the window edge and the
    border coincide.  A decoy slightly farther on the other side of the query is what a window that misses the
    partner's cell would report.  Each query is repeated 32 times: one tile = one query, searched staged.  Filler
    points on face +z set the first cap (chord^2 = 12 / n for k = 1): ~0.0055 rad for C >= 64."""
    n_fill = {1: 10000, 2: 10000, 7: 40000}.get(cells, 400000)  # few cells: keep the filler's cells small enough
    width = (np.pi / 2) / cells
    spacing = 5.5 * math.sqrt(12.0 / n_fill)  # no other configuration within twice the cap of a query
    step = max(1, int(math.ceil(spacing / width)))
    borders = []
    for centre in (0.0, np.pi / 2, np.pi, -np.pi / 2):
        for m in range(0, cells + 1, step):
            borders.append(centre - np.pi / 4 + m * width)
    borders = np.unique(np.round(np.mod(np.asarray(borders) + np.pi, 2 * np.pi) - np.pi, 12))
    keep = np.concatenate([[True], np.diff(borders) > spacing * 0.99])
    borders = borders[keep]
    if borders.size > 1 and (borders[0] + 2 * np.pi - borders[-1]) < spacing:
        borders = borders[:-1]
    n = n_fill + 3 * borders.size
    t2 = float(np.float32(6.0 * 2 / n))
    margin = 4.2e-7 * math.sqrt(t2) + 1e-6 * t2 + 1e-13
    rho = 2.0 * math.asin(math.sqrt(t2 - 6.0 * margin) / 2.0)  # farthest k-th neighbour the first cap accepts
    partner = np.float32(borders)
    if variant:
        partner = np.nextafter(partner, np.float32(np.inf * variant))
    side = np.where(np.arange(borders.size) % 2 == 0, -1.0, 1.0)  # query below / above the border, alternating
    q_lon = partner.astype(np.float64) + side * (rho - 8e-7)
    decoy = q_lon + side * rho
    lat = np.zeros(borders.size)
    rng = np.random.default_rng(cells)
    ref = np.concatenate([
        np.stack([lat, partner], axis=1), np.stack([lat, decoy], axis=1),
        np.stack([rng.uniform(1.2, 1.4, n_fill), rng.uniform(-np.pi, np.pi, n_fill)], axis=1),  # filler: on face +z
        np.stack([np.full(borders.size, -1.0), borders], axis=1),  # pad: n is what t2 was computed from
    ]).astype(np.float32)  # fmt: skip
    assert ref.shape[0] == n
    q = np.stack([lat, q_lon], axis=1).astype(np.float32)
    return ref, q


@pytest.mark.gpu
@pytest.mark.parametrize("cells", [1, 2, 7, 64, 1024, 2048])
def test_knn_window_edge_at_cell_borders(ops, cells, monkeypatch):
    monkeypatch.setenv("AGX_KNN_BIN", "0")
    for variant in (0, 1, -1):
        ref, q = _window_edge_case(cells, variant)
        rep = np.repeat(q, 32, axis=0)
        ei, _, st = run_knn(ops, ref, rep, 1, cells=cells)
        assert st[3] > 0 and st[2] == 0  # staged, answered by the first cap
        want, _ = oracle_knn(ref, q, 1)
        got = ei[0].reshape(q.shape[0], 32)
        assert (got == got[:, :1]).all()
        np.testing.assert_array_equal(got[:, 0], want[0], err_msg=f"variant {variant}")
        assert (want[0] < q.shape[0]).all()  # every query's answer is its partner on the border


# ------------------------------------------------------------------------------------------------
# 5. odd shapes
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_knn_partial_tiles_dst_base_and_output_maps(ops):
    ref = x_deg(*grids.uniform_sphere(5000, seed=91))
    allq = x_deg(*grids.uniform_sphere(1017, seed=92))
    for nq in (1, 31, 33, 1017):
        q = allq[:nq]
        for k in (3, 33):
            ei, _, _ = run_knn(ops, ref, q, k)
            np.testing.assert_array_equal(canon(ei), oracle_knn(ref, q, k)[0], err_msg=f"nq={nq} k={k}")
    q, k = allq[:40], 4
    with ops.NeighbourIndex(dev(ref), hint_k=k) as ix:
        plain = ix.knn(dev(q), k).cpu().numpy()
        base = INT32_MAX - q.shape[0] - 1
        ei = ix.knn(dev(q), k, dst_base=base).cpu().numpy()
        np.testing.assert_array_equal(ei[0], plain[0])
        np.testing.assert_array_equal(ei[1].astype(np.int64), base + plain[1])
        assert ei[1].max() == INT32_MAX - 2
        with pytest.raises(ValueError, match="exceeds int32"):
            ix.knn(dev(q), k, dst_base=INT32_MAX - q.shape[0])
    rng = np.random.default_rng(93)
    src_sel = np.sort(rng.choice(20000, size=ref.shape[0], replace=False)).astype(np.int64)
    dst_sel = np.sort(rng.choice(50000, size=allq.shape[0], replace=False)).astype(np.int64)
    for k in (7, 33):
        with ops.NeighbourIndex(dev(ref), hint_k=k) as ix:
            plain = ix.knn(dev(allq), k).cpu().numpy()
            with ops.output_maps(dev(src_sel), dev(dst_sel)):
                fused = ix.knn(dev(allq), k).cpu().numpy()
        np.testing.assert_array_equal(fused, np.stack([src_sel[plain[0]], dst_sel[plain[1]]]).astype(np.int32))


# ------------------------------------------------------------------------------------------------
# 6 + 7. max_radius with k > 1, and the order inside a row
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3, 7, 17])
def test_knn_max_radius_contract(ops, k):
    """Queries whose k-th neighbour is within the limit: exact, equal to the unlimited search.  Every other query:
    every reference point within the limit is reported with its exact rdist, the other slots are -1 / +inf or points
    beyond the limit, no index twice, and the row is ascending (rdist, index) - in the staged and the per-thread
    `limited` branches alike."""
    # a sparse 3000 km patch (100 km spacing: ~7 points within the limit) around a dense 200 km core (10 km)
    ref = np.concatenate([x_deg(*grids.lam_patch(30, 30, 100.0)), x_deg(*grids.lam_patch(20, 20, 10.0))])
    rng = np.random.default_rng(100 + k)
    inside = ref[rng.choice(ref.shape[0], 600, replace=False)] + rng.normal(scale=2e-3, size=(600, 2)).astype(np.float32)
    q = np.concatenate([x_deg(*grids.uniform_sphere(3000, seed=101)), inside.astype(np.float32)])
    limit = 150.0 / 6371.0
    thr = math.sin(0.5 * limit) ** 2
    full_ei, full_rd, _ = run_knn(ops, ref, q, k, return_rdist=True)
    lim_ei, lim_rd, _ = run_knn(ops, ref, q, k, return_rdist=True, max_radius=limit)
    lim_src, full_src = lim_ei[0].reshape(-1, k), full_ei[0].reshape(-1, k)
    exact = full_rd[:, k - 1] <= thr
    assert exact.sum() > 100 and (~exact).sum() > 1000
    np.testing.assert_array_equal(lim_src[exact], full_src[exact])
    np.testing.assert_array_equal(lim_rd[exact], full_rd[exact])
    assert_rows_ascending(lim_src, lim_rd)
    assert_rdist_exact(ref, q, lim_src, lim_rd)
    offsets, within, _ = X.Grid(ref, cell_rad=limit).radius(q, limit)
    partial = 0
    for i in np.nonzero(~exact)[0]:
        row = lim_src[i]
        have = row[row >= 0]
        assert np.unique(have).size == have.size
        w = within[offsets[i] : offsets[i + 1]]
        assert w.size < k
        partial += w.size > 0
        assert set(w.tolist()) <= set(have.tolist()), i
        others = np.isin(row, w, invert=True) & (row >= 0)
        assert (lim_rd[i][others] > thr * (1 - 1e-12)).all(), i
    if k >= 7:
        assert partial > 20  # queries with some, but fewer than k, points inside the limit


# ------------------------------------------------------------------------------------------------
# 8 + 9. cut-off: duplicates, cube geometry, the threshold, the tile -> warp hand-off
# ------------------------------------------------------------------------------------------------
MODES = [(t, b) for t in ("0", "1") for b in ("0", "1")]


def oracle_cutoff(ref, q, radius):
    """``exact_search.cutoff_edges`` with a grid no finer than 0.01 rad (its memory grows as 1 / cell^2)."""
    offsets, src, near = X.Grid(ref, cell_rad=max(radius, 0.01)).radius(q, radius)
    dst = np.repeat(np.arange(q.shape[0], dtype=np.int32), np.diff(offsets))
    return np.stack([src, dst]), near


def _radius_all_modes(ops, monkeypatch, ref, q, radius, hint=None):
    outs = {}
    for tile, binned in MODES:
        monkeypatch.setenv("AGX_RADIUS_TILE", tile)
        monkeypatch.setenv("AGX_RADIUS_BIN", binned)
        stats = ops.new_stats("cuda")
        with ops.NeighbourIndex(dev(ref), hint_radius=radius if hint is None else hint) as ix:
            outs[(tile, binned)] = (ix.radius(dev(q), radius, stats=stats).cpu().numpy(), stats.cpu().numpy())
    for key, (ei, st) in outs.items():
        np.testing.assert_array_equal(ei, outs[("0", "0")][0], err_msg=str(key))
        assert st[1] == outs[("0", "0")][1][1], key
    return outs[("1", "0")]


def _threshold_pairs(radius: float) -> np.ndarray:
    """References at longitude +-radius on the equator, for a query at (0, 0): their rdist is sin(radius / 2)^2 - the
    threshold itself - when the device's float64 sin returns the C library's bits at radius / 2."""
    if radius <= 0.0:
        return np.zeros((0, 2), dtype=np.float32)
    x = 0.5 * radius
    if torch.sin(torch.tensor([x], dtype=torch.float64, device="cuda")).item() != math.sin(x):
        return np.zeros((0, 2), dtype=np.float32)
    return np.array([[0.0, radius], [0.0, -radius]], dtype=np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("radius", [0.0, 1e-7, "cell", 0.3, 1.5, 1.57, 2.0])
def test_cutoff_duplicates_geometry_and_threshold(ops, monkeypatch, radius):
    base = x_deg(*grids.uniform_sphere(2000, seed=111))
    special = ulp_neighbours(np.concatenate([_cube_edges_and_corners(5), _special_longitudes(), _cell_borders(64, 6, 3, 7)]))
    if radius == "cell":
        with ops.NeighbourIndex(dev(base), hint_radius=0.05) as ix:
            radius = (np.pi / 2) / ix.cells_per_face
    radius = float(np.float32(radius))  # representable: the threshold pairs sit exactly on it
    pairs = _threshold_pairs(radius)
    ref = np.concatenate([base, np.repeat(base[:50], 3, axis=0), special, pairs])
    q = np.concatenate([base[:200], special[::3], np.zeros((1, 2), dtype=np.float32)])
    ei, st = _radius_all_modes(ops, monkeypatch, ref, q, radius)
    want, near = oracle_cutoff(ref, q, radius)
    np.testing.assert_array_equal(canon(ei), want)
    assert st[1] == near
    if pairs.size:
        assert near >= 2
        n = ref.shape[0]
        kept = ei[0][ei[1] == q.shape[0] - 1]
        assert {n - 2, n - 1} <= set(kept.tolist())  # rdist == sin^2(r/2): inclusive
    assert (np.diff(ei[1]) >= 0).all()


@pytest.mark.gpu
def test_cutoff_tile_to_warp_handoff(ops, monkeypatch):
    """Query tiles that mix degree <= 6 (sparse background) and degree > 320 (a dense cluster): identical output in
    every mode, equal to the oracle, grouped by query in ascending order."""
    n_bg = 50000
    background = x_deg(*grids.uniform_sphere(n_bg, seed=121))
    rng = np.random.default_rng(122)
    centre = np.array([0.2, 0.9])
    cluster = (centre + rng.normal(scale=2e-3, size=(3000, 2))).astype(np.float32)
    ref = np.concatenate([background, cluster])
    radius = float(np.arccos(1.0 - 2.0 * 4 / n_bg))
    line = np.stack([np.full(256, centre[0]), centre[1] + np.linspace(-0.15, 0.15, 256)], axis=1).astype(np.float32)
    ei, _ = _radius_all_modes(ops, monkeypatch, ref, line, radius)
    want, _ = oracle_cutoff(ref, line, radius)
    np.testing.assert_array_equal(canon(ei), want)
    deg = np.bincount(ei[1], minlength=line.shape[0])
    tiles = deg.reshape(-1, 32)
    assert ((tiles.min(axis=1) <= 6) & (tiles.max(axis=1) > 320)).any()
    assert (np.diff(ei[1]) >= 0).all()


# ------------------------------------------------------------------------------------------------
# 10. counting backbone
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, SCAN_TILE - 1, SCAN_TILE, SCAN_TILE + 1, 3 * SCAN_TILE + 5, 5_000_000])
def test_exclusive_scan_past_2_to_32(n):
    from anemoi_graphs_b200 import _cabi

    lib = _cabi.load_library()
    rng = np.random.default_rng(n)
    counts = (INT32_MAX - rng.integers(0, 1000, size=n)).astype(np.int32)
    offsets = torch.full((n + 1,), -7, dtype=torch.int64, device="cuda")
    total = c_int64()
    cd = dev(counts)
    _cabi.check(lib.agx_exclusive_scan(cd.data_ptr(), n, offsets.data_ptr(), byref(total), _cabi.current_stream()))
    want = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(counts.astype(np.int64), out=want[1:])
    np.testing.assert_array_equal(offsets.cpu().numpy(), want)
    assert total.value == want[-1]
    if n > 2:
        assert want[-1] > 2**32


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 3, 4, 31, 32, 33, 1_000_003])
@pytest.mark.parametrize("fill", ["zero", "all", "sparse"])
def test_compact_flags(ops, n, fill):
    rng = np.random.default_rng(n)
    flags = {"zero": np.zeros(n), "all": np.ones(n), "sparse": rng.random(n) < 0.01}[fill].astype(np.uint8)
    if fill == "sparse":
        flags[[0, n - 1]] = rng.integers(1, 256, size=2)  # any non-zero byte counts, at both ends
    lst, count = ops.compact_flags(dev(flags))
    want = np.nonzero(flags)[0]
    assert int(count.item()) == want.size
    np.testing.assert_array_equal(lst.cpu().numpy()[: want.size], want)
