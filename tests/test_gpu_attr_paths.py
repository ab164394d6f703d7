"""Adversarial parity of the edge attribute kernel (K5: ``EdgeLength`` / ``EdgeDirection`` and their normalisation)
along every code path: both node forms per side, the paired (J = 2) and scalar (J = 1) lanes, the walk by target of a
regular-k list, the split statistics -> apply form with several statistics sets (a multi-GPU build), the flag modes
and the list-driven patch pass of the provisional-numbering decoder, and the in-place scaling pass at every
16-byte misalignment.

Every result is compared with ``oracle/ref_path`` (the reference's own numpy / scipy arithmetic) at the DESIGN section 4
tolerances: 1e-6 relative, absolute 1e-6 of the array's largest magnitude for ``unit-range`` and inverted lengths and
for direction components near 0; bit-identity where two paths of the kernel are claimed to agree bit for bit.  Where
the reference reduces a float32 array in float32 (the ``l1`` / ``l2`` / ``unit-std`` divisor of lengths and of
non-rotated directions), that divisor's own rounding error, measured against float64, is added to the 1e-6.

Listed exceptions:
* coincident endpoints, and exactly antipodal ones, have no defined direction (the reference returns amplified rounding
  noise): their lengths are checked, their directions are not, and they stay out of the sets whose directions are
  normalised;
* the two epsilon nudges (``|v|^2 < 1e-10`` for a target near a pole and for a rotated source near the pole, i.e. an
  edge shorter than ~1e-5 rad) are exercised clearly on both sides; points inside the band 0.25e-10 < |v|^2 < 4e-10,
  where the kernel and the reference could round the test differently, are kept out of the inputs;
* near-constant attributes, whose standard deviation sits at rounding level, are not generated: ``np.std`` there is
  noise.  The exact ``std == 0`` cases (one edge, two equal edges) are tested."""

import numpy as np
import pytest
import torch

from oracle import ref_path as R

pytestmark = pytest.mark.gpu

ATTR_RTOL = 1e-6
FOLD_RTOL = 3e-7  # the same statistics folded in a different association (sum-based norms only)
NORMS = [None, "l1", "l2", "unit-max", "unit-range", "unit-std"]
ORDER_FREE = (None, "unit-max", "unit-range")  # no sum in the parameters: bit-identical across association orders
NO_VALUE = [0.0, 0.0, 1e300, -1e300]  # the statistics of an empty edge set
F32_HALF_PI = np.float32(np.pi / 2)
SWITCH = 2.0 * np.arctan(0.0625)  # atan2_short: the series below tan(d/2) = 1/16, the library above


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def ops():
    from anemoi_graphs_b200 import ops as _ops

    return _ops


@pytest.fixture(scope="module")
def lib(ops):
    return ops.load_library()


def _check(rc):
    from anemoi_graphs_b200 import _cabi

    _cabi.check(rc)


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------------------------
# geometry
# ------------------------------------------------------------------------------------------------
def destination(lat, lon, d, bearing):
    """float64 great-circle destination from (lat, lon) at angular distance d and the given bearing."""
    s = np.clip(np.sin(lat) * np.cos(d) + np.cos(lat) * np.sin(d) * np.cos(bearing), -1.0, 1.0)
    lat2 = np.arcsin(s)
    lon2 = lon + np.arctan2(np.sin(bearing) * np.sin(d) * np.cos(lat), np.cos(d) - np.sin(lat) * s)
    return lat2, lon2


def wrap_pi(lon):
    return (np.asarray(lon) + np.pi) % (2 * np.pi) - np.pi


def f32(lat, lon) -> np.ndarray:
    return np.stack([np.asarray(lat, dtype=np.float64), np.asarray(lon, dtype=np.float64)], axis=1).astype(np.float32)


def sep64(s: np.ndarray, t: np.ndarray) -> np.ndarray:
    """float64 great-circle separation of float32 (lat, lon) rows."""
    s, t = s.astype(np.float64), t.astype(np.float64)
    a = np.sin((t[:, 0] - s[:, 0]) / 2) ** 2 + np.cos(s[:, 0]) * np.cos(t[:, 0]) * np.sin((t[:, 1] - s[:, 1]) / 2) ** 2
    return 2 * np.arcsin(np.sqrt(np.clip(a, 0.0, 1.0)))


def pole_vn(x: np.ndarray) -> np.ndarray:
    """|v|^2 of direction_vec(p, z^) for the float32 unit vector of each (lat, lon) row (the target-side nudge test)."""
    p = R.latlon_rad_to_cartesian((x[:, 0], x[:, 1]), 1.0).astype(np.float64)
    return p[:, 0] ** 2 + p[:, 1] ** 2


def haversine_switch_side(s: np.ndarray, t: np.ndarray) -> np.ndarray:
    """True where the kernel takes the short-edge series: sqrt(a) <= sqrt(1 - a) / 16 with numpy's float32 ``a``."""
    dlat, dlon = t[:, 0] - s[:, 0], t[:, 1] - s[:, 1]
    a = np.sin(dlat / np.float32(2)) ** 2 + np.cos(s[:, 0]) * np.cos(t[:, 0]) * np.sin(dlon / np.float32(2)) ** 2
    assert a.dtype == np.float32
    return np.sqrt(a).astype(np.float64) <= 0.0625 * np.sqrt(np.float32(1) - a).astype(np.float64)


def adversarial_pairs(seed: int = 11):
    """(src (E, 2), dst (E, 2)) float32 pairs whose length AND direction are defined (see the module docstring)."""
    rng = np.random.default_rng(seed)
    pairs = []

    def add(lat, lon, d, bearing):
        lat2, lon2 = destination(lat, lon, d, bearing)
        pairs.append((f32(lat, lon), f32(lat2, wrap_pi(lon2))))

    # separations 1e-7 .. pi - 1e-3, random start points and orientations
    d = np.logspace(-7, np.log10(np.pi - 1e-3), 200)
    n = d.size
    add(np.arcsin(rng.uniform(-1, 1, n)), rng.uniform(-np.pi, np.pi, n), d, rng.uniform(0, 2 * np.pi, n))
    # both sides of the atan2_short switch, on meridians: dlat steps through the float32 values around the switch
    for lat0, lon0 in ((0.0, 0.3), (-0.5, -2.0), (0.7, 3.1)):
        t_lat = np.float32(lat0 + SWITCH)
        steps = [t_lat]
        for to in (np.inf, -np.inf):
            v = t_lat
            for _ in range(8):
                v = np.nextafter(v, np.float32(to))
                steps.append(v)
        steps = np.array(steps, dtype=np.float32)
        pairs.append((f32(np.full(steps.size, lat0), np.full(steps.size, lon0)), np.stack([steps, np.full(steps.size, np.float32(lon0))], 1)))
    # targets at and near both poles (cos(lat) on both sides of the target nudge), sources 1e-6 .. 1 rad away
    for pole in (1.0, -1.0):
        for off in (0.0, 3e-6, 3e-5, 1e-3):
            t_lat = np.float32(pole * (np.pi / 2 - off))
            m = 24
            dd = np.logspace(-6, 0, m)
            t_lon = rng.uniform(-np.pi, np.pi, m)
            tl = np.full(m, float(t_lat))
            s_lat, s_lon = destination(tl, t_lon, dd, rng.uniform(0, 2 * np.pi, m))
            pairs.append((f32(s_lat, wrap_pi(s_lon)), f32(tl, t_lon)))
    # the date line: [-pi, pi] and [0, 2 pi) conventions, mixed, with |dlon| > pi
    m = 16
    lat = rng.uniform(-1.2, 1.2, m)
    dl = np.logspace(-5, -0.5, m)
    s = f32(lat, np.pi - dl / 2)
    for t in (f32(lat + 1e-3, -np.pi + dl / 2), f32(lat - 1e-3, np.pi + dl / 2), f32(lat, -np.pi + dl / 3)):
        pairs.append((s, t))
    pairs.append((f32(lat, dl / 2), f32(lat + 2e-3, 2 * np.pi - dl / 2)))  # [0, 2 pi): dlon close to 2 pi
    pairs.append((f32(lat, -np.pi + dl), f32(lat, 2 * np.pi - dl)))  # mixed conventions: dlon close to 3 pi
    # near-antipodal with a finite length
    m = 16
    lat, lon = np.arcsin(rng.uniform(-0.9, 0.9, m)), rng.uniform(-np.pi, np.pi, m)
    add(lat, lon, np.pi - np.logspace(-3, -1, m), rng.uniform(0, 2 * np.pi, m))
    src = np.concatenate([p[0] for p in pairs])
    dst = np.concatenate([p[1] for p in pairs])
    # the listed exceptions: coincident (after the float32 rounding), NaN / antipodal, inside a nudge band
    sep = sep64(src, dst)
    keep = (sep > 0) & (sep < np.pi - 1e-4) & ~np.isnan(R.haversine_distance(src, dst))
    keep &= ~((sep > 0.5e-5) & (sep < 2e-5))  # the rotated-source nudge: |q_xy|^2 ~ sep^2
    vn = pole_vn(dst)
    keep &= ~((vn > 0.25e-10) & (vn < 4e-10))
    return src[keep], dst[keep]


def degenerate_pairs(seed: int = 12):
    """Pairs with a length but no direction: coincident endpoints, and antipodal ones whose float32 ``a`` is <= 1."""
    rng = np.random.default_rng(seed)
    m = 64
    lat, lon = np.arcsin(rng.uniform(-1, 1, m)), rng.uniform(-np.pi, np.pi, m)
    same = f32(lat, lon)
    src = [same, f32([F32_HALF_PI, -F32_HALF_PI], [0.0, 1.0])]
    dst = [same.copy(), f32([F32_HALF_PI, -F32_HALF_PI], [0.0, 1.0])]
    anti_s, anti_t = antipodal_candidates(rng)
    length = R.haversine_distance(anti_s, anti_t)
    src.append(anti_s[~np.isnan(length)])
    dst.append(anti_t[~np.isnan(length)])
    return np.concatenate(src), np.concatenate(dst)


def antipodal_candidates(rng):
    m = 256
    lat, lon = rng.uniform(-1.4, 1.4, m), rng.uniform(-np.pi, np.pi, m)
    return f32(lat, lon), f32(-lat, wrap_pi(lon + np.pi))


def nan_pairs(seed: int = 13):
    """Antipodal pairs whose float32 haversine ``a`` exceeds 1: NaN length in the reference."""
    s, t = antipodal_candidates(np.random.default_rng(seed))
    bad = np.isnan(R.haversine_distance(s, t))
    assert bad.sum() >= 4
    return s[bad], t[bad]


def edge_set(src: np.ndarray, dst: np.ndarray, seed: int):
    """Node sets (src, dst) and a (2, E) int32 list over them with the columns in random order."""
    perm = np.random.default_rng(seed).permutation(src.shape[0])
    ei = np.stack([np.arange(src.shape[0]), np.arange(src.shape[0])])[:, perm].astype(np.int32)
    return src, dst, ei


def regular_set(k: int, n_t: int, seed: int, dst_base: int = 0):
    """A KNN-shaped list: target i = dst_base + i owns the columns [i k, (i + 1) k).  Targets include both poles, at
    and near them; the sources lie 1e-6 .. 1 rad away at random bearings (pole offsets and edge lengths outside the
    nudge bands)."""
    rng = np.random.default_rng(seed)
    t_lat = np.arcsin(rng.uniform(-1, 1, n_t))
    t_lat[:8] = np.array([1, -1, 1, -1, 1, -1, 1, -1]) * (np.pi / 2 - np.array([0, 0, 3e-6, 3e-6, 3e-5, 3e-5, 1e-3, 1e-3]))
    tx = f32(t_lat, rng.uniform(-np.pi, np.pi, n_t))
    d = np.exp(rng.uniform(np.log(1e-6), 0.0, (n_t, k)))
    d[(d > 0.5e-5) & (d < 2e-5)] *= 4.0
    s_lat, s_lon = destination(np.repeat(tx[:, 0].astype(np.float64), k), np.repeat(tx[:, 1].astype(np.float64), k),
                               d.ravel(), rng.uniform(0, 2 * np.pi, n_t * k))  # fmt: skip
    sx = f32(s_lat, wrap_pi(s_lon))
    perm = rng.permutation(n_t * k)  # the source numbering is not the edge order
    sx_nodes = np.empty_like(sx)
    sx_nodes[perm] = sx
    ei = np.stack([perm, dst_base + np.repeat(np.arange(n_t), k)]).astype(np.int32)
    tx_nodes = np.concatenate([np.zeros((dst_base, 2), np.float32), tx])
    return sx_nodes, tx_nodes, ei


# ------------------------------------------------------------------------------------------------
# the reference: raw values once per edge set, each norm applied as R.edge_length / R.edge_direction do
# ------------------------------------------------------------------------------------------------
class Ref:
    def __init__(self, sx, tx, ei):
        s, t = sx[ei[0]], tx[ei[1]]
        self.len_raw = R.haversine_distance(s, t)[:, np.newaxis]
        self.dir_raw = {rot: R.edge_directions_raw(s.T, t.T, rot).T for rot in (True, False)}

    def length(self, norm, invert=False):
        out = R.normalise(self.len_raw, norm).astype(np.float32)
        return 1 - out if invert else out

    def direction(self, norm, rotated):
        return R.normalise(self.dir_raw[rotated], norm).astype(np.float32)


def assert_len(got, want, norm, msg="", invert=False, rtol=ATTR_RTOL):
    """unit-range and 1 - v end in differences of nearly equal float32 numbers: absolute 1e-6 of the largest value."""
    finite = want[np.isfinite(want)]
    atol = ATTR_RTOL * np.abs(finite).max() if ((invert or norm == "unit-range") and finite.size) else 0.0
    np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, err_msg=f"length {norm} {msg}")


def assert_dir(got, want, norm, msg="", defined=None, rtol=ATTR_RTOL):
    if defined is not None:
        got, want = got[defined], want[defined]
    finite = want[np.isfinite(want)]
    atol = ATTR_RTOL * np.abs(finite).max() if finite.size else 0.0
    np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, err_msg=f"direction {norm} {msg}")


def reference_divisor_rtol(v: np.ndarray, norm) -> float:
    """The reference's own rounding in its divisor.  Lengths and non-rotated directions are float32 arrays there and
    numpy reduces them in float32 (np.sum, np.linalg.norm, np.std): a signed sum can cancel, a sum of squares over a
    million values drifts by ~1e-5.  The kernel reduces in float64; this is added to the 1e-6."""
    if v.dtype != np.float32 or norm not in ("l1", "l2", "unit-std"):
        return 0.0
    v64 = v.astype(np.float64)
    exact = {"l1": v64.sum(), "l2": np.sqrt((v64 * v64).sum()), "unit-std": v64.std()}[norm]
    ref = {"l1": np.sum(v), "l2": np.linalg.norm(v), "unit-std": np.std(v)}[norm]
    return abs(float(ref) - exact) / abs(exact) if exact else 0.0


def bits_equal(a, b, msg=""):
    np.testing.assert_array_equal(np.asarray(a).view(np.int32), np.asarray(b).view(np.int32), err_msg=msg)


def close_or_bits(a, b, norm, msg=""):
    """The same attributes from two association orders of the statistics."""
    if norm in ORDER_FREE:
        bits_equal(a, b, msg)
    else:
        np.testing.assert_allclose(a, b, rtol=FOLD_RTOL, atol=0, err_msg=msg)


# ------------------------------------------------------------------------------------------------
# calls through the C ABI
# ------------------------------------------------------------------------------------------------
class Call:
    """One attribute configuration on one edge set, with the (2, E) list and the outputs possibly starting at an odd
    column of wider arrays (what the gathered multi-GPU path passes).  Outputs outside the block are guarded."""

    GUARD = 7.25

    def __init__(self, ops, sx, tx, ei, ts=True, tt=True, off=0, pad=None):
        self.ops, self.lib = ops, ops.load_library()
        self.src, self.dst = ops.NodeTables(dev(sx), tabulate=ts), ops.NodeTables(dev(tx), tabulate=tt)
        self.nodes = ops._node_inputs(self.src, self.dst)
        self.E, self.off = int(ei.shape[1]), off
        if pad is None:
            pad = (off + self.E) % 2  # an even width: with off = 0 both index rows are 8-byte aligned (paired lanes)
        wide = np.zeros((2, off + self.E + pad), dtype=np.int32)
        wide[:, off : off + self.E] = ei
        self.ei = dev(wide)
        self.ws = ops._attr_workspace(self.ei.device)

    def col(self, row, lo=0):
        return self.ei[row].data_ptr() + 4 * (self.off + lo)

    def outputs(self):
        n = self.ei.shape[1]
        self.out_len = torch.full((n,), self.GUARD, dtype=torch.float32, device="cuda")
        self.out_dir = torch.full((n, 2), self.GUARD, dtype=torch.float32, device="cuda")

    def len_ptr(self, lo=0):
        return self.out_len.data_ptr() + 4 * (self.off + lo)

    def dir_ptr(self, lo=0):
        return self.out_dir.data_ptr() + 8 * (self.off + lo)

    def result(self):
        """(len (E, 1), dir (E, 2)) of the block; the columns around it must be untouched."""
        ln, dr = self.out_len.cpu().numpy(), self.out_dir.cpu().numpy()
        a, b = self.off, self.off + self.E
        outside = np.concatenate([ln[:a], ln[b:], dr[:a].ravel(), dr[b:].ravel()])
        assert (outside == self.GUARD).all(), "an attribute was written outside its block"
        return ln[a:b, None].copy(), dr[a:b].copy()

    def one(self, len_norm=None, invert=False, dir_norm=None, rotated=True, regular_k=0, length=True, direction=True):
        """agx_edge_attrs: the single-call form."""
        codes = self.ops.NORM_CODES
        self.outputs()
        _check(self.lib.agx_edge_attrs(
            self.col(0), self.col(1), self.E, *self.nodes, codes[len_norm] if length else -1, int(invert),
            self.len_ptr(), codes[dir_norm] if direction else -1, int(rotated), self.dir_ptr(), self.ws.data_ptr(),
            regular_k, _stream()))  # fmt: skip
        return self.result()

    def stats(self, lo, hi, st, rotated):
        """agx_edge_attrs_stats over the columns [lo, hi) into the 8 doubles at st."""
        _check(self.lib.agx_edge_attrs_stats(
            self.col(0, lo), self.col(1, lo), hi - lo, *self.nodes, 1, 1, int(rotated), self.len_ptr(lo),
            self.dir_ptr(lo), st, self.ws.data_ptr(), None, 0, None, None, 0, _stream()))  # fmt: skip

    def apply(self, lo, hi, len_norm, invert, dir_norm, rotated, stats, n_sets):
        codes = self.ops.NORM_CODES
        _check(self.lib.agx_edge_attrs_apply(
            hi - lo, codes[len_norm], int(invert), self.len_ptr(lo), codes[dir_norm], int(rotated), self.dir_ptr(lo),
            stats.data_ptr(), n_sets, self.E, self.ws.data_ptr(), _stream()))  # fmt: skip

    def sharded(self, bounds, len_norm, invert, dir_norm, rotated):
        """Blocks [bounds[r], bounds[r + 1]) evaluated as the ranks of a multi-GPU build would: statistics per block
        into a (W, 8) tensor, then every block normalised with all W sets."""
        w = len(bounds) - 1
        st = torch.full((w, 8), float("nan"), dtype=torch.float64, device="cuda")
        self.outputs()
        for r in range(w):
            self.stats(bounds[r], bounds[r + 1], st[r].data_ptr(), rotated)
        for r in range(w):
            self.apply(bounds[r], bounds[r + 1], len_norm, invert, dir_norm, rotated, st, w)
        return (*self.result(), st.cpu().numpy(), bounds)

    def blocks(self, bounds, invert, rotated):
        """Every block in its own agx_edge_attrs call without a norm: how the ranks of a multi-GPU build evaluate
        an un-normalised edge set (no statistics to exchange)."""
        self.outputs()
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            _check(self.lib.agx_edge_attrs(
                self.col(0, lo), self.col(1, lo), hi - lo, *self.nodes, 0, int(invert), self.len_ptr(lo), 0,
                int(rotated), self.dir_ptr(lo), self.ws.data_ptr(), 0, _stream()))  # fmt: skip
        return self.result()


def check_all(got_len, got_dir, ref, len_norm, invert, dir_norm, rotated, msg, dir_defined=None):
    rtol = ATTR_RTOL + reference_divisor_rtol(ref.len_raw, len_norm)
    assert_len(got_len, ref.length(len_norm, invert), len_norm, msg, invert, rtol)
    if dir_defined is None or dir_norm is None:
        rtol = ATTR_RTOL + reference_divisor_rtol(ref.dir_raw[rotated], dir_norm)
        assert_dir(got_dir, ref.direction(dir_norm, rotated), dir_norm, msg, dir_defined, rtol)


CONFIGS = [(n, inv, rot) for n in NORMS for inv in (False, True) for rot in (True, False)]


@pytest.fixture(scope="module")
def adversarial():
    sx, tx = adversarial_pairs()
    return edge_set(sx, tx, seed=21)


# ------------------------------------------------------------------------------------------------
# the reference side and the geometry itself
# ------------------------------------------------------------------------------------------------
def test_adversarial_geometry_covers_every_branch():
    """The inputs really sit on both sides of every switch the kernel has (checked on the float32 values)."""
    src, dst = adversarial_pairs()
    sep = sep64(src, dst)
    assert sep.min() < 1e-6 and sep.max() > np.pi - 2e-3
    near = np.abs(sep - SWITCH) < 1e-5
    side = haversine_switch_side(src[near], dst[near])
    assert side.sum() >= 3 and (~side).sum() >= 3, "pairs on both sides of tan(d/2) = 1/16"
    assert (sep < 0.5e-5).sum() >= 10 and ((sep > 2e-5) & (sep < 1e-3)).sum() >= 10, "both sides of the source nudge"
    vn = pole_vn(dst)
    assert (vn < 0.25e-10).sum() >= 40 and ((vn > 4e-10) & (vn < 1e-8)).sum() >= 40, "both sides of the target nudge"
    assert (dst[:, 0] == F32_HALF_PI).sum() >= 20 and (dst[:, 0] == -F32_HALF_PI).sum() >= 20
    dlon = dst[:, 1].astype(np.float64) - src[:, 1]
    assert (dlon > np.pi).sum() >= 10 and (dlon < -np.pi).sum() >= 10 and (dst[:, 1] > np.pi).sum() >= 10
    s_d, t_d = degenerate_pairs()
    assert (sep64(s_d, t_d) == 0).sum() >= 60 and (sep64(s_d, t_d) > np.pi - 1e-4).sum() >= 4


# ------------------------------------------------------------------------------------------------
# node forms, column offsets, edge counts, every norm
# ------------------------------------------------------------------------------------------------
def test_every_norm_and_node_form_on_adversarial_edges(ops, adversarial):
    """All 6 norms x invert x rotated, the four source / target node forms (bit-identical), against the reference."""
    sx, tx, ei = adversarial
    ref = Ref(sx, tx, ei)
    calls = [Call(ops, sx, tx, ei, ts, tt) for ts in (True, False) for tt in (True, False)]
    for norm, inv, rot in CONFIGS:
        outs = [c.one(norm, inv, norm, rot) for c in calls]
        for ln, dr in outs[1:]:
            bits_equal(ln, outs[0][0], f"{norm} {inv} {rot}: node forms")
            bits_equal(dr, outs[0][1], f"{norm} {inv} {rot}: node forms")
        check_all(*outs[0], ref, norm, inv, norm, rot, f"inv={inv} rot={rot}")


@pytest.mark.parametrize("off", [0, 1, 2, 3])
def test_edge_counts_and_column_offsets(ops, adversarial, off):
    """E in {0 .. 129} through the paired lanes (off = 0, even width) and the scalar lanes (odd starts), with the
    scaling pass's head / tail at every 16-byte misalignment; the columns around the block stay untouched."""
    sx, tx, ei_all = adversarial
    for i, e in enumerate((0, 1, 2, 3, 31, 32, 33, 63, 64, 65, 129)):
        ei = ei_all[:, :e]
        ref = Ref(sx, tx, ei)
        call = Call(ops, sx, tx, ei, ts=bool(i & 1), tt=bool(i & 2), off=off)
        paired = Call(ops, sx, tx, ei, ts=bool(i & 1), tt=bool(i & 2))
        for norm, inv, rot in CONFIGS:
            ln, dr = call.one(norm, inv, norm, rot)
            assert ln.shape == (e, 1) and dr.shape == (e, 2)
            if e:
                check_all(ln, dr, ref, norm, inv, norm, rot, f"E={e} off={off} inv={inv} rot={rot}")
            if e and off:
                base = paired.one(norm, inv, norm, rot)
                close_or_bits(ln, base[0], norm, f"E={e} off={off}: J = 1 vs J = 2")
                close_or_bits(dr, base[1], norm, f"E={e} off={off}: J = 1 vs J = 2")


def test_million_edges_fold_many_block_partials(ops):
    """~1 M edges: k_attr_fold folds more than 256 block partials per thread slot."""
    rng = np.random.default_rng(31)
    n = 1 << 20
    lat, lon = np.arcsin(rng.uniform(-1, 1, n)), rng.uniform(-np.pi, np.pi, n)
    s_lat, s_lon = destination(lat, lon, np.exp(rng.uniform(np.log(1e-4), np.log(2.0), n)), rng.uniform(0, 2 * np.pi, n))
    sx, tx, ei = edge_set(f32(s_lat, wrap_pi(s_lon)), f32(lat, lon), seed=32)
    ref = Ref(sx, tx, ei)
    call = Call(ops, sx, tx, ei, ts=False, tt=True)
    for norm in NORMS:
        ln, dr = call.one(norm, False, norm, True)
        check_all(ln, dr, ref, norm, False, norm, True, "1M")
    ln, dr = call.one("unit-std", True, "l2", False)
    check_all(ln, dr, ref, "unit-std", True, "l2", False, "1M")


# ------------------------------------------------------------------------------------------------
# NaN, std == 0, max == min
# ------------------------------------------------------------------------------------------------
def test_nan_length_propagates_through_every_norm_and_shard(ops, golden):
    """An antipodal pair's NaN length makes every normalised length NaN, as numpy's sum / amax / amin / std do in
    the reference - for the golden vectors (row 9) and for a random set with a few such pairs, in every path."""
    g = golden("attr_vectors")
    s_nan, t_nan = nan_pairs()
    sx, tx = adversarial_pairs()
    sets = {"golden": (g["src"], g["dst"], np.stack([np.arange(14)] * 2).astype(np.int32))}
    sets["random"] = edge_set(np.concatenate([sx, s_nan]), np.concatenate([tx, t_nan]), seed=41)
    for name, (s, t, ei) in sets.items():
        ref = Ref(s, t, ei)
        e = ei.shape[1]
        for norm in NORMS:
            want = ref.length(norm)
            if norm is not None:
                assert np.isnan(want).all()
            for off in (0, 1):
                ln, _ = Call(ops, s, t, ei, off=off).one(norm, False, None, True)
                assert_len(ln, want, norm, f"{name} off={off}")
                ln, _ = Call(ops, s, t, ei, off=off).one(norm, True, None, True)
                assert_len(ln, ref.length(norm, True), norm, f"{name} inverted off={off}", invert=True)
            if norm is not None:
                ln, _, _, _ = Call(ops, s, t, ei, off=1).sharded([0, 1, e // 2, e], norm, False, "l1", True)
                assert np.isnan(ln).all(), f"{name} {norm}: sharded"


def test_exact_zero_std_and_zero_range(ops):
    """One edge, and two equal edges: std == 0, so ``unit-std`` returns the values unchanged; ``unit-range`` with
    max == min is 0 / 0 = NaN, in the reference and here."""
    s = f32([0.3, 0.3], [0.1, 0.1])
    t = f32([0.35, 0.35], [0.2, 0.2])
    for e in (1, 2):
        ei = np.stack([np.arange(e), np.arange(e)]).astype(np.int32)
        ref = Ref(s, t, ei)
        assert float(np.std(ref.len_raw)) == 0.0
        for off in (0, 1):
            call = Call(ops, s, t, ei, off=off)
            for norm in NORMS:
                ln, dr = call.one(norm, False, norm, False)
                check_all(ln, dr, ref, norm, False, norm, False, f"E={e}")
            ln, _ = call.one("unit-std", False, None, True)
            bits_equal(ln, ref.len_raw.astype(np.float32), "unit-std with std == 0")
            ln, _ = call.one("unit-range", False, None, True)
            assert np.isnan(ln).all()


def test_degenerate_pairs_lengths(ops):
    """Coincident endpoints (length 0) and antipodal pairs with a finite float32 ``a`` (length pi or close): lengths
    with every norm; directions only where they are defined."""
    s, t, ei = edge_set(*degenerate_pairs(), seed=51)
    ref = Ref(s, t, ei)
    sep = sep64(s[ei[0]], t[ei[1]])
    defined = (sep > 1e-6) & (sep < np.pi - 1e-4)
    for norm, inv, rot in CONFIGS:
        ln, dr = Call(ops, s, t, ei, off=1).one(norm, inv, None, rot)
        check_all(ln, dr, ref, norm, inv, None, rot, f"inv={inv}", dir_defined=defined)


# ------------------------------------------------------------------------------------------------
# walk by target (regular k)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 3, 7, 33, 64])
def test_regular_k_walk_by_target(ops, k):
    """k_edge_attrs_regular against the reference and against the edge-centric kernel on the same list: bit-identical
    where no sum enters the parameters, within 3e-7 otherwise (the per-block association differs)."""
    sx, tx, ei = regular_set(k, n_t=max(40, 2048 // k), seed=60 + k)
    ref = Ref(sx, tx, ei)
    for ts, tt in ((True, True), (False, False), (True, False)):
        call = Call(ops, sx, tx, ei, ts, tt)
        for norm, inv, rot in CONFIGS:
            ln, dr = call.one(norm, inv, norm, rot, regular_k=k)
            check_all(ln, dr, ref, norm, inv, norm, rot, f"k={k} inv={inv} rot={rot}")
            base = call.one(norm, inv, norm, rot)
            close_or_bits(ln, base[0], norm, f"k={k} {norm}: regular vs edge-centric")
            close_or_bits(dr, base[1], norm, f"k={k} {norm}: regular vs edge-centric")


# ------------------------------------------------------------------------------------------------
# the split statistics -> apply form: W shards simulated on one GPU
# ------------------------------------------------------------------------------------------------
def shard_bounds(e: int, w: int, rng) -> list[int]:
    """w blocks of [0, e) that start at odd columns; from w = 3 on one block is empty."""
    if w == e + 1:
        return [0] + list(range(e + 1))  # an empty first block, then one edge per block
    cuts = sorted(int(c) | 1 for c in rng.integers(1, e - 1, w - 1))
    if w >= 3:
        cuts[1] = cuts[0]
    return [0] + cuts + [e]


@pytest.mark.parametrize("w", [2, 3, 7, "E+1"])
def test_sharded_statistics_fold_and_unnormalised_blocks(ops, adversarial, w):
    """Blocks at odd column boundaries, empty ones included ({0, 0, 1e300, -1e300}); every norm through
    statistics -> apply, and the un-normalised blocks in one agx_edge_attrs call each.  Equal to the one-call result -
    bit for bit where no sum enters the parameters - and to the reference."""
    sx, tx, ei = adversarial
    if w == "E+1":
        ei = ei[:, :65]
    e = ei.shape[1]
    bounds = shard_bounds(e, e + 1 if w == "E+1" else w, np.random.default_rng(70))
    assert len(bounds) - 1 == (e + 1 if w == "E+1" else w) and bounds[0] == 0 and bounds[-1] == e
    ref = Ref(sx, tx, ei)
    call = Call(ops, sx, tx, ei, off=1, pad=0)
    whole = {}
    for rot in (True, False):  # the statistics of the whole set in one call
        st = torch.empty(8, dtype=torch.float64, device="cuda")
        call.outputs()
        call.stats(0, e, st.data_ptr(), rot)
        whole[rot] = st.cpu().numpy()
    norms = NORMS if w != "E+1" else ["unit-range", "unit-std"]
    for norm in norms:
        for inv, rot in ((False, True), (True, False)):
            one = call.one(norm, inv, norm, rot)
            ln, dr, st, b = call.sharded(bounds, norm, inv, norm, rot)
            msg = f"W={w} {norm} inv={inv} rot={rot}"
            close_or_bits(ln, one[0], norm, msg)
            close_or_bits(dr, one[1], norm, msg)
            check_all(ln, dr, ref, norm, inv, norm, rot, msg)
            empty = [r for r in range(len(b) - 1) if b[r] == b[r + 1]]
            assert empty or w == 2
            for r in empty:
                np.testing.assert_array_equal(st[r], NO_VALUE * 2)
            np.testing.assert_allclose(st[:, [0, 1, 4, 5]].sum(0), whole[rot][[0, 1, 4, 5]], rtol=1e-12, err_msg=msg)
            np.testing.assert_array_equal(st[:, [2, 6]].min(0), whole[rot][[2, 6]], err_msg=msg)
            np.testing.assert_array_equal(st[:, [3, 7]].max(0), whole[rot][[3, 7]], err_msg=msg)
    for inv, rot in ((False, True), (True, False)):
        ln, dr = call.blocks(bounds, inv, rot)
        one = call.one(None, inv, None, rot)
        msg = f"W={w} un-normalised blocks inv={inv} rot={rot}"
        bits_equal(ln, one[0], msg)
        bits_equal(dr, one[1], msg)
        check_all(ln, dr, ref, None, inv, None, rot, msg)


# ------------------------------------------------------------------------------------------------
# flag modes and the list-driven patch pass on a KNN result
# ------------------------------------------------------------------------------------------------
def _flag_lists(n_t: int, rng) -> dict:
    some = np.sort(rng.choice(n_t, size=max(2, n_t // 9), replace=False))
    return {"empty": np.zeros(0, int), "last": np.array([n_t - 1]), "every": np.arange(n_t), "some": some}


@pytest.mark.parametrize("k", [3, 7])
def test_flag_modes_and_target_list_of_one_stats_entry_point(ops, lib, k):
    """"skip" with regular_k, then the list pass (lists of 0, 1 = the last target, every target, some) with a flag
    pointer offset as in a sharded decoder; also "only" without a list.  The two statistics sets add up to the whole
    set's, and apply(n_stat_sets = 2) equals the one-call result and the reference."""
    base = 5
    sx, tx, ei = regular_set(k, n_t=300, seed=80 + k, dst_base=base)
    n_t, e = 300, ei.shape[1]
    ref = Ref(sx, tx, ei)
    call = Call(ops, sx, tx, ei, ts=True, tt=False)
    ws = call.ws.data_ptr()
    whole = torch.empty(8, dtype=torch.float64, device="cuda")
    call.outputs()
    call.stats(0, e, whole.data_ptr(), True)
    whole_rot = whole.cpu().numpy()
    call.stats(0, e, whole.data_ptr(), False)
    whole_norot = whole.cpu().numpy()
    for name, listed in _flag_lists(n_t, np.random.default_rng(k)).items():
        flags = torch.zeros(n_t, dtype=torch.uint8, device="cuda")
        flags[dev(listed.astype(np.int64))] = 1
        f_list, f_count = ops.compact_flags(flags)
        assert int(f_count.item()) == listed.size
        flagged_edges = np.repeat(np.isin(np.arange(n_t), listed), k)
        for mode in ("list", "only", "only_k"):
            for norm, inv, rot in ((n, i, r) for n, i, r in CONFIGS if i == (n in ("l1", "unit-range"))):
                st = torch.tensor([NO_VALUE * 2] * 2, dtype=torch.float64, device="cuda")
                call.outputs()
                _check(lib.agx_edge_attrs_stats(
                    call.col(0), call.col(1), e, *call.nodes, 1, 1, int(rot), call.len_ptr(), call.dir_ptr(),
                    st[0].data_ptr(), ws, flags.data_ptr() - base, 1, None, None, k, _stream()))  # fmt: skip
                fe = torch.from_numpy(flagged_edges).cuda()
                call.out_len[fe] = float("nan")  # what the second pass must overwrite
                call.out_dir[fe] = float("nan")
                if mode == "list":
                    _check(lib.agx_edge_attrs_stats(
                        call.col(0), call.col(1), e, *call.nodes, 1, 1, int(rot), call.len_ptr(), call.dir_ptr(),
                        st[1].data_ptr(), ws, None, 2, f_list.data_ptr(), f_count.data_ptr(), k, _stream()))  # fmt: skip
                else:
                    _check(lib.agx_edge_attrs_stats(
                        call.col(0), call.col(1), e, *call.nodes, 1, 1, int(rot), call.len_ptr(), call.dir_ptr(),
                        st[1].data_ptr(), ws, flags.data_ptr() - base, 2, None, None, k if mode == "only_k" else 0,
                        _stream()))  # fmt: skip
                s = st.cpu().numpy()
                w = whole_rot if rot else whole_norot
                msg = f"k={k} list={name} {mode} {norm} inv={inv} rot={rot}"
                np.testing.assert_allclose(s[0, [0, 1, 4, 5]] + s[1, [0, 1, 4, 5]], w[[0, 1, 4, 5]], rtol=1e-12, err_msg=msg)
                np.testing.assert_array_equal(np.minimum(s[0, [2, 6]], s[1, [2, 6]]), w[[2, 6]], err_msg=msg)
                np.testing.assert_array_equal(np.maximum(s[0, [3, 7]], s[1, [3, 7]]), w[[3, 7]], err_msg=msg)
                if listed.size == 0:
                    np.testing.assert_array_equal(s[1], NO_VALUE * 2)
                call.apply(0, e, norm, inv, norm, rot, st, 2)
                ln, dr = call.result()
                one = call.one(norm, inv, norm, rot, regular_k=k)
                close_or_bits(ln, one[0], norm, msg)
                close_or_bits(dr, one[1], norm, msg)
                check_all(ln, dr, ref, norm, inv, norm, rot, msg)
        # the production path: ops.DeferredEdgeAttributes with the list, regular_k and the flag offset
        for norm in ("unit-std", "unit-range", "l2"):
            job = ops.DeferredEdgeAttributes(call.ei, call.src, call.dst, flags, length_norm=norm, direction_norm=norm,
                                             flag_list=f_list, flag_count=f_count, regular_k=k, flag_base=base)  # fmt: skip
            job.raw()
            fe = torch.from_numpy(flagged_edges).cuda()
            job.out_len[fe] = float("nan")
            job.out_dir[fe] = float("nan")
            job.patch()
            job.apply()
            one = call.one(norm, False, norm, True, regular_k=k)
            close_or_bits(job.out_len.cpu().numpy(), one[0], norm, f"deferred k={k} {name} {norm}")
            close_or_bits(job.out_dir.cpu().numpy(), one[1], norm, f"deferred k={k} {name} {norm}")
            check_all(job.out_len.cpu().numpy(), job.out_dir.cpu().numpy(), ref, norm, False, norm, True, "deferred")


# ------------------------------------------------------------------------------------------------
# argument checks
# ------------------------------------------------------------------------------------------------
def test_out_dir_must_be_8_byte_aligned_in_every_work_set(ops, lib, adversarial):
    """A direction output 4 bytes off an 8-byte boundary is refused by every entry point before any device work
    (the kernels store each direction as one float2)."""
    from anemoi_graphs_b200._cabi import AGX_ERR_ARG

    sx, tx, ei = adversarial
    ei = ei[:, :33]
    call = Call(ops, sx, tx, ei)
    call.outputs()
    e, ws = call.E, call.ws.data_ptr()
    bad = call.out_dir.data_ptr() + 4
    st = torch.tensor([NO_VALUE * 2] * 2, dtype=torch.float64, device="cuda")
    flags = torch.ones(e, dtype=torch.uint8, device="cuda")
    f_list, f_count = ops.compact_flags(torch.ones(e, dtype=torch.uint8, device="cuda"))
    before = call.out_dir.clone()
    a, b, s = call.col(0), call.col(1), _stream()
    rcs = {
        "agx_edge_attrs": lib.agx_edge_attrs(a, b, e, *call.nodes, 3, 0, call.len_ptr(), 3, 1, bad, ws, 0, s),
        "agx_edge_attrs regular": lib.agx_edge_attrs(a, b, e, *call.nodes, 0, 0, call.len_ptr(), 0, 1, bad, ws, 1, s),
        "agx_edge_attrs_stats all": lib.agx_edge_attrs_stats(
            a, b, e, *call.nodes, 1, 1, 1, call.len_ptr(), bad, st[0].data_ptr(), ws, None, 0, None, None, 0, s),
        "agx_edge_attrs_stats skip": lib.agx_edge_attrs_stats(
            a, b, e, *call.nodes, 1, 1, 1, call.len_ptr(), bad, st[0].data_ptr(), ws, flags.data_ptr(), 1, None, None, 0, s),
        "agx_edge_attrs_stats only": lib.agx_edge_attrs_stats(
            a, b, e, *call.nodes, 1, 1, 1, call.len_ptr(), bad, st[0].data_ptr(), ws, flags.data_ptr(), 2, None, None, 0, s),
        "agx_edge_attrs_stats list": lib.agx_edge_attrs_stats(
            a, b, e, *call.nodes, 1, 1, 1, call.len_ptr(), bad, st[1].data_ptr(), ws, None, 2, f_list.data_ptr(),
            f_count.data_ptr(), 1, s),
        "agx_edge_attrs_apply": lib.agx_edge_attrs_apply(e, 3, 0, call.len_ptr(), 3, 1, bad, st.data_ptr(), 2, e, ws, s),
    }  # fmt: skip
    assert rcs == {name: AGX_ERR_ARG for name in rcs}
    torch.cuda.synchronize()
    assert torch.equal(call.out_dir, before) and (call.out_len == Call.GUARD).all()
