"""SphericalAreaWeights on cutout node sets: a global O-grid with a cap cut out of it and a finer O-grid's points
inside a smaller cap, which leaves an empty ring like a cutout's ``min_distance_km``.  The cells on both sides of the
ring are not closed by their 63 nearest neighbours, so they go through the wide pass (``agx_voronoi_areas_wide``)."""

import numpy as np
import pytest
import torch

from oracle import ref_path as R

pytestmark = pytest.mark.gpu

RAW_RTOL = 1e-9  # as test_gpu_node_attributes.py: float64 areas, scipy's half-spaces and solid-angle formula
ATTR_RTOL = 1e-6
# scipy's calculate_areas takes each area as the difference of two entries of ONE running sum (np.cumsum) of the
# triangle solid angles of the whole sphere, which climbs to 4 pi: every area carries the rounding of that sum, up
# to ~5e-15 sr whatever the cell's size - 2e-9 relative for an O1280 cell (2e-6 sr), 2e-8 for an O2560 one, against
# 1e-13 when the same float64 triangle terms are summed per cell.  So each cell is checked against scipy wherever
# scipy agrees with its own diagram evaluated in extended precision (``_hull_areas_extended``), and every cell
# against that extended evaluation, both at RAW_RTOL.
SCIPY_SELF_RTOL = 1e-10

# case: (global O-grid, regional O-grid, regional cap (deg), empty ring (deg), centre lat, centre lon)
CASES = {
    "A": (48, 1280, 10.0, 0.3, 50.0, 10.0),
    "B": (24, 2560, 3.0, 0.5, 0.0, 0.0),  # km-scale ratio; the patch crosses the 0/360 meridian
    "C": (32, 1280, 10.0, 0.5, 90.0, 0.0),  # over the pole: the regional part is north of 80 degrees
    "D": (96, 1280, 8.0, 0.3, 0.0, 0.0),
    "E": (24, 1280, 10.0, 0.3, 50.0, 10.0),  # case A's patch under a coarser global grid
}
WIDER_THAN_32 = ("B", "E")  # the cases whose widest scipy region has more than 32 vertices


def _unit(lat_deg, lon_deg):
    la, lo = np.deg2rad(lat_deg), np.deg2rad(lon_deg)
    return np.stack([np.cos(la) * np.cos(lo), np.cos(la) * np.sin(lo), np.sin(la)], -1)


def cutout(n_global, n_regional, cap, gap, lat0, lon0, regional_only=False):
    """float32 (N, 2) radians: the global points farther than cap + gap from the centre, then the regional points
    within cap of it."""
    from anemoi_graphs_b200 import grids

    centre = _unit(np.float64(lat0), np.float64(lon0))
    parts = []
    for n, keep in ((n_global, lambda a: a > cap + gap), (n_regional, lambda a: a <= cap)):
        lat, lon = grids.octahedral_grid(n)
        ang = np.rad2deg(np.arccos(np.clip(_unit(lat, lon) @ centre, -1.0, 1.0)))
        parts.append((lat[keep(ang)], lon[keep(ang)]))
    if regional_only:
        parts = parts[1:]
    lat = np.concatenate([p[0] for p in parts])
    lon = np.concatenate([p[1] for p in parts])
    return grids.latlon_deg_to_x(lat, lon).numpy()


def _hull_areas_extended(points, sv):
    """The areas of scipy's diagram with its vertices recomputed from the float32 generators in long double: each
    vertex the unit normal of its hull facet (a, b, c), then the same Van Oosterom - Strackee sum over the same sorted
    regions."""
    P = points.astype(np.longdouble)
    a, b, c = (P[sv._simplices[:, j]] for j in range(3))
    nrm = np.cross(b - a, c - a)
    nrm /= np.sqrt((nrm * nrm).sum(1))[:, None]
    nrm *= np.sign((nrm * a).sum(1))[:, None]
    out = np.zeros(len(P), dtype=np.longdouble)
    for i, region in enumerate(sv.regions):
        v = nrm[region]
        w = np.roll(v, 1, axis=0)
        num = (P[i] * np.cross(v, w)).sum(1)
        den = 1 + (P[i] * v).sum(1) + (v * w).sum(1) + (w * P[i]).sum(1)
        out[i] = np.abs(2 * np.arctan2(num, den)).sum()
    return out.astype(np.float64)


def _scipy(x):
    """scipy's areas, the same diagram in extended precision, and scipy's widest region."""
    from scipy.spatial import SphericalVoronoi

    points = R.latlon_rad_to_cartesian((x[:, 0], x[:, 1]))
    sv = SphericalVoronoi(points, 1.0, np.array([0, 0, 0]))
    want = sv.calculate_areas()  # sorts the regions
    return want, _hull_areas_extended(points, sv), max(len(r) for r in sv.regions)


@pytest.fixture(scope="module", params=sorted(CASES))
def case(request):
    x = cutout(*CASES[request.param])
    return (request.param, x, *_scipy(x))


def test_cutout_areas_match_scipy(case):
    from anemoi_graphs_b200 import ops

    name, x, want, extended, widest = case
    got = ops.voronoi_areas(torch.from_numpy(x).cuda()).cpu().numpy()
    info = dict(ops.voronoi_wide)
    # the set needs the new pass: its cells are not closed by their 63 nearest neighbours (the k <= 64 passes raise)
    assert info["cells"] > 0 and info["rounds"] >= 1, info
    if name in WIDER_THAN_32:  # a coarse cell bordered by more fine cells than k_voronoi_areas' 32-edge polygon holds
        assert widest > 32
    wide = np.zeros(len(x), dtype=bool)
    wide[info["generators"].long().cpu().numpy()] = True
    scipy_exact = np.abs(want - extended) <= SCIPY_SELF_RTOL * extended
    # the cells of the wide pass and every other cell where scipy agrees with its own hull: scipy at 1e-9, no atol
    for sel, what in ((wide & scipy_exact, "wide-pass"), (~wide & scipy_exact, "other")):
        bad = np.flatnonzero(sel & ~np.isclose(got, want, rtol=RAW_RTOL, atol=0))
        assert bad.size == 0, f"case {name}: {bad.size} {what} cells differ from scipy: {bad[:5]} {got[bad[:5]]} {want[bad[:5]]}"
    # every cell, scipy's rounded ones included: its hull in extended precision at 1e-9
    bad = np.flatnonzero(~np.isclose(got, extended, rtol=RAW_RTOL, atol=0))
    assert bad.size == 0, f"case {name}: {bad.size} cells differ from the extended hull: {bad[:5]}"
    assert (got > 0).all()
    np.testing.assert_allclose(got.sum(), 4 * np.pi, rtol=1e-7)
    again = ops.voronoi_areas(torch.from_numpy(x).cuda()).cpu().numpy()
    assert np.array_equal(got.view(np.int64), again.view(np.int64))


def test_cutout_through_graph_creator():
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.graph import HeteroData

    x = cutout(*CASES["A"])
    lat, lon = np.rad2deg(x[:, 0].astype(np.float64)), np.rad2deg(x[:, 1].astype(np.float64))
    T = "anemoi.graphs."
    recipe = {
        "nodes": {
            "data": {
                "node_builder": {"_target_": T + "nodes.LatLonNodes", "latitudes": lat, "longitudes": lon},
                "attributes": {"area_weight": {"_target_": T + "nodes.attributes.SphericalAreaWeights", "norm": "unit-max"}},
            },
        },
        "edges": [],
    }
    graph = GraphCreator(recipe).update_graph(HeteroData())
    want = R.spherical_area_weights(graph["data"].x.numpy(), "unit-max")
    got = graph["data"]["area_weight"]
    assert got.dtype == torch.float32
    np.testing.assert_allclose(got.numpy(), want, rtol=ATTR_RTOL)


def test_regional_part_alone_still_raises():
    """A limited-area set on its own: its boundary cells reach round the back of the sphere."""
    from anemoi_graphs_b200 import ops

    x = cutout(*CASES["A"], regional_only=True)
    with pytest.raises(NotImplementedError):
        ops.voronoi_areas(torch.from_numpy(x).cuda())


@pytest.mark.parametrize("n", [96, 1280])
def test_global_grids_skip_the_wide_pass(n):
    from anemoi_graphs_b200 import grids, ops

    x = grids.latlon_deg_to_x(*grids.octahedral_grid(n)).cuda()
    ops.timeline = ops.Timeline()
    try:
        ops.voronoi_areas(x)
        spans = ops.timeline.counts()
    finally:
        ops.timeline = None
    assert ops.voronoi_wide["cells"] == 0
    assert "voronoi_areas_wide" not in spans and "voronoi_areas" in spans
