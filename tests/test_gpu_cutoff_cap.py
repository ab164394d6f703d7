"""``CutOffEdges(max_num_neighbours=M)`` / ``ReversedCutOffEdges(max_num_neighbours=M)``: the capped cut-off search.

A query with at most M sources within the radius keeps its cut-off set, columns and order as without the cap; any
other query keeps the M nearest by float64 ``rdist``, ties at the M-th boundary to the lower source index (the KNN
rule).  Checked against ``capped_cutoff_edges`` below (the exact-search oracle's cut-off sets and KNN tie groups,
pinned to sklearn here on the CPU), the uncapped builder, and the intersection of ``CutOffEdges`` with
``KNNEdges(M)``.  Constructor and recipe validation run without a GPU."""

import math

import numpy as np
import pytest
import torch
from sklearn.neighbors import NearestNeighbors

from anemoi_graphs_b200 import grids
from oracle import exact_search as X
from oracle import ref_path as R

T = "anemoi.graphs."
ATTR_RTOL = 1e-6  # DESIGN.md section 4


def x_deg(lat, lon) -> np.ndarray:
    return grids.latlon_deg_to_x(np.asarray(lat, dtype=np.float64), np.asarray(lon, dtype=np.float64)).numpy()


def canon(ei) -> np.ndarray:
    ei = ei.cpu().numpy() if isinstance(ei, torch.Tensor) else np.asarray(ei)
    return R.canonical_sort(ei)


def capped_cutoff_edges(source_x, target_x, radius: float, M: int, tau: float = X.TIE_TAU, extra: int = 8):
    """``CutOffEdges(max_num_neighbours=M)`` restated on ``oracle/exact_search``: a target keeps its cut-off set
    (``Grid.radius``) when it has at most ``M`` members, else the ``M`` nearest of them under the KNN tie rule
    (``Grid.knn`` + ``knn_tie_groups``: the tie group of the M-th smallest rdist is filled from the lowest source index).
    Returns ``(edge_index sorted by (dst, src), info)``; ``info["capped"]`` / ``info["tied"]`` are the capped target ids
    and those with a tie at the boundary.  Raises when a tie group reaches past the ``M + extra`` candidates fetched, as
    ``knn_edges_canonical`` does."""
    offsets, src, _ = X.Grid(source_x, cell_rad=max(radius, 0.01)).radius(target_x, radius, tau)
    counts = np.diff(offsets)
    nq = counts.size
    capped = np.nonzero(counts > M)[0]
    under = np.stack([src[np.repeat(counts <= M, counts)], np.repeat(np.arange(nq, dtype=np.int32), counts * (counts <= M))])
    tied, chosen = np.empty(0, dtype=np.int64), np.empty((0, M), dtype=np.int32)
    if capped.size:
        n_src = np.asarray(source_x).shape[0]
        kk = min(n_src, M + extra)
        ind, rd = X.Grid(source_x).knn(np.asarray(target_x)[capped], kk)
        thr = math.sin(0.5 * radius) ** 2
        rd = np.where(rd <= thr, rd, np.inf)  # only the cut-off set competes: candidates past it join no tie group
        chosen, tied_rows, report = X.knn_tie_groups(ind, rd, M, tau)
        open_ended = [r["query"] for r in report if r["group_open_ended"] and kk < n_src]
        if open_ended:
            raise RuntimeError(f"tie group wider than extra={extra} for queries {capped[open_ended[:5]]}; raise `extra`")
        tied = capped[tied_rows]
    over = np.stack([chosen.reshape(-1), np.repeat(capped.astype(np.int32), M)])
    edge_index = np.concatenate([under, over], axis=1).astype(np.int32)
    return R.canonical_sort(edge_index), {"capped": capped, "tied": tied, "counts": counts}


def sklearn_capped(src, q, radius, M) -> np.ndarray:
    """sklearn ``radius_neighbors``, then per row a stable sort by (rdist, index) and the first M."""
    dist, ind = NearestNeighbors(metric="haversine").fit(src).radius_neighbors(q, radius=radius)
    cols = []
    for i in range(q.shape[0]):
        o = np.lexsort((ind[i], np.sin(0.5 * dist[i]) ** 2))[:M]
        cols.append(np.stack([ind[i][o], np.full(o.size, i)]))
    return R.canonical_sort(np.concatenate(cols, axis=1).astype(np.int32))


def tie_cloud():
    """Sources with exact ties at many boundaries: every source three times, plus the mirror images (lon -> -lon) of
    a random set around queries on the meridian lon = 0 (bit-equal rdist)."""
    base = x_deg(*grids.uniform_sphere(1500, seed=31))
    mirror = base.copy()
    mirror[:, 1] = -mirror[:, 1]
    src = np.concatenate([np.repeat(base[:300], 3, axis=0), base, mirror])
    lat = np.linspace(-1.4, 1.4, 60, dtype=np.float32)
    q = np.concatenate([np.stack([lat, np.zeros_like(lat)], axis=1), base[:200]])
    return src, q


# ------------------------------------------------------------------------------------------------
# CPU: the oracle, constructors, recipes
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1, 2, 5, 16, 1000])
def test_oracle_equals_sklearn(M):
    src = x_deg(*grids.uniform_sphere(3000, seed=1))
    q = x_deg(*grids.uniform_sphere(400, seed=2))
    for radius in (0.05, 0.12):
        got, info = capped_cutoff_edges(src, q, radius, M)
        np.testing.assert_array_equal(got, sklearn_capped(src, q, radius, M))
    assert (info["capped"].size > 0) == (M < 1000)


@pytest.mark.parametrize("M", [1, 2, 3, 4, 7])
def test_oracle_equals_sklearn_with_exact_ties(M):
    src, q = tie_cloud()
    got, info = capped_cutoff_edges(src, q, 0.08, M, extra=16)
    np.testing.assert_array_equal(got, sklearn_capped(src, q, 0.08, M))
    assert info["tied"].size > 0 and set(info["tied"]) <= set(info["capped"])


BAD = [(0, "must be positive"), (-1, "must be positive"), (2.5, "must be an integer"), (True, "must be an integer"),
       ("64", "must be an integer")]  # fmt: skip


def test_constructor_validation():
    from anemoi_graphs_b200.edges import CutOffEdges, ReversedCutOffEdges

    for cls in (CutOffEdges, ReversedCutOffEdges):
        assert cls("a", "b", 0.6).max_num_neighbours is None
        assert cls("a", "b", 0.6, max_num_neighbours=64).max_num_neighbours == 64
        for bad, msg in BAD:
            with pytest.raises(AssertionError, match=f"Maximum number of neighbours {msg}"):
                cls("a", "b", 0.6, max_num_neighbours=bad)


def _recipe(builder: dict) -> dict:
    return {
        "nodes": {"hidden": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": 5}}},
        "edges": [{"source_name": "hidden", "target_name": "hidden", "edge_builders": [builder]}],
    }


def test_recipe_validation():
    from anemoi_graphs_b200.create import GraphCreator

    for name in ("CutOffEdges", "ReversedCutOffEdges"):
        GraphCreator(_recipe({"_target_": T + f"edges.{name}", "cutoff_factor": 0.6}))
        GraphCreator(_recipe({"_target_": T + f"edges.{name}", "cutoff_factor": 0.6, "max_num_neighbours": 64}))
        for bad, msg in BAD:
            with pytest.raises(AssertionError, match=f"Maximum number of neighbours {msg}"):
                GraphCreator(_recipe({"_target_": T + f"edges.{name}", "cutoff_factor": 0.6, "max_num_neighbours": bad}))


# ------------------------------------------------------------------------------------------------
# GPU: the search itself
# ------------------------------------------------------------------------------------------------
def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


MODES = [(t, b) for t in ("0", "1") for b in ("0", "1")]


def run_capped(ref, q, radius, M, dst_base=0, maps=None):
    """(edge_index as the kernels wrote it, stats) of one capped search."""
    from anemoi_graphs_b200 import ops

    stats = ops.new_stats("cuda")
    with ops.NeighbourIndex(dev(ref), hint_radius=radius) as ix:
        qd = dev(q)
        offsets, total, counts = ix.radius_capped(qd, radius, M)
        out = torch.empty((2, total), dtype=torch.int32, device="cuda")
        if maps is None:
            ix.radius_fill(qd, radius, offsets, total, out, 0, dst_base=dst_base, stats=stats, counts=counts,
                           max_neighbours=M)  # fmt: skip
        else:
            with ops.output_maps(*maps):
                ix.radius_fill(qd, radius, offsets, total, out, 0, dst_base=dst_base, stats=stats, counts=counts,
                               max_neighbours=M)  # fmt: skip
    return out.cpu().numpy(), stats.cpu().numpy()


def run_uncapped(ref, q, radius):
    from anemoi_graphs_b200 import ops

    stats = ops.new_stats("cuda")
    with ops.NeighbourIndex(dev(ref), hint_radius=radius) as ix:
        return ix.radius(dev(q), radius, stats=stats).cpu().numpy(), stats.cpu().numpy()


def check_capped(ref, q, radius, M, monkeypatch, extra=8):
    """Every K3 mode gives the same bits; equal to the oracle; under-cap queries keep their uncapped columns in order;
    capped queries come in ascending (rdist, index); stats 0 / 1 as uncapped, 2 / 3 = capped / tied queries."""
    want, info = capped_cutoff_edges(ref, q, radius, M, extra=extra)
    outs = {}
    for tile, binned in MODES:
        monkeypatch.setenv("AGX_RADIUS_TILE", tile)
        monkeypatch.setenv("AGX_RADIUS_BIN", binned)
        outs[(tile, binned)] = run_capped(ref, q, radius, M), run_uncapped(ref, q, radius)
    (ei, st), (full, fst) = outs[("0", "0")]
    for key, ((e, s), (f, _)) in outs.items():
        np.testing.assert_array_equal(e, ei, err_msg=str(key))
        np.testing.assert_array_equal(f, full, err_msg=str(key))
        np.testing.assert_array_equal(s, st, err_msg=str(key))
    np.testing.assert_array_equal(canon(ei), want)
    assert st[0] == fst[0] and st[1] == fst[1]
    assert st[2] == info["capped"].size and st[3] == info["tied"].size
    counts = info["counts"]
    under = np.isin(ei[1], np.nonzero(counts <= M)[0])
    np.testing.assert_array_equal(ei[:, under], full[:, np.isin(full[1], np.nonzero(counts <= M)[0])])
    assert (np.diff(ei[1]) >= 0).all()  # grouped by query
    capped = ~under
    if capped.any():
        # ascending rdist; the kept members of the boundary's tie group (within 2^-40 of each other) come by index
        rd = X.pair_rdist(q[ei[1][capped]], ref[ei[0][capped]])
        qq = ei[1][capped]
        ok = rd[1:] >= rd[:-1] * (1.0 - 2.0 * X.TIE_TAU)
        assert (ok | (qq[1:] != qq[:-1])).all()
    return ei, st, info


def clustered_cloud(seed: int):
    rng = np.random.default_rng(seed)
    lat, lon = grids.uniform_sphere(40, seed=seed)
    centres = np.stack([np.deg2rad(lat), np.deg2rad(lon)], axis=1)
    pts = [centres[i] + rng.normal(scale=s, size=(n, 2)) for i, (n, s) in enumerate(zip(rng.integers(20, 2000, 40),
                                                                                        rng.uniform(1e-3, 3e-2, 40)))]  # fmt: skip
    pts = np.concatenate(pts)
    pts[:, 0] = np.clip(pts[:, 0], -1.5, 1.5)
    return np.concatenate([pts.astype(np.float32), x_deg(*grids.uniform_sphere(5000, seed=seed + 1))])


@pytest.fixture(scope="module")
def o96():
    dx = x_deg(*grids.octahedral_grid(96))
    hx, _ = R.tri_nodes(5)
    return dx, np.ascontiguousarray(hx, dtype=np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 3, 16, 64, 65, 200, 1000])
@pytest.mark.parametrize("factor", [0.6, 1.5, 4.0])
def test_o96_parity(o96, M, factor, monkeypatch):
    dx, hx = o96
    radius = R.cutoff_radius(hx, factor)
    ei, st, info = check_capped(dx, hx, radius, M, monkeypatch)
    if M >= info["counts"].max():
        assert st[2] == 0
        np.testing.assert_array_equal(ei, run_uncapped(dx, hx, radius)[0])  # the cap does not bind: unchanged
    if M <= 64:
        with torch.no_grad():
            from anemoi_graphs_b200 import ops

            with ops.NeighbourIndex(dev(dx), hint_k=M) as ix:
                knn = ix.knn(dev(hx), M).cpu().numpy()
        cut = run_uncapped(dx, hx, radius)[0]
        both = np.intersect1d(cut[0].astype(np.int64) << 32 | cut[1], knn[0].astype(np.int64) << 32 | knn[1])
        inter = np.stack([both >> 32, both & 0xFFFFFFFF]).astype(np.int32)
        np.testing.assert_array_equal(canon(ei), R.canonical_sort(inter))


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 3, 16, 64, 65, 200, 1000])
def test_clustered_cloud_parity(M, monkeypatch):
    ref = clustered_cloud(7)
    q = clustered_cloud(8)[::7]
    for radius in (2e-3, 2e-2, 8e-2):
        check_capped(ref, q, radius, M, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 2, 3, 4, 7])
def test_ties_go_to_the_lower_index(M, monkeypatch):
    src, q = tie_cloud()
    ei, st, info = check_capped(src, q, 0.08, M, monkeypatch, extra=16)
    assert st[3] > 0 and st[3] == info["tied"].size and st[2] == info["capped"].size
    np.testing.assert_array_equal(canon(ei), sklearn_capped(src, q, 0.08, M))


@pytest.mark.gpu
def test_long_segments_dst_base_and_output_maps(monkeypatch):
    """One query with > 1e5 candidates; dst_base != 0; masked node sets through the output maps."""
    rng = np.random.default_rng(5)
    dense = (np.array([0.3, 1.0]) + rng.normal(scale=4e-3, size=(150000, 2))).astype(np.float32)
    ref = np.concatenate([dense, x_deg(*grids.uniform_sphere(20000, seed=6))])
    q = np.concatenate([np.array([[0.3, 1.0]], dtype=np.float32), dense[:500:5], x_deg(*grids.uniform_sphere(300, seed=7))])
    radius = 0.03
    for M in (64, 1000):
        ei, st, info = check_capped(ref, q, radius, M, monkeypatch)
        assert info["counts"][0] > 100000
    want, _ = capped_cutoff_edges(ref, q, radius, 64)
    got, _ = run_capped(ref, q, radius, 64, dst_base=1000)
    np.testing.assert_array_equal(canon(got - np.array([[0], [1000]], dtype=np.int32)), want)
    src_sel = np.sort(rng.choice(ref.shape[0] * 2, ref.shape[0], replace=False))
    dst_sel = np.sort(rng.choice(q.shape[0] * 3, q.shape[0], replace=False))
    got, _ = run_capped(ref, q, radius, 64, maps=(dev(src_sel), dev(dst_sel)))
    np.testing.assert_array_equal(canon(got), R.canonical_sort(np.stack([src_sel[want[0]], dst_sel[want[1]]]).astype(np.int32)))


# ------------------------------------------------------------------------------------------------
# GPU: the builders
# ------------------------------------------------------------------------------------------------
def _graph(o96, masks=False):
    from anemoi_graphs_b200.graph import HeteroData

    g = HeteroData()
    for name, x in zip(("data", "hidden"), o96):
        g[name].x = torch.from_numpy(x)
        g[name]["m"] = torch.from_numpy(((x[:, 1] < 1.0) | (x[:, 0] > 0.3)).reshape(-1, 1))
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("M", [4, 16])
@pytest.mark.parametrize("masked", [False, True])
def test_builders_forward_reversed_masks_and_attributes(o96, M, masked):
    from anemoi_graphs_b200.edges import CutOffEdges, ReversedCutOffEdges

    dx, hx = o96
    g = _graph(o96)
    m = "m" if masked else None
    fwd = CutOffEdges("data", "hidden", 0.6, source_mask_attr_name=m, target_mask_attr_name=m, max_num_neighbours=M)
    fwd.update_graph(g, {"len": {"_target_": T + "edges.attributes.EdgeLength"},
                         "dirs": {"_target_": T + "edges.attributes.EdgeDirection"}})  # fmt: skip
    rev = ReversedCutOffEdges("hidden", "data", 0.6, source_mask_attr_name=m, target_mask_attr_name=m,
                              max_num_neighbours=M)  # fmt: skip
    rev.update_graph(g)
    ei = g[("data", "to", "hidden")].edge_index.numpy()
    np.testing.assert_array_equal(g[("hidden", "to", "data")].edge_index.numpy(), np.ascontiguousarray(ei[::-1]))
    s_sel = np.nonzero(g["data"]["m"].numpy().ravel())[0] if masked else np.arange(dx.shape[0])
    t_sel = np.nonzero(g["hidden"]["m"].numpy().ravel())[0] if masked else np.arange(hx.shape[0])
    want, info = capped_cutoff_edges(dx[s_sel], hx[t_sel], fwd.radius, M)
    assert info["capped"].size > 0  # the largest degree is 20
    want = R.canonical_sort(np.stack([s_sel[want[0]], t_sel[want[1]]]).astype(np.int32))
    np.testing.assert_array_equal(canon(ei), want)
    np.testing.assert_allclose(g[("data", "to", "hidden")]["len"].numpy(), R.edge_length(dx, hx, ei), rtol=ATTR_RTOL, atol=0)
    want_d = R.edge_direction(dx, hx, ei)
    np.testing.assert_allclose(g[("data", "to", "hidden")]["dirs"].numpy(), want_d, rtol=ATTR_RTOL,
                               atol=ATTR_RTOL * np.abs(want_d).max())  # fmt: skip


@pytest.mark.gpu
@pytest.mark.parametrize("resident", [False, True])
def test_provisional_indexed_side(o96, resident, monkeypatch):
    """TriNodes indexed (sources of a forward cut-off, targets of a reversed one): the lazily ordered build equals the
    one with the order sorted first, bit for bit."""
    from anemoi_graphs_b200 import device as agx_device
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.graph import HeteroData

    recipe = {
        "nodes": {"hidden": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": 5}}},
        "edges": [
            {"source_name": "hidden", "target_name": "data", "edge_builders": [
                {"_target_": T + "edges.CutOffEdges", "cutoff_factor": 6.0, "max_num_neighbours": 3}]},
            {"source_name": "data", "target_name": "hidden", "edge_builders": [
                {"_target_": T + "edges.ReversedCutOffEdges", "cutoff_factor": 6.0, "max_num_neighbours": 2}]},
        ],
    }  # fmt: skip

    def run(lazy):
        monkeypatch.setattr(agx_device, "LAZY_NODE_ORDER", lazy)
        prev = agx_device.set_resident(resident)
        try:
            g = HeteroData()
            g["data"].x = torch.from_numpy(o96[0]).cuda() if resident else torch.from_numpy(o96[0])
            g["data"].node_type = "LatLonNodes"
            g = GraphCreator(recipe).update_graph(g)
            torch.cuda.synchronize()
            return g
        finally:
            agx_device.set_resident(prev)

    a, b = run(True), run(False)
    hx = b["hidden"].x.cpu().numpy()
    for key in (("hidden", "to", "data"), ("data", "to", "hidden")):
        np.testing.assert_array_equal(a[key].edge_index.cpu().numpy(), b[key].edge_index.cpu().numpy())
    want, info = capped_cutoff_edges(hx, o96[0], R.cutoff_radius(o96[0], 6.0), 3)
    assert info["tied"].size > 0  # the mesh's mirror symmetry: ties at the boundary, decided by the final numbering
    np.testing.assert_array_equal(canon(a[("hidden", "to", "data")].edge_index), want)


@pytest.mark.gpu
def test_cli_prints_capped_counts(tmp_path, capsys):
    import yaml

    from anemoi_graphs_b200.__main__ import main

    recipe = {
        "nodes": {
            "data": {"node_builder": {"_target_": T + "nodes.ReducedGaussianGridNodes", "grid": "o96"}},
            "hidden": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": 5}},
        },
        "edges": [{"source_name": "data", "target_name": "hidden", "edge_builders": [
            {"_target_": T + "edges.CutOffEdges", "cutoff_factor": 0.6, "max_num_neighbours": 4}]}],
    }  # fmt: skip
    (tmp_path / "r.yaml").write_text(yaml.safe_dump(recipe))
    dx = x_deg(*grids.octahedral_grid(96))
    hx, _ = R.tri_nodes(5)
    want, info = capped_cutoff_edges(dx, hx, R.cutoff_radius(hx, 0.6), 4)
    assert want.shape[1] < 62980 and info["capped"].size > 0  # 62 980 uncapped
    assert main(["create", str(tmp_path / "r.yaml"), str(tmp_path / "g.pt")]) == 0
    out = capsys.readouterr().out
    assert f" {want.shape[1]} " in out, out


@pytest.mark.gpu
@pytest.mark.parametrize("res,capped_share", [(6, 1.0), (7, 0.4)])
def test_full_size_o1280(res, capped_share):
    from anemoi_graphs_b200.edges import CutOffEdges

    dx = x_deg(*grids.octahedral_grid(1280))
    hx, _ = R.tri_nodes(res)
    hx = np.ascontiguousarray(hx, dtype=np.float32)
    g = _graph((dx, hx))
    b = CutOffEdges("data", "hidden", 0.6, max_num_neighbours=64)
    b.update_graph(g)
    want, info = capped_cutoff_edges(dx, hx, b.radius, 64)
    assert info["capped"].size >= capped_share * hx.shape[0] * 0.99
    np.testing.assert_array_equal(canon(g[("data", "to", "hidden")].edge_index), want)
