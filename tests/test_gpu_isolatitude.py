"""``IsolatitudeAreaWeights`` (newer anemoi-graphs releases) on the GPU: each node gets the area of its latitude band
over the number of nodes in its row.

The rule (DESIGN.md section 4; upstream parity unverified) is restated below in numpy - ``np.unique`` on the float64 of
the float32 latitudes, the midpoint boundaries closed by the poles, the product form of the band area - and the device
route is checked against it on every kind of node set the package lays out in rows, on unsorted input, at the edge
cases of the rule and through a recipe.  The reference's own self-checks and the recipe validation run without a GPU."""

import numpy as np
import pytest
import torch

from anemoi_graphs_b200 import grids
from oracle import healpix_restated as H
from oracle import ref_path as R

T = "anemoi.graphs."
RAW_RTOL = 1e-14  # float64 weights: the same operations in the same order; CUDA's cos / sin are within 2 ulp of libm's
NORM_RTOL = 1e-12
NORMS = [None, "l1", "l2", "unit-max", "unit-range", "unit-std"]


def reference(x) -> tuple[np.ndarray, int, np.ndarray]:
    """float64 (n,) weights, R and the per-row counts (north to south) of the float32 (n, 2) radians ``x``."""
    lat = np.asarray(x, dtype=np.float32)[:, 0].astype(np.float64) + 0.0  # -0.0 + 0.0 is +0.0: one equatorial row
    rows, inverse, counts = np.unique(lat, return_inverse=True, return_counts=True)  # ascending
    phi, counts = rows[::-1], counts[::-1]  # phi_0 > phi_1 > ... > phi_{R-1}
    n_rows = int(phi.shape[0])
    b = np.empty(n_rows + 1)
    b[0], b[n_rows] = np.pi / 2, -np.pi / 2
    b[1:n_rows] = (phi[:-1] + phi[1:]) / 2
    area = 4 * np.pi * np.cos((b[:-1] + b[1:]) / 2) * np.sin((b[:-1] - b[1:]) / 2)
    return (area / counts)[n_rows - 1 - inverse.reshape(-1)], n_rows, counts


def octahedral_x(n: int) -> np.ndarray:
    return grids.latlon_deg_to_x(*grids.octahedral_grid(n)).numpy()


def latlon_1deg_x() -> np.ndarray:
    """A regular 1-degree grid with 360 nodes at each pole."""
    lat, lon = np.meshgrid(np.arange(90.0, -91.0, -1.0), np.arange(0.0, 360.0, 1.0), indexing="ij")
    return grids.latlon_deg_to_x(lat.ravel(), lon.ravel()).numpy()


def x_of(name: str):
    """The node sets of the parity test, float32 (n, 2) radians (CUDA tensors where the device generates them)."""
    from anemoi_graphs_b200 import ops

    kind, _, arg = name.partition(":")
    if kind == "O":  # the grids ReducedGaussianGridNodes generates
        return ops.octahedral_nodes(int(arg))
    if kind == "healpix":  # nested order: latitudes are not monotone
        return ops.healpix_nodes(int(arg))
    if kind == "latlon1":
        return torch.from_numpy(latlon_1deg_x())
    if kind == "lam":
        return grids.latlon_deg_to_x(*grids.lam_patch())
    return grids.latlon_deg_to_x(*grids.uniform_sphere(int(arg)))


# ------------------------------------------------------------------------------------------------
# the reference and the recipe (CPU)
# ------------------------------------------------------------------------------------------------
def test_class_resolves_and_constructs():
    from anemoi_graphs_b200.config import resolve_target
    from anemoi_graphs_b200.nodes.attributes import BaseNodeAttribute, IsolatitudeAreaWeights

    assert resolve_target(T + "nodes.attributes.IsolatitudeAreaWeights") is IsolatitudeAreaWeights
    attr = IsolatitudeAreaWeights()
    assert isinstance(attr, BaseNodeAttribute) and attr.norm is None and attr.dtype == "float32"
    attr = IsolatitudeAreaWeights(norm="unit-max", dtype="float64")
    assert attr.norm == "unit-max" and attr.dtype == "float64"


def _attr_recipe(norm: str | None = "unit-max") -> dict:
    from test_gpu_reduced_gaussian import _recipe

    attrs = {"area": {"_target_": T + "nodes.attributes.IsolatitudeAreaWeights", "norm": norm}}
    recipe = _recipe({"_target_": T + "nodes.ReducedGaussianGridNodes", "grid": "o96"}, 5, attrs)
    recipe["nodes"]["hidden"]["attributes"] = attrs
    return recipe


def test_graph_creator_accepts_the_class():
    from anemoi_graphs_b200.create import GraphCreator

    GraphCreator(_attr_recipe())
    GraphCreator(_attr_recipe(None))


@pytest.mark.parametrize("n", [1, 16, 96, 1280])
def test_reference_octahedral_rows(n):
    w, n_rows, counts = reference(octahedral_x(n))
    assert n_rows == 2 * n
    i = np.arange(1, n + 1)
    np.testing.assert_array_equal(counts, np.concatenate([4 * i + 16, (4 * i + 16)[::-1]]))
    np.testing.assert_allclose(w.sum(), 4 * np.pi, rtol=1e-13)


def test_reference_row_counts():
    for res in (2, 5, 7):
        w, n_rows, _ = reference(H.healpix_nodes_x(res))
        assert n_rows == 4 * 2**res - 1, res
        np.testing.assert_allclose(w.sum(), 4 * np.pi, rtol=1e-13)
    w, n_rows, counts = reference(latlon_1deg_x())
    assert n_rows == 181 and (counts == 360).all()
    np.testing.assert_allclose(w.sum(), 4 * np.pi, rtol=1e-13)
    # 100 000 random points: almost every node is its own row, 92 pairs share a float32 latitude
    w, n_rows, counts = reference(grids.latlon_deg_to_x(*grids.uniform_sphere(100_000)).numpy())
    assert n_rows == 99_908 and int((counts == 2).sum()) == 92 and int(counts.max()) == 2
    np.testing.assert_allclose(w.sum(), 4 * np.pi, rtol=1e-13)
    w, n_rows, _ = reference(grids.latlon_deg_to_x(*grids.lam_patch()).numpy())
    assert n_rows == 1000
    np.testing.assert_allclose(w.sum(), 4 * np.pi, rtol=1e-13)


# ------------------------------------------------------------------------------------------------
# the kernel (GPU)
# ------------------------------------------------------------------------------------------------
def _assert_parity(x, got: torch.Tensor, n_rows: int) -> None:
    want, want_rows, _ = reference(x.cpu().numpy() if isinstance(x, torch.Tensor) else x)
    assert got.dtype == torch.float64 and got.shape == want.shape and got.is_cuda
    assert n_rows == want_rows
    rel = np.abs(got.cpu().numpy() - want) / want
    assert rel.max() <= RAW_RTOL, (float(rel.max()), int(rel.argmax()))


@pytest.mark.gpu
@pytest.mark.parametrize(
    "name", ["O:1", "O:16", "O:96", "O:320", "O:1280", "healpix:2", "healpix:5", "healpix:7", "latlon1", "lam",
             "sphere:100000"],
)  # fmt: skip
def test_parity(name):
    from anemoi_graphs_b200 import ops

    x = x_of(name)
    got, n_rows = ops.isolatitude_areas(x)
    _assert_parity(x, got, n_rows)


@pytest.mark.gpu
def test_shuffled_nodes_give_the_shuffled_weights():
    from anemoi_graphs_b200 import ops

    x = ops.octahedral_nodes(96)
    perm = torch.randperm(x.shape[0], generator=torch.Generator().manual_seed(7)).cuda()
    got, n_rows = ops.isolatitude_areas(x)
    shuffled, shuffled_rows = ops.isolatitude_areas(x[perm])
    assert shuffled_rows == n_rows == 192
    assert torch.equal(shuffled, got[perm])


@pytest.mark.gpu
def test_edge_cases():
    from anemoi_graphs_b200 import ops

    # -0.0 and +0.0 are one row
    x = torch.tensor([[0.0, 0.1], [-0.0, 0.2], [0.5, 0.0], [-0.0, 3.0], [-0.7, 1.0]], dtype=torch.float32)
    assert torch.signbit(x[1, 0])
    got, n_rows = ops.isolatitude_areas(x)
    assert n_rows == 3 and got[0] == got[1] == got[3]
    _assert_parity(x, got, n_rows)
    # duplicate nodes share their row
    x = torch.tensor([[0.3, 1.0], [0.3, 1.0], [0.3, 1.0], [-1.2, 2.0], [-1.2, 2.0]], dtype=torch.float32)
    got, n_rows = ops.isolatitude_areas(x)
    assert n_rows == 2 and got[0] == got[1] == got[2] and got[3] == got[4]
    _assert_parity(x, got, n_rows)
    # one node: the whole sphere
    got, n_rows = ops.isolatitude_areas(torch.tensor([[0.25, 0.5]]))
    assert n_rows == 1 and got.shape == (1,)
    np.testing.assert_allclose(got.cpu().numpy(), [4 * np.pi], rtol=1e-15)
    # no node
    got, n_rows = ops.isolatitude_areas(torch.empty((0, 2)))
    assert n_rows == 0 and got.shape == (0,) and got.dtype == torch.float64 and got.is_cuda
    # nodes at float32(pi/2) = 1.5707963705 > pi/2 are valid; the outer boundaries stay at +-pi/2
    half_pi = np.float32(np.pi / 2)
    x = torch.tensor([[half_pi, 0.0], [0.0, 0.0], [-half_pi, 0.0]])
    got, n_rows = ops.isolatitude_areas(x)
    assert n_rows == 3
    _assert_parity(x, got, n_rows)
    np.testing.assert_allclose(float(got.sum()), 4 * np.pi, rtol=1e-15)


@pytest.mark.gpu
def test_rejections_leave_the_library_usable():
    from anemoi_graphs_b200 import _cabi, ops

    x = ops.octahedral_nodes(16)
    for bad in (float("nan"), 1.6, -1.6, float("inf")):
        y = x.clone()
        y[100, 0] = bad
        with pytest.raises(ValueError, match="NaN or its magnitude exceeds"):
            ops.isolatitude_areas(y)
    above = np.nextafter(np.float32(np.pi / 2), np.float32(2))
    with pytest.raises(ValueError, match="NaN or its magnitude exceeds"):
        ops.isolatitude_areas(torch.tensor([[0.0, 0.0], [above, 0.0]]))
    got, n_rows = ops.isolatitude_areas(x)
    _assert_parity(x, got, n_rows)
    lib, stream = _cabi.load_library(), _cabi.current_stream()
    out = torch.empty(x.shape[0], dtype=torch.float64, device="cuda")
    assert lib.agx_isolatitude_areas(None, x.shape[0], _cabi.ptr(out), None, stream) == _cabi.AGX_ERR_ARG
    assert b"NULL" in lib.agx_last_error()
    assert lib.agx_isolatitude_areas(_cabi.ptr(x), x.shape[0], None, None, stream) == _cabi.AGX_ERR_ARG
    for n in (-1, 2**31):
        assert lib.agx_isolatitude_areas(_cabi.ptr(x), n, _cabi.ptr(out), None, stream) == _cabi.AGX_ERR_ARG
    assert lib.agx_isolatitude_areas(_cabi.ptr(x), x.shape[0], _cabi.ptr(out), None, stream) == _cabi.AGX_OK
    assert torch.equal(out, got)


# ------------------------------------------------------------------------------------------------
# the attribute (GPU)
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("resident", [False, True])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_norms_through_compute(resident, dtype):
    from anemoi_graphs_b200.graph import HeteroData
    from anemoi_graphs_b200.nodes.attributes import IsolatitudeAreaWeights

    x = torch.from_numpy(octahedral_x(96))
    graph = HeteroData()
    graph["data"].x = x.cuda() if resident else x
    graph["data"].node_type = "LatLonNodes"
    raw = reference(x.numpy())[0][:, None]
    for norm in NORMS:
        got = IsolatitudeAreaWeights(norm=norm, dtype=dtype).compute(graph, "data")
        assert got.is_cuda == resident and got.shape == (x.shape[0], 1) and got.dtype == getattr(torch, dtype)
        want = R.normalise(raw, norm)
        if dtype == "float32":  # the cast may round a value 1e-12 away from the reference's to the neighbouring float
            np.testing.assert_allclose(got.cpu().numpy(), want.astype(np.float32), rtol=2**-23, atol=0)
        else:
            atol = NORM_RTOL if norm == "unit-range" else 0  # unit-range maps the smallest weight to 0
            np.testing.assert_allclose(got.cpu().numpy(), want, rtol=NORM_RTOL, atol=atol)


@pytest.mark.gpu
def test_recipe_data_and_lazily_ordered_hidden_nodes():
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.graph import HeteroData

    got = GraphCreator(_attr_recipe()).update_graph(HeteroData())
    recipe = _attr_recipe()
    for nodes in recipe["nodes"].values():
        del nodes["attributes"]
    want = GraphCreator(recipe).update_graph(HeteroData())
    for name in ("data", "hidden"):
        x = got[name].x
        assert torch.equal(x, want[name].x)
        expected = R.normalise(reference(x.numpy())[0][:, None], "unit-max").astype(np.float32)
        area = got[name]["area"]
        assert area.dtype == torch.float32 and area.shape == (x.shape[0], 1)
        np.testing.assert_allclose(area.numpy(), expected, rtol=2**-23, atol=0)
    # the attribute on the hidden nodes resolves their order before the edges are built, so columns come grouped by final
    # target index instead of the icosphere's vertex numbering: the same edges, compared in canonical (dst, src) order
    for key in (("data", "to", "hidden"), ("hidden", "to", "hidden"), ("hidden", "to", "data")):
        assert got[key].edge_index.shape == want[key].edge_index.shape, key
        orders = [torch.from_numpy(np.lexsort((g[key].edge_index[0].numpy(), g[key].edge_index[1].numpy()))) for g in (got, want)]
        for attr in ("edge_index", "edge_length", "edge_dirs"):
            a, b = got[key][attr], want[key][attr]
            a, b = (a[:, orders[0]], b[:, orders[1]]) if attr == "edge_index" else (a[orders[0]], b[orders[1]])
            assert torch.equal(a, b), (key, attr)
