"""``ReducedGaussianGridNodes`` (newer anemoi-graphs releases) on the GPU: octahedral grids O<N> from two kernels.

The latitudes are checked against 30-digit mpmath roots of P_2N and against numpy's ``leggauss``; the grids bit for bit
against ``grids.latlon_deg_to_x(*grids.octahedral_grid(N))``, the generator ``bench.py`` and the other tests use; the
documentation's O96 -> TriNodes(5) recipe against the same recipe over ``LatLonNodes``.  Constructor and recipe
validation run without a GPU."""

import mpmath
import numpy as np
import pytest
import torch

from anemoi_graphs_b200 import grids
from oracle import ref_path as R

T = "anemoi.graphs."
LAT_MPMATH_TOL = 2e-12  # degrees, against the exact roots (DESIGN.md section 4)
LAT_LEGGAUSS_TOL = 5e-12  # degrees, against numpy's leggauss, whose own error near the poles reaches 3e-12 at N = 1280


# ------------------------------------------------------------------------------------------------
# constructor and recipe validation (CPU)
# ------------------------------------------------------------------------------------------------
def test_constructor_validation():
    from anemoi_graphs_b200.nodes import ReducedGaussianGridNodes
    from anemoi_graphs_b200.nodes.builders.base import BaseNodeBuilder

    for grid in ("o96", "O96"):
        builder = ReducedGaussianGridNodes(grid, "data")
        assert isinstance(builder, BaseNodeBuilder)
        assert builder.grid == grid and builder.n == 96 and builder.name == "data"
    for bad in (96, None, "o", "o0", "x96", "o9.5", " o96", "o-96", "96"):
        with pytest.raises(AssertionError):
            ReducedGaussianGridNodes(bad, "data")
    for classic in ("n320", "N320"):
        with pytest.raises(NotImplementedError, match="classic reduced Gaussian grids"):
            ReducedGaussianGridNodes(classic, "data")


def _recipe(data_builder: dict, hidden_resolution: int = 5, data_attributes: dict | None = None) -> dict:
    """The documentation's encoder / processor / decoder recipe: CutOff 0.6, MultiScale x_hops 1, KNN 3."""
    attrs = {
        "edge_length": {"_target_": T + "edges.attributes.EdgeLength", "norm": "unit-std"},
        "edge_dirs": {"_target_": T + "edges.attributes.EdgeDirection", "norm": "unit-std"},
    }
    data = {"node_builder": data_builder}
    if data_attributes:
        data["attributes"] = data_attributes
    return {
        "nodes": {
            "data": data,
            "hidden": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": hidden_resolution}},
        },
        "edges": [
            {"source_name": "data", "target_name": "hidden", "attributes": attrs,
             "edge_builders": [{"_target_": T + "edges.CutOffEdges", "cutoff_factor": 0.6}]},
            {"source_name": "hidden", "target_name": "hidden", "attributes": attrs,
             "edge_builders": [{"_target_": T + "edges.MultiScaleEdges", "x_hops": 1}]},
            {"source_name": "hidden", "target_name": "data", "attributes": attrs,
             "edge_builders": [{"_target_": T + "edges.KNNEdges", "num_nearest_neighbours": 3}]},
        ],
    }  # fmt: skip


def _grid_recipe(grid) -> dict:
    return _recipe({"_target_": T + "nodes.ReducedGaussianGridNodes", "grid": grid})


def test_recipe_validation():
    from anemoi_graphs_b200.config import resolve_target
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.nodes import ReducedGaussianGridNodes

    assert resolve_target(T + "nodes.ReducedGaussianGridNodes") is ReducedGaussianGridNodes
    GraphCreator(_grid_recipe("o96"))
    GraphCreator(_grid_recipe("O1280"))
    for classic in ("n320", "N96"):
        with pytest.raises(NotImplementedError, match="classic reduced Gaussian grids"):
            GraphCreator(_grid_recipe(classic))
    for bad in (96, "o", "o0", "x96", "o9.5", None):
        with pytest.raises(AssertionError):
            GraphCreator(_grid_recipe(bad))


# ------------------------------------------------------------------------------------------------
# kernels (GPU)
# ------------------------------------------------------------------------------------------------
def mp_latitudes(n: int) -> list:
    """The northern N roots of P_2N as latitudes in degrees, north to south, to 30 digits: Newton in theta (the
    colatitude) from numpy's leggauss nodes, three steps of the three-term recurrence at 30 digits."""
    m = 2 * n
    x0 = np.polynomial.legendre.leggauss(m)[0][::-1][:n]
    out = []
    with mpmath.workdps(30):
        for x in x0:
            theta = mpmath.acos(mpmath.mpf(float(x)))
            for _ in range(3):
                c = mpmath.cos(theta)
                p0, p1 = mpmath.mpf(1), c
                for j in range(2, m + 1):
                    p0, p1 = p1, ((2 * j - 1) * c * p1 - (j - 1) * p0) / j
                theta -= p1 * mpmath.sin(theta) / (m * (c * p1 - p0))
            out.append(90 - theta * 180 / mpmath.pi)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 16, 96])
def test_latitudes_against_mpmath(n):
    from anemoi_graphs_b200 import ops

    lat = ops.gaussian_latitudes(n)
    assert lat.dtype == torch.float64 and lat.shape == (2 * n,) and lat.is_cuda
    assert torch.equal(lat.flip(0), -lat)  # south rows: the exact negation of the north rows
    got = lat.cpu().numpy()
    with mpmath.workdps(30):
        err = [abs(float(mpmath.mpf(float(g)) - want)) for g, want in zip(got[:n], mp_latitudes(n))]
    assert max(err) <= LAT_MPMATH_TOL, (max(err), int(np.argmax(err)))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [320, 1280])
def test_latitudes_against_leggauss(n):
    from anemoi_graphs_b200 import ops

    lat = ops.gaussian_latitudes(n)
    assert torch.equal(lat.flip(0), -lat)
    np.testing.assert_allclose(lat.cpu().numpy(), grids.gaussian_latitudes_deg(n), rtol=0, atol=LAT_LEGGAUSS_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 16, 48, 96, 320, 1280, 2560])
def test_octahedral_grid_bit_for_bit(n):
    from anemoi_graphs_b200 import ops

    got = ops.octahedral_nodes(n)
    assert got.dtype == torch.float32 and got.shape == (4 * n * (n + 9), 2) and got.is_cuda
    want = grids.latlon_deg_to_x(*grids.octahedral_grid(n)).numpy()
    np.testing.assert_array_equal(got.cpu().numpy().view(np.int32), want.view(np.int32))


@pytest.mark.gpu
def test_kernel_arguments_are_checked():
    from anemoi_graphs_b200 import _cabi, ops

    for n in (0, -3):
        with pytest.raises(ValueError, match="must be >= 1"):
            ops.gaussian_latitudes(n)
        with pytest.raises(ValueError, match="must be >= 1"):
            ops.octahedral_nodes(n)
    # O23165 is the largest grid whose 4N(N + 9) points int32 node indices hold
    with pytest.raises(ValueError, match="more than int32 node indices hold"):
        ops.octahedral_nodes(23166)
    lib, stream = _cabi.load_library(), _cabi.current_stream()
    lat = ops.gaussian_latitudes(4)
    out = torch.empty((4 * 4 * 13, 2), dtype=torch.float32, device="cuda")
    assert lib.agx_gaussian_latitudes(23165, None, stream) == _cabi.AGX_ERR_ARG
    assert b"NULL" in lib.agx_last_error()
    assert lib.agx_octahedral_nodes(4, None, _cabi.ptr(out), stream) == _cabi.AGX_ERR_ARG
    assert lib.agx_octahedral_nodes(4, _cabi.ptr(lat), None, stream) == _cabi.AGX_ERR_ARG
    assert lib.agx_octahedral_nodes(4, _cabi.ptr(lat), _cabi.ptr(out), stream) == _cabi.AGX_OK
    np.testing.assert_array_equal(out.cpu().numpy(), grids.latlon_deg_to_x(*grids.octahedral_grid(4)).numpy())


# ------------------------------------------------------------------------------------------------
# node builder and recipes (GPU)
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_builder_host_and_device_resident():
    from anemoi_graphs_b200 import device as agx_device
    from anemoi_graphs_b200.graph import HeteroData
    from anemoi_graphs_b200.nodes import ReducedGaussianGridNodes

    want = grids.latlon_deg_to_x(*grids.octahedral_grid(24))
    graph = ReducedGaussianGridNodes("O24", "data").update_graph(HeteroData(), {})
    x = graph["data"].x
    assert not x.is_cuda and x.dtype == torch.float32 and torch.equal(x, want)
    assert graph["data"].node_type == "ReducedGaussianGridNodes"
    prev = agx_device.set_resident(True)
    try:
        graph = ReducedGaussianGridNodes("o24", "data").update_graph(HeteroData(), {})
    finally:
        agx_device.set_resident(prev)
    x = graph["data"].x
    assert x.is_cuda and x.dtype == torch.float32 and torch.equal(x.cpu(), want)


@pytest.mark.gpu
def test_o96_recipe_equals_the_latlon_recipe():
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.graph import HeteroData

    lat, lon = grids.octahedral_grid(96)
    got = GraphCreator(_grid_recipe("o96")).update_graph(HeteroData())
    want = GraphCreator(_recipe({"_target_": T + "nodes.LatLonNodes", "latitudes": lat, "longitudes": lon})).update_graph(
        HeteroData()
    )
    assert got["data"].node_type == "ReducedGaussianGridNodes"
    assert torch.equal(got["data"].x, want["data"].x) and torch.equal(got["hidden"].x, want["hidden"].x)
    counts = {("data", "to", "hidden"): 62_980, ("hidden", "to", "hidden"): 81_900, ("hidden", "to", "data"): 120_960}
    for key, count in counts.items():
        assert got[key].edge_index.shape == (2, count), key
        for attr in ("edge_index", "edge_length", "edge_dirs"):
            assert torch.equal(got[key][attr], want[key][attr]), (key, attr)


@pytest.mark.gpu
def test_o48_area_weights_through_the_recipe():
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.graph import HeteroData

    attributes = {
        "area_raw": {"_target_": T + "nodes.attributes.SphericalAreaWeights", "norm": None, "dtype": "float64"},
        "area_weight": {"_target_": T + "nodes.attributes.SphericalAreaWeights", "norm": "unit-max"},
    }
    recipe = _recipe({"_target_": T + "nodes.ReducedGaussianGridNodes", "grid": "o48"}, 3, attributes)
    graph = GraphCreator(recipe).update_graph(HeteroData())
    x = graph["data"].x.numpy()
    assert x.shape == (4 * 48 * 57, 2)
    np.testing.assert_allclose(graph["data"]["area_raw"].numpy(), R.spherical_area_weights(x, None, "float64"), rtol=1e-9)
    np.testing.assert_allclose(graph["data"]["area_weight"].numpy(), R.spherical_area_weights(x, "unit-max"), rtol=1e-6)


@pytest.mark.gpu
def test_create_command_on_the_o96_recipe(tmp_path, capsys):
    import yaml

    from anemoi_graphs_b200.__main__ import main

    recipe = tmp_path / "o96.yaml"
    recipe.write_text(yaml.safe_dump(_grid_recipe("o96")))
    assert main(["create", str(recipe), str(tmp_path / "o96.pt")]) == 0
    out = capsys.readouterr().out
    for count in ("62980", "81900", "120960"):
        assert f" {count} " in out, out
