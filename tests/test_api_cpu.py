"""Host-side logic that needs no GPU: constructor validation mirrored from the reference's tests
(tests/edges/test_knn.py:15-31, test_cutoff.py:15-31, test_multiscale_edges.py:21-35,
tests/generate/test_masks.py), recipe handling, the C-ABI symbol table, shard arithmetic."""

import ctypes
import re

import numpy as np
import pytest
import torch

from anemoi_graphs_b200 import _cabi
from anemoi_graphs_b200 import device as agx_device
from anemoi_graphs_b200.config import DotDict, instantiate, resolve_target
from anemoi_graphs_b200.create import GraphCreator
from anemoi_graphs_b200.edges import CutOffEdges, KNNEdges, MultiScaleEdges
from anemoi_graphs_b200.edges.attributes import EdgeDirection, EdgeLength
from anemoi_graphs_b200.generate.masks import KNNAreaMaskBuilder
from anemoi_graphs_b200.graph import HeteroData
from anemoi_graphs_b200.nodes import HexNodes, LatLonNodes, TriNodes


def test_knn_init():
    KNNEdges("test_nodes1", "test_nodes2", 3)
    for bad in (-1, 4.5, None, "hello"):
        with pytest.raises(AssertionError):
            KNNEdges("test_nodes1", "test_nodes2", bad)


def test_cutoff_init():
    CutOffEdges("test_nodes1", "test_nodes2", 0.5)
    CutOffEdges("test_nodes1", "test_nodes2", 1)
    for bad in (-0.5, "hello", None):
        with pytest.raises(AssertionError):
            CutOffEdges("test_nodes1", "test_nodes2", bad)


def test_multiscale_init():
    assert isinstance(MultiScaleEdges("test_nodes", "test_nodes", 1), MultiScaleEdges)
    for bad in (-1, 0, 1.5, "1"):
        with pytest.raises(AssertionError):
            MultiScaleEdges("test_nodes", "test_nodes", bad)
    with pytest.raises(AssertionError):
        MultiScaleEdges("test_nodes1", "test_nodes2", 1)


def test_multiscale_rejects_other_node_types():
    graph = HeteroData()
    graph["data"].x = torch.zeros((4, 2))
    graph["data"].node_type = "LatLonNodes"
    with pytest.raises(AssertionError):
        MultiScaleEdges("data", "data", 1).update_graph(graph)


def test_mask_builder_init():
    KNNAreaMaskBuilder("nodes", 100)
    for bad in (-1, "hello", None):
        with pytest.raises(AssertionError):
            KNNAreaMaskBuilder("nodes", bad)


def test_node_builders_host_side():
    b = LatLonNodes([0.0, 10.0], [5.0, 350.0], name="n")
    x = b.get_coordinates()
    assert x.dtype == torch.float32 and x.shape == (2, 2)
    np.testing.assert_allclose(x.numpy(), np.deg2rad([[0, 5], [10, 350]]), rtol=1e-6)
    with pytest.raises(AssertionError):
        LatLonNodes([0.0], [1.0, 2.0], name="n")
    assert TriNodes(3, "h").resolutions == [0, 1, 2, 3]
    assert TriNodes([1, 3], "h").resolutions == [1, 3]
    assert HexNodes(2, "h").resolutions == [0, 1, 2]
    if not torch.cuda.is_available():  # no CPU fallback: generating cells without a device must fail loudly
        with pytest.raises(RuntimeError, match="CUDA"):
            HexNodes(1, "h").create_nodes()


def test_attribute_ctor_and_norm_validation():
    assert EdgeLength(norm="l1", invert=True).invert is True
    assert EdgeDirection(luse_rotated_features=False).luse_rotated_features is False


def test_recipe_targets_resolve_to_this_package():
    for target, cls in (
        ("anemoi.graphs.edges.KNNEdges", KNNEdges),
        ("anemoi.graphs.edges.CutOffEdges", CutOffEdges),
        ("anemoi.graphs.edges.MultiScaleEdges", MultiScaleEdges),
        ("anemoi.graphs.edges.attributes.EdgeLength", EdgeLength),
        ("anemoi.graphs.edges.attributes.EdgeDirection", EdgeDirection),
        ("anemoi.graphs.nodes.TriNodes", TriNodes),
        ("anemoi.graphs.nodes.LatLonNodes", LatLonNodes),
    ):
        assert resolve_target(target) is cls
    k = instantiate(DotDict({"_target_": "anemoi.graphs.edges.KNNEdges", "num_nearest_neighbours": 4}),
                    source_name="a", target_name="b")  # fmt: skip
    assert isinstance(k, KNNEdges) and k.name == ("a", "to", "b")


def test_graph_creator_legacy_edge_builder_key(tmp_path):
    recipe = tmp_path / "r.yaml"
    recipe.write_text(
        "nodes: {}\n"
        "edges:\n"
        "  - source_name: a\n    target_name: b\n"
        "    edge_builder: {_target_: anemoi.graphs.edges.KNNEdges, num_nearest_neighbours: 3}\n"
        "    source_mask_attr_name: m\n"
    )
    with pytest.warns(DeprecationWarning):
        creator = GraphCreator(recipe)
    cfg = creator.config.edges[0].edge_builders[0]
    assert cfg.source_mask_attr_name == "m" and cfg.target_mask_attr_name is None


def test_compute_requires_cuda_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    graph = HeteroData()
    graph["a"].x = torch.zeros((4, 2))
    graph["b"].x = torch.zeros((4, 2))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        KNNEdges("a", "b", 2).update_graph(graph)


def test_cabi_library_matches_the_header_and_abi_version():
    header = (_cabi.LIB_PATH.parents[2] / "include" / "agx_b200.h").read_text()
    declared = set(re.findall(r"\b(agx_[a-z0-9_]+)\s*\(", header)) - {"agx_index"}
    assert declared == set(_cabi.SIGNATURES), declared ^ set(_cabi.SIGNATURES)
    lib = _cabi.load_library()
    for name in declared:
        assert isinstance(getattr(lib, name), ctypes._CFuncPtr)
    assert lib.agx_abi_version() == _cabi.ABI_VERSION == 4
    assert lib.agx_edge_attrs_workspace() > 16
    assert lib.agx_multiscale_scratch_per_node(8, 1) == 9 * 7


def test_shard_ranges_partition():
    for n in (0, 1, 7, 163842, 6599680):
        for w in (1, 2, 3, 8):
            r = [agx_device.shard_range(n, k, w) for k in range(w)]
            assert r[0][0] == 0 and r[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(r, r[1:]))
            assert max(b - a for a, b in r) - min(b - a for a, b in r) <= 1


def test_node_ordering_equals_reference_expression():
    """generate/utils.py:30-33 of the reference, restated in oracle/ref_path.py, vs the contiguous-column form."""
    from anemoi_graphs_b200.generate.utils import get_coordinates_ordering
    from oracle import ref_path as R
    from oracle import trimesh_icosphere as TM

    for res in range(7):
        coords = R.cartesian_to_latlon_rad(TM.icosphere(res)[0])
        want = R.coordinates_ordering(coords)
        np.testing.assert_array_equal(get_coordinates_ordering(coords), want)
        np.testing.assert_array_equal(
            get_coordinates_ordering(lat=np.ascontiguousarray(coords[:, 0]), lon=np.ascontiguousarray(coords[:, 1])), want
        )


def test_graph_descriptor_on_a_saved_graph(tmp_path, capsys):
    """describe.py:20-225 - sizes, isolated-node counts and attribute statistics of a saved graph."""
    from anemoi_graphs_b200.describe import GraphDescriptor
    from anemoi_graphs_b200.graph import HeteroData

    g = HeteroData()
    g["a"].x = torch.tensor([[0.1, 0.2], [0.3, 6.0], [-0.5, 3.0]], dtype=torch.float32)
    g["a"].node_type = "LatLonNodes"
    g["a"]["w"] = torch.tensor([[1.0], [2.0], [3.0]])
    g["b"].x = torch.tensor([[0.0, 0.0], [1.0, 1.0]], dtype=torch.float32)
    g["b"].node_type = "LatLonNodes"
    store = g[("a", "to", "b")]
    store.edge_index = torch.tensor([[0, 0, 2], [1, 1, 1]], dtype=torch.int32)
    store.edge_type = "KNNEdges"
    store["edge_length"] = torch.tensor([[1.0], [2.0], [4.0]])
    path = tmp_path / "graph.pt"
    torch.save(g, path)
    d = GraphDescriptor(path)
    assert d.total_size == (6 + 3 + 4) * 4 + 6 * 4 + 3 * 4
    nodes = {row[0]: row for row in d.get_node_summary()}
    assert nodes["a"][1] == 3 and nodes["a"][2] == "w" and nodes["a"][3] == 1
    np.testing.assert_allclose(nodes["a"][4:], np.rad2deg([-0.5, 0.3, 0.2, 6.0]), rtol=1e-6)
    (edges,) = d.get_edge_summary()
    assert edges[:6] == ["a", "b", 3, 1, 1, 1] and edges[6] == "edge_length(1D)"
    table = d.get_attribute_table()
    assert [r[:3] for r in table] == [["Node", "a", "w"], ["Edge", "a-->b", "edge_length"]]
    np.testing.assert_allclose(table[1][4:], [1.0, 7.0 / 3.0, 4.0, np.std([1.0, 2.0, 4.0], ddof=1)], rtol=1e-6)
    d.describe()
    out = capsys.readouterr().out
    assert "Nodes summary" in out and "Edges summary" in out and "Graph ready." in out


class _MockZarrDataset:
    """reference tests/conftest.py MockZarrDataset."""

    def __init__(self, latitudes, longitudes, grids=None):
        self.latitudes = latitudes
        self.longitudes = longitudes
        self.num_nodes = len(latitudes)
        if grids is not None:
            self.grids = grids


def test_zarr_dataset_nodes_and_dataset_masks(monkeypatch):
    """reference tests/nodes/test_zarr.py + test_cutout_nodes.py: the dataset-backed node builder and masks are pure
    input adaptors over ``anemoi.datasets.open_dataset`` (mocked, as in the reference's tests)."""
    from anemoi_graphs_b200.graph import HeteroData
    from anemoi_graphs_b200.nodes import ZarrDatasetNodes
    from anemoi_graphs_b200.nodes.attributes import BooleanAndMask, BooleanNot, BooleanOrMask, CutOutMask
    from anemoi_graphs_b200.nodes.builders import from_file

    lats, lons = [-0.15, 0, 0.15], [0, 0.25, 0.5, 0.75]
    coords = 2 * np.pi * np.array([[lat, lon] for lat in lats for lon in lons])
    ds = _MockZarrDataset(coords[:, 0], coords[:, 1], grids=(4, 8))
    monkeypatch.setattr(from_file, "open_dataset", lambda *a, **k: ds)
    builder = ZarrDatasetNodes({"cutout": ["lam.zarr", "global.zarr"]}, name="test_nodes")
    graph = builder.update_graph(HeteroData(), {})
    x = graph["test_nodes"].x
    assert x.dtype == torch.float32 and x.shape == (12, 2) and graph["test_nodes"].node_type == "ZarrDatasetNodes"
    np.testing.assert_allclose(x.numpy(), np.deg2rad(coords), rtol=1e-6)
    assert graph["test_nodes"]["_dataset"] == {"cutout": ["lam.zarr", "global.zarr"]}
    mask = CutOutMask().compute(graph, "test_nodes")
    assert mask.dtype == torch.bool and mask.shape == (12, 1) and mask[:, 0].tolist() == [True] * 4 + [False] * 8
    graph["test_nodes"]["interior"] = torch.tensor([True, False] * 6)
    both = BooleanAndMask([CutOutMask(), "interior"]).compute(graph, "test_nodes")[:, 0].tolist()
    assert both == [True, False, True, False] + [False] * 8
    either = BooleanOrMask([BooleanNot(CutOutMask()), "interior"]).compute(graph, "test_nodes")[:, 0].tolist()
    assert either == [True, False, True, False] + [True] * 8
    with pytest.raises(AssertionError):
        BooleanNot(["interior", "interior"]).compute(graph, "test_nodes")


# ------------------------------------------------------------------------------------------------
# advisor findings, round 1
# ------------------------------------------------------------------------------------------------
def test_edge_bookkeeping_stays_off_the_tensor(tmp_path):
    """Provisional-row / tie-fixup / shard bookkeeping lives in a side table: a tagged edge_index pickles
    (``torch.save`` of a device-resident graph) and the entry dies with the tensor."""
    import gc
    import threading

    import torch

    from anemoi_graphs_b200 import device as D

    class FakeProvisional:  # holds what the real one holds: something that cannot be pickled
        done = False
        lock = threading.RLock()

    t = torch.arange(10, dtype=torch.int32).reshape(2, 5)
    prov = FakeProvisional()
    D.tag_rows(t, prov, None)
    D.edge_meta(t, create=True).fixup = prov
    D.edge_meta(t).local = (0, 5, [5])
    assert D.row_tags(t) == (prov, None)
    assert not [k for k in vars(t) if k.startswith("_agx")]
    torch.save({"edge_index": t}, tmp_path / "g.pt")  # TypeError: cannot pickle '_thread.RLock' before the fix
    back = torch.load(tmp_path / "g.pt", weights_only=False)["edge_index"]
    assert torch.equal(back, t) and D.edge_meta(back) is None
    key = id(t)
    del t, back
    gc.collect()
    assert key not in D._edge_meta


def test_boolean_masks_of_mixed_shapes_do_not_broadcast():
    import torch

    from anemoi_graphs_b200.graph import HeteroData
    from anemoi_graphs_b200.nodes.attributes import BooleanAndMask, BooleanNot, BooleanOrMask

    g = HeteroData()
    n = 7
    g["n"].x = torch.zeros((n, 2))
    g["n"]["a"] = torch.tensor([1, 1, 0, 0, 1, 0, 1], dtype=torch.bool)[:, None]  # a stored attribute: (N, 1)
    g["n"]["b"] = torch.tensor([1, 0, 1, 0, 1, 1, 0], dtype=torch.bool)[:, None]
    nested = BooleanNot("b")  # a mask object: raw values (N,)
    both = BooleanAndMask(["a", nested]).compute(g, "n")
    either = BooleanOrMask(["a", nested]).compute(g, "n")
    assert both.shape == (n, 1) and either.shape == (n, 1)
    a, nb = g["n"]["a"][:, 0], ~g["n"]["b"][:, 0]
    assert torch.equal(both[:, 0], a & nb) and torch.equal(either[:, 0], a | nb)
    g["n"]["ragged"] = torch.ones((n, 2), dtype=torch.bool)
    with pytest.raises(ValueError, match="one value per node"):
        BooleanAndMask(["a", "ragged"]).compute(g, "n")


def test_foreign_plugins_get_a_flushed_graph(monkeypatch):
    """A reference-style plugin (not one of the package's device-aware classes) is only called after ``flush()``."""
    from anemoi_graphs_b200 import device as D
    from anemoi_graphs_b200.edges.attributes import EdgeLength
    from anemoi_graphs_b200.edges.builder import KNNEdges

    class ForeignAttribute:
        def compute(self, graph, name):
            return None

    assert D.is_device_aware(EdgeLength()) and D.is_device_aware(KNNEdges("a", "b", 3))
    assert not D.is_device_aware(ForeignAttribute())
    calls = []
    monkeypatch.setattr(D, "flush", lambda: calls.append("flush"))
    D.flush_for(EdgeLength())
    assert calls == []
    D.flush_for(ForeignAttribute())
    assert calls == ["flush"]


def test_recipe_is_validated_up_front():
    from anemoi_graphs_b200.create import GraphCreator

    T = "anemoi.graphs."
    ok = {"nodes": {"h": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": 1}}},
          "edges": [{"source_name": "h", "target_name": "h", "edge_builders": [{"_target_": T + "edges.KNNEdges", "num_nearest_neighbours": 3}]}]}  # fmt: skip
    GraphCreator(ok)
    bad = {"nodes": {"h": {"node_builder": {"_target_": T + "nodes.ICONNodes", "name": "x", "grid_filename": "f", "max_level": 1}}}, "edges": []}
    with pytest.raises(ImportError):
        GraphCreator(bad)
    ok["edges"][0]["edge_builders"][0]["num_nearest_neighbours"] = 65
    with pytest.raises(NotImplementedError, match="65 > 64"):
        GraphCreator(ok)


def test_prelaunch_mode_rule(monkeypatch):
    """AGX_PRELAUNCH_TAIL: "auto" queues the post-sort work behind stream gates for device-resident graphs only (the
    measured rule, DESIGN.md section 3); "1" / "0" (or a bool set by a test) force it."""
    from anemoi_graphs_b200 import device as D

    prev = D.set_resident(False)
    try:
        for mode, resident, want in (("auto", False, False), ("auto", True, True), ("1", False, True), ("0", True, False),
                                     (True, False, True), (False, True, False)):  # fmt: skip
            monkeypatch.setattr(D, "PRELAUNCH_TAIL", mode)
            D.set_resident(resident)
            assert D._prelaunch_wanted() is want, (mode, resident)
    finally:
        D.set_resident(prev)


def test_known_rows_are_emitted_only_for_single_unmasked_knn_builders(monkeypatch):
    """GraphCreator._emit_known_rows (host-resident graphs): the a-priori target row is sent ahead only where a builder
    will adopt it - ONE unmasked KNNEdges on a node pair without edges yet, over a host node set the graph arrived with."""
    import torch

    from anemoi_graphs_b200 import device as D
    from anemoi_graphs_b200.create import GraphCreator
    from anemoi_graphs_b200.graph import HeteroData

    T = "anemoi.graphs."
    knn = {"_target_": T + "edges.KNNEdges", "num_nearest_neighbours": 3}
    masked = dict(knn, target_mask_attr_name="m")
    cut = {"_target_": T + "edges.CutOffEdges", "cutoff_factor": 0.6}

    def recipe(*edge_cfgs):
        return {"nodes": {"hidden": {"node_builder": {"_target_": T + "nodes.TriNodes", "resolution": 1}}},
                "edges": [{"source_name": s, "target_name": t, "edge_builders": list(b), "attributes": {}} for s, t, b in edge_cfgs]}  # fmt: skip

    emitted = []
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(D, "emit_regular_target_row", lambda n, k: emitted.append((n, k)))
    monkeypatch.setattr(GraphCreator, "EARLY_ROW_MIN_TARGETS", 4)
    graph = HeteroData()
    graph["data"].x = torch.zeros((10, 2))
    graph["tiny"].x = torch.zeros((2, 2))

    def rows(*edge_cfgs):
        emitted.clear()
        GraphCreator(recipe(*edge_cfgs))._emit_known_rows(graph)
        return list(emitted)

    assert rows(("hidden", "data", [knn])) == [(10, 3)]
    assert rows(("hidden", "data", [masked])) == []  # a mask changes which targets have edges
    assert rows(("hidden", "data", [knn, cut])) == []  # merged builders: sorted unique columns
    assert rows(("hidden", "data", [cut])) == []
    assert rows(("data", "hidden", [knn])) == []  # the target set is generated by this recipe: unknown size, device side
    assert rows(("hidden", "tiny", [knn])) == []  # not worth a separate copy
    prev = D.set_resident(True)
    try:
        assert rows(("hidden", "data", [knn])) == []  # device-resident graphs copy nothing
    finally:
        D.set_resident(prev)


def test_committed_bench_lines_keep_the_contract():
    """The bench lines kept under profiles/ carry every key the driver's contract names (bench.py prints them; a renamed
    key would silently turn a measured number into an unmeasured one)."""
    import json
    import pathlib

    import bench

    root = pathlib.Path(__file__).resolve().parents[1] / "profiles"
    base = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"}  # fmt: skip
    for name, with_cpu in (("r02_bench_n1_final.json", False), ("r02_bench_n1_slow_box.json", True)):
        line = json.loads((root / name).read_text())
        assert base <= set(line), base - set(line)
        assert line["metric"] == bench.METRIC and line["unit"] == "edges/s" and line["higher_is_better"] is True
        assert line["vs_baseline"] is None and line["data"] == "synthetic" and line["n_gpus"] == 1
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic", "fp32"} <= set(line["roofline"])
        assert abs(line["roofline"]["frac"] - line["roofline"]["achieved"] / line["roofline"]["peak"]) < 1e-3
        assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
        assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
        assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(line["clocks"]) and line["gpu_launches"] > 0
        assert line["config"] == bench.workload_config(
            "o1280_res7", 6599680, 163842,
            {bench.EDGE_KEYS[0]: 10394844, bench.EDGE_KEYS[1]: 1310700, bench.EDGE_KEYS[2]: 19799040},
        )
        # value and ms_per_step describe the same time
        edges = sum(line["config"]["edges"].values())
        assert abs(line["value"] - edges / (line["ms_per_step"] * 1e-3)) / line["value"] < 1e-3
        if with_cpu:
            assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"])
