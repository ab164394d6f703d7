"""``export_to_sparse`` without a GPU: the command line, and the errors ``edge_set_to_sparse`` / ``GraphExporter`` /
``agx_edges_to_csr`` raise before any kernel runs."""

import ctypes
import warnings

import pytest
import torch

from anemoi_graphs_b200 import _cabi
from anemoi_graphs_b200.graph import HeteroData

KEY = ("a", "to", "b")


def graph(attrs=None):
    g = HeteroData()
    g["a"].x = torch.zeros((5, 2))
    g["b"].x = torch.zeros((4, 2))
    g[KEY].edge_index = torch.tensor([[0, 1, 4], [3, 3, 0]], dtype=torch.int32)
    for name, value in (attrs or {}).items():
        g[KEY][name] = value
    return g


def test_command_line(monkeypatch, tmp_path):
    from anemoi_graphs_b200 import export
    from anemoi_graphs_b200.__main__ import main

    calls = []

    class Recorder:
        def __init__(self, *args):
            calls.append(args)

        def export(self):
            return []

    monkeypatch.setattr(export, "GraphExporter", Recorder)
    assert main(["export_to_sparse", "g.pt", str(tmp_path)]) == 0
    assert main(["export_to_sparse", "g.pt", "out", "--edges-name", "data", "hidden", "--edges-attribute-name", "w",
                 "--edges-name", "hidden", "data"]) == 0  # fmt: skip
    assert calls == [("g.pt", str(tmp_path), None, None), ("g.pt", "out", [["data", "hidden"], ["hidden", "data"]], "w")]
    with pytest.raises(SystemExit):
        main(["export_to_sparse", "g.pt", "out", "--edges-name", "data"])  # SOURCE TARGET: two names


def test_errors_before_any_kernel(tmp_path):
    from anemoi_graphs_b200.export import GraphExporter
    from anemoi_graphs_b200.export import edge_set_to_sparse

    g = graph({"w2": torch.ones((3, 2)), "w64": torch.ones(3, dtype=torch.float64), "w": torch.ones((3, 1))})
    with pytest.raises(ValueError, match=r"'w2'.*\(3, 2\)"):
        edge_set_to_sparse(g, KEY, "w2")
    with pytest.raises(ValueError, match=r"'w64'.*float32 or bool"):
        edge_set_to_sparse(g, KEY, "w64")
    with pytest.raises(KeyError, match="no attribute 'nothing'"):
        edge_set_to_sparse(g, KEY, "nothing")
    with pytest.raises(KeyError, match="no edge set"):
        edge_set_to_sparse(g, ("b", "to", "a"))
    with pytest.raises(ValueError, match="named"):
        edge_set_to_sparse(g, ("a", "b", "c", "d"))
    g[KEY]["edge_shard"] = {"rank": 1, "world": 2, "counts": [3, 3], "replicated": False}
    with pytest.raises(NotImplementedError, match="AGX_OUTPUT=gather"):
        edge_set_to_sparse(g, KEY, "w")
    assert "_agx_edge_index" not in g[KEY] and set(g[KEY].keys()) == {"edge_index", "w2", "w64", "w", "edge_shard"}

    with pytest.raises(KeyError, match="no edge set"):
        GraphExporter(graph(), tmp_path / "x", edges_name=[("a", "c")]).export()
    assert not (tmp_path / "x").exists()
    # every requested edge set lacks the attribute: a warning naming them, and no file
    with pytest.warns(UserWarning, match=r"without the attribute 'w'.*\('a', 'to', 'b'\)"):
        assert GraphExporter(graph(), tmp_path / "y", edge_attribute_name="w").export() == []
    assert list((tmp_path / "y").iterdir()) == []


def test_saved_graph_with_unknown_edge_set_raises(tmp_path):
    from anemoi_graphs_b200.__main__ import main

    torch.save(graph(), tmp_path / "g.pt")
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        with pytest.raises(KeyError, match="'b', 'to', 'a'"):
            main(["export_to_sparse", str(tmp_path / "g.pt"), str(tmp_path / "out"), "--edges-name", "b", "a"])


def test_abi_rejects_bad_arguments_before_device_work():
    lib = _cabi.load_library()
    nnz = ctypes.c_int64(-1)
    rc = lib.agx_edges_to_csr(None, None, 2**31, 10, None, None, 0, None, None, None, ctypes.byref(nnz), None)
    assert rc == _cabi.AGX_ERR_ARG and b"2^31" in lib.agx_last_error()
    rc = lib.agx_edges_to_csr(None, None, 10, 10, None, None, 3, None, None, None, ctypes.byref(nnz), None)
    assert rc == _cabi.AGX_ERR_ARG and b"value_kind" in lib.agx_last_error()
    rc = lib.agx_edges_to_csr(None, None, 10, 10, None, None, 1, None, None, None, ctypes.byref(nnz), None)
    assert rc == _cabi.AGX_ERR_ARG and b"NULL" in lib.agx_last_error()
    assert nnz.value == -1
