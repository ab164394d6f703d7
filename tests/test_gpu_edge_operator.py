"""Edge sets as operators: ``export.EdgeSetOperator``, ``export.apply_edge_set`` and ``ops.csr_spmm`` against a float64
scipy ``csr @ x`` on the same CSR.

The kernel sums each row in float32, left to right in ascending source order (``acc = fmaf(w, x, acc)`` from +0), so
every element lies within ``nnz_row * 2^-24 * sum |w| |x|`` of the float64 product, plus one bf16 ulp when the field is
bf16 (rounded once at the end).  ``torch.sparse.mm`` on the tensor ``edge_set_to_sparse`` returns must lie within the
same bound.  The order is fixed, so the bits repeat from call to call, between host- and device-resident graphs, and
between an aligned field and a copy of it at an offset that breaks 16-byte alignment.
"""

import numpy as np
import pytest
import torch

from anemoi_graphs_b200.export import EdgeSetOperator, apply_edge_set
from test_gpu_sparse_export import KEY, build, coords, host_graph, on_device, varied_float32, with_duplicates

F_SET = [1, 3, 4, 31, 32, 33, 64, 129]
DTYPES = {"float32": torch.float32, "bfloat16": torch.bfloat16}


def csr_arrays(op: EdgeSetOperator):
    """Host (indptr, indices, data) of the operator's CSR."""
    return tuple(t.cpu().numpy() for t in (op._indptr, op._indices, op._data))


def reference(csr, shape, x: torch.Tensor):
    """(float64 product, per-element bound) for the host CSR ``csr`` and the field ``x``."""
    from scipy.sparse import csr_matrix

    indptr, indices, data = csr
    m = csr_matrix((data.astype(np.float64), indices, indptr), shape=shape)
    x64 = x.detach().cpu().to(torch.float64).numpy()
    x2 = x64.reshape(x64.shape[0], -1)
    with np.errstate(invalid="ignore"):
        ref = m @ x2
        bound = (np.diff(indptr) * 2.0**-24)[:, None] * (abs(m) @ np.abs(x2))
    return ref.reshape((shape[0], *x64.shape[1:])), bound.reshape((shape[0], *x64.shape[1:]))


def bf16_ulp(v: np.ndarray) -> np.ndarray:
    return 2.0 ** (np.floor(np.log2(np.maximum(np.abs(v), 2.0**-126))) - 7)


def assert_within(y: torch.Tensor, ref: np.ndarray, bound: np.ndarray, bf16: bool) -> None:
    got = y.detach().cpu().to(torch.float64).numpy()
    assert got.shape == ref.shape
    tol = bound + (bf16_ulp(np.maximum(np.abs(ref), np.abs(np.nan_to_num(got)))) if bf16 else 0.0)
    finite = np.isfinite(ref)
    with np.errstate(invalid="ignore"):  # inf - inf where both are inf
        err = np.abs(got - ref)
    assert (err[finite] <= tol[finite]).all(), f"max excess {np.max(err[finite] - tol[finite])}"
    np.testing.assert_array_equal(got[~finite], ref[~finite])  # NaN where NaN, inf of the same sign


def field(rng, n: int, f: int | None, dtype: torch.dtype) -> torch.Tensor:
    """A (n, f) field, or (n,) for f = None, of signed values over four decades."""
    shape = (n,) if f is None else (n, f)
    v = rng.standard_normal(shape) * 10.0 ** rng.integers(-2, 2, shape)
    return torch.from_numpy(v.astype(np.float32)).to(dtype)


def bits(t: torch.Tensor) -> bytes:
    t = t.detach().cpu()
    return (t.view(torch.int16) if t.dtype == torch.bfloat16 else t).numpy().tobytes()


# ------------------------------------------------------------------------------------------------
# graphs built by GraphCreator, device-resident and host-resident
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def graphs():
    return {"device": build(True), "host": build(False)}


@pytest.mark.gpu
def test_knn_gaussian_weights_operator(graphs):
    from anemoi_graphs_b200.export import edge_set_to_sparse

    key = ("data", "to", "hidden")
    rng = np.random.default_rng(0)
    x = field(rng, 40320, 16, torch.float32).cuda()
    results = {}
    for where, g in graphs.items():
        op = EdgeSetOperator(g, key, "w")
        assert op.shape == (10242, 40320)
        csr = csr_arrays(op)
        assert (np.diff(csr[0]) == 4).all()
        y = op(x)
        assert y.is_cuda and y.dtype == torch.float32 and y.shape == (10242, 16)
        assert_within(y, *reference(csr, op.shape, x), bf16=False)
        assert bits(op(x)) == bits(y)  # two calls, bit-identical
        y_host = op(x.cpu())  # a host field gives a host result
        assert not y_host.is_cuda and bits(y_host) == bits(y)
        assert bits(apply_edge_set(g, key, x, "w")) == bits(y)
        const = torch.full((40320, 3), 2.5, device="cuda")
        c = op(const)
        _, bound = reference(csr, op.shape, const)
        assert (np.abs(c.cpu().numpy().astype(np.float64) - 2.5) <= bound + 2.5 * 4 * 2.0**-24).all()  # rows sum to 1
        results[where] = y
    assert bits(results["device"]) == bits(results["host"])
    m = edge_set_to_sparse(graphs["device"], key, "w")
    ref, bound = reference(csr_arrays(EdgeSetOperator(graphs["device"], key, "w")), (10242, 40320), x)
    assert_within(torch.sparse.mm(m, x), ref, bound, bf16=False)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_cutoff_operator_of_ones(graphs, dtype):
    from anemoi_graphs_b200.export import edge_set_to_sparse

    key = ("hidden", "to", "data")
    rng = np.random.default_rng(1)
    x = field(rng, 10242, 8, DTYPES[dtype]).cuda()
    results = []
    for g in graphs.values():
        op = EdgeSetOperator(g, key)
        assert op.shape == (40320, 10242)
        csr = csr_arrays(op)
        assert (csr[2] == 1.0).all() and (np.diff(csr[0]) == 0).any()  # ones, and data nodes out of every hidden node's reach
        y = op(x)
        assert y.dtype == DTYPES[dtype]
        assert_within(y, *reference(csr, op.shape, x), bf16=dtype == "bfloat16")
        results.append(bits(y))
    assert results[0] == results[1]
    if dtype == "float32":
        m = edge_set_to_sparse(graphs["device"], key)
        assert_within(torch.sparse.mm(m, x), *reference(csr, (40320, 10242), x), bf16=False)


# ------------------------------------------------------------------------------------------------
# hand-made edge lists
# ------------------------------------------------------------------------------------------------
N_SRC, N_DST = 12_000, 200


def hand_made_graph(seed: int = 7):
    """N_SRC source and N_DST target nodes: duplicate pairs, a quarter of the target rows empty, and target 0 with
    11 000 distinct sources; float32 weights over eight decades."""
    rng = np.random.default_rng(seed)
    ei = with_duplicates(rng, N_SRC, N_DST, 6000, 1000, 5, rng.choice(np.arange(1, N_DST), 150, replace=False))
    long_row = np.stack([rng.choice(N_SRC, 11_000, replace=False), np.zeros(11_000, dtype=np.int64)]).astype(np.int32)
    ei = np.concatenate([ei, long_row], axis=1)
    ei = np.ascontiguousarray(ei[:, rng.permutation(ei.shape[1])])
    w = varied_float32(rng, ei.shape[1])
    return host_graph(coords(N_SRC, 1), coords(N_DST, 2), ei, {"w": w.reshape(-1, 1), "m": (w > 0).reshape(-1, 1)})


@pytest.fixture(scope="module")
def hand_made():
    g = hand_made_graph()
    return {"host": g, "device": on_device(g)}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("f", F_SET + [None])
def test_feature_widths(hand_made, f, dtype):
    rng = np.random.default_rng(100 + (f or 0))
    ops_ = {where: EdgeSetOperator(g, KEY, "w") for where, g in hand_made.items()}
    csr = csr_arrays(ops_["device"])
    lengths = np.diff(csr[0])
    assert lengths[0] > 10_000 and (lengths == 0).sum() >= 40 and csr[1].size < hand_made["host"][KEY].edge_index.shape[1]
    x = field(rng, N_SRC, f, DTYPES[dtype]).cuda()
    y = ops_["device"](x)
    assert y.shape == ((N_DST,) if f is None else (N_DST, f)) and y.dtype == x.dtype
    ref, bound = reference(csr, (N_DST, N_SRC), x)
    assert_within(y, ref, bound, bf16=dtype == "bfloat16")
    empty = lengths == 0
    assert (y.cpu().float().numpy()[empty] == 0).all() and not np.signbit(y.cpu().float().numpy()[empty]).any()
    assert bits(ops_["device"](x)) == bits(y)  # two calls
    assert bits(ops_["host"](x)) == bits(y)  # host-resident graph
    if dtype == "float32":
        from anemoi_graphs_b200.export import edge_set_to_sparse

        m = edge_set_to_sparse(hand_made["device"], KEY, "w")
        x2 = x.reshape(N_SRC, -1)
        assert_within(torch.sparse.mm(m, x2), ref.reshape(N_DST, -1), bound.reshape(N_DST, -1), bf16=False)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("f", [4, 8, 64, 129])
def test_field_at_an_unaligned_offset(hand_made, f, dtype):
    """A contiguous field whose first element sits one element past a 16-byte boundary: same bits as an aligned copy."""
    rng = np.random.default_rng(200 + f)
    op = EdgeSetOperator(hand_made["device"], KEY, "w")
    base = field(rng, N_SRC * f + 1, None, DTYPES[dtype]).cuda()
    x = base[1:].view(N_SRC, f)
    assert x.is_contiguous() and x.data_ptr() % 16 != 0
    aligned = x.clone()
    assert aligned.data_ptr() % 16 == 0
    y = op(x)
    assert bits(y) == bits(op(aligned))
    assert_within(y, *reference(csr_arrays(op), op.shape, x), bf16=dtype == "bfloat16")
    xt = field(rng, f, N_SRC, DTYPES[dtype]).cuda().t()  # not contiguous
    assert bits(op(xt)) == bits(op(xt.contiguous()))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_nan_and_inf_reach_only_their_rows(hand_made, dtype):
    rng = np.random.default_rng(9)
    op = EdgeSetOperator(hand_made["device"], KEY, "w")
    csr = csr_arrays(op)
    s = np.unique(csr[1][csr[0][1] :])[[5, 50, 51, 500]]  # sources that rows other than the long row 0 reference
    x = field(rng, N_SRC, 5, DTYPES[dtype])
    x[s[0], 0] = float("nan")
    x[s[1], 1] = float("inf")
    x[s[2], 2] = float("-inf")
    x[s[3], 3] = float("inf")
    x[s[3], 4] = float("nan")
    y = op(x.cuda()).cpu()
    ref, bound = reference(csr, op.shape, x)
    assert_within(y, ref, bound, bf16=dtype == "bfloat16")
    rows = np.repeat(np.arange(N_DST), np.diff(csr[0]))
    for col, src in ((0, s[0]), (1, s[1]), (2, s[2]), (3, s[3]), (4, s[3])):
        hit = np.zeros(N_DST, dtype=bool)
        hit[rows[csr[1] == src]] = True
        assert hit.any() and (~np.isfinite(y[:, col].float().numpy()) == hit).all()


@pytest.mark.gpu
def test_edge_set_without_entries_and_empty_fields():
    from anemoi_graphs_b200 import _cabi

    g = on_device(host_graph(coords(30, 1), coords(20, 2), np.zeros((2, 0), dtype=np.int32), {"w": np.zeros(0, np.float32)}))
    op = EdgeSetOperator(g, KEY, "w")
    y = op(torch.randn(30, 6, device="cuda"))
    assert y.shape == (20, 6) and (y == 0).all() and not torch.signbit(y).any()
    g = on_device(hand_made_graph())
    op = EdgeSetOperator(g, KEY, "w")
    for x in (torch.empty(N_SRC, 0, device="cuda"), torch.empty(N_SRC, 0, dtype=torch.bfloat16)):
        before = _cabi.launch_count()
        y = op(x)
        assert _cabi.launch_count() == before  # F = 0: no launch
        assert y.shape == (N_DST, 0) and y.dtype == x.dtype and y.device == x.device


# ------------------------------------------------------------------------------------------------
# errors
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_operator_errors():
    g = on_device(hand_made_graph())
    op = EdgeSetOperator(g, KEY, "w")
    with pytest.raises(ValueError, match=rf"{N_SRC - 1} rows.*{N_SRC} nodes"):
        op(torch.zeros(N_SRC - 1, 4, device="cuda"))
    for dtype in (torch.float64, torch.float16, torch.int32):
        with pytest.raises(ValueError, match="float32 or bfloat16"):
            op(torch.zeros(N_SRC, 4, dtype=dtype, device="cuda"))
    with pytest.raises(ValueError, match=rf"\({N_SRC}, 2, 2\)"):
        op(torch.zeros(N_SRC, 2, 2, device="cuda"))
    with pytest.raises(ValueError, match=rf"{N_SRC + 1} rows.*{N_SRC} nodes"):
        apply_edge_set(g, KEY, torch.zeros(N_SRC + 1), "w")
    with pytest.raises(ValueError, match="'m'.*bool"):
        EdgeSetOperator(g, KEY, "m")
    g[KEY]["w2"] = torch.ones(g[KEY].edge_index.shape[1], 2, device="cuda")
    with pytest.raises(ValueError, match=r"'w2'.*, 2\)"):
        EdgeSetOperator(g, KEY, "w2")
    g[KEY]["w64"] = torch.ones(g[KEY].edge_index.shape[1], dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError, match="'w64'.*float32 or bool"):
        EdgeSetOperator(g, KEY, "w64")
    with pytest.raises(KeyError, match="nowhere"):
        EdgeSetOperator(g, ("src", "nowhere"))
    with pytest.raises(KeyError, match="'missing'"):
        EdgeSetOperator(g, KEY, "missing")
    g[KEY]["edge_shard"] = {"rank": 0, "world": 2, "counts": [1, 1], "replicated": False}
    for attr in (None, "w"):
        with pytest.raises(NotImplementedError, match="gather"):
            EdgeSetOperator(g, KEY, attr)


@pytest.mark.gpu
def test_kernel_argument_rejection():
    from anemoi_graphs_b200 import _cabi, ops

    lib, stream = _cabi.load_library(), _cabi.current_stream()
    indptr = torch.tensor([0, 2, 2, 3], dtype=torch.int64, device="cuda")
    indices = torch.tensor([0, 4, 1], dtype=torch.int32, device="cuda")
    data = torch.tensor([0.5, 0.25, 2.0], device="cuda")
    x = torch.arange(10, dtype=torch.float32, device="cuda").reshape(5, 2)
    out = torch.full((3, 2), -1.0, device="cuda")
    p = {k: _cabi.ptr(v) for k, v in {"indptr": indptr, "indices": indices, "data": data, "x": x, "out": out}.items()}
    ok = (p["indptr"], p["indices"], p["data"], 3, 5, p["x"], 2, 0, p["out"], stream)

    def call(**change):
        args = list(ok)
        for name, value in change.items():
            args[["indptr", "indices", "data", "n_rows", "n_cols", "x", "n_features", "dtype", "out"].index(name)] = value
        return lib.agx_csr_spmm(*args)

    for name in ("indptr", "indices", "data", "x", "out"):
        assert call(**{name: None}) == _cabi.AGX_ERR_ARG
    for name in ("n_rows", "n_cols", "n_features"):
        assert call(**{name: -1}) == _cabi.AGX_ERR_ARG
    assert call(n_cols=2**31) == _cabi.AGX_ERR_ARG
    for dtype in (-1, 2, 7):
        assert call(dtype=dtype) == _cabi.AGX_ERR_ARG
    assert call(x=p["x"] + 2) == _cabi.AGX_ERR_ARG  # not aligned to its float32 elements
    assert (out == -1.0).all()  # nothing written
    assert call(n_cols=4) == _cabi.AGX_ERR_ARG and "outside [0, n_cols = 4)" in lib.agx_last_error().decode()
    assert call() == _cabi.AGX_OK
    torch.testing.assert_close(out, torch.tensor([[0.5 * 0 + 0.25 * 8, 0.5 * 1 + 0.25 * 9], [0, 0], [4.0, 6.0]], device="cuda"))
    assert call(n_rows=0) == _cabi.AGX_OK and call(n_features=0) == _cabi.AGX_OK
    bad = torch.tensor([0, -1, 1], dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="outside"):
        ops.csr_spmm(indptr, bad, data, x, 3)
    np.testing.assert_array_equal(ops.csr_spmm(indptr, indices, data, x, 3).cpu().numpy(), out.cpu().numpy())
