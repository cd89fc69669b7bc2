"""Cosine and cityblock graphs against the CPU oracle beyond the golden cases: float64 rows, feature counts around
the warp width and the kernel flavours' operand limits, offsets that stress the rounding of the float32 search copy,
all-zero rows, the reference's metric-less fallback search (quirk H9), exact graphs at tile-edge shapes, and the
"data" edge lengths of G.shortest_path at widths around numpy's summation blocks."""
import math
import warnings

import numpy as np
import pytest
from scipy import sparse

import graphtools_b200 as gt
from graphtools_b200 import dense, pipeline, synth
from oracle import graph_oracle as go
from tests.parity import compare_dense, compare_sparse
from tests.test_shortest_path_gpu import assert_bitwise, oracle as sp_oracle

pytestmark = pytest.mark.gpu

N = 3000
NQ = 200


@pytest.fixture(params=["auto", "tc", "tc16", "tch", "tch1", "simt"])
def impl(request, monkeypatch):
    monkeypatch.setenv("GTB_SEARCH_IMPL", request.param)
    return request.param


def expected_impl(want, d):
    """knn_kernel's fallback order at N = 3000 (too few reference tiles for the seeded one-product flavour under
    auto): the first flavour whose resident query tile holds d features."""
    fits = {"tch1": d <= 126, "tch": d <= 510, "tc16": d <= 127, "tc": d <= 103}
    order = {"auto": ("tch", "tc16", "tc"), "tch1": ("tch1", "tch", "tc16", "tc"), "tch": ("tch", "tc16", "tc"),
             "tc16": ("tc16", "tc"), "tc": ("tc", "tc16"), "simt": ()}[want]
    return next((c for c in order if fits[c]), "simt")


def _graph(X, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return gt.Graph(X, verbose=0, **kw)


def _f64(X, seed):
    """float64 rows that float32 cannot hold: the search copy is then a rounded copy of the rows."""
    rng = np.random.default_rng(seed)
    return X.astype(np.float64) * (1 + 1e-9 * rng.normal(size=X.shape))


def _compare_graph(K, P, K_ref, P_ref, thresh, tie, what):
    """K against the oracle; P on every row when nothing was exempted, else on the rows whose K row agrees."""
    r = compare_sparse(K, K_ref, thresh=thresh, what=what + ".K", tie=tie)
    if r["n_exempt"] == 0:
        compare_sparse(P, P_ref, what=what + ".P")
        return r
    K, K_ref, P, P_ref = (sparse.csr_matrix(m) for m in (K, K_ref, P, P_ref))
    same = [i for i in range(K.shape[0])
            if np.array_equal(K[i].indices, K_ref[i].indices) and np.allclose(K[i].data, K_ref[i].data, rtol=1e-5)]
    assert len(same) > 0.9 * K.shape[0], what
    compare_sparse(P[same], P_ref[same], what=what + ".P (agreeing rows)")
    return r


def _assert_no_fallback(g):
    """The oracle's search never went to its metric-less brute-force index with rows left to do."""
    for sc in g.schedules:
        assert not (sc["fallback"] and sc["todo"].size), "case drifted into the metric-less fallback regime"


# --------------------------------------------------------------------------- A1: kNN sweep
# isotropic data: a decay per width that puts rows beyond every candidate list (radius pass) while the reference's
# search stays below N / 2.  2-D cosine stays at decay 1: below 1, (d / bw)^decay turns the rounding noise of the
# reference's own self-distances (~1e-16, bw ~1e-5) into value errors above rtol, and at decay >= 1 its rows are too
# short for the radius pass.
ISO_DECAY = {("cosine", 2): 1, ("cosine", 3): 1, ("cosine", 31): 10, ("cosine", 33): 10, ("cosine", 100): 20,
             ("cosine", 129): 40, ("cosine", 300): 40, ("cosine", 510): 40, ("cityblock", 1): 2,
             ("cityblock", 3): 5, ("cityblock", 31): 20, ("cityblock", 33): 20, ("cityblock", 129): 40,
             ("cityblock", 300): 40}
_SWEEP = {}


def sweep_case(metric, dtype, d, kind):
    """(X, Y, params, K_ref, P_ref, Kyx_ref) of one sweep case, built once per module."""
    key = (metric, dtype, d, kind)
    if key not in _SWEEP:
        if kind == "iso" and metric == "cosine" and d == 2:
            # directions on a jittered grid: random angles put pairs ~1e-6 rad apart, whose cosine distance (~1e-13)
            # carries a relative rounding error of ~1e-3 in the reference itself, which a decay below 1 passes on
            rng = np.random.default_rng(d)
            theta = 2 * np.pi * (rng.permutation(N) + 0.6 * rng.random(N)) / N
            X = ((0.5 + np.abs(rng.normal(size=N)))[:, None] * np.stack([np.cos(theta), np.sin(theta)], 1))
            X = X.astype(np.float32)
            params = dict(knn=5, decay=ISO_DECAY[(metric, d)], thresh=1e-4)
        elif kind == "iso":
            X = np.random.default_rng(d).normal(size=(N, d)).astype(np.float32)
            params = dict(knn=5, decay=ISO_DECAY[(metric, d)], thresh=1e-4)
        else:
            X, _ = synth.gaussian_mixture(N, d, n_clusters=6, intrinsic_dim=4, seed=d)
            params = dict(knn=5, decay=40, thresh=1e-4)
        X = _f64(X, d) if dtype == "float64" else X
        X64 = X.astype(np.float64)
        Y = X[:NQ] + np.asarray(0.02 * np.random.default_rng(d + 1).normal(size=(NQ, d)), dtype=X.dtype)
        K_ref, P_ref, g = go.knn_graph(X64, distance=metric, return_oracle=True, **params)
        Kyx_ref = g.kernel_to_data(Y.astype(np.float64))
        _assert_no_fallback(g)
        _SWEEP[key] = (X, Y, params, K_ref, P_ref, Kyx_ref)
    return _SWEEP[key]


def _run_sweep(metric, dtype, d, kind, want):
    X, Y, params, K_ref, P_ref, Kyx_ref = sweep_case(metric, dtype, d, kind)
    G = _graph(X, distance=metric, **params)
    K, P = G.kernel, G.diff_op
    st = pipeline.stats()
    assert st["impl"] == ("simt" if metric == "cityblock" else expected_impl(want, d)), st
    if kind == "iso" and not (metric == "cosine" and d == 2):
        assert st["radius_rows"] > 0, st
    what = "%s %s d=%d %s %s" % (metric, dtype, d, kind, want)
    _compare_graph(K, P, K_ref, P_ref, params["thresh"], dict(X=X, knn=6, metric=metric), what)
    compare_sparse(G.build_kernel_to_data(Y), Kyx_ref, thresh=params["thresh"], what=what + ".Kyx",
                   tie=dict(X=X, Y=Y, knn=5, metric=metric))


@pytest.mark.parametrize("kind", ["clustered", "iso"])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("d", [2, 3, 31, 33, 100, 129, 300, 510])
def test_cosine_knn_sweep(d, dtype, kind, impl):
    _run_sweep("cosine", dtype, d, kind, impl)


@pytest.mark.parametrize("kind", ["clustered", "iso"])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("d", [1, 3, 31, 33, 129, 300])
def test_cityblock_knn_sweep(d, dtype, kind):
    _run_sweep("cityblock", dtype, d, kind, "auto")


# --------------------------------------------------------------------------- A2: offsets
@pytest.mark.parametrize("dtype,offset", [("float64", 1e4), ("float32", 1e3)])
def test_cityblock_offset(dtype, offset):
    """Cityblock rows far from the origin: the float32 search copy is not centred, so its rounding (an ulp of ~1e-3
    at 1e4) is large against the spread of ~1; the certification must account for it."""
    X, _ = synth.gaussian_mixture(N, 31, n_clusters=6, intrinsic_dim=4, seed=7)
    X = (X.astype(np.float64) + offset) if dtype == "float64" else (X + np.float32(offset))
    if dtype == "float64":
        X = _f64(X, 7)
    Y = X[:NQ] + 0.01
    K_ref, P_ref, g = go.knn_graph(X.astype(np.float64), knn=5, decay=40, thresh=1e-4, distance="cityblock",
                                   return_oracle=True)
    _assert_no_fallback(g)
    G = _graph(X, knn=5, decay=40, thresh=1e-4, distance="cityblock")
    _compare_graph(G.kernel, G.diff_op, K_ref, P_ref, 1e-4, dict(X=X, knn=6, metric="cityblock"), "cityblock offset")
    compare_sparse(G.build_kernel_to_data(Y), g.kernel_to_data(Y.astype(np.float64)), thresh=1e-4,
                   what="cityblock offset Kyx", tie=dict(X=X, Y=Y, knn=5, metric="cityblock"))


def test_cosine_offset(impl):
    """Cosine distances of ~1e-3 (an offset of 10 in every coordinate makes the rows nearly parallel): the search copy
    is normalised and centred in float64 before its rounding.  The reference stays well conditioned there: with
    decay 40, decay (d / bw)^decay <= 40 (-ln thresh) ~ 370 times its relative distance error (~1e-16 / 1e-3) is
    ~4e-11, far below rtol, so the test measures the kernels and not sklearn's formula against ours."""
    X, _ = synth.gaussian_mixture(N, 31, n_clusters=6, intrinsic_dim=4, seed=9)
    X = _f64(X, 9) + 10.0
    D = np.sort(1 - (X[:200] / np.linalg.norm(X[:200], axis=1, keepdims=True)) @
                (X / np.linalg.norm(X, axis=1, keepdims=True)).T, axis=1)
    assert 1e-4 < np.median(D[:, 6]) < 1e-2, np.median(D[:, 6])
    Y = X[:NQ] + 0.01 * np.random.default_rng(10).normal(size=(NQ, 31))
    K_ref, P_ref, g = go.knn_graph(X, knn=5, decay=40, thresh=1e-4, distance="cosine", return_oracle=True)
    _assert_no_fallback(g)
    G = _graph(X, knn=5, decay=40, thresh=1e-4, distance="cosine")
    _compare_graph(G.kernel, G.diff_op, K_ref, P_ref, 1e-4, dict(X=X, knn=6, metric="cosine"), "cosine offset")
    compare_sparse(G.build_kernel_to_data(Y), g.kernel_to_data(Y), thresh=1e-4, what="cosine offset Kyx",
                   tie=dict(X=X, Y=Y, knn=5, metric="cosine"))


# --------------------------------------------------------------------------- A3: all-zero rows (cosine)
def _zero_row_data(dtype):
    X, _ = synth.gaussian_mixture(600, 20, n_clusters=4, intrinsic_dim=5, seed=17)
    X = _f64(X, 17) if dtype == "float64" else X
    X[17] = 0
    X[400] = 0
    return X


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_cosine_zero_rows_knn(dtype, impl):
    """An all-zero row is at cosine distance 1 from every row (sklearn's normalize leaves it at zero): its kernel row
    covers every point, and no NaN reaches the other rows."""
    X = _zero_row_data(dtype)
    K_ref, P_ref, g = go.knn_graph(X.astype(np.float64), knn=5, decay=40, thresh=1e-4, distance="cosine",
                                   return_oracle=True)
    _assert_no_fallback(g)
    G = _graph(X, knn=5, decay=40, thresh=1e-4, distance="cosine")
    K, P = G.kernel, G.diff_op
    assert np.isfinite(K.data).all() and np.isfinite(P.data).all()
    assert K[17].nnz == 600 and math.isclose(K[17, 17], math.exp(-1), rel_tol=1e-12)
    compare_sparse(K, K_ref, thresh=1e-4, what="zero rows K")
    compare_sparse(P, P_ref, thresh=1e-4, what="zero rows P")
    Y = X[:50] + np.asarray(0.01, dtype=X.dtype)
    Y[[0, 9]] = 0
    Kyx = G.build_kernel_to_data(Y)
    assert np.isfinite(Kyx.data).all() and Kyx[9].nnz == 600
    compare_sparse(Kyx, g.kernel_to_data(Y.astype(np.float64)), thresh=1e-4, what="zero query rows Kyx")


@pytest.mark.parametrize("thresh", [1e-4, 0])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_cosine_zero_rows_exact(dtype, thresh):
    """Exact graphs: scipy's cosine distance from a zero row is NaN and the reference maps its kernel value to 1, so
    the zero rows and columns of K are all ones; np.partition sorts NaN last, so the other rows' bandwidths ignore
    them."""
    X = _zero_row_data(dtype)[:300]
    X64 = X.astype(np.float64)
    G = _graph(X, graphtype="exact", knn=5, decay=40, thresh=thresh, distance="cosine")
    K_ref = go.finish_kernel(go.exact_kernel(X64, knn=5, decay=40, distance="cosine", thresh=thresh))
    K = G.kernel
    K = K.toarray() if sparse.issparse(K) else np.asarray(K)
    assert np.isfinite(K).all() and (K[17] == 1).all() and (K[:, 17] == 1).all()
    compare_dense(K, K_ref, thresh=thresh, what="exact zero rows K")
    P = G.diff_op
    compare_dense(P.toarray() if sparse.issparse(P) else P, np.asarray(go.diff_op(K_ref)), thresh=thresh,
                  what="exact zero rows P")
    Y = X[:30] + np.asarray(0.01, dtype=X.dtype)
    Y[[0, 5]] = 0
    Kyx = np.asarray(G.build_kernel_to_data(Y))
    Kyx_ref = go.exact_kernel_to_data(X64, Y.astype(np.float64), knn=5, decay=40, distance="cosine", thresh=thresh)
    assert np.isfinite(Kyx).all() and (Kyx[5] == 1).all()
    compare_dense(Kyx, Kyx_ref, thresh=thresh, what="exact zero query rows Kyx")


# --------------------------------------------------------------------------- A4: metric-less fallback search (H9)
def _mixture64(n, d, seed):
    X, _ = synth.gaussian_mixture(n, d, n_clusters=2, intrinsic_dim=None, seed=seed)
    return X.astype(np.float64)


def _assert_fallback(g, branch):
    sc = g.schedules[-1]
    assert sc["fallback"] and sc["todo"].size > 0 and sc["branch"] == branch, sc


@pytest.mark.parametrize("metric,n,d,seed,decay,branch", [
    ("cityblock", 400, 10, 3, 10, "radius"),
    ("cosine", 400, 50, 5, 10, "radius"),
    ("cosine", 200, 10, 5, 5, "kneighbors"),
    ("cosine", 400, 50, 5, 5, "radius"),          # Euclidean distances beyond the cosine radius: K = I
    ("cosine", 1000, 50, 0, 5, "kneighbors"),     # the escalation loop runs (216 wide) and ends above N / 2
])
def test_fallback_in_sample(metric, n, d, seed, decay, branch):
    """When the reference's search grows beyond N / 2 neighbours, the remaining rows are searched with Euclidean
    distances (graphs.py:945-948): their kernel rows hold Euclidean distances over the metric's bandwidth."""
    X = _mixture64(n, d, seed)
    K_ref, P_ref, g = go.knn_graph(X, knn=5, decay=decay, thresh=1e-3, distance=metric, return_oracle=True)
    _assert_fallback(g, branch)
    G = _graph(X, knn=5, decay=decay, thresh=1e-3, distance=metric)
    K, P = G.kernel, G.diff_op
    compare_sparse(K, K_ref, what="fallback K")
    compare_sparse(P, P_ref, what="fallback P")


def test_fallback_out_of_sample():
    X = _mixture64(300, 10, 3)
    Y = X[:120] + np.random.default_rng(4).normal(scale=0.05, size=(120, 10))
    g = go.KnnOracle(X, knn=5, decay=10, thresh=1e-3, distance="cityblock")
    Kyx_ref = g.kernel_to_data(Y)
    _assert_fallback(g, "radius")
    G = _graph(X, knn=5, decay=10, thresh=1e-3, distance="cityblock")
    compare_sparse(G.build_kernel_to_data(Y), Kyx_ref, what="fallback Kyx")


def test_fallback_mnn_small_batches():
    """Each MNN batch runs its own search with the batch's N, so small batches reach the fallback too."""
    X = _mixture64(600, 10, 3)
    idx = np.repeat([0, 1, 2], 200)
    g = go.KnnOracle(X[idx == 0], knn=5, decay=10, thresh=1e-3, distance="cityblock")
    g.kernel()
    g.kernel_to_data(X[idx == 1], knn=5)
    assert any(sc["fallback"] and sc["todo"].size for sc in g.schedules)
    K_ref = go.finish_kernel(go.mnn_kernel(X, idx, knn=5, decay=10, thresh=1e-3, distance="cityblock"), "mnn", 0.5)
    G = _graph(X, sample_idx=idx, knn=5, decay=10, thresh=1e-3, distance="cityblock", kernel_symm="mnn", theta=0.5)
    compare_sparse(G.kernel, K_ref, what="fallback MNN K")
    compare_sparse(G.diff_op, go.diff_op(K_ref), what="fallback MNN P")


# --------------------------------------------------------------------------- A5: exact graphs and dense_distances
EXACT_METRICS = ["euclidean", "cosine", "cityblock"]


@pytest.mark.parametrize("d", [1, 15, 16, 17, 129])
@pytest.mark.parametrize("n", [5, 63, 64, 65, 130, 700])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("metric", EXACT_METRICS)
def test_exact_graph_shapes(metric, dtype, n, d):
    """Tile edges (DT = 64 outputs), feature chunks (DK = 16) and both precisions of the dense kernel, in-sample
    with each symmetrisation and out of sample with 40 and 150 query rows.  (Cosine on one feature is only the sign
    of the value: left out.)"""
    if metric == "cosine" and d == 1:
        pytest.skip("cosine distance of one feature is degenerate (0 or 2)")
    rng = np.random.default_rng(n * 1000 + d)
    X = rng.normal(size=(n, d)).astype(np.float32) + 0.5
    X = _f64(X, n + d) if dtype == "float64" else X
    X64 = X.astype(np.float64)
    knn = min(5, n - 2)
    for k, thresh in enumerate((1e-4, 0.0)):
        symm, theta = [("+", None), ("*", None), ("mnn", 0.3)][(n + d + k) % 3]
        G = _graph(X, graphtype="exact", knn=5, decay=20, thresh=thresh, distance=metric, kernel_symm=symm,
                   theta=theta)
        K_ref = go.finish_kernel(go.exact_kernel(X64, knn=knn, decay=20, distance=metric, thresh=thresh), symm, theta)
        K = G.kernel
        K = K.toarray() if sparse.issparse(K) else np.asarray(K)
        what = "exact %s %s n=%d d=%d thresh=%g %s" % (metric, dtype, n, d, thresh, symm)
        compare_dense(K, K_ref, thresh=thresh, what=what + " K")
        P = G.diff_op
        compare_dense(P.toarray() if sparse.issparse(P) else P, np.asarray(go.diff_op(K_ref)), thresh=thresh,
                      what=what + " P")
        for nq in (40, 150):
            Y = (X[rng.integers(0, n, nq)] + np.asarray(0.1 * rng.normal(size=(nq, d)), dtype=X.dtype))
            Kyx_ref = go.exact_kernel_to_data(X64, Y.astype(np.float64), knn=knn, decay=20, distance=metric,
                                              thresh=thresh)
            compare_dense(np.asarray(G.build_kernel_to_data(Y)), Kyx_ref, thresh=thresh, what=what + " Kyx%d" % nq)


def _gamma(k):
    u = 2.0 ** -53
    return k * u / (1 - k * u)


@pytest.mark.parametrize("d", [1, 15, 16, 17, 129, 1000])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("metric", EXACT_METRICS)
def test_dense_distances_error_bound(metric, dtype, d):
    """dense_distances against a long-double evaluation of the same inputs, u = 2^-53 (the long-double reference's
    own error, ~2^-64 relative, is negligible).

    Euclidean: each difference q_k - r_k is rounded once (exact for float32 inputs), each square and the d-term
    sum accumulate by fma: the squared distance carries a relative error of at most gamma(d + 2) (all terms are
    non-negative, no cancellation); the square root halves it and adds one rounding, so gamma(d + 2) bounds the
    relative error of the distance.  Cityblock: one rounding per difference, fabs is exact, d - 1 additions of
    non-negative terms: gamma(d + 2) relative again.  Cosine: the dot product's error is at most gamma(d) |q| |r|,
    each squared norm's gamma(d) relative, the square roots, product and quotient add 3 roundings, so the cosine c
    is off by at most gamma(2 d + 4) absolutely; 1 - c adds 2u absolutely.  1 - c cancels, so the bound is absolute,
    gamma(2 d + 8)."""
    rng = np.random.default_rng(d + (dtype == "float64"))
    Xq = rng.normal(size=(70, d)).astype(np.float32) + 0.25
    Xr = rng.normal(size=(130, d)).astype(np.float32) - 0.1
    if dtype == "float64":
        Xq, Xr = _f64(Xq, 1), _f64(Xr, 2)
    import torch
    dev = pipeline._dev()
    D = dense.dense_distances(torch.from_numpy(Xq).to(dev), torch.from_numpy(Xr).to(dev), metric).cpu().numpy()
    q, r = Xq.astype(np.longdouble), Xr.astype(np.longdouble)
    if metric == "euclidean":
        R = np.sqrt(((q[:, None, :] - r[None, :, :]) ** 2).sum(-1))
    elif metric == "cityblock":
        R = np.abs(q[:, None, :] - r[None, :, :]).sum(-1)
    else:
        R = 1 - (q @ r.T) / (np.sqrt((q * q).sum(1))[:, None] * np.sqrt((r * r).sum(1))[None, :])
    err = np.abs(D.astype(np.longdouble) - R)
    if metric == "cosine":
        assert float(err.max()) <= _gamma(2 * d + 8), (float(err.max()), _gamma(2 * d + 8))
    else:
        rel = err / R
        assert float(rel.max()) <= _gamma(d + 2), (float(rel.max()), _gamma(d + 2))


# --------------------------------------------------------------------------- A6: shortest-path "data" lengths
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("d", [1, 3, 7, 8, 9, 127, 128, 129, 136, 257, 1000])
def test_shortest_path_data_lengths_widths(d, dtype):
    """numpy's pairwise summation of the squared differences, in the dtype of data_nu, at widths below, at and beyond
    its blocks of 8 and 128 (the d > 128 recursion of sqdist_pairwise), bit for bit."""
    rng = np.random.default_rng(d)
    X = rng.normal(size=(300, d)).astype(np.float32)
    X = _f64(X, d) if dtype == "float64" else X
    G = _graph(X, knn=5, decay=None)
    assert G.data_nu.dtype == np.dtype(dtype)
    assert_bitwise(G.shortest_path(distance="data"), sp_oracle(G, distance="data"), "data d=%d %s" % (d, dtype))
