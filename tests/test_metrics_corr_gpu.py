"""sqeuclidean and correlation graphs against the CPU oracle: the kNN sweep over every search flavour, the identities
that tie them to the Euclidean and cosine graphs, per-row offsets, constant rows, the reference's metric-less
fallback search (quirk H9), exact graphs at tile edges, landmark and MNN graphs, shortest paths and the duplicate
warning for affine copies."""
import re
import warnings

import numpy as np
import pytest
from scipy import sparse
from scipy.spatial.distance import cdist

import graphtools_b200 as gt
from graphtools_b200 import dense, pipeline, synth
from oracle import graph_oracle as go
from tests.parity import compare_dense, compare_sparse
from tests.test_metrics_gpu import (N, NQ, _assert_fallback, _assert_no_fallback, _compare_graph, _f64, _gamma,
                                    _graph, _mixture64, expected_impl)
from tests.test_shortest_path_gpu import assert_bitwise, oracle as sp_oracle

pytestmark = pytest.mark.gpu

IMPLS = ["auto", "tc", "tc16", "tch", "tch1", "simt"]


def _centred(X):
    X = np.asarray(X, dtype=np.float64)
    return X - X.mean(axis=1, keepdims=True)


def _tie(metric, X, knn, Y=None):
    """Tie exemption in a metric with the same ordering: cosine of the centred rows for correlation, Euclidean for
    sqeuclidean."""
    if metric == "correlation":
        return dict(X=_centred(X), Y=None if Y is None else _centred(Y), knn=knn, metric="cosine")
    return dict(X=X, Y=Y, knn=knn, metric="euclidean")


# --------------------------------------------------------------------------- 1: kNN sweep over every flavour
# isotropic data: a decay per width whose raw rows run past the 64-entry candidate lists (so the radius pass runs)
# while the reference's search stays below N / 2.  3-D correlation is 2-D cosine (rows centred to a plane): decay 1,
# as for 2-D cosine.  2-D correlation is not swept: a centred 2-D row is +-(a, -a), every distance is 0 or 2.
ISO_DECAY = {("sqeuclidean", 2): 2, ("sqeuclidean", 3): 3, ("sqeuclidean", 31): 10, ("sqeuclidean", 33): 10,
             ("sqeuclidean", 100): 20, ("sqeuclidean", 129): 20, ("sqeuclidean", 300): 40, ("sqeuclidean", 510): 40,
             ("correlation", 3): 1, ("correlation", 31): 10, ("correlation", 33): 10, ("correlation", 100): 20,
             ("correlation", 129): 20, ("correlation", 300): 40, ("correlation", 510): 40}


def _sweep_case(metric, dtype, d, kind):
    if kind == "iso":
        X = np.random.default_rng(d).normal(size=(N, d)).astype(np.float32)
        params = dict(knn=5, decay=ISO_DECAY[(metric, d)], thresh=1e-4)
    else:
        X, _ = synth.gaussian_mixture(N, d, n_clusters=6, intrinsic_dim=4, seed=d)
        params = dict(knn=5, decay=40, thresh=1e-4)
    X = _f64(X, d) if dtype == "float64" else X
    Y = X[:NQ] + np.asarray(0.02 * np.random.default_rng(d + 1).normal(size=(NQ, d)), dtype=X.dtype)
    K_ref, P_ref, g = go.knn_graph(X.astype(np.float64), distance=metric, return_oracle=True, **params)
    Kyx_ref = g.kernel_to_data(Y.astype(np.float64))
    _assert_no_fallback(g)
    long_rows = int(np.diff(g.kernel().indptr).max()) > 64
    return X, Y, params, K_ref, P_ref, Kyx_ref, long_rows


@pytest.mark.parametrize("kind", ["clustered", "iso"])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("d", [2, 3, 31, 33, 100, 129, 300, 510])
@pytest.mark.parametrize("metric", ["sqeuclidean", "correlation"])
def test_knn_sweep(metric, d, dtype, kind, monkeypatch):
    """Every search flavour against the oracle; K, P and the out-of-sample kernel bit-identical across flavours."""
    if metric == "correlation" and d == 2:
        pytest.skip("correlation of two features is degenerate (0 or 2)")
    X, Y, params, K_ref, P_ref, Kyx_ref, long_rows = _sweep_case(metric, dtype, d, kind)
    if kind == "iso" and not (metric == "correlation" and d == 3):
        assert long_rows, "iso case does not reach the radius pass"
    first = None
    for want in IMPLS:
        monkeypatch.setenv("GTB_SEARCH_IMPL", want)
        G = _graph(X, distance=metric, **params)
        K, P = G.kernel, G.diff_op
        st = pipeline.stats()
        assert st["impl"] == expected_impl(want, d), (want, st)
        if long_rows:
            assert st["radius_rows"] > 0, st
        Kyx = G.build_kernel_to_data(Y)
        what = "%s %s d=%d %s %s" % (metric, dtype, d, kind, want)
        if first is None:
            _compare_graph(K, P, K_ref, P_ref, params["thresh"], _tie(metric, X, 6), what)
            compare_sparse(Kyx, Kyx_ref, thresh=params["thresh"], what=what + ".Kyx", tie=_tie(metric, X, 5, Y))
            first = (K, P, Kyx)
        else:
            for a, b, name in zip(first, (K, P, Kyx), ("K", "P", "Kyx")):
                assert (a != b).nnz == 0 and np.array_equal(a.data, b.data), what + " " + name + " differs from auto"


# --------------------------------------------------------------------------- 2: cross-identities
def _clustered(n=N, d=40, seed=11, dtype=np.float32):
    X, _ = synth.gaussian_mixture(n, d, n_clusters=6, intrinsic_dim=5, seed=seed)
    return X.astype(dtype)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_sqeuclidean_binary_is_euclidean_bitwise(dtype):
    X = _clustered(dtype=dtype)
    for knn_max in (None, 8):
        K = _graph(X, knn=5, decay=None, knn_max=knn_max, distance="sqeuclidean").kernel
        Ke = _graph(X, knn=5, decay=None, knn_max=knn_max, distance="euclidean").kernel
        assert (K != Ke).nnz == 0 and np.array_equal(K.indices, Ke.indices) and np.array_equal(K.data, Ke.data)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_sqeuclidean_decay_is_euclidean_double_decay(dtype):
    X = _clustered(dtype=dtype)
    for a in (5, 20):
        G = _graph(X, knn=5, decay=a, thresh=1e-4, distance="sqeuclidean")
        Ge = _graph(X, knn=5, decay=2 * a, thresh=1e-4, distance="euclidean")
        K, Ke = G.kernel, Ge.kernel
        assert np.array_equal(K.indptr, Ke.indptr) and np.array_equal(K.indices, Ke.indices)
        assert np.allclose(K.data, Ke.data, rtol=1e-12, atol=0)
        assert np.allclose(G.diff_op.data, Ge.diff_op.data, rtol=1e-12, atol=0)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_correlation_is_cosine_of_centred_rows(dtype):
    """32 float32 values sum exactly in float64 and the division by 32 is exact, so every row mean is exact on the
    device and on the host: the correlation graph and the cosine graph of the host-centred rows see the same
    centred values."""
    X = _clustered(d=32).astype(dtype) + dtype(3.0)
    G = _graph(X, knn=5, decay=40, thresh=1e-4, distance="correlation")
    Gc = _graph(_centred(X), knn=5, decay=40, thresh=1e-4, distance="cosine")
    K, Kc = G.kernel, Gc.kernel
    assert np.array_equal(K.indptr, Kc.indptr) and np.array_equal(K.indices, Kc.indices)
    assert np.allclose(K.data, Kc.data, rtol=1e-12, atol=0)
    assert np.allclose(G.diff_op.data, Gc.diff_op.data, rtol=1e-12, atol=0)


# --------------------------------------------------------------------------- 3: per-row offsets
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("offset", [1e3, 1e4])
def test_correlation_row_offsets(offset, dtype):
    """Each row shifted by its own offset, 1e3 or 1e4 times the spread: correlation ignores it, but a search copy
    rounded to float32 before centring would keep only ~3 digits of the row's shape."""
    X, _ = synth.gaussian_mixture(N, 31, n_clusters=6, intrinsic_dim=4, seed=21)
    X = X.astype(np.float64)
    X = X + offset * X.std() * np.random.default_rng(22).uniform(1, 2, size=(N, 1))
    X = _f64(X, 21) if dtype == "float64" else X.astype(np.float32)
    Y = X[:NQ] + np.asarray(0.01 * X.std(axis=1, keepdims=True)[:NQ]
                            * np.random.default_rng(23).normal(size=(NQ, 31)), dtype=X.dtype)
    K_ref, P_ref, g = go.knn_graph(X.astype(np.float64), knn=5, decay=40, thresh=1e-4, distance="correlation",
                                   return_oracle=True)
    _assert_no_fallback(g)
    G = _graph(X, knn=5, decay=40, thresh=1e-4, distance="correlation")
    _compare_graph(G.kernel, G.diff_op, K_ref, P_ref, 1e-4, _tie("correlation", X, 6), "offset %g %s" % (offset, dtype))
    compare_sparse(G.build_kernel_to_data(Y), g.kernel_to_data(Y.astype(np.float64)), thresh=1e-4,
                   what="offset Kyx", tie=_tie("correlation", X, 5, Y))


# --------------------------------------------------------------------------- 4: constant rows
def _with_constant_rows(n=300, d=16, dtype=np.float64):
    X = _clustered(n, d, seed=31, dtype=dtype)
    X[7] = 0.0
    X[150] = 2.0
    X[151] = 0.25
    return X


def test_constant_rows_rejected_by_searches():
    X = _with_constant_rows()
    with pytest.raises(ValueError, match="3 of 300 rows are constant"):
        _graph(X, knn=5, decay=20, distance="correlation")
    with pytest.raises(ValueError, match="3 of 300 rows are constant"):
        _graph(X, knn=5, decay=20, distance="correlation", sample_idx=np.arange(300) % 2, kernel_symm="mnn",
               theta=0.5)
    with pytest.raises(ValueError, match="rows are constant"):
        _graph(X, graphtype="exact", knn=5, decay=20, distance="correlation", n_landmark=20, random_landmarking=True,
               random_state=1).landmark_op
    Xc = _clustered(300, 16, seed=31, dtype=np.float64)
    G = _graph(Xc, knn=5, decay=20, distance="correlation")
    Y = Xc[:10].copy()
    Y[3] = 1.0
    with pytest.raises(ValueError, match="1 of 10 rows are constant"):
        G.extend_to_data(Y)
    with pytest.raises(ValueError, match="1 of 10 rows are constant"):
        G.build_kernel_to_data(Y)


@pytest.mark.parametrize("symm", ["+", "*", "mnn", None])
@pytest.mark.parametrize("thresh", [1e-4, 0])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_constant_rows_exact(dtype, thresh, symm):
    """Exact graphs: scipy's correlation distance from a constant row is NaN, which the reference maps to affinity 1;
    np.partition sorts NaN last, so the other rows' bandwidths ignore them.  (Constants with an exact np.mean.)"""
    X = _with_constant_rows(dtype=dtype)
    X64 = X.astype(np.float64)
    theta = 0.3 if symm == "mnn" else None
    G = _graph(X, graphtype="exact", knn=5, decay=20, thresh=thresh, distance="correlation", kernel_symm=symm,
               theta=theta)
    K_ref = go.finish_kernel(go.exact_kernel(X64, knn=5, decay=20, distance="correlation", thresh=thresh), symm, theta)
    K = G.kernel
    K = K.toarray() if sparse.issparse(K) else np.asarray(K)
    assert np.isfinite(K).all()
    compare_dense(K, K_ref, thresh=thresh, what="exact constant rows K %s %g" % (symm, thresh))
    P = G.diff_op
    compare_dense(P.toarray() if sparse.issparse(P) else P, np.asarray(go.diff_op(K_ref)), thresh=thresh,
                  what="exact constant rows P")
    Y = X[:30] + np.asarray(0.01, dtype=X.dtype) * X[30:60]
    Y[[2, 9]] = 1.0
    Kyx_ref = go.exact_kernel_to_data(X64, Y.astype(np.float64), knn=5, decay=20, distance="correlation",
                                      thresh=thresh)
    compare_dense(np.asarray(G.build_kernel_to_data(Y)), Kyx_ref, thresh=thresh, what="exact constant query rows")


# --------------------------------------------------------------------------- 5: metric-less fallback search (H9)
@pytest.mark.parametrize("metric,n,d,seed,decay,branch", [
    ("sqeuclidean", 400, 50, 5, 10, "radius"),
    ("sqeuclidean", 400, 10, 3, 5, "radius"),
    ("sqeuclidean", 200, 10, 5, 3, "kneighbors"),
    ("sqeuclidean", 1000, 50, 0, 5, "kneighbors"),
    ("correlation", 400, 50, 5, 10, "radius"),
    ("correlation", 400, 10, 3, 3, "radius"),
    ("correlation", 200, 10, 5, 3, "kneighbors"),
    ("correlation", 1000, 50, 0, 5, "kneighbors"),
])
def test_fallback_in_sample(metric, n, d, seed, decay, branch):
    """Rows the reference finishes on its metric-less index hold Euclidean distances of the raw rows (not squared,
    not centred) over the metric's own bandwidth."""
    X = _mixture64(n, d, seed)
    K_ref, P_ref, g = go.knn_graph(X, knn=5, decay=decay, thresh=1e-3, distance=metric, return_oracle=True)
    _assert_fallback(g, branch)
    G = _graph(X, knn=5, decay=decay, thresh=1e-3, distance=metric)
    compare_sparse(G.kernel, K_ref, what="fallback K")
    compare_sparse(G.diff_op, P_ref, what="fallback P")
    assert pipeline.stats()["euclidean_fallback_rows"] > 0


@pytest.mark.parametrize("metric,decay", [("sqeuclidean", 5), ("correlation", 3)])
def test_fallback_out_of_sample(metric, decay):
    X = _mixture64(300, 10, 3)
    Y = X[:120] + np.random.default_rng(4).normal(scale=0.05, size=(120, 10))
    g = go.KnnOracle(X, knn=5, decay=decay, thresh=1e-3, distance=metric)
    Kyx_ref = g.kernel_to_data(Y)
    _assert_fallback(g, "radius")
    G = _graph(X, knn=5, decay=decay, thresh=1e-3, distance=metric)
    compare_sparse(G.build_kernel_to_data(Y), Kyx_ref, what="fallback Kyx")


@pytest.mark.parametrize("metric", ["sqeuclidean", "correlation"])
def test_fallback_mnn_small_batches(metric):
    X = _mixture64(600, 10, 3)
    idx = np.repeat([0, 1, 2], 200)
    g = go.KnnOracle(X[idx == 0], knn=5, decay=3, thresh=1e-3, distance=metric)
    g.kernel()
    g.kernel_to_data(X[idx == 1], knn=5)
    assert any(sc["fallback"] and sc["todo"].size for sc in g.schedules)
    K_ref = go.finish_kernel(go.mnn_kernel(X, idx, knn=5, decay=3, thresh=1e-3, distance=metric), "mnn", 0.5)
    G = _graph(X, sample_idx=idx, knn=5, decay=3, thresh=1e-3, distance=metric, kernel_symm="mnn", theta=0.5)
    compare_sparse(G.kernel, K_ref, what="fallback MNN K")
    compare_sparse(G.diff_op, go.diff_op(K_ref), what="fallback MNN P")


# --------------------------------------------------------------------------- 6: exact graphs and dense_distances
@pytest.mark.parametrize("d", [15, 16, 17])
@pytest.mark.parametrize("n", [63, 64, 65, 129])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("metric", ["sqeuclidean", "correlation"])
def test_exact_graph_shapes(metric, dtype, n, d):
    """Tile edges (DT = 64) and feature chunks (DK = 16) on the sparse route (thresh > 0) and the dense one
    (thresh = 0, and a callable bandwidth), in-sample with each symmetrisation and out of sample."""
    rng = np.random.default_rng(n * 1000 + d)
    X = rng.normal(size=(n, d)).astype(np.float32) + 0.5
    X = _f64(X, n + d) if dtype == "float64" else X
    X64 = X.astype(np.float64)
    knn = min(5, n - 2)
    bw_fn = lambda D: np.median(D, axis=1)                   # noqa: E731
    for k, (thresh, bw) in enumerate(((1e-4, None), (0.0, None), (1e-4, bw_fn))):
        symm, theta = [("+", None), ("*", None), ("mnn", 0.3)][(n + d + k) % 3]
        G = _graph(X, graphtype="exact", knn=5, decay=20, thresh=thresh, distance=metric, kernel_symm=symm,
                   theta=theta, bandwidth=bw)
        K_ref = go.finish_kernel(go.exact_kernel(X64, knn=knn, decay=20, distance=metric, thresh=thresh,
                                                 bandwidth=bw), symm, theta)
        K = G.kernel
        K = K.toarray() if sparse.issparse(K) else np.asarray(K)
        what = "exact %s %s n=%d d=%d thresh=%g %s bw=%s" % (metric, dtype, n, d, thresh, symm, bw is not None)
        compare_dense(K, K_ref, thresh=thresh, what=what + " K")
        P = G.diff_op
        compare_dense(P.toarray() if sparse.issparse(P) else P, np.asarray(go.diff_op(K_ref)), thresh=thresh,
                      what=what + " P")
        Y = X[rng.integers(0, n, 40)] + np.asarray(0.1 * rng.normal(size=(40, d)), dtype=X.dtype)
        Kyx_ref = go.exact_kernel_to_data(X64, Y.astype(np.float64), knn=knn, decay=20, distance=metric,
                                          thresh=thresh, bandwidth=bw)
        compare_dense(np.asarray(G.build_kernel_to_data(Y)), Kyx_ref, thresh=thresh, what=what + " Kyx")


@pytest.mark.parametrize("d", [2, 15, 16, 17, 129, 1000])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("metric", ["sqeuclidean", "correlation"])
def test_dense_distances_against_cdist(metric, dtype, d):
    """sqeuclidean: the Euclidean sum without the square root, relative error <= gamma(d + 1) against scipy (whose own
    error is as large: both terms, doubled).  correlation: the cosine bound of test_metrics_gpu (gamma(2 d + 8)
    absolute) on the centred rows, plus the centring: each centred element carries <= gamma(d + 1) |x|_inf of its
    row's mean rounding on either side, at most gamma(d + 1) |x|_inf sqrt(d) / |x - mean| in the cosine, twice."""
    import torch
    rng = np.random.default_rng(d + (dtype == "float64"))
    Xq = rng.normal(size=(70, d)).astype(np.float32) + 0.25
    Xr = rng.normal(size=(130, d)).astype(np.float32) - 0.1
    if dtype == "float64":
        Xq, Xr = _f64(Xq, 1), _f64(Xr, 2)
    dev = pipeline._dev()
    D = dense.dense_distances(torch.from_numpy(Xq).to(dev), torch.from_numpy(Xr).to(dev), metric).cpu().numpy()
    R = cdist(Xq.astype(np.float64), Xr.astype(np.float64), metric)
    if metric == "sqeuclidean":
        assert float((np.abs(D - R) / R).max()) <= 2 * _gamma(d + 1)
    else:
        def cond(X):
            X = X.astype(np.float64)
            return np.abs(X).max(1) * np.sqrt(d) / np.linalg.norm(_centred(X), axis=1)
        bound = 2 * _gamma(2 * d + 8) + 4 * _gamma(d + 1) * (cond(Xq)[:, None] + cond(Xr)[None, :])
        assert (np.abs(D - R) <= bound).all(), float((np.abs(D - R) / bound).max())


# --------------------------------------------------------------------------- 7: landmark, MNN, shortest paths
@pytest.mark.parametrize("metric", ["sqeuclidean", "correlation"])
def test_landmark_random(metric):
    X = _clustered(2000, 20, seed=41, dtype=np.float64)
    K_ref, _ = go.knn_graph(X, knn=5, decay=20, thresh=1e-4, distance=metric)
    clusters = go.random_landmark_clusters(X, 50, 42, distance=metric)
    op_ref, pnm_ref = go.landmark_operator(K_ref, clusters)
    G = _graph(X, knn=5, decay=20, thresh=1e-4, distance=metric, n_landmark=50, random_landmarking=True,
               random_state=42)
    assert np.array_equal(G.clusters, clusters)
    compare_dense(G.landmark_op, op_ref, what=metric + " landmark_op")
    compare_sparse(G.transitions, pnm_ref, what=metric + " transitions")


@pytest.mark.parametrize("metric", ["sqeuclidean", "correlation"])
def test_mnn_graph(metric):
    X = _clustered(900, 20, seed=43, dtype=np.float64)
    idx = np.repeat([0, 1, 2], 300)
    K_ref = go.finish_kernel(go.mnn_kernel(X, idx, knn=5, decay=20, thresh=1e-4, distance=metric), "mnn", 0.5)
    G = _graph(X, sample_idx=idx, knn=5, decay=20, thresh=1e-4, distance=metric, kernel_symm="mnn", theta=0.5)
    compare_sparse(G.kernel, K_ref, thresh=1e-4, what=metric + " MNN K")
    compare_sparse(G.diff_op, go.diff_op(K_ref), thresh=1e-4, what=metric + " MNN P")


def test_shortest_path_on_correlation_graph():
    X = _clustered(1500, 20, seed=45, dtype=np.float32)
    G = _graph(X, knn=5, decay=20, thresh=1e-4, distance="correlation")
    assert_bitwise(G.shortest_path(), sp_oracle(G), "correlation affinity")
    Gb = _graph(X, knn=5, decay=None, distance="correlation")
    assert_bitwise(Gb.shortest_path(distance="constant"), sp_oracle(Gb, distance="constant"), "correlation constant")


# --------------------------------------------------------------------------- 8: duplicate warning
def test_affine_copies_named_in_duplicate_warning():
    """Under correlation y = a x + b (a > 0) is at distance 0 from x without being equal to it.  Integer rows with
    an exact mean (d = 16) and a square centred norm make every distance of the pairs exactly 0, themselves included,
    on the device and in scipy."""
    rng = np.random.default_rng(51)
    X = rng.normal(size=(400, 16)).astype(np.float32)
    base = np.tile(np.array([1.0, -1.0], dtype=np.float32), 8)      # centred, |base|^2 = 16
    X[10] = 3.0 + base
    X[200] = 2 * X[10] + 8.0
    X[300] = 5.0 - base                                                # a < 0: distance 2
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        gt.Graph(X, knn=5, decay=20, thresh=1e-4, distance="correlation", verbose=0).kernel
    msgs = [str(x.message) for x in w if "zero distance" in str(x.message)]
    assert msgs and re.search(r"samples 10 and 200\.", msgs[0]), msgs
    assert cdist(X[[10]].astype(np.float64), X[[200]].astype(np.float64), "correlation")[0, 0] == 0.0


# --------------------------------------------------------------------------- radius wider than the data
@pytest.mark.parametrize("impl", ["tch", "tc"])
def test_radius_wider_than_the_data(impl, monkeypatch):
    """A kernel support radius beyond every point (here a fixed bandwidth 20 x the data's diameter; the reference's
    Euclidean fallback rows of a sqeuclidean graph divide by a squared-unit bandwidth the same way): the radius pass
    must return every reference point and no padded column (n = 1000 is padded to 1024 reference rows)."""
    monkeypatch.setenv("GTB_SEARCH_IMPL", impl)
    X = _mixture64(1000, 50, 0)
    bw = 20 * float(np.sqrt(((X - X.mean(0)) ** 2).sum(1).max()))
    G = _graph(X, knn=5, decay=5, thresh=1e-3, bandwidth=bw)
    assert pipeline.stats()["impl"] == impl and pipeline.stats()["radius_rows"] == 1000
    K_ref, P_ref = go.knn_graph(X, knn=5, decay=5, thresh=1e-3, bandwidth=bw)
    assert G.kernel.nnz == 1000 * 1000
    compare_sparse(G.kernel, K_ref, what="wide radius K")
    compare_sparse(G.diff_op, P_ref, what="wide radius P")
