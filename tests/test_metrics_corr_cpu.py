"""Host-side pieces of the sqeuclidean and correlation metrics, checked without a GPU: the names graphs accept, the
constant-row test, the correlation search copy, and the identities of the reference (scipy / sklearn through the CPU
oracle) that the device paths rely on."""
import warnings

import numpy as np
import pytest
import torch
from scipy.spatial.distance import cdist, pdist

import graphtools_b200 as gt
from graphtools_b200 import pipeline, synth
from oracle import graph_oracle as go
from tests.parity import compare_dense, compare_sparse


def _data(n=80, d=6, seed=0):
    return np.random.default_rng(seed).normal(size=(n, d))


@pytest.mark.parametrize("graphtype", ["knn", "exact"])
@pytest.mark.parametrize("distance", ["sqeuclidean", "correlation"])
def test_new_metrics_are_accepted(distance, graphtype):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        G = gt.Graph(_data(), graphtype=graphtype, knn=5, decay=20, distance=distance, initialize=False, verbose=0)
    assert G.distance == distance


@pytest.mark.parametrize("graphtype", ["knn", "exact"])
@pytest.mark.parametrize("distance", ["minkowski", "chebyshev", "braycurtis"])
def test_other_metrics_still_raise(distance, graphtype):
    with pytest.raises(NotImplementedError, match="euclidean, cosine and cityblock"):
        gt.Graph(_data(), graphtype=graphtype, knn=5, decay=20, distance=distance, initialize=False, verbose=0)


def test_degenerate_rows_on_host_arrays():
    from scipy import sparse
    X = _data(10, 5)
    X[2] = 0.0
    X[4] = 3.25
    X[7] = [1.0, 1.0, 1.0, 1.0, 1.0 + 2 ** -20]         # not constant, however close
    want = np.zeros(10, dtype=bool)
    want[[2, 4]] = True
    for A in (X, X.astype(np.float32)):
        assert np.array_equal(pipeline.degenerate_rows(A, "correlation"), want)
    assert np.array_equal(pipeline.degenerate_rows(sparse.csr_matrix(X), "correlation"), want)
    assert torch.equal(pipeline.degenerate_rows(torch.from_numpy(X), "correlation"), torch.from_numpy(want))
    assert np.array_equal(pipeline.degenerate_rows(X, "cosine"), np.arange(10) == 2)
    for metric in ("euclidean", "sqeuclidean", "cityblock"):
        assert pipeline.degenerate_rows(X, metric) is None
    pipeline.reject_constant_rows(X, "cosine")            # only correlation searches reject them
    with pytest.raises(ValueError, match="2 of 10 rows are constant"):
        pipeline.reject_constant_rows(X, "correlation")
    with pytest.raises(ValueError, match="1 of 3 rows are constant"):
        pipeline.reject_constant_rows(torch.from_numpy(X[3:6]), "correlation")


@pytest.mark.parametrize("offset", [0.0, 1e4])
def test_correlation_operand_centres_rows_before_rounding(offset):
    """The search copy is built from the row-centred, row-normalised rows in float64 and rounded once: with a per-row
    offset 1e4 times the spread, centring after the float32 rounding would leave an error of ~1e-3 of the spread.
    ``X`` keeps the original rows."""
    rng = np.random.default_rng(3)
    X = rng.normal(size=(40, 9)) + offset * rng.normal(size=(40, 1))
    Xt = torch.from_numpy(X)
    op = pipeline.SearchOperand(Xt, metric="correlation")
    assert op.X is Xt and op.metric == "correlation"
    C = X - X.mean(axis=1, keepdims=True)
    U = C / np.linalg.norm(C, axis=1, keepdims=True)
    want = U - U.mean(axis=0)
    assert np.allclose(op.mean.numpy(), U.mean(axis=0), rtol=0, atol=1e-10)   # row means round differently
    assert np.abs(op.Xs.numpy().astype(np.float64) - want).max() <= 2 ** -23
    # squared Euclidean distances of the unit rows are 2 x the correlation distances
    D = cdist(X, X, "correlation")
    assert np.allclose(cdist(U, U, "sqeuclidean"), 2 * D, rtol=0, atol=1e-12)


def test_sqeuclidean_operand_is_euclidean():
    X = torch.from_numpy(_data(30, 7))
    a, b = pipeline.SearchOperand(X, metric="sqeuclidean"), pipeline.SearchOperand(X, metric="euclidean")
    assert torch.equal(a.Xs, b.Xs) and torch.equal(a.mean, b.mean)
    assert pipeline.METRIC_CODE["sqeuclidean"] == 3 and pipeline.METRIC_CODE["correlation"] == 4


# --------------------------------------------------------------------------- the reference's identities
def test_scipy_correlation_is_cosine_of_centred_rows():
    X = _data(50, 13, 5) + 7.0
    C = X - X.mean(axis=1, keepdims=True)
    assert np.array_equal(pdist(X, "correlation"), pdist(C, "cosine"))
    Y = _data(20, 13, 6)
    assert np.array_equal(cdist(Y, X, "correlation"), cdist(Y - Y.mean(axis=1, keepdims=True), C, "cosine"))
    X[4] = 2.0                                               # constant row: NaN distances
    D = cdist(X, X, "correlation")
    assert np.isnan(D[4]).all() and np.isnan(D[:, 4]).all() and np.isfinite(np.delete(D, 4, 0)[:, :4]).all()


def test_oracle_correlation_knn_is_cosine_knn_of_centred_rows():
    """sklearn's cosine search evaluates 1 - x^.y^ on normalised rows, scipy's correlation 1 - x.y / (|x||y|):
    the same distances up to rounding, which decay 20 amplifies to ~1e-11."""
    X, _ = synth.gaussian_mixture(400, 12, n_clusters=3, intrinsic_dim=4, seed=2)
    X = X.astype(np.float64) + 3.0
    C = X - X.mean(axis=1, keepdims=True)
    K, P = go.knn_graph(X, knn=5, decay=20, thresh=1e-4, distance="correlation")
    Kc, Pc = go.knn_graph(C, knn=5, decay=20, thresh=1e-4, distance="cosine")
    compare_sparse(K, Kc, rtol=1e-9, what="correlation vs cosine of centred rows")
    compare_sparse(P, Pc, rtol=1e-9, what="P")


def test_oracle_sqeuclidean_decay_is_euclidean_double_decay():
    """Bandwidth and radius are in squared units: exp(-(s / s_k)^a) = exp(-(r / r_k)^(2 a)) for s = r^2.  With
    decay=None the neighbour sets are the Euclidean ones."""
    X, _ = synth.gaussian_mixture(400, 10, n_clusters=3, intrinsic_dim=4, seed=4)
    X = X.astype(np.float64)
    K, P = go.knn_graph(X, knn=5, decay=10, thresh=1e-4, distance="sqeuclidean")
    Ke, Pe = go.knn_graph(X, knn=5, decay=20, thresh=1e-4, distance="euclidean")
    compare_sparse(K, Ke, rtol=1e-9, what="sqeuclidean decay 10 vs euclidean decay 20")
    Kb, _ = go.knn_graph(X, knn=5, decay=None, distance="sqeuclidean")
    Kbe, _ = go.knn_graph(X, knn=5, decay=None, distance="euclidean")
    assert (Kb != Kbe).nnz == 0
    Kx = go.exact_kernel(X[:150], knn=5, decay=10, distance="sqeuclidean", thresh=0)
    Kxe = go.exact_kernel(X[:150], knn=5, decay=20, distance="euclidean", thresh=0)
    compare_dense(Kx, Kxe, rtol=1e-9, what="exact sqeuclidean vs euclidean")
