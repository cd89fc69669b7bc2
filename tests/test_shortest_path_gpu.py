"""G.shortest_path on the device against the reference wrapper (base.py:934-988) applied with scipy to the graph's
own host K and data_nu.

Bit identity is required for method="D": the device traversal computes the fixpoint of float64 relaxations, which
is what Dijkstra returns for non-negative lengths.  For "affinity" the oracle takes -log(K_ij) correctly rounded
(mpmath): the device computes that value, while numpy's log depends on the host (SVML on AVX-512 CPUs is off by one
ulp on ~0.2 % of inputs), so against numpy's own log the result is only required to agree within rounding."""
import pickle
import warnings

import mpmath
import numpy as np
import pytest
from scipy import sparse
from scipy.sparse.csgraph import shortest_path as scipy_shortest_path

import graphtools_b200 as gt
from graphtools_b200 import paths, synth

pytestmark = pytest.mark.gpu


def _log_cr(x):
    mpmath.mp.prec = 120
    return np.array([float(mpmath.log(mpmath.mpf(float(v)))) if v > 0 else -np.inf for v in x])


def oracle(G, method="D", distance=None, numpy_log=False):
    if distance is None:
        distance = "affinity" if G.weighted else "data"
    K = G.K
    with np.errstate(divide="ignore"):
        if distance == "constant":
            L = K
        elif distance == "data":
            L = sparse.coo_matrix(K)
            X = G.data_nu
            L.data = np.sqrt(np.sum((X[L.row] - X[L.col]) ** 2, axis=1))
        else:
            L = sparse.csr_matrix(K, copy=True)
            L.data = -1 * (np.log(L.data) if numpy_log else _log_cr(L.data))
    if method == "FW":
        L = sparse.csr_matrix(L)
    D = scipy_shortest_path(L, method=method)
    D = (D + D.T) / 2
    D[D == 0] = np.inf
    D[np.arange(D.shape[0]), np.arange(D.shape[0])] = 0
    return D


def _graph(X, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return gt.Graph(X, verbose=0, **kw)


def _digits(n=None):
    from sklearn.datasets import load_digits
    return load_digits().data.astype(np.float32)[:n]


def assert_bitwise(D, R, what):
    assert D.shape == R.shape and D.dtype == np.float64, what
    same = (D == R) | (np.isinf(D) & np.isinf(R))
    bad = np.argwhere(~same)
    assert bad.shape[0] == 0, "%s: %d entries differ, first %s: %r vs %r" % (
        what, bad.shape[0], bad[0], D[tuple(bad[0])], R[tuple(bad[0])])
    assert np.array_equal(D, D.T), what + ": not bitwise symmetric"


@pytest.fixture(scope="module")
def digits_weighted():
    return _graph(_digits(), knn=5, decay=40)


def test_digits_affinity_bitwise(digits_weighted):
    G = digits_weighted
    assert G.weighted
    D = G.shortest_path()
    assert_bitwise(D, oracle(G), "digits affinity")
    assert_bitwise(G.shortest_path(method="auto", distance="affinity"), D, "explicit arguments")
    # against numpy's own log: same inf pattern, within rounding
    R = oracle(G, numpy_log=True)
    fin = np.isfinite(R)
    assert np.array_equal(fin, np.isfinite(D))
    assert np.allclose(D[fin], R[fin], rtol=1e-13, atol=0)


def test_run_to_run_bit_identity(digits_weighted):
    D1 = digits_weighted.shortest_path()
    D2 = digits_weighted.shortest_path()
    assert np.array_equal(D1, D2)


def test_digits_unweighted_data_and_constant():
    G = _graph(_digits(), knn=5, decay=None)
    assert not G.weighted
    assert_bitwise(G.shortest_path(), oracle(G, distance="data"), "digits data")
    assert_bitwise(G.shortest_path(distance="constant"), oracle(G, distance="constant"), "digits constant")


def test_disconnected_clusters_give_inf_blocks():
    rng = np.random.default_rng(3)
    X = np.concatenate([rng.normal(size=(400, 8)), rng.normal(size=(300, 8)) + 1000.0]).astype(np.float32)
    G = _graph(X, knn=5, decay=40)
    D = G.shortest_path()
    assert_bitwise(D, oracle(G), "two clusters")
    assert np.isinf(D[:400, 400:]).all() and np.isinf(D[400:, :400]).all()
    assert np.isfinite(D[:400, :400]).all()
    assert paths.stats()["components"] >= 2


def test_asymmetric_kernel():
    G = _graph(_digits(), knn=5, decay=40, kernel_symm=None)
    K = G.K
    assert abs(K - K.T).max() > 0
    assert_bitwise(G.shortest_path(), oracle(G), "kernel_symm=None")


def test_mnn_graph():
    X = _digits(900)
    G = _graph(X, knn=5, decay=40, sample_idx=np.arange(900) % 3, kernel_symm="mnn", theta=0.7)
    assert type(G).__name__ == "MNNGraph"
    assert_bitwise(G.shortest_path(), oracle(G), "mnn")


def test_exact_graph_with_threshold():
    G = _graph(_digits(700), graphtype="exact", knn=5, decay=40, thresh=1e-4)
    assert type(G).__name__ == "TraditionalGraph" and isinstance(G.K, np.ndarray)
    assert_bitwise(G.shortest_path(), oracle(G), "exact thresh")


def test_precomputed_adjacency_graph():
    from scipy.spatial.distance import pdist, squareform
    X = _digits(500).astype(np.float64)
    Dx = squareform(pdist(X))
    A = (Dx < np.percentile(Dx, 3)).astype(float)
    np.fill_diagonal(A, 0)
    G = _graph(A, precomputed="adjacency", decay=None)
    assert not G.weighted
    assert_bitwise(G.shortest_path(), oracle(G, distance="data"), "adjacency data")
    assert_bitwise(G.shortest_path(distance="constant"), oracle(G, distance="constant"), "adjacency constant")
    with pytest.raises(ValueError, match="only valid for weighted graphs"):
        G.shortest_path(distance="affinity")


def test_duplicate_points_zero_length_paths_become_inf():
    X = _digits(500)
    X = np.concatenate([X, X[:40]])
    Gu = _graph(X, knn=5, decay=None)
    D = Gu.shortest_path()
    assert_bitwise(D, oracle(Gu, distance="data"), "duplicates data")
    assert np.isinf(D[np.arange(40), 500 + np.arange(40)]).all()
    Gw = _graph(X, knn=5, decay=40)
    assert_bitwise(Gw.shortest_path(), oracle(Gw), "duplicates affinity")


def test_landmark_graph_kernel():
    X, _ = synth.gaussian_mixture(1500, 20, n_clusters=4, intrinsic_dim=5, seed=7)
    G = _graph(X, knn=5, decay=40, n_landmark=100, random_landmarking=True, random_state=1)
    assert type(G).__name__ == "kNNLandmarkGraph"
    assert_bitwise(G.shortest_path(), oracle(G), "landmark kernel")


def test_20k_points_several_batches():
    X, _ = synth.gaussian_mixture(20000, 30, n_clusters=6, intrinsic_dim=6, seed=11)
    G = _graph(X, knn=5, decay=None)
    D = G.shortest_path()
    st = paths.stats()
    assert st["batches"] >= 20
    assert_bitwise(D, oracle(G, distance="data"), "20k data")


def test_floyd_warshall_within_rounding():
    G = _graph(_digits(600), knn=5, decay=40)
    D = G.shortest_path(method="FW")
    R = oracle(G, method="FW")
    assert np.array_equal(np.isinf(D), np.isinf(R))
    fin = np.isfinite(R)
    assert np.allclose(D[fin], R[fin], rtol=1e-12, atol=0)


def test_negative_lengths_raise():
    # a precomputed affinity without self-loops has degrees below 1, so anisotropy pushes K above 1 and -log(K) < 0
    A = np.zeros((8, 8))
    for i in range(7):
        A[i, i + 1] = A[i + 1, i] = 0.2
    G = _graph(A, precomputed="affinity", decay=None, anisotropy=1)
    assert G.weighted and G.K.max() > 1
    with pytest.raises(NotImplementedError, match="negative edge lengths"):
        G.shortest_path()


def test_error_paths(digits_weighted):
    with pytest.raises(ValueError, match="Expected `distance` in"):
        digits_weighted.shortest_path(distance="geodesic")
    with pytest.raises(NotImplementedError, match="only implemented for unweighted graphs"):
        digits_weighted.shortest_path(distance="data")
    with pytest.raises(NotImplementedError, match="only implemented for unweighted graphs"):
        digits_weighted.shortest_path(distance="constant")
    with pytest.raises(ValueError, match="unrecognized method"):
        digits_weighted.shortest_path(method="Dijkstra")


def test_pickle_roundtrip(digits_weighted, tmp_path):
    D = digits_weighted.shortest_path()
    path = tmp_path / "g.pkl"
    digits_weighted.to_pickle(str(path))
    with open(path, "rb") as f:
        G2 = pickle.load(f)
    assert np.array_equal(G2.shortest_path(), D)
