"""Pins oracle/graph_oracle.py to the unmodified reference: every golden fixture
(tests/golden/*.npz, produced by oracle/make_golden.py from /root/reference) must be
reproduced BIT-FOR-BIT by the oracle's restatement on the same float32-exact inputs."""
import numpy as np
import pytest
from scipy import sparse
from threadpoolctl import threadpool_limits

from oracle import graph_oracle as go
from tests.golden_util import GOLDEN_THREADS, Case, csr_equal, names


@pytest.fixture(autouse=True)
def _golden_threads():
    with threadpool_limits(limits=GOLDEN_THREADS, user_api="blas"):
        yield


def _raw_kernel(case):
    p, X = case.params, case.X.astype(np.float64)
    if case.cls.startswith("kNN"):
        g = go.KnnOracle(X, knn=p.get("knn", 5), decay=p.get("decay", 40), knn_max=p.get("knn_max"),
                         bandwidth=p.get("bandwidth"), bandwidth_scale=p.get("bandwidth_scale", 1.0),
                         thresh=p.get("thresh", 1e-4), distance=p.get("distance", "euclidean"),
                         n_jobs=GOLDEN_THREADS)
        return g.kernel(), g
    if case.cls.startswith("Traditional"):
        return go.exact_kernel(X, knn=p.get("knn", 5), decay=p.get("decay", 40), bandwidth=p.get("bandwidth"),
                               bandwidth_scale=p.get("bandwidth_scale", 1.0), thresh=p.get("thresh", 1e-4),
                               distance=p.get("distance", "euclidean")), None
    if case.cls.startswith("MNN"):
        return go.mnn_kernel(X, p["sample_idx"], knn=p.get("knn", 5), decay=p.get("decay", 40),
                             thresh=p.get("thresh", 1e-4), beta=p.get("beta", 1), n_jobs=GOLDEN_THREADS), None
    raise AssertionError(case.cls)


def _same(A, B):
    if sparse.issparse(A) or sparse.issparse(B):
        return csr_equal(A, B)
    return np.array_equal(np.asarray(A), np.asarray(B))


@pytest.mark.parametrize("name", names())
def test_oracle_reproduces_reference(name):
    case = Case(name)
    p = case.params
    R, g = _raw_kernel(case)
    if case.has("R"):
        assert _same(R, case.mat("R")), "raw kernel differs from reference"
    K = go.finish_kernel(R, p.get("kernel_symm", "+"), p.get("theta"), p.get("anisotropy", 0))
    if case.has("K"):
        assert _same(K, case.mat("K")), "kernel differs from reference"
        assert _same(go.diff_op(K), case.mat("P")), "diff_op differs from reference"
        assert np.array_equal(go.kernel_degree(K), case.z["degree"])
    if "clusters" in case.z.files:
        X = case.X.astype(np.float64)
        if p.get("random_landmarking"):
            clusters = go.random_landmark_clusters(X, p["n_landmark"], p["random_state"],
                                                   distance=p.get("distance", "euclidean"))
        else:
            clusters = go.spectral_clusters(K, p["n_landmark"], p.get("n_svd", 100), p["random_state"])
        assert np.array_equal(clusters, case.z["clusters"])
        op, pnm = go.landmark_operator(K, clusters)
        assert _same(op, case.mat("landmark_op"))
        assert _same(pnm, case.mat("transitions"))
    if "Y" in case.z.files:
        Y = case.z["Y"].astype(np.float64)
        if case.cls.startswith("kNN"):
            Kyx = g.kernel_to_data(Y)
        else:
            Kyx = go.exact_kernel_to_data(case.X.astype(np.float64), Y, knn=p.get("knn", 5),
                                          decay=p.get("decay", 40), thresh=p.get("thresh", 1e-4),
                                          distance=p.get("distance", "euclidean"))
        assert _same(Kyx, case.mat("Kyx"))
        if "clusters" in case.z.files:
            assert _same(go.landmark_extend(Kyx, case.z["clusters"]), case.mat("ext"))
        else:
            assert _same(go.diff_op(Kyx), case.mat("ext"))
