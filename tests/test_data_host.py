"""Host-side contract of the Data front-end (reference graphtools/base.py:72-424), mirroring the reference's own
test/test_data.py: argument parsing, error and warning text, accepted containers, transform / inverse_transform.
No GPU needed: graphs are created with initialize=False, and the PCA front-end is the reference's scikit-learn call
(GTB_PCA=host)."""
import numbers
import warnings

import numpy as np
import pytest
from scipy import sparse
from scipy.spatial.distance import pdist, squareform
from sklearn.datasets import load_digits

import graphtools_b200 as gt

DATA = load_digits().data[:400]


@pytest.fixture(autouse=True)
def _host_pca(monkeypatch):
    """The host front-end on every machine: with a GPU present GTB_PCA=auto would reduce on the device, whose
    factors agree with scikit-learn's to rounding only (tests/test_pca_gpu.py), not bit for bit."""
    monkeypatch.setenv("GTB_PCA", "host")


def build(data=DATA, **kw):
    kw.setdefault("initialize", False)
    kw.setdefault("verbose", 0)
    kw.setdefault("random_state", 42)
    return gt.Graph(data, **kw)


def _raises(exc, text, fn):
    with pytest.raises(exc) as ei:
        fn()
    assert text in str(ei.value), str(ei.value)


def _warns(cat, text, fn):
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        out = fn()
    assert any(issubclass(w.category, cat) and text in str(w.message) for w in rec), [str(w.message) for w in rec]
    return out


# ---- parameters (test_data.py:32-196)
def test_1d_and_3d_data():
    _raises(ValueError, "Expected 2D array, got 1D array instead (shape: ({},).)".format(DATA.shape[0]),
            lambda: build(DATA[:, 0], n_pca=20))
    _raises(ValueError, "Reshape your data either using array.reshape(-1, 1) if your data has a single feature or "
                        "array.reshape(1, -1) if it contains a single sample.", lambda: build(DATA[:, 0], n_pca=20))
    _raises(ValueError, "Expected 2D array, got 3D array instead (shape: ({0}, 64, 1).)".format(DATA.shape[0]),
            lambda: build(DATA[:, :, None], n_pca=20))


def test_n_pca_parsing():
    assert build(n_pca=0).n_pca is None and build(n_pca=False).n_pca is None
    _raises(ValueError, "n_pca must be an integer 0 <= n_pca < min(n_samples,n_features), or in [None, False, True, "
                        "'auto'].", lambda: build(n_pca="foobar"))
    _raises(ValueError, "n_pca was not an instance of numbers.Number, could not be cast to False, and not None. Please "
                        "supply an integer 0 <= n_pca < min(n_samples,n_features) or None", lambda: build(n_pca=[]))
    _raises(ValueError, "n_pca cannot be negative. Please supply an integer 0 <= n_pca < min(n_samples,n_features) or "
                        "None", lambda: build(n_pca=-1))
    _warns(RuntimeWarning, "Cannot perform PCA to fractional 1.5 dimensions. Rounding to 2", lambda: build(n_pca=1.5))
    _warns(RuntimeWarning, "Cannot perform PCA to {0} dimensions on data with min(n_samples, n_features) = {0}".format(
        DATA.shape[1]), lambda: build(n_pca=DATA.shape[1]))
    _warns(RuntimeWarning, "Cannot perform PCA to {0} dimensions on data with min(n_samples, n_features) = {0}".format(
        DATA.shape[1] - 1), lambda: build(DATA[: DATA.shape[1] - 1], n_pca=DATA.shape[1] - 1))


def test_rank_threshold_parsing():
    for bad in ("foobar", -1, []):
        _raises(ValueError, "rank_threshold must be positive float or 'auto'.",
                lambda: build(n_pca=True, rank_threshold=bad))
    with pytest.raises(ValueError, match=r"Supplied threshold ([0-9\.]*) was greater than maximum singular value "
                                         r"([0-9\.]*) for the data matrix"):
        build(n_pca=True, rank_threshold=np.linalg.norm(DATA) ** 2)
    g = _warns(RuntimeWarning, "n_pca = 10, therefore rank_threshold of -1 will not be used. To use rank thresholding, "
                               "set n_pca = True", lambda: build(n_pca=10, rank_threshold=-1))
    assert g.n_pca == 10


def test_adaptive_n_pca():
    assert isinstance(build(n_pca=True).n_pca, numbers.Number)
    g = build(n_pca=True, rank_threshold=0.1)
    assert isinstance(g.n_pca, numbers.Number) and isinstance(g.rank_threshold, numbers.Number)
    g = build(n_pca=True, rank_threshold="auto")
    assert isinstance(g.n_pca, numbers.Number) and isinstance(g.rank_threshold, numbers.Number)
    nxt = np.sort(g.data_pca.singular_values_)[2]
    assert g.n_pca > build(n_pca=True, rank_threshold=nxt).n_pca
    build(n_pca=True, rank_threshold="AUTO")
    build(n_pca="auto")
    build(n_pca="AUTO")
    assert g.data_nu.shape == (DATA.shape[0], g.n_pca)
    assert np.allclose(g.data_nu, g.transform(g.data))


def test_precomputed_with_pca():
    _warns(RuntimeWarning, "n_pca cannot be given on a precomputed graph. Setting n_pca=None",
           lambda: build(squareform(pdist(DATA)), precomputed="distance", n_pca=20))


# ---- containers (test_data.py:199-240)
def test_pandas_inputs():
    pd = pytest.importorskip("pandas")
    G = build(pd.DataFrame(DATA))
    assert isinstance(G.data, np.ndarray)
    Xs = pd.DataFrame(DATA).astype(pd.SparseDtype(float, fill_value=0))
    G = build(Xs)
    assert sparse.issparse(G.data) and isinstance(G.data_nu, sparse.csr_matrix)


# ---- transform / inverse_transform (test_data.py:242-530)
def _shape_msg(shape, G):
    return "data of shape {0} cannot be transformed to graph built on data of shape {1}".format(shape, G.data.shape)


@pytest.mark.parametrize("n_pca", [20, None])
def test_transform_dense(n_pca):
    G = build(n_pca=n_pca)
    assert np.all(G.data_nu == G.transform(G.data))
    _raises(ValueError, _shape_msg((DATA.shape[0],), G), lambda: G.transform(G.data[:, 0]))
    _raises(ValueError, _shape_msg((DATA.shape[0], 1, 15), G), lambda: G.transform(G.data[:, None, :15]))
    _raises(ValueError, _shape_msg((DATA.shape[0], 15), G), lambda: G.transform(G.data[:, :15]))


@pytest.mark.parametrize("n_pca", [20, None])
def test_transform_sparse(n_pca):
    G = build(sparse.coo_matrix(DATA), n_pca=n_pca)
    if n_pca:
        assert np.all(G.data_nu == G.transform(G.data))
    else:
        assert (G.data_nu != G.transform(G.data)).nnz == 0
    _raises(ValueError, _shape_msg((DATA.shape[0], 1), G), lambda: G.transform(sparse.csr_matrix(DATA)[:, 0]))
    _raises(ValueError, _shape_msg((DATA.shape[0], 15), G), lambda: G.transform(sparse.csr_matrix(DATA)[:, :15]))


def test_inverse_transform_dense_pca():
    G = build(n_pca=DATA.shape[1] - 1)
    np.testing.assert_allclose(G.data, G.inverse_transform(G.data_nu), atol=1e-12)
    np.testing.assert_allclose(G.data[:, -1, None], G.inverse_transform(G.data_nu, columns=-1), atol=1e-12)
    np.testing.assert_allclose(G.data[:, 5:7], G.inverse_transform(G.data_nu, columns=[5, 6]), atol=1e-12)
    with pytest.raises(IndexError):
        G.inverse_transform(G.data_nu, columns=DATA.shape[1])
    for bad in (G.data[:, 0], G.data[:, None, :15], G.data[:, :15]):
        _raises(ValueError, "data of shape {} cannot be inverse transformed from graph built on reduced data of shape "
                            "({}, {})".format(bad.shape, G.data_nu.shape[0], G.data_nu.shape[1]),
                lambda: G.inverse_transform(bad))


def test_inverse_transform_no_pca():
    G = build(n_pca=None)
    np.testing.assert_allclose(DATA[:, 5:7], G.inverse_transform(G.data_nu, columns=[5, 6]), atol=1e-12)
    assert np.all(G.data == G.inverse_transform(G.data_nu))
    with pytest.raises(IndexError):
        G.inverse_transform(G.data_nu, columns=DATA.shape[1])
    for bad in (G.data[:, 0], G.data[:, None, :15], G.data[:, :15]):
        _raises(ValueError, "data of shape {} cannot be inverse transformed from graph built on reduced data of shape "
                            "({}, {})".format(bad.shape, DATA.shape[0], DATA.shape[1]), lambda: G.inverse_transform(bad))


def test_set_params():
    G = build(n_pca=20)
    assert G.get_params()["n_pca"] == 20 and G.get_params()["random_state"] == 42
    G.set_params(random_state=13)
    assert G.random_state == 13
    _raises(ValueError, "Cannot update n_pca. Please create a new graph", lambda: G.set_params(n_pca=10))
    G.set_params(n_pca=G.n_pca)


@pytest.mark.parametrize("as_sparse", [False, True])
def test_transform_adaptive_pca(as_sparse):
    """test_data.py:465-530: rank-thresholded PCA is consistent with the fixed-n_pca graph of the same rank."""
    X = sparse.csr_matrix(DATA) if as_sparse else DATA
    G = build(X, n_pca=True, random_state=42)
    assert np.all(G.data_nu == G.transform(G.data))
    bad = sparse.csr_matrix(DATA)[:, :15] if as_sparse else DATA[:, :15]
    _raises(ValueError, _shape_msg(bad.shape, G) + ". Expected shape ({}, {})".format(DATA.shape[0], DATA.shape[1]),
            lambda: G.transform(bad))
    G2 = build(X, n_pca=True, rank_threshold=G.rank_threshold, random_state=42)
    assert np.allclose(G2.data_nu, G2.transform(G2.data)) and np.allclose(G2.data_nu, G.transform(G.data))
    G3 = build(X, n_pca=G2.n_pca, random_state=42)
    assert np.allclose(G3.data_nu, G3.transform(G3.data)) and np.allclose(G3.data_nu, G2.transform(G2.data))


def test_inverse_transform_sparse_svd():
    """test_data.py:374-410: TruncatedSVD has no mean_; inverse_transform(columns=...) still works."""
    G = build(sparse.csr_matrix(DATA), n_pca=DATA.shape[1] - 1)
    np.testing.assert_allclose(DATA, G.inverse_transform(G.data_nu), atol=1e-12)
    np.testing.assert_allclose(DATA[:, -1, None], G.inverse_transform(G.data_nu, columns=-1), atol=1e-12)
    np.testing.assert_allclose(DATA[:, 5:7], G.inverse_transform(G.data_nu, columns=[5, 6]), atol=1e-12)
    with pytest.raises(IndexError):
        G.inverse_transform(G.data_nu, columns=DATA.shape[1])
