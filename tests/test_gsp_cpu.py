"""Graph signal filtering without a device (graphtools_b200/gsp.py): the Chebyshev recurrence and Lanczos driven by a
host product, against polynomial identities, numpy's eigh and the numpy restatement of pygsp's cheby_op; the shape
rules and the argument errors."""
import warnings

import numpy as np
import pytest
import torch
from scipy import sparse

import graphtools_b200 as gt
from graphtools_b200 import gsp, pipeline
from tests import gsp_reference as ref


def _random_kernel(n, seed, p=0.05):
    rng = np.random.default_rng(seed)
    A = sparse.random(n, n, density=p, random_state=rng, data_rvs=rng.random)
    W = sparse.triu(A, 1)
    W = (W + W.T).tocsr()
    W = W + sparse.diags(np.ones(n))           # K with its diagonal stored, as the graph builds store it
    W = sparse.csr_matrix(W)
    W.sort_indices()
    return W


def _csr(L):
    return pipeline.DeviceCSR(torch.from_numpy(L.indptr.astype(np.int64)), torch.from_numpy(L.indices),
                              torch.from_numpy(L.data), L.shape)


def _host_step(L):
    """The product of gtb_spmm_cheb / gtb_spmm_cheb_acc with scipy and numpy, in their rounding order."""
    def step(vals, Y, Z, alpha, beta, gamma, out, coef=None, R=None):
        assert out.data_ptr() != Y.data_ptr()
        A = sparse.csr_matrix((vals.numpy(), L.indices, L.indptr), shape=L.shape)
        Yh, Zh = Y.numpy(), Z.numpy()
        out.copy_(torch.from_numpy(alpha * A.dot(Yh) + beta * Yh + gamma * Zh))
        if coef is not None:
            for a in range(coef.shape[0]):
                R[a] = torch.from_numpy(R[a].numpy() + coef[a].item() * out.numpy())
    return step


def _filter(L, s, kernels, order, lmax):
    c = gsp.cheby_coeff(kernels, order, lmax)
    return gsp.cheby_op(_host_step(L), _csr(L), torch.from_numpy(s), c, lmax).numpy()


@pytest.fixture(scope="module")
def graph():
    K = _random_kernel(300, 1)
    L, dw = ref.laplacian(K, "combinatorial")
    lam, U = np.linalg.eigh(L.toarray())
    return K, L, dw, lam, U


@pytest.mark.parametrize("order", [2, 3, 10, 30])
def test_polynomial_kernel_is_reproduced(graph, order):
    _, L, _, lam, _ = graph
    s = np.random.default_rng(order).normal(size=(L.shape[0], 3))
    got = _filter(L, s, [lambda x: 1 + 2 * x + 0.5 * x ** 2], order, 1.01 * lam[-1])[0]
    Ls = L @ s
    want = s + 2 * Ls + 0.5 * (L @ Ls)
    assert np.linalg.norm(got - want) <= 1e-12 * np.linalg.norm(want)


@pytest.mark.parametrize("lap_type", ["combinatorial", "normalized"])
def test_heat_filter_matches_eigendecomposition(graph, lap_type):
    K = graph[0]
    L, _ = ref.laplacian(K, lap_type)
    lam, U = np.linalg.eigh(L.toarray())
    lmax = 1.01 * lam[-1]
    s = np.random.default_rng(2).normal(size=(L.shape[0], 4))
    taus = [1.0, 10.0, 60.0]
    got = _filter(L, s, gsp.heat_kernel(taus, lmax), 30, lmax)
    for i, tau in enumerate(taus):
        want = U @ (np.exp(-tau * lam / lmax)[:, None] * (U.T @ s))
        assert np.abs(got[i] - want).max() <= 1e-6


@pytest.mark.parametrize("order", [1, 2, 5, 30])
def test_recurrence_follows_cheby_op_bit_for_bit(graph, order):
    # the Python side of the recurrence (T1, the first two terms, the factor values) in pygsp's rounding order
    K = graph[0]
    L, _ = ref.laplacian(K, "normalized")
    lmax = 1.7
    s = np.random.default_rng(order).normal(size=(L.shape[0], 5))
    kernels = [ref.heat(10.0, lmax), lambda x: 1 / (1 + x)]
    got = _filter(L, s, kernels, order, lmax)
    c = np.stack([ref.cheby_coeff(h, order, lmax) for h in kernels])
    assert np.array_equal(gsp.cheby_coeff(kernels, order, lmax), c)
    want = ref.cheby_op(L, c, s, lmax)
    for i in range(2):
        assert np.array_equal(got[i], want[i])


def test_laplacian_restatement_is_pygsp_laplacian(graph):
    K, L, dw, _, _ = graph
    W = K - sparse.diags(K.diagonal())
    assert np.abs(dw - np.asarray(W.sum(axis=1)).ravel()).max() <= 1e-14 * dw.max()
    assert np.abs((sparse.diags(dw) - W - L).toarray()).max() == 0
    Ln, _ = ref.laplacian(K, "normalized")
    d = 1 / np.sqrt(dw)
    assert np.abs((sparse.identity(K.shape[0]) - sparse.diags(d) @ W @ sparse.diags(d) - Ln).toarray()).max() <= 1e-15


# ------------------------------------------------------------------------------------------------ Lanczos
def _lanczos(A, **kw):
    At = torch.from_numpy(A)
    v0 = torch.from_numpy(np.random.default_rng(0).normal(size=A.shape[0]))
    return gsp.lanczos(lambda v, out: out.copy_(At @ v), v0, **kw)


@pytest.mark.parametrize("lap_type", ["combinatorial", "normalized"])
def test_lanczos_top_ritz_value_within_its_residual(graph, lap_type):
    L, _ = ref.laplacian(graph[0], lap_type)
    A = L.toarray()
    lam = np.linalg.eigvalsh(A)
    theta, steps, residual, reason = _lanczos(A)
    assert reason == "residual" and steps < gsp.LANCZOS_MAX_STEPS
    assert residual <= gsp.LANCZOS_RTOL * theta
    assert theta <= lam[-1] + 1e-12 and lam[-1] - theta <= residual
    assert lam[-1] <= gsp.bound_lmax(theta, lap_type, 1.0) or lap_type == "combinatorial"


def test_lanczos_step_cap_ends_the_iteration():
    rng = np.random.default_rng(4)
    V, _ = np.linalg.qr(rng.normal(size=(500, 500)))
    A = (V * np.linspace(0, 2, 500)) @ V.T
    theta, steps, residual, reason = _lanczos((A + A.T) / 2, rtol=0.0)
    assert (steps, reason) == (gsp.LANCZOS_MAX_STEPS, "max_steps") and gsp.LANCZOS_MAX_STEPS == 200
    assert 0 < residual and theta <= 2 + 1e-12


def test_lanczos_stops_at_an_invariant_subspace():
    rng = np.random.default_rng(5)
    V, _ = np.linalg.qr(rng.normal(size=(100, 100)))
    A = (V * np.repeat([0.0, 1.0, 3.0], [40, 30, 30])) @ V.T
    theta, steps, _, reason = _lanczos((A + A.T) / 2, rtol=0.0)
    assert reason == "invariant" and steps == 3 and abs(theta - 3) <= 1e-12
    assert _lanczos(np.zeros((5, 5)))[1:] == (1, 0.0, "residual")


def test_bound_clamps():
    # a bipartite graph: the normalized Laplacian's top eigenvalue is exactly 2, so 1.01 theta exceeds the bound
    n = 40
    K = sparse.csr_matrix(sparse.diags([np.ones(n - 1), np.ones(n - 1)], [-1, 1]))
    L, dw = ref.laplacian(K, "normalized")
    theta = _lanczos(L.toarray())[0]
    assert theta > 2 / gsp.LMAX_FACTOR
    assert gsp.bound_lmax(theta, "normalized", dw.max()) == 2.0
    assert gsp.bound_lmax(theta, "combinatorial", 0.9) == 1.8
    assert gsp.bound_lmax(1.0, "combinatorial", 3.0) == gsp.LMAX_FACTOR


# ------------------------------------------------------------------------------------------------ shapes, errors
@pytest.mark.parametrize("one_d", [True, False])
@pytest.mark.parametrize("bank", [True, False])
def test_output_shape_rules(one_d, bank):
    F, n, f = (3 if bank else 1), 7, (1 if one_d else 4)
    R = torch.arange(F * n * f, dtype=torch.float64).reshape(F, n, f)
    out = gsp.arrange(R, one_d, bank)
    want = {(True, True): (n, F), (True, False): (n,), (False, True): (n, f, F), (False, False): (n, f)}
    assert tuple(out.shape) == want[(one_d, bank)]
    for a in range(F):
        for i in range(n):
            for k in range(f):
                idx = (i,) + (() if one_d else (k,)) + ((a,) if bank else ())
                assert out[idx] == R[a, i, k]


def test_argument_errors():
    with pytest.raises(ValueError, match="Unknown Laplacian type"):
        gsp.check_lap_type("random_walk")
    for bad in (None, 3, [], [np.exp, 2]):
        with pytest.raises(ValueError, match="kernel must be a callable"):
            gsp.check_kernels(bad)
    assert gsp.check_kernels(np.exp) == ([np.exp], False)
    assert gsp.check_kernels([np.exp]) == ([np.exp], True)
    for bad in (0, -1, 2.0, True, "3"):
        with pytest.raises(ValueError, match="integer order >= 1"):
            gsp.check_order(bad)
    for bad in (0, -1.0, np.inf, np.nan):
        with pytest.raises(ValueError, match="lmax > 0"):
            gsp.check_lmax(bad)
    for bad in (np.zeros((5, 2, 2)), np.zeros(())):
        with pytest.raises(ValueError, match=r"shape \[N\] or \[N, f\]"):
            gsp.check_signal(bad, 5)
    for bad in (np.zeros(4), np.zeros((6, 2)), np.zeros((5, 0)), torch.zeros(3)):
        with pytest.raises(ValueError, match="n_samples = 5"):
            gsp.check_signal(bad, 5)
    for bad in (np.array([0, 1, np.nan, 2, 3]), torch.tensor([[0.0], [np.inf], [1], [2], [3]])):
        with pytest.raises(ValueError, match="non-finite"):
            gsp.check_signal(bad, 5)
    with pytest.raises(ValueError, match=r"kernel 1 returned shape \(\) for 4 points"):
        gsp.cheby_coeff([np.exp, lambda x: 1.0], 3, 2.0)
    with pytest.raises(ValueError, match="kernel 0 returned non-finite"):
        gsp.cheby_coeff([lambda x: np.full_like(x, np.inf)], 3, 2.0)
    for bad in ([], "a", [[1.0, 2.0]]):
        with pytest.raises(ValueError, match="tau"):
            gsp.heat_kernel(bad, 1.0)
    assert callable(gsp.heat_kernel(10, 1.0)) and len(gsp.heat_kernel([1, 2], 1.0)) == 2
    assert len(gsp.heat_kernel(np.array([5.0]), 1.0)) == 1


def test_graph_methods_reject_before_touching_the_device():
    X = np.random.default_rng(0).normal(size=(50, 4))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        G = gt.Graph(X, knn=3, kernel_symm=None, initialize=False, verbose=0)
        H = gt.Graph(X, knn=3, initialize=False, verbose=0)
    for call in (lambda: G.laplacian(), lambda: G.estimate_lmax(), lambda: G.filter(X[:, 0], np.exp),
                 lambda: G.heat_filter(X[:, 0], lmax=1.0)):
        with pytest.raises(ValueError, match="kernel_symm=None"):
            call()
    with pytest.raises(ValueError, match="Unknown Laplacian type"):
        H.estimate_lmax("rw")
    with pytest.raises(ValueError, match="Unknown Laplacian type"):
        H.heat_filter(X[:, 0], lap_type="rw")
    with pytest.raises(ValueError, match="kernel must be a callable"):
        H.filter(X[:, 0], "heat")
    with pytest.raises(ValueError, match="order >= 1"):
        H.filter(X[:, 0], np.exp, order=0)
