"""Graph signal filtering on the device: the Laplacian assembly (csrc/gsp.cu), the fused filter step
gtb_spmm_cheb_acc (csrc/spmm.cu), G.estimate_lmax and G.filter / G.heat_filter, against the numpy / scipy
restatement of pygsp 0.5 in tests/gsp_reference.py."""
import pickle
import warnings

import numpy as np
import pytest
import torch
from scipy import sparse
from scipy.sparse.csgraph import connected_components
from scipy.sparse.linalg import eigsh

import graphtools_b200 as gt
from graphtools_b200 import _engine as E
from graphtools_b200 import gsp, synth
from tests import gsp_reference as ref
from tests.test_diffusion_map_gpu import _random_csr

pytestmark = pytest.mark.gpu

LAP_TYPES = ["combinatorial", "normalized"]


def _graph(X, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return gt.Graph(X, verbose=0, **kw)


def _digits(n=None):
    from sklearn.datasets import load_digits
    return load_digits().data.astype(np.float32)[:n]


def _affinity(n, zero_diagonal=False, isolated=None):
    from scipy.spatial.distance import pdist, squareform
    D = squareform(pdist(_digits(n).astype(np.float64)))
    A = np.exp(-(D / np.median(D)) ** 2)
    A[A < 1e-3] = 0
    if zero_diagonal:
        np.fill_diagonal(A, 0)
    if isolated is not None:
        A[isolated, :] = 0
        A[:, isolated] = 0
    return A


def _mixture(n, seed=3):
    return synth.gaussian_mixture(n, 20, n_clusters=4, intrinsic_dim=10, seed=seed, center_scale=0.5)[0]


GRAPHS = {
    "digits": lambda: _graph(_digits(), knn=5, decay=40),
    "digits_binary": lambda: _graph(_digits(), knn=5, decay=None),
    "anisotropy": lambda: _graph(_digits(), knn=5, decay=40, anisotropy=1),
    "cosine": lambda: _graph(_digits(), knn=5, decay=40, distance="cosine"),
    "mnn": lambda: _graph(_digits(900), knn=5, decay=40, sample_idx=np.arange(900) % 3, kernel_symm="mnn",
                          theta=0.7),
    "exact_dense": lambda: _graph(_digits(700), graphtype="exact", knn=5, decay=40, thresh=0),
    "landmark": lambda: _graph(synth.gaussian_mixture(1500, 20, n_clusters=4, intrinsic_dim=5, seed=7)[0], knn=5,
                               decay=40, n_landmark=100, random_landmarking=True, random_state=1),
    "precomputed_zero_diagonal": lambda: _graph(_affinity(500, zero_diagonal=True), precomputed="affinity"),
    "isolated_vertex": lambda: _graph(_affinity(300, isolated=7), precomputed="affinity"),
}


# ------------------------------------------------------------------------------------------------ the kernel
@pytest.fixture(scope="module")
def csr():
    A = _random_csr(4000, 11)
    dev = torch.device("cuda")
    return A, (torch.from_numpy(A.indptr.astype(np.int64)).to(dev), torch.from_numpy(A.indices).to(dev),
               torch.from_numpy(A.data).to(dev))


def _acc(Ad, n, Y, Z, alpha, beta, gamma, out, coef, R):
    indptr, idx, val = Ad
    E.call("gtb_spmm_cheb_acc", indptr, idx, val, n, Y, Y.stride(0), Y.shape[1], alpha, beta, gamma, Z, Z.stride(0),
           out, out.stride(0), coef, coef.shape[0], R, R.stride(1), R.stride(0))


@pytest.mark.parametrize("f", [1, 2, 3, 8, 17, 33, 64, 65, 130])
@pytest.mark.parametrize("F", [1, 3, 8])
def test_fused_step_bit_identical_to_scipy_and_numpy(csr, f, F):
    A, Ad = csr
    n = A.shape[0]
    rng = np.random.default_rng(f * 10 + F)
    Yh, Zh, R0 = rng.normal(size=(n, f)), rng.normal(size=(n, f)), rng.normal(size=(F, n, f))
    ch = rng.normal(size=F)
    coef = torch.from_numpy(ch).cuda()
    for alpha, beta, gamma in [(1.0, 0.0, -1.0), (0.83, -0.41, 0.27)]:
        S = alpha * (A @ Yh) + beta * Yh + gamma * Zh
        want = [R0[a] + ch[a] * S for a in range(F)]
        Y, Z = torch.from_numpy(Yh).cuda(), torch.from_numpy(Zh).cuda()
        Rbuf = torch.full((F, n, f + 3), np.nan, dtype=torch.float64, device="cuda")   # ldr > f, stride > n ldr
        R = Rbuf[:, :, :f]
        R.copy_(torch.from_numpy(R0))
        out = torch.full((n, f), np.nan, dtype=torch.float64, device="cuda")
        _acc(Ad, n, Y, Z, alpha, beta, gamma, out, coef, R)
        assert np.array_equal(out.cpu().numpy(), S)
        for a in range(F):
            assert np.array_equal(R[a].cpu().numpy(), want[a])
        assert torch.isnan(Rbuf[:, :, f:]).all()
        R.copy_(torch.from_numpy(R0))
        _acc(Ad, n, Y, Z, alpha, beta, gamma, Z, coef, R)                        # out aliasing Z
        assert np.array_equal(Z.cpu().numpy(), S)
        for a in range(F):
            assert np.array_equal(R[a].cpu().numpy(), want[a])


def test_fused_step_rejects_overlaps(csr):
    A, Ad = csr
    n, f = A.shape[0], 8
    dev = "cuda"
    Y, Z, out = (torch.randn((n, f), dtype=torch.float64, device=dev) for _ in range(3))
    coef = torch.ones(3, dtype=torch.float64, device=dev)
    R = torch.zeros((3, n, f), dtype=torch.float64, device=dev)
    for what, RR in [("Y", Y), ("Z", Z), ("out", out)]:
        with pytest.raises(E.EngineError, match="R must not overlap"):
            _acc(Ad, n, Y, Z, 1.0, 0.0, -1.0, out, coef[:1], RR.reshape(1, n, f))
    big = torch.zeros((n + 1, f), dtype=torch.float64, device=dev)
    with pytest.raises(E.EngineError, match="R must not overlap"):
        _acc(Ad, n, Y, Z, 1.0, 0.0, -1.0, big[:n], coef[:1], big[1:].reshape(1, n, f))
    with pytest.raises(E.EngineError, match="blocks of R overlap"):
        _acc(Ad, n, Y, Z, 1.0, 0.0, -1.0, out, coef, torch.as_strided(R, (3, n, f), (f, f, 1)))
    with pytest.raises(E.EngineError, match="coef must not overlap"):
        _acc(Ad, n, Y, Z, 1.0, 0.0, -1.0, out, R.reshape(-1)[:3], R)
    with pytest.raises(E.EngineError, match="out must not overlap Y"):
        _acc(Ad, n, Y, Z, 1.0, 0.0, -1.0, Y, coef, R)
    with pytest.raises(E.EngineError, match="Z itself"):
        _acc(Ad, n, Y, big[:n], 1.0, 0.0, -1.0, big[1:], coef, R)


# ------------------------------------------------------------------------------------------------ the Laplacian
def _host_kernel(G):
    return sparse.csr_matrix(G.K)


@pytest.mark.parametrize("name", list(GRAPHS))
def test_laplacian_matches_restatement(name):
    G = GRAPHS[name]()
    if name == "exact_dense":
        assert isinstance(G.K, np.ndarray)
    if name == "landmark":
        assert type(G).__name__ == "kNNLandmarkGraph"
    K = _host_kernel(G)
    if name == "precomputed_zero_diagonal":
        assert (K.diagonal() == 0).all()                   # every diagonal entry of L is inserted
    dw_ref = ref.degrees(K)
    W = K - sparse.diags(K.diagonal())
    for lap_type in LAP_TYPES:
        L = G.laplacian(lap_type)
        L_ref, _ = ref.laplacian(K, lap_type)
        assert isinstance(L, sparse.csr_matrix) and L.dtype == np.float64
        assert L.indices.dtype == np.int32 and L.has_sorted_indices
        assert np.array_equal(L.indptr, L_ref.indptr) and np.array_equal(L.indices, L_ref.indices)
        assert abs(L - L_ref).max() == 0
        dw = gsp.laplacian_device(G, lap_type)[1].cpu().numpy()
        assert np.array_equal(dw, dw_ref)
        assert np.abs(dw - np.asarray(W.sum(axis=1)).ravel()).max() <= 1e-14 * max(dw.max(), 1.0)
    if name == "isolated_vertex":
        assert dw_ref[7] == 0
        for lap_type in LAP_TYPES:
            L = G.laplacian(lap_type)
            assert L.indptr[8] - L.indptr[7] == 1 and L[7, 7] == 0 and L.has_sorted_indices


# ------------------------------------------------------------------------------------------------ the filter
@pytest.fixture(scope="module")
def digits_graph():
    return GRAPHS["digits"]()


def _reference_filter(G, lap_type, s, kernels, order, lmax):
    L_ref, _ = ref.laplacian(_host_kernel(G), lap_type)
    c = np.stack([ref.cheby_coeff(h, order, lmax) for h in kernels])
    return ref.cheby_op(L_ref, c, s, lmax)


@pytest.mark.parametrize("lap_type", LAP_TYPES)
@pytest.mark.parametrize("order", [1, 2, 30, 50])
@pytest.mark.parametrize("width", [None, 20])
def test_heat_filter_bit_identical_to_cheby_op(digits_graph, lap_type, order, width):
    G = digits_graph
    n = G.K.shape[0]
    rng = np.random.default_rng(order)
    s = rng.normal(size=n if width is None else (n, width))
    lmax = G.estimate_lmax(lap_type)
    taus = [1.0, 10.0, 30.0, 60.0]
    want = _reference_filter(G, lap_type, s, [ref.heat(t, lmax) for t in taus], order, lmax)
    got = G.heat_filter(s, tau=10.0, order=order, lap_type=lap_type)
    assert got.shape == s.shape and np.array_equal(got, want[1])
    bank = G.heat_filter(s, tau=taus, order=order, lap_type=lap_type)
    assert bank.shape == s.shape + (4,)
    for i in range(4):
        assert np.array_equal(bank[..., i], want[i])


def test_filter_with_own_kernels_and_device_output(digits_graph):
    G = digits_graph
    n = G.K.shape[0]
    labels = np.random.default_rng(0).integers(0, 3, size=n)
    onehot = np.eye(3)[labels]
    kernels = [lambda x: 1 / (1 + 2 * x), lambda x: np.exp(-x ** 2)]
    lmax = 1.5 * G.estimate_lmax()
    want = _reference_filter(G, "combinatorial", onehot, kernels, 30, lmax)
    got = G.filter(torch.from_numpy(onehot).cuda(), kernels, order=30, lmax=lmax, return_device=True)
    assert isinstance(got, torch.Tensor) and got.is_cuda and tuple(got.shape) == (n, 3, 2)
    for i in range(2):
        assert np.array_equal(got[..., i].cpu().numpy(), want[i])
    single = G.filter(onehot, kernels[0], order=30, lmax=lmax)
    assert np.array_equal(single, want[0])


def test_meld_style_heat_filter_on_200k_connected_mixture():
    G = _graph(_mixture(200000), knn=5, decay=40)
    K = _host_kernel(G)
    assert connected_components(K, directed=False)[0] == 1
    labels = np.random.default_rng(1).integers(0, 4, size=K.shape[0])
    onehot = np.eye(4)[labels]
    lmax = G.estimate_lmax()
    got = G.heat_filter(onehot, tau=60, order=50)
    want = _reference_filter(G, "combinatorial", onehot, [ref.heat(60, lmax)], 50, lmax)[0]
    assert np.array_equal(got, want)


# ------------------------------------------------------------------------------------------------ the bound
@pytest.mark.parametrize("name", ["digits", "mixture_10k"])
def test_estimate_lmax_brackets_the_top_eigenvalue(name, digits_graph):
    G = digits_graph if name == "digits" else _graph(_mixture(10000), knn=5, decay=40)
    for lap_type in LAP_TYPES:
        lam = eigsh(G.laplacian(lap_type), k=1, which="LA", tol=1e-12)[0][0]
        lmax = G.estimate_lmax(lap_type)
        assert isinstance(lmax, float) and lam <= lmax <= 1.02 * lam
        assert gsp.estimate_lmax(G, lap_type) == lmax                     # reproducible from call to call
        st = gsp.stats()
        assert 1 <= st["lanczos_steps"] <= gsp.LANCZOS_MAX_STEPS
        assert G.__dict__["_lmax"][lap_type] == lmax


def test_caches_pickle_and_use_pygsp(digits_graph):
    G = digits_graph
    G.laplacian("normalized")
    lmax = G.estimate_lmax("normalized")
    assert "normalized" in G.__dict__["_dev_laplacian"]
    H = pickle.loads(pickle.dumps(G))
    assert "_dev_laplacian" not in H.__dict__ and H.__dict__["_lmax"]["normalized"] == lmax
    assert abs(H.laplacian("normalized") - G.laplacian("normalized")).max() == 0
    with pytest.raises(NotImplementedError):
        gt.Graph(_digits(200), knn=5, use_pygsp=True, verbose=0)


def test_errors_on_the_device(digits_graph):
    G = digits_graph
    n = G.K.shape[0]
    with pytest.raises(ValueError, match="n_samples"):
        G.heat_filter(np.ones(n + 1))
    with pytest.raises(ValueError, match=r"shape \[N\] or \[N, f\]"):
        G.heat_filter(np.ones((n, 2, 2)))
    s = np.ones(n)
    s[5] = np.nan
    with pytest.raises(ValueError, match="non-finite"):
        G.filter(s, np.exp)
    with pytest.raises(ValueError, match="lmax > 0"):
        G.filter(np.ones(n), np.exp, lmax=0.0)
    with pytest.raises(ValueError, match="returned non-finite"):
        G.filter(np.ones(n), lambda x: np.full_like(x, np.nan))
    with pytest.raises(ValueError, match="returned shape"):
        G.filter(np.ones(n), lambda x: x[:3])
    with pytest.raises(ValueError, match="kernel_symm=None"):
        _graph(_digits(300), knn=5, decay=40, kernel_symm=None).heat_filter(np.ones(300))
    E_ = _graph(np.eye(50), precomputed="affinity")               # a graph without edges
    assert E_.estimate_lmax() == 0.0 and E_.estimate_lmax("normalized") == 0.0
    with pytest.raises(ValueError, match="lmax > 0"):
        E_.heat_filter(np.ones(50))
