"""G.diffusion_eigs / G.diffusion_map on the device, and the Chebyshev filter-step kernel gtb_spmm_cheb.

The eigenpairs are checked on the host against scipy's eigsh on the graph's own diff_aff.  Single-vector Lanczos
finds one copy of a multiple eigenvalue at a time, and a disconnected graph has the eigenvalue 1 once per
component, so the reference runs eigsh on each connected component and merges the spectra."""
import math
import warnings

import numpy as np
import pytest
import torch
from scipy import sparse
from scipy.sparse.csgraph import connected_components
from scipy.sparse.linalg import eigsh

import graphtools_b200 as gt
from graphtools_b200 import _engine as E
from graphtools_b200 import eigen, synth

pytestmark = pytest.mark.gpu

TOL = 1e-10


def _graph(X, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return gt.Graph(X, verbose=0, **kw)


def _digits(n=None):
    from sklearn.datasets import load_digits
    return load_digits().data.astype(np.float32)[:n]


# ------------------------------------------------------------------------------------------------ the kernel
def _random_csr(n, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 24, size=n)
    lens[rng.random(n) < 0.1] = 0                             # empty rows
    lens[n // 3] = 1500                                       # one row longer than 1000
    rows = [np.sort(rng.choice(n, size=m, replace=False)) for m in lens]
    indptr = np.concatenate([[0], np.cumsum(lens)])
    A = sparse.csr_matrix((rng.normal(size=indptr[-1]), np.concatenate(rows).astype(np.int32), indptr), shape=(n, n))
    assert A.has_sorted_indices
    return A


@pytest.fixture(scope="module")
def csr():
    A = _random_csr(4000, 11)
    dev = torch.device("cuda")
    return A, (torch.from_numpy(A.indptr.astype(np.int64)).to(dev), torch.from_numpy(A.indices).to(dev),
               torch.from_numpy(A.data).to(dev))


def _cheb(Ad, n, Y, Z, alpha, beta, gamma, out):
    indptr, idx, val = Ad
    E.call("gtb_spmm_cheb", indptr, idx, val, n, Y, Y.stride(0), Y.shape[1], alpha, beta, gamma, Z, Z.stride(0), out,
           out.stride(0))


@pytest.mark.parametrize("b", [1, 2, 3, 8, 16, 17, 32, 33, 64, 100, 130])
@pytest.mark.parametrize("coef", [(1.37, 0.0, 0.0), (0.83, -0.41, 0.27), (-1.9, 0.0, 0.66), (2.5, 0.31, 0.0)])
def test_kernel_bit_identical_to_scipy_and_numpy(csr, b, coef):
    A, Ad = csr
    n = A.shape[0]
    rng = np.random.default_rng(b)
    Yh, Zh = rng.normal(size=(n, b)), rng.normal(size=(n, b))
    alpha, beta, gamma = coef
    ref = alpha * (A @ Yh) + beta * Yh + gamma * Zh
    Y, Z = torch.from_numpy(Yh).cuda(), torch.from_numpy(Zh).cuda()
    out = torch.full((n, b), np.nan, dtype=torch.float64, device="cuda")
    _cheb(Ad, n, Y, Z, alpha, beta, gamma, out)
    assert np.array_equal(out.cpu().numpy(), ref)
    _cheb(Ad, n, Y, Z, alpha, beta, gamma, Z)                 # out aliasing Z: the recurrence's buffer rotation
    assert np.array_equal(Z.cpu().numpy(), ref)


def test_kernel_rejects_out_overlapping_y(csr):
    A, Ad = csr
    n = A.shape[0]
    Y = torch.randn((n, 16), dtype=torch.float64, device="cuda")
    with pytest.raises(E.EngineError, match="overlap"):
        _cheb(Ad, n, Y, Y.clone(), 1.0, 0.5, 0.25, Y)
    big = torch.randn((n + 1, 16), dtype=torch.float64, device="cuda")
    with pytest.raises(E.EngineError, match="overlap"):
        _cheb(Ad, n, big[:n], big[1:].clone(), 1.0, 0.5, 0.25, big[1:])


def test_kernel_rejects_out_partially_overlapping_z(csr):
    A, Ad = csr
    n = A.shape[0]
    Y = torch.randn((n, 16), dtype=torch.float64, device="cuda")
    zbuf = torch.randn((n + 1, 16), dtype=torch.float64, device="cuda")
    with pytest.raises(E.EngineError, match="Z itself"):
        _cheb(Ad, n, Y, zbuf[:n], 1.0, 0.5, 0.25, zbuf[1:])       # shifted by one row
    wide = torch.randn((n, 32), dtype=torch.float64, device="cuda")
    with pytest.raises(E.EngineError, match="Z itself"):                # same pointer, other leading dimension
        _cheb(Ad, n, Y, wide[:, :16], 1.0, 0.5, 0.25, torch.as_strided(wide, (n, 16), (16, 1)))


# ------------------------------------------------------------------------------------------------ eigenpairs
def _reference(A, k):
    """Top k + 1 eigenpairs of the symmetric A: eigsh(which="LA", tol=1e-12) on each connected component."""
    A = sparse.csr_matrix(A)
    n_comp, lab = connected_components(A, directed=False)
    vals, vecs = [], []
    for c in range(n_comp):
        idx = np.flatnonzero(lab == c)
        B = A[idx][:, idx]
        kk = min(k + 1, len(idx))
        if len(idx) <= 2 * kk + 2:
            w, V = np.linalg.eigh(B.toarray())
            w, V = w[-kk:], V[:, -kk:]
        else:
            w, V = eigsh(B, kk, which="LA", tol=1e-12)
        full = np.zeros((A.shape[0], len(w)))
        full[idx] = V
        vals.append(w)
        vecs.append(full)
    w, V = np.concatenate(vals), np.concatenate(vecs, axis=1)
    order = np.argsort(-w, kind="stable")[:k + 1]
    return w[order], V[:, order], n_comp


def _sin_angle(U, V):
    """sin of the largest principal angle between the spans of the orthonormal U and V."""
    return float(np.linalg.norm(U - V @ (V.T @ U), 2))


def check_pairs(G, w, psi, k, tol=TOL, reference=True):
    n = G.kernel_degree.shape[0]
    assert w.shape == (k,) and w.dtype == np.float64 and psi.shape == (n, k) and psi.dtype == np.float64
    assert np.all(np.diff(w) <= 0)
    A = sparse.csr_matrix(G.diff_aff)
    d = G.kernel_degree.ravel()
    phi = np.sqrt(d)[:, None] * psi
    assert np.linalg.norm(A @ phi - phi * w, axis=0).max() <= tol * (1 + 1e-3)
    assert np.abs(phi.T @ phi - np.eye(k)).max() <= 1e-10
    piv = np.abs(psi).argmax(axis=0)
    assert np.all(psi[piv, np.arange(k)] > 0), "sign rule"
    if not reference:
        return
    lam, V, n_comp = _reference(A, k)
    assert np.abs(w - lam[:k]).max() <= 1e-10
    # groups of eigenvalues inside the top k that a gap separates from the rest of the spectrum
    lo = 0
    for hi in range(1, k + 1):
        if lam[hi - 1] - lam[hi] <= 1e-8:
            continue
        delta = min(lam[hi - 1] - lam[hi], lam[lo - 1] - lam[lo] if lo else np.inf)
        size = hi - lo
        assert _sin_angle(phi[:, lo:hi], V[:, lo:hi]) <= math.sqrt(size) * tol / delta + 1e-9, (lo, hi, delta)
        lo = hi
    if n_comp == 1:
        # the stationary pair: psi[:, 0] is constant, i.e. phi[:, 0] lies along sqrt(d) -- in the D-norm, as closely
        # as the gap to the second eigenvalue allows
        delta = lam[0] - lam[1]
        u = np.sqrt(d) / np.linalg.norm(np.sqrt(d))
        assert _sin_angle(phi[:, :1], u[:, None]) <= tol / delta + 1e-9


def _precomputed_affinity(n):
    from scipy.spatial.distance import pdist, squareform
    D = squareform(pdist(_digits(n).astype(np.float64)))
    return np.exp(-(D / np.median(D)) ** 2)


GRAPHS = {
    "digits": lambda: _graph(_digits(), knn=5, decay=40),
    "mixture_10k": lambda: _graph(synth.gaussian_mixture(10000, 20, n_clusters=4, intrinsic_dim=10, seed=3,
                                                         center_scale=0.5)[0], knn=5, decay=40),
    "anisotropy": lambda: _graph(_digits(), knn=5, decay=40, anisotropy=1),
    "cosine": lambda: _graph(_digits(), knn=5, decay=40, distance="cosine"),
    "mnn": lambda: _graph(_digits(900), knn=5, decay=40, sample_idx=np.arange(900) % 3, kernel_symm="mnn",
                          theta=0.7),
    "exact_dense": lambda: _graph(_digits(700), graphtype="exact", knn=5, decay=40, thresh=0),
    "precomputed": lambda: _graph(_precomputed_affinity(500), precomputed="affinity"),
    "landmark": lambda: _graph(synth.gaussian_mixture(1500, 20, n_clusters=4, intrinsic_dim=5, seed=7)[0], knn=5,
                               decay=40, n_landmark=100, random_landmarking=True, random_state=1),
}


@pytest.mark.parametrize("name", list(GRAPHS))
def test_eigenpairs_against_eigsh(name):
    G = GRAPHS[name]()
    if name == "exact_dense":
        assert isinstance(G.K, np.ndarray)
    if name == "landmark":
        assert type(G).__name__ == "kNNLandmarkGraph"
    if name == "mnn":
        assert type(G).__name__ == "MNNGraph"
    w, psi = G.diffusion_eigs(k=10, tol=TOL, random_state=0)
    check_pairs(G, w, psi, 10)
    assert abs(w[0] - 1) <= 1e-12


def test_disconnected_graph_gives_eigenvalue_one_per_component():
    rng = np.random.default_rng(3)
    X = np.concatenate([rng.normal(size=(400, 8)), rng.normal(size=(300, 8)) + 1000.0,
                        rng.normal(size=(350, 8)) - 1000.0]).astype(np.float32)
    G = _graph(X, knn=5, decay=40)
    n_comp, lab = connected_components(sparse.csr_matrix(G.K), directed=False)
    assert n_comp == 3
    w, psi = G.diffusion_eigs(k=6, tol=TOL, random_state=1)
    check_pairs(G, w, psi, 6)
    assert np.abs(w[:3] - 1).max() <= 1e-12 and w[3] < 1 - 1e-6
    d = G.kernel_degree.ravel()
    ind = np.stack([np.where(lab == c, np.sqrt(d), 0.0) for c in range(3)], axis=1)
    ind /= np.linalg.norm(ind, axis=0)
    phi = np.sqrt(d)[:, None] * psi[:, :3]
    assert _sin_angle(phi, ind) <= 1e-9


@pytest.fixture(scope="module")
def digits_graph():
    return GRAPHS["digits"]()


@pytest.mark.parametrize("t", [0, 1, 3])
def test_diffusion_map_is_scaled_eigenvectors(digits_graph, t):
    Y = digits_graph.diffusion_map(n_components=3, t=t, random_state=42)
    w, psi = digits_graph.diffusion_eigs(k=4, random_state=42)
    assert Y.shape == (psi.shape[0], 3)
    assert np.array_equal(Y, psi[:, 1:4] * w[1:4] ** t)


def test_same_random_state_is_bit_identical(digits_graph):
    w1, psi1 = digits_graph.diffusion_eigs(k=8, random_state=7)
    w2, psi2 = digits_graph.diffusion_eigs(k=8, random_state=7)
    assert np.array_equal(w1, w2) and np.array_equal(psi1, psi2)
    assert eigen.stats()["filter_steps"] > 0


def test_errors(digits_graph):
    G = _graph(_digits(300), knn=5, decay=40, kernel_symm=None)
    with pytest.raises(ValueError, match="kernel_symm=None"):
        G.diffusion_eigs(3)
    n = digits_graph.kernel_degree.shape[0]
    for k in (0, n, n + 5):
        with pytest.raises(ValueError, match="1 <= k < n_samples"):
            digits_graph.diffusion_eigs(k)
    with pytest.raises(ValueError, match="t >= 0"):
        digits_graph.diffusion_map(2, t=-1)
    A = _precomputed_affinity(60)
    A[7, :] = 0
    A[:, 7] = 0
    Gz = _graph(A, precomputed="affinity")
    with pytest.raises(ValueError, match="row 7 .*zero degree"):
        Gz.diffusion_eigs(3)
    with pytest.raises(eigen.NoConvergence) as err:
        digits_graph.diffusion_eigs(10, tol=1e-15, maxiter=1, random_state=0)
    assert err.value.n_converged < 10 and err.value.max_residual > 1e-15


def test_200k_connected_mixture():
    # overlapping clusters: one component, so the wanted eigenvalues sit just below 1 instead of all being 1
    X, _ = synth.gaussian_mixture(200000, 20, n_clusters=4, intrinsic_dim=10, seed=3, center_scale=0.5)
    G = _graph(X, knn=5, decay=40)
    assert connected_components(sparse.csr_matrix(G.K), directed=False)[0] == 1
    w, psi = G.diffusion_eigs(k=10, tol=TOL, random_state=0)
    check_pairs(G, w, psi, 10, reference=False)
