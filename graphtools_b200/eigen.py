"""Leading eigenpairs of the diffusion operator on the device: ``G.diffusion_eigs(k)`` and ``G.diffusion_map``.

P = D^-1 K is similar to the symmetric A = D^-1/2 K D^-1/2 (``G.diff_aff``): for every eigenpair (w, phi) of A,
psi = D^-1/2 phi is a right eigenvector of P with the same eigenvalue, and orthonormal phi give psi^T D psi = I.
Diffusion maps, spectral clustering and Laplacian eigenmaps need the top of that spectrum, which for a kNN graph
sits just below 1 -- a Krylov-type method needs many operator products there, and those products are what the
device is good at.

The solver is block Chebyshev-filtered subspace iteration (ChFSI; Zhou & Saad 2007) on A.  The spectrum of A lies
in [-1, 1] and its top eigenvalue is exactly 1 with eigenvector sqrt(d), so no spectral bound has to be estimated;
a block handles the eigenvalue 1 of a disconnected graph (one per component) and tight clusters near 1.  Every
outer iteration

1. orthonormalises the block (``spectral._cholesky_qr``, CholeskyQR2),
2. forms W = A Q and H = Q^T W, symmetrised as (H + H^T) / 2 (the ``diff_aff`` values can be asymmetric by an ulp),
3. computes eigh(H), the Ritz vectors and their residual norms ||A x_i - theta_i x_i||_2,
4. stops when the top k residuals are <= tol (||A||_2 = 1, so the tolerance is relative), and otherwise applies a
   degree-m Chebyshev filter that damps [-1, c] and scales the polynomial to 1 at the top of the spectrum.

Each filter step is one call of ``gtb_spmm_cheb`` (csrc/spmm.cu): Y_{j+1} = alpha_j (A Y_j) + beta_j Y_j +
gamma_j Y_{j-1}, the scaled three-term recurrence, rotating two buffers.  The rules, fixed here:

* block width b = k + max(8, k // 2), rounded up to a multiple of 8 (whole double2 lane pairs in the kernel),
  capped at N;
* start block: column 0 is sqrt(d), the eigenvector of eigenvalue 1 (exact for a connected graph, inside the
  eigenspace otherwise); the other columns are standard normal, drawn on the device from a ``torch.Generator``
  seeded with ``spectral._seed_of(random_state)``;
* cut c = the smallest Ritz value of the block, clamped to [CUT_MIN, CUT_MAX].  The upper clamp keeps the filter
  working when the whole block already sits at 1 (more components than columns): damping [-1, theta_b] with
  theta_b within rounding of 1 would damp nothing;
* degree m = the largest degree <= DEGREE_MAX whose amplification T_m(s0) of the top of the spectrum over the cut
  stays <= GROWTH_MAX (at least 1).  That bounds the condition number the filter gives the block, which CholeskyQR2
  needs to be below ~1e8;
* ``maxiter`` counts outer iterations (Rayleigh-Ritz steps); the default is DEFAULT_MAXITER.

The solver takes the filter step as a callable so that the CPU tests can run it with a torch product; the product
path always passes the CUDA kernel.  It is not sharded: a row-sharded build gathers its kernel on the local GPU
first, as ``G.diffuse`` does.
"""
import math
import numbers

import numpy as np
import torch

from . import _engine as E
from . import pipeline
from .pca import _svd_flip_v
from .spectral import _cholesky_qr, _seed_of, diff_aff_values

CUT_MIN = -0.9
CUT_MAX = 1.0 - 1e-3
GROWTH_MAX = 1e4
DEGREE_MAX = 64
DEFAULT_MAXITER = 1000
_STATS = {}


class NoConvergence(RuntimeError):
    """The top k Ritz pairs did not all reach the tolerance within ``maxiter`` outer iterations."""

    def __init__(self, n_converged, k, max_residual, iterations):
        super().__init__("diffusion eigenpairs: {} of {} pairs converged after {} iterations; largest residual "
                         "{:.3e}".format(n_converged, k, iterations, max_residual))
        self.n_converged, self.k, self.max_residual, self.iterations = n_converged, k, max_residual, iterations


def stats():
    """Counters of the last solve: n, nnz, block width, outer iterations, filter steps."""
    return dict(_STATS)


def block_width(k, n):
    return int(min(n, -(-(k + max(8, k // 2)) // 8) * 8))


def filter_degree(c):
    """Chebyshev degree for the cut c (see the module rules)."""
    s0 = (3.0 - c) / (1.0 + c)                       # the top of the spectrum, 1, on the interval's [-1, 1] scale
    return int(min(DEGREE_MAX, max(1, math.floor(math.acosh(GROWTH_MAX) / math.acosh(s0)))))


def cheb_coefficients(c, m):
    """(alpha, beta, gamma) of the m steps of the scaled recurrence that evaluates p_m(A) Y with
    p_m(t) = T_m((t - cc) / e) / T_m((1 - cc) / e), e = (c + 1) / 2, cc = (c - 1) / 2: |p_m| <= 1 / T_m(s0) on the
    damped interval [-1, c] and p_m(1) = 1.  Step j computes alpha (A Y_j) + beta Y_j + gamma Y_{j-1}."""
    e, cc = (c + 1.0) / 2.0, (c - 1.0) / 2.0
    sigma1 = e / (1.0 - cc)
    coef = [(sigma1 / e, -sigma1 * cc / e, 0.0)]
    tau, sigma = 2.0 / sigma1, sigma1
    for _ in range(1, m):
        s_new = 1.0 / (tau - sigma)
        coef.append((2.0 * s_new / e, -2.0 * s_new * cc / e, -sigma * s_new))
        sigma = s_new
    return coef


def chebyshev_filter(step, X, work, c, m):
    """p_m(A) X (module rules) by m filter steps.  Overwrites X and ``work``; returns the one holding the result."""
    cur, prev, out = X, X, work                      # first step: gamma = 0, Z is X itself
    for alpha, beta, gamma in cheb_coefficients(c, m):
        step(cur, prev, alpha, beta, gamma, out)
        prev, cur = cur, out
        out = prev                                   # the next step writes over Y_{j-1}, its own Z
    return cur


def chfsi(step, X, k, tol, maxiter):
    """Top k eigenpairs of the symmetric A with spectrum in [-1, 1] and top eigenvalue 1, by block Chebyshev-
    filtered subspace iteration from the start block X [n, b] (overwritten).

    ``step(Y, Z, alpha, beta, gamma, out)`` must write alpha (A Y) + beta Y + gamma Z into ``out``, which may be Z
    but never Y.  Returns (w float64 numpy [k] descending, phi [n, k] orthonormal, on X's device); raises
    NoConvergence."""
    n, b = X.shape
    W = torch.empty_like(X)
    work = torch.empty_like(X)
    _STATS.update(block=b, iterations=0, filter_steps=0)
    # row-major blocks throughout: the Householder fallback of _cholesky_qr returns a column-major Q
    Q = _cholesky_qr(X).contiguous()
    r = np.full(k, np.inf)
    for it in range(1, maxiter + 1):
        step(Q, Q, 1.0, 0.0, 0.0, W)                               # W = A Q
        H = Q.T @ W
        H = (H + H.T) * 0.5
        theta, S = np.linalg.eigh(H.cpu().numpy())
        theta, S = theta[::-1].copy(), torch.from_numpy(S[:, ::-1].copy()).to(X.device)
        X = Q @ S                                                  # Ritz vectors, descending Ritz values
        R = W @ S - X * torch.from_numpy(theta).to(X.device)
        r = torch.linalg.vector_norm(R[:, :k], dim=0).cpu().numpy()
        _STATS.update(iterations=it, max_residual=float(r.max()))
        if (r <= tol).all():
            return theta[:k], X[:, :k]
        if it == maxiter:
            break
        c = min(max(float(theta[-1]), CUT_MIN), CUT_MAX)
        m = filter_degree(c)
        Q = _cholesky_qr(chebyshev_filter(step, X, work, c, m)).contiguous()   # a new tensor: `work` is free
        _STATS["filter_steps"] += m
    raise NoConvergence(int((r <= tol).sum()), k, float(r.max()), maxiter)


def _cheb_step(K, vals):
    def step(Y, Z, alpha, beta, gamma, out):
        E.call("gtb_spmm_cheb", K.indptr, K.indices, vals, K.shape[0], Y, Y.stride(0), Y.shape[1], alpha, beta,
               gamma, Z, Z.stride(0), out, out.stride(0))
    return step


def diffusion_eigs(G, k=10, tol=1e-8, maxiter=None, random_state=None):
    """(w float64 [k] descending, psi float64 [N, k]): the k largest eigenvalues of P = D^-1 K and right
    eigenvectors psi = D^-1/2 phi, phi orthonormal eigenvectors of G.diff_aff; the entry of largest magnitude in
    every column of psi is positive."""
    if G.kernel_symm is None:
        raise ValueError("diffusion eigenpairs need a symmetric kernel; this graph was built with kernel_symm=None")
    G._ensure_built()
    K = G._dev_kernel
    if not isinstance(K, pipeline.DeviceCSR):
        from .paths import dense_to_csr
        K = dense_to_csr(K.contiguous())
    n = K.shape[0]
    if not isinstance(k, numbers.Integral) or not 1 <= k < n:
        raise ValueError("Expected 1 <= k < n_samples = {}. Got k = {}".format(n, k))
    if not tol > 0:
        raise ValueError("Expected tol > 0. Got {}".format(tol))
    maxiter = DEFAULT_MAXITER if maxiter is None else maxiter
    if not isinstance(maxiter, numbers.Integral) or maxiter < 1:
        raise ValueError("Expected an integer maxiter >= 1. Got {}".format(maxiter))
    degree = G._dev_degree
    zero = torch.nonzero(degree <= 0)
    if zero.shape[0]:
        raise ValueError("row {} of the kernel has zero degree: P = D^-1 K is undefined".format(int(zero[0, 0])))
    vals = diff_aff_values(K, degree)
    b = block_width(k, n)
    dev = degree.device
    gen = torch.Generator(device=dev)
    gen.manual_seed(_seed_of(random_state))
    X = torch.randn((n, b), dtype=torch.float64, device=dev, generator=gen)
    sqrt_d = torch.sqrt(degree)
    X[:, 0] = sqrt_d
    _STATS.clear()
    _STATS.update(n=n, nnz=K.nnz)
    w, phi = chfsi(_cheb_step(K, vals), X, k, tol, maxiter)
    _, psi_t = _svd_flip_v(phi, (phi / sqrt_d[:, None]).T)
    return w, psi_t.T.cpu().numpy()


def diffusion_map(G, n_components=2, t=1, tol=1e-8, maxiter=None, random_state=None):
    """Diffusion-map coordinates psi[:, 1:n+1] * w[1:n+1] ** t (Coifman & Lafon): the stationary pair is dropped."""
    if not isinstance(n_components, numbers.Integral) or n_components < 1:
        raise ValueError("Expected an integer n_components >= 1. Got {}".format(n_components))
    if not t >= 0:
        raise ValueError("Expected t >= 0. Got {}".format(t))
    w, psi = diffusion_eigs(G, n_components + 1, tol=tol, maxiter=maxiter, random_state=random_state)
    return psi[:, 1:] * w[1:] ** t
