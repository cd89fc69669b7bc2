"""The diffusion-map eigensolver (graphtools_b200/eigen.py) with a torch filter step on the host, against
numpy.linalg.eigh on dense symmetric matrices with spectrum in [-1, 1]; and the Chebyshev recurrence coefficients
against the scaled polynomial evaluated directly."""
import math

import numpy as np
import pytest
import torch
from numpy.polynomial import chebyshev

from graphtools_b200 import eigen

TOL = 1e-10


def _matrix(spectrum, seed):
    rng = np.random.default_rng(seed)
    V, _ = np.linalg.qr(rng.normal(size=(len(spectrum), len(spectrum))))
    A = (V * np.asarray(spectrum)) @ V.T
    return (A + A.T) / 2


def _host_step(A):
    def step(Y, Z, alpha, beta, gamma, out):
        assert out.data_ptr() != Y.data_ptr()
        out.copy_(alpha * (A @ Y) + beta * Y + gamma * Z)
    return step


def _solve(A, k, seed=0, maxiter=eigen.DEFAULT_MAXITER):
    n = A.shape[0]
    gen = torch.Generator().manual_seed(seed)
    X = torch.randn((n, eigen.block_width(k, n)), dtype=torch.float64, generator=gen)
    w, phi = eigen.chfsi(_host_step(torch.from_numpy(A)), X, k, TOL, maxiter)
    return w, phi.numpy()


def _principal_angle_sin(U, V):
    """sin of the largest principal angle between the spans of the orthonormal U and V: ||(I - V V^T) U||_2."""
    return float(np.linalg.norm(U - V @ (V.T @ U), 2))


def _check(A, k, w, phi):
    lam, V = np.linalg.eigh(A)
    lam, V = lam[::-1], V[:, ::-1]
    assert w.shape == (k,) and phi.shape == (A.shape[0], k)
    assert np.all(np.diff(w) <= 0)
    assert np.abs(w - lam[:k]).max() <= TOL
    assert np.linalg.norm(A @ phi - phi * w, axis=0).max() <= TOL
    assert np.abs(phi.T @ phi - np.eye(k)).max() <= TOL
    # every group of eigenvalues inside the top k that a gap delta separates from the rest of the spectrum
    lo = 0
    for hi in range(1, k + 1):
        delta = min(lam[hi - 1] - lam[hi], lam[lo - 1] - lam[lo] if lo else np.inf)
        if lam[hi - 1] - lam[hi] > 1e-6:
            size = hi - lo
            assert _principal_angle_sin(phi[:, lo:hi], V[:, lo:hi]) <= math.sqrt(size) * TOL / delta + 1e-9
            lo = hi


def test_clustered_eigenvalues_just_below_one():
    rng = np.random.default_rng(1)
    spec = np.concatenate([1 - 1e-4 * np.arange(6), 0.99 - 1.99 * rng.random(394)])
    A = _matrix(spec, 2)
    w, phi = _solve(A, 6)
    _check(A, 6, w, phi)
    assert eigen.stats()["filter_steps"] > 0


def test_multiple_eigenvalue_one():
    rng = np.random.default_rng(3)
    spec = np.concatenate([[1.0, 1.0, 1.0, 0.95, 0.9], 0.8 - 1.8 * rng.random(295)])
    A = _matrix(spec, 4)
    w, phi = _solve(A, 5)
    _check(A, 5, w, phi)
    assert np.abs(w[:3] - 1).max() <= 1e-12


def test_eigenvalues_near_minus_one_are_damped():
    rng = np.random.default_rng(5)
    spec = np.concatenate([[1.0, 0.6, 0.55, 0.5], -1 + 1e-3 * rng.random(150), 0.4 - 1.3 * rng.random(146)])
    A = _matrix(spec, 6)
    w, phi = _solve(A, 4)
    _check(A, 4, w, phi)
    assert w.min() > 0.45


def test_no_convergence_reports_progress():
    A = _matrix(np.concatenate([1 - 1e-4 * np.arange(6), np.linspace(0.99, -1, 194)]), 7)
    with pytest.raises(eigen.NoConvergence) as err:
        _solve(A, 6, maxiter=1)
    assert err.value.k == 6 and err.value.n_converged < 6 and err.value.max_residual > TOL
    assert isinstance(err.value, RuntimeError)


@pytest.mark.parametrize("c", [-0.9, -0.3, 0.2, 0.9, 0.99, eigen.CUT_MAX])
def test_recurrence_reproduces_scaled_chebyshev_polynomial(c):
    m = eigen.filter_degree(c)
    coef = eigen.cheb_coefficients(c, m)
    assert len(coef) == m and coef[0][2] == 0.0
    t = np.linspace(-1, 1, 2001)
    prev = cur = np.ones_like(t)
    for alpha, beta, gamma in coef:
        prev, cur = cur, alpha * (t * cur) + beta * cur + gamma * prev
    e, cc = (c + 1) / 2, (c - 1) / 2
    direct = chebyshev.chebval((t - cc) / e, [0] * m + [1]) / chebyshev.chebval((1 - cc) / e, [0] * m + [1])
    np.testing.assert_allclose(cur, direct, rtol=1e-9, atol=1e-12)
    assert abs(cur[-1] - 1) < 1e-12                        # scaled to 1 at the top of the spectrum
    damped = t <= c
    growth = math.cosh(m * math.acosh((3 - c) / (1 + c)))
    assert np.abs(cur[damped]).max() <= 1 / growth * (1 + 1e-9)
    assert growth <= eigen.GROWTH_MAX or m == 1


def test_block_width_and_degree_rules():
    assert eigen.block_width(10, 10 ** 6) == 24
    assert eigen.block_width(11, 10 ** 6) == 24
    assert eigen.block_width(40, 10 ** 6) == 64
    assert eigen.block_width(5, 9) == 9
    assert 1 <= eigen.filter_degree(eigen.CUT_MIN) <= eigen.filter_degree(0.5) <= eigen.filter_degree(eigen.CUT_MAX)
    assert eigen.filter_degree(eigen.CUT_MAX) == eigen.DEGREE_MAX
