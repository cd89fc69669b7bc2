"""numpy / scipy restatement of pygsp 0.5's graph-signal scheme, the oracle of tests/test_gsp_*.py:
``Graph.compute_laplacian`` on W = K without its diagonal, ``compute_cheby_coeff`` and ``cheby_op``, written out with
pygsp's operation order."""
import numpy as np
from scipy import sparse


def degrees(K):
    """dw: the off-diagonal values of every row of the CSR K added sequentially in column order, from +0.0 (a loop over
    row positions, vectorised across rows)."""
    K = sparse.csr_matrix(K)
    lens = np.diff(K.indptr)
    dw = np.zeros(K.shape[0])
    for t in range(int(lens.max())):
        live = np.flatnonzero(lens > t)
        p = K.indptr[live] + t
        keep = K.indices[p] != live
        dw[live[keep]] = dw[live[keep]] + K.data[p[keep]]
    return dw


def laplacian(K, lap_type):
    """L on K's off-diagonal pattern plus one diagonal entry per row (scipy CSR, sorted int32 indices)."""
    K = sparse.csr_matrix(K)
    n = K.shape[0]
    dw = degrees(K)
    rows = np.repeat(np.arange(n), np.diff(K.indptr))
    off = K.indices != rows
    r, c, w = rows[off], K.indices[off], K.data[off]
    if lap_type == "combinatorial":
        offv, diag = -w, dw
    else:
        with np.errstate(divide="ignore"):
            s = np.where(dw == 0, 0.0, 1.0 / np.sqrt(dw))
        offv, diag = -((s[r] * w) * s[c]), np.where(dw == 0, 0.0, 1.0)
    R = np.concatenate([r, np.arange(n)])
    C = np.concatenate([c, np.arange(n)])
    V = np.concatenate([offv, diag])
    order = np.lexsort((C, R))
    indptr = np.concatenate([[0], np.cumsum(np.bincount(R, minlength=n))]).astype(np.int32)
    L = sparse.csr_matrix((V[order], C[order].astype(np.int32), indptr), shape=(n, n))
    return L, dw


def cheby_coeff(h, m, lmax):
    """compute_cheby_coeff(f, m): c[0 .. m] for one kernel."""
    N = m + 1
    a1 = (lmax - 0) / 2
    a2 = (lmax + 0) / 2
    c = np.zeros(m + 1)
    tmpN = np.arange(N)
    num = np.cos(np.pi * (tmpN + 0.5) / N)
    for o in range(m + 1):
        c[o] = 2. / N * np.dot(h(a1 * num + a2), np.cos(np.pi * o * (tmpN + 0.5) / N))
    return c


def cheby_op(L, c, signal, lmax):
    """cheby_op(G, c, signal) for c [Nscales, M]: list of the Nscales results, each shaped like ``signal``."""
    c = np.atleast_2d(c)
    Nscales, M = c.shape
    a1 = float(lmax - 0) / 2.
    a2 = float(lmax + 0) / 2.
    twf_old = signal
    twf_cur = (L.dot(signal) - a2 * signal) / a1
    r = [0.5 * c[i, 0] * twf_old + c[i, 1] * twf_cur for i in range(Nscales)]
    factor = 2 / a1 * (L - a2 * sparse.eye(L.shape[0]))
    for k in range(2, M):
        twf_new = factor.dot(twf_cur) - twf_old
        for i in range(Nscales):
            r[i] += c[i, k] * twf_new
        twf_old = twf_cur
        twf_cur = twf_new
    return r


def heat(tau, lmax):
    return lambda x: np.exp(-tau * x / lmax)
