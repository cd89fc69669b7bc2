"""Graph signal processing on the device: ``G.laplacian``, ``G.estimate_lmax``, ``G.filter`` and ``G.heat_filter``.

These are the computations behind the reference's PyGSP bridge (``use_pygsp=True``, which stays out of scope): the
graph Laplacian, a bound on its largest eigenvalue and Chebyshev-approximated spectral filters of a block of signals
-- the heat filter of one-hot sample labels that MELD-style analyses run, for example.  The scheme is pygsp 0.5's
(``Graph.compute_laplacian``, ``Graph.estimate_lmax``, ``filters.approximations.compute_cheby_coeff`` and
``cheby_op``), with the same operation order, so a filter is bit-identical to that code on the host run with the same
lmax (signed zeros aside).

Laplacian (csrc/gsp.cu): W = K without its diagonal, dw_i = the sum of row i of W added sequentially in column order;
combinatorial L = D - W, normalized L = I - D^-1/2 W D^-1/2 with L_ij = -((s_i W_ij) s_j), s_i = 1 / sqrt(dw_i); a
vertex with dw_i = 0 gets s_i = 0 and L_ii = 0.  L stores K's off-diagonal pattern plus one diagonal entry per row.

Spectral bound, fixed here (pygsp's "Lanczos estimate times 1.01"):

* Lanczos on L with full reorthogonalisation (classical Gram-Schmidt, twice), from a standard normal vector drawn on
  the device from a ``torch.Generator`` seeded with LANCZOS_SEED, so the value is reproducible from call to call;
* it stops at step m when the top Ritz pair's residual beta_m |s_m| <= LANCZOS_RTOL * theta, at an invariant
  subspace (beta_m <= INVARIANT_RTOL * ||T_m||, or m = N), or after LANCZOS_MAX_STEPS steps;
* lmax = min(LMAX_FACTOR * theta, bound), bound = 2 for normalized and 2 max(dw) for combinatorial Laplacians
  (Gershgorin); the value is cached on the graph per Laplacian type.

Filter (pygsp's cheby_op, a1 = a2 = lmax / 2, M = order + 1 coefficients per kernel):

* coefficients on the host: c_o = 2 / M * sum_n h(a1 cos(pi (n + 1/2) / M) + a2) cos(pi o (n + 1/2) / M);
* T1 = (L s - a2 s) / a1: one ``gtb_spmm_cheb`` launch (1, -a2, 0) and a division;
* r = 0.5 c_0 s + c_1 T1 per kernel, and the factor values (2 / a1) (L_ij - [i = j] a2) on L's pattern: one-off
  elementwise operations in pygsp's rounding order;
* every step k = 2 ... order, T_k = factor T_{k-1} - T_{k-2} and r += c_k T_k for all kernels at once, is one
  ``gtb_spmm_cheb_acc`` launch (1, 0, -1), rotating two buffers.

The recurrence and Lanczos take the product as a callable, as ``eigen.chfsi`` does, so that the CPU tests can run them
with a torch product; the graph methods always pass the CUDA kernels.  Nothing here is sharded: a row-sharded build
gathers its kernel on the local GPU first (a collective call), as ``G.diffuse`` does.
"""
import numbers

import numpy as np
import torch

from . import _engine as E
from . import pipeline

LAP_TYPES = {"combinatorial": 0, "normalized": 1}
LANCZOS_SEED = 0
LANCZOS_RTOL = 1e-3
LANCZOS_MAX_STEPS = 200
INVARIANT_RTOL = 1e-12
LMAX_FACTOR = 1.01
_STATS = {}


def stats():
    """Counters of the last call: n, nnz of L, and for a bound Lanczos steps, residual, theta and the stop reason."""
    return dict(_STATS)


def check_lap_type(lap_type):
    if lap_type not in LAP_TYPES:
        raise ValueError("Unknown Laplacian type {}. Choose from 'combinatorial' or 'normalized'.".format(lap_type))


# ------------------------------------------------------------------------------------------------ the Laplacian
def _kernel_csr(G):
    if G.kernel_symm is None:
        raise ValueError("graph signal filtering needs a symmetric Laplacian; this graph was built with "
                         "kernel_symm=None")
    G._ensure_built()
    K = G._dev_kernel
    if not isinstance(K, pipeline.DeviceCSR):
        from .paths import dense_to_csr
        K = dense_to_csr(K.contiguous())
    return K


def laplacian_device(G, lap_type="combinatorial"):
    """(L DeviceCSR, dw float64 [N]) in HBM, cached on the graph under ``_dev_laplacian``."""
    check_lap_type(lap_type)
    cache = G.__dict__.setdefault("_dev_laplacian", {})
    if lap_type not in cache:
        K = _kernel_csr(G)
        n = K.shape[0]
        dw = pipeline._empty((n,), torch.float64)
        length = pipeline._empty((n,), torch.int32)
        E.call("gtb_laplacian_count", K.indptr, K.indices, K.data, n, dw, length)
        lptr = pipeline.exclusive_scan(length)
        nnz = int(lptr[-1].item())
        lidx = pipeline._empty((nnz,), torch.int32)
        lval = pipeline._empty((nnz,), torch.float64)
        E.call("gtb_laplacian_fill", K.indptr, K.indices, K.data, n, dw, lptr, LAP_TYPES[lap_type], lidx, lval)
        cache[lap_type] = (pipeline.DeviceCSR(lptr, lidx, lval, (n, n)), dw)
    return cache[lap_type]


def laplacian(G, lap_type="combinatorial"):
    return laplacian_device(G, lap_type)[0].to_scipy()


# ------------------------------------------------------------------------------------------------ the bound
def lanczos(matvec, v0, rtol=LANCZOS_RTOL, max_steps=LANCZOS_MAX_STEPS):
    """Top Ritz value of the symmetric operator behind ``matvec(v, out)`` (out = A v, both 1-D) by Lanczos with full
    reorthogonalisation from v0 (module rules).  Returns (theta, steps, residual, reason)."""
    n = v0.shape[0]
    m_max = min(int(max_steps), n)
    V = v0.new_empty((m_max, n))
    V[0] = v0 / torch.linalg.vector_norm(v0)
    w = torch.empty_like(v0)
    alpha, beta = [], []
    for j in range(m_max):
        matvec(V[j], w)
        a = float(torch.dot(V[j], w))
        w -= a * V[j]
        if j:
            w -= beta[-1] * V[j - 1]
        for _ in range(2):
            w -= V[:j + 1].T @ (V[:j + 1] @ w)
        b = float(torch.linalg.vector_norm(w))
        alpha.append(a)
        T = np.diag(alpha) + np.diag(beta, 1) + np.diag(beta, -1)
        ritz, S = np.linalg.eigh(T)
        theta, residual = float(ritz[-1]), b * abs(float(S[-1, -1]))
        if residual <= rtol * theta:
            return theta, j + 1, residual, "residual"
        if b <= INVARIANT_RTOL * float(np.abs(ritz).max()) or j + 1 == n:
            return theta, j + 1, residual, "invariant"
        if j + 1 == m_max:
            return theta, j + 1, residual, "max_steps"
        beta.append(b)
        V[j + 1] = w / b


def _matvec(L):
    def matvec(v, out):
        y, o = v.reshape(-1, 1), out.reshape(-1, 1)
        E.call("gtb_spmm_cheb", L.indptr, L.indices, L.data, L.shape[0], y, 1, 1, 1.0, 0.0, 0.0, y, 1, o, 1)
    return matvec


def estimate_lmax(G, lap_type="combinatorial"):
    """min(LMAX_FACTOR * theta, bound) (module rules); not cached here (``BaseGraph.estimate_lmax`` caches)."""
    L, dw = laplacian_device(G, lap_type)
    gen = torch.Generator(device=dw.device)
    gen.manual_seed(LANCZOS_SEED)
    v0 = torch.randn(L.shape[0], dtype=torch.float64, device=dw.device, generator=gen)
    theta, steps, residual, reason = lanczos(_matvec(L), v0)
    _STATS.clear()
    _STATS.update(n=L.shape[0], nnz=L.nnz, lanczos_steps=steps, residual=residual, theta=theta, stop=reason)
    return bound_lmax(theta, lap_type, float(dw.max()))


def bound_lmax(theta, lap_type, dw_max):
    """min(LMAX_FACTOR * theta, bound): bound = 2 (normalized) or 2 max(dw) (combinatorial)."""
    return min(LMAX_FACTOR * theta, 2.0 if lap_type == "normalized" else 2.0 * dw_max)


# ------------------------------------------------------------------------------------------------ the filter
def cheby_coeff(kernels, order, lmax):
    """pygsp's compute_cheby_coeff for each kernel: float64 [len(kernels), order + 1]."""
    m = order + 1
    a1 = (lmax - 0) / 2
    a2 = (lmax + 0) / 2
    tmpN = np.arange(m)
    num = np.cos(np.pi * (tmpN + 0.5) / m)
    c = np.zeros((len(kernels), m))
    for i, h in enumerate(kernels):
        y = np.asarray(h(a1 * num + a2), dtype=np.float64)
        if y.shape != (m,):
            raise ValueError("kernel {} returned shape {} for {} points; expected ({},)".format(i, y.shape, m, m))
        if not np.isfinite(y).all():
            raise ValueError("kernel {} returned non-finite values on [0, lmax]".format(i))
        for o in range(m):
            c[i, o] = 2. / m * np.dot(y, np.cos(np.pi * o * (tmpN + 0.5) / m))
    return c


def factor_values(L, a1, a2):
    """(2 / a1) (L_ij - [i = j] a2) on L's pattern, in pygsp's rounding order."""
    n = L.shape[0]
    rows = torch.repeat_interleave(torch.arange(n, device=L.data.device), L.indptr[1:] - L.indptr[:-1])
    diag = L.indices == rows
    vals = L.data.clone()
    vals[diag] = L.data[diag] - a2
    return (2 / a1) * vals


def cheby_op(step, L, s, c, lmax):
    """pygsp's cheby_op on the block s [N, f] (not modified) for the coefficients c [F, M]: R [F, N, f].

    ``step(vals, Y, Z, alpha, beta, gamma, out, coef=None, R=None)`` must write (alpha (A Y) + beta Y) + gamma Z
    into ``out`` (which may be Z, never Y), A = L's pattern with the values ``vals``; with ``coef`` (a [F] tensor on
    s's device) it then adds coef[a] * out into R[a] for every a."""
    F, m = c.shape
    a1 = float(lmax - 0) / 2.
    a2 = float(lmax + 0) / 2.
    old = s.clone()                                   # T0; the recurrence writes over it
    cur = torch.empty_like(s)
    step(L.data, old, old, 1.0, -a2, 0.0, cur)
    # a 0-dim tensor on the device: torch divides by a host scalar as a product with its reciprocal
    cur = cur / torch.tensor(a1, dtype=s.dtype, device=s.device)
    R = s.new_empty((F,) + tuple(s.shape))
    for i in range(F):
        R[i] = float(0.5 * c[i, 0]) * old + float(c[i, 1]) * cur
    if m > 2:
        vals = factor_values(L, a1, a2)
        coef = torch.from_numpy(np.ascontiguousarray(c[:, 2:].T)).to(s.device)
        for k in range(2, m):
            step(vals, cur, old, 1.0, 0.0, -1.0, old, coef[k - 2], R)
            old, cur = cur, old
    return R


def _device_step(L):
    def step(vals, Y, Z, alpha, beta, gamma, out, coef=None, R=None):
        n, f = Y.shape
        if coef is None:
            E.call("gtb_spmm_cheb", L.indptr, L.indices, vals, n, Y, Y.stride(0), f, alpha, beta, gamma, Z,
                   Z.stride(0), out, out.stride(0))
        else:
            E.call("gtb_spmm_cheb_acc", L.indptr, L.indices, vals, n, Y, Y.stride(0), f, alpha, beta, gamma, Z,
                   Z.stride(0), out, out.stride(0), coef, coef.shape[0], R, R.stride(1), R.stride(0))
    return step


def check_signal(signal, n):
    """Shape of a [N] or [N, f] signal (numpy-like or torch), with its finiteness checked."""
    shape = tuple(signal.shape) if isinstance(signal, torch.Tensor) else np.shape(signal)
    if len(shape) not in (1, 2):
        raise ValueError("Expected a signal of shape [N] or [N, f]. Got shape {}".format(shape))
    if shape[0] != n or (len(shape) == 2 and shape[1] == 0):
        raise ValueError("signal must have n_samples = {} rows and at least one column. Got shape {}"
                         .format(n, shape))
    finite = torch.isfinite(signal).all() if isinstance(signal, torch.Tensor) else \
        np.isfinite(np.asarray(signal, dtype=np.float64)).all()
    if not bool(finite):
        raise ValueError("signal has non-finite values")
    return shape


def check_kernels(kernel):
    """(list of kernels, bank?) for a callable or a list of callables."""
    bank = isinstance(kernel, (list, tuple))
    kernels = list(kernel) if bank else [kernel]
    if not kernels or not all(callable(h) for h in kernels):
        raise ValueError("kernel must be a callable h(lambda) or a non-empty list of them. Got {!r}".format(kernel))
    return kernels, bank


def check_order(order):
    if not isinstance(order, numbers.Integral) or isinstance(order, bool) or order < 1:
        raise ValueError("Expected an integer order >= 1. Got {}".format(order))


def check_lmax(lmax):
    lmax = float(lmax)
    if not (np.isfinite(lmax) and lmax > 0):
        raise ValueError("Expected a finite lmax > 0. Got {} (a graph without edges has nothing to filter)"
                         .format(lmax))
    return lmax


def arrange(R, one_d, bank):
    """R [F, N, f] in the caller's layout: the signal's shape, with a trailing axis of size F for a bank."""
    if one_d:
        return R[:, :, 0].T if bank else R[0, :, 0]
    return R.permute(1, 2, 0) if bank else R[0]


def filter(G, signal, kernel, order=30, lap_type="combinatorial", lmax=None, return_device=False):
    check_lap_type(lap_type)
    kernels, bank = check_kernels(kernel)
    check_order(order)
    L, _ = laplacian_device(G, lap_type)
    n = L.shape[0]
    shape = check_signal(signal, n)
    if isinstance(signal, torch.Tensor):
        x = signal.to(device=pipeline._dev(), dtype=torch.float64).reshape(n, -1).contiguous()
    else:
        x = pipeline.to_device(np.ascontiguousarray(np.asarray(signal, dtype=np.float64).reshape(n, -1)))
    lmax = check_lmax(G.estimate_lmax(lap_type) if lmax is None else lmax)
    c = cheby_coeff(kernels, order, lmax)
    R = cheby_op(_device_step(L), L, x, c, lmax)
    _STATS.clear()
    _STATS.update(n=n, nnz=L.nnz, f=x.shape[1], kernels=len(kernels), order=order, lmax=lmax, steps=order - 1)
    out = arrange(R, len(shape) == 1, bank).contiguous()
    return out if return_device else out.cpu().numpy()


def heat_kernel(tau, lmax):
    """pygsp's Heat: h(lambda) = exp(-tau lambda / lmax); a list of kernels for a sequence of tau."""
    try:
        taus = np.asarray(tau, dtype=np.float64)
    except (TypeError, ValueError):
        taus = np.zeros((0, 0))
    if taus.ndim > 1 or taus.size == 0:
        raise ValueError("Expected a number or a non-empty sequence of numbers for tau. Got {!r}".format(tau))
    kernels = [(lambda x, t=float(t): np.exp(-t * x / lmax)) for t in taus.ravel()]
    return kernels if taus.ndim == 1 else kernels[0]


def heat_filter(G, signal, tau=10, order=30, lap_type="combinatorial", lmax=None, return_device=False):
    check_lap_type(lap_type)
    if lmax is None:
        lmax = G.estimate_lmax(lap_type)
    return filter(G, signal, heat_kernel(tau, lmax), order=order, lap_type=lap_type, lmax=lmax,
                  return_device=return_device)
