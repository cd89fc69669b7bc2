"""Spectral landmark selection on the device (SURVEY section 8f rank 1; reference graphtools/graphs.py:1216-1230).

The reference clusters the samples with scikit-learn on the host:
``randomized_svd(diff_aff, n_svd)`` -> ``MiniBatchKMeans(n_landmark, init_size=3 n_landmark, n_init=1,
batch_size=10000).fit_predict(diff_op . VT^T)``.  At 1M samples that is minutes of single-node CPU time, two orders
of magnitude more than the whole kernel build on the GPU.  This module runs the same two algorithms in HBM:

* randomized range finder + SVD (Halko et al., as in sklearn.utils.extmath.randomized_svd: ``n_oversamples=10``,
  ``n_iter = 7 if n_svd < 0.1 N else 4``, one normalisation per product, sign convention of ``svd_flip``).  The
  sparse products ``diff_aff . Q`` are csrc/spmm.cu (diff_aff is symmetric, so ``A^T Q = A Q`` and ``Q^T A =
  (A Q)^T``); the tall-skinny normalisations are Cholesky-QR on 110 x 110 Gram matrices (plain library
  GEMM / Cholesky calls).
* mini-batch k-means with sklearn's hyper-parameters and stopping rule (k-means++ on ``init_size`` samples, EWA
  inertia with ``max_no_improvement=10``, low-count centre reassignment every ``10 n_clusters`` samples); the
  assignment step -- nearest centre of every batch sample, and the final labelling of all N samples -- is the fused
  distance / top-1 kernel (exact float64 argmin).

Random streams (``GTB_SPECTRAL_RNG``): ``numpy`` (default) draws every random number on the HOST from the same
``numpy.random.RandomState(seed)`` streams, in the same order, as scikit-learn does -- the Gaussian test matrix of
``randomized_svd`` ([N, n_svd + 10]: 3.7 s of single-thread MT19937 at 1M samples, the price of starting from the
reference's own matrix), the validation / init subsets, the k-means++ draws, every mini-batch and every
reassignment of ``MiniBatchKMeans``.  The run then follows the reference's trajectory up to floating-point
summation order: V agrees with sklearn's to rounding and the clusters agree except for samples that sit on a
boundary (tests/test_spectral_gpu.py reports the agreement).  ``torch`` uses device generators instead (no host
draw; same algorithms, unrelated clusters).  The host path (``GTB_SPECTRAL=host``) stays the bit-exact pin; this
path is selected with ``GTB_SPECTRAL=device`` and by ``auto`` above landmark.SPECTRAL_AUTO_N samples.
"""
import math

import numpy as np
import torch

from . import _engine as E
from . import pipeline


def rng_mode():
    import os
    mode = os.environ.get("GTB_SPECTRAL_RNG", "numpy")
    if mode not in ("numpy", "torch"):
        raise ValueError("GTB_SPECTRAL_RNG must be numpy or torch (got %r)" % (mode,))
    return mode


def _check_random_state(seed):
    from sklearn.utils import check_random_state
    return check_random_state(seed)


class _Draws:
    """The random draws of the two algorithms behind one interface: numpy RandomState on the host (scikit-learn's
    streams and call order) or torch device generators."""

    def __init__(self, random_state, mode, salt=0):
        self.mode = mode
        self.dev = pipeline._dev()
        if mode == "numpy":
            self.rs = _check_random_state(random_state)
        else:
            self.gen = torch.Generator(device=self.dev)
            self.gen.manual_seed(_seed_of(random_state) + salt)

    def normal(self, n, k):
        if self.mode == "numpy":
            return torch.from_numpy(self.rs.normal(size=(n, k))).to(self.dev)
        return torch.randn((n, k), dtype=torch.float64, device=self.dev, generator=self.gen)

    def randint(self, high, size):
        if self.mode == "numpy":
            return torch.from_numpy(self.rs.randint(0, high, size)).to(self.dev)
        return torch.randint(0, high, (size,), device=self.dev, generator=self.gen)

    def first_center(self, n):
        if self.mode == "numpy":          # random_state.choice(n, p=sample_weight / sample_weight.sum())
            return int(self.rs.choice(n, p=np.full(n, 1.0 / n)))
        return int(torch.randint(0, n, (1,), device=self.dev, generator=self.gen).item())

    def uniform(self, size):
        if self.mode == "numpy":
            return torch.from_numpy(self.rs.uniform(size=size)).to(self.dev)
        return torch.rand((size,), dtype=torch.float64, device=self.dev, generator=self.gen)

    def choice_no_replace(self, n, size):
        if self.mode == "numpy":
            return torch.from_numpy(self.rs.choice(n, replace=False, size=size)).to(self.dev)
        return torch.randperm(n, device=self.dev, generator=self.gen)[:size]


def _seed_of(random_state):
    if random_state is None:
        return int(np.random.SeedSequence().entropy % (2 ** 31))
    if isinstance(random_state, np.random.RandomState):
        return int(random_state.randint(0, 2 ** 31 - 1))
    return int(random_state) % (2 ** 31)


def _cholesky_qr(A, passes=2):
    """Orthonormal basis of the columns of tall-skinny ``A`` [n, k] (k ~ 110): Q = A R^-1 with R from the Cholesky
    factor of the k x k Gram matrix, applied twice (CholeskyQR2) so the loss of orthogonality of the first pass
    (kappa^2 eps) is removed.  R^-1 is formed explicitly (k x k triangular solve against the identity) so the tall
    operand only ever goes through GEMMs.  Falls back to Householder QR when the Gram matrix is numerically
    singular."""
    Q = A
    k = A.shape[1]
    eye = torch.eye(k, dtype=A.dtype, device=A.device)
    for _ in range(passes):
        G = Q.T @ Q
        L, info = torch.linalg.cholesky_ex(G)
        if int(info.item()) != 0:
            return torch.linalg.qr(A, mode="reduced")[0]
        Rinv = torch.linalg.solve_triangular(L.T, eye, upper=True)        # R = L^T, Q = A R^-1
        Q = Q @ Rinv
    return Q


def diff_aff_values(K, degree):
    """Values of D^-1/2 K D^-1/2 on K's structure (base.py:668-698)."""
    vals = K.data.clone()
    E.call("gtb_anisotropy", K.indptr, K.indices, vals, degree, 0.5, K.shape[0])
    return vals


def randomized_svd_vt(K, degree, n_components, random_state=None, n_oversamples=10, n_iter="auto"):
    """(singular values [n_components], VT [n_components, N]) of diff_aff = D^-1/2 K D^-1/2, device tensors."""
    return randomized_svd_sym(K, diff_aff_values(K, degree), n_components, random_state, n_oversamples, n_iter)


def randomized_svd_sym(K, A, n_components, random_state=None, n_oversamples=10, n_iter="auto"):
    """Randomized SVD of the SYMMETRIC sparse matrix with K's structure and values ``A`` (None = K's own)."""
    n = K.shape[0]
    k = int(min(n_components + n_oversamples, n))
    if n_iter == "auto":
        n_iter = 7 if n_components < 0.1 * n else 4
    Q = _Draws(random_state, rng_mode()).normal(n, k)     # sklearn: random_state.normal(size=(A.shape[1], k))
    for _ in range(int(n_iter)):
        Q = _cholesky_qr(pipeline.spmm(K, Q, A), passes=1)      # A Q
        Q = _cholesky_qr(pipeline.spmm(K, Q, A), passes=1)      # A^T Q (A symmetric)
    Q = _cholesky_qr(pipeline.spmm(K, Q, A), passes=2)
    Bt = pipeline.spmm(K, Q, A)                                  # B^T = A^T Q = A Q   [N, k]
    # thin SVD of B = Bt^T through a QR of Bt:  Bt = Q2 R2  ->  B = R2^T Q2^T = Uh S (Q2 W)^T
    Q2 = _cholesky_qr(Bt, passes=2)
    R2 = Q2.T @ Bt
    Uh, s, Wt = torch.linalg.svd(R2.T, full_matrices=False)
    Vt = (Q2 @ Wt.T).T                                           # [k, N]
    # svd_flip (u-based): the largest-magnitude entry of every left singular vector is positive
    U = Q @ Uh
    piv = U.abs().argmax(dim=0)
    signs = torch.sign(U[piv, torch.arange(k, device=U.device)])
    signs[signs == 0] = 1.0
    Vt = Vt * signs[:, None]
    return s[:n_components], Vt[:n_components].contiguous()


# ----------------------------------------------------------------------------------------------- k-means
def assign_nearest(X, centers):
    """Index of the nearest centre of every row of X (float64 [n, d]) -- the fused distance / top-1 kernel with the
    exact float64 re-evaluation -- and the squared distance to it."""
    ref = pipeline.SearchOperand(centers.contiguous())
    qry = pipeline.SearchOperand(X, mean=ref.mean)
    nearest, _ = pipeline.knn_kernel(ref, qry, knn=1, decay=None)
    labels = nearest.indices.to(torch.int64)
    d2 = ((X - centers[labels]) ** 2).sum(dim=1)
    return labels, d2


def _kmeans_plusplus(X, n_clusters, draws):
    """k-means++ seeding with sklearn's greedy local trials (2 + log k candidates per step;
    sklearn.cluster._kmeans._kmeans_plusplus, same draws in the same order)."""
    n = X.shape[0]
    dev = X.device
    n_trials = 2 + int(math.log(n_clusters))
    centers = torch.empty((n_clusters, X.shape[1]), dtype=X.dtype, device=dev)
    first = draws.first_center(n)
    centers[0] = X[first]
    closest = ((X - X[first]) ** 2).sum(dim=1)
    xn = (X * X).sum(dim=1)
    for c in range(1, n_clusters):
        pot = closest.sum()
        r = draws.uniform(n_trials) * pot
        cand = torch.searchsorted(torch.cumsum(closest, 0), r).clamp_(max=n - 1)
        Xc = X[cand]                                                         # [t, d]
        d2 = (xn[None, :] + (Xc * Xc).sum(dim=1)[:, None] - 2.0 * (Xc @ X.T)).clamp_(min=0)
        d2 = torch.minimum(d2, closest[None, :])
        best = torch.argmin(d2.sum(dim=1))
        closest = d2[best]
        centers[c] = Xc[best]
    return centers


def minibatch_kmeans(X, n_clusters, init_size=None, batch_size=10000, max_iter=100, max_no_improvement=10,
                     reassignment_ratio=0.01, random_state=None):
    """Labels [N] (int64 device tensor) and centres of a mini-batch k-means run with sklearn's schedule."""
    n, d = X.shape
    dev = X.device
    draws = _Draws(random_state, rng_mode(), salt=1)     # sklearn: check_random_state(self.random_state), a fresh stream
    batch_size = int(min(batch_size, n))
    init_size = int(min(n, max(3 * batch_size if init_size is None else init_size, n_clusters)))
    draws.randint(n, init_size)                          # validation_indices: drawn first, only scores the n_init runs
    init_idx = draws.randint(n, init_size) if init_size < n else torch.arange(n, device=dev)
    centers = _kmeans_plusplus(X[init_idx], n_clusters, draws)
    counts = torch.zeros((n_clusters,), dtype=torch.float64, device=dev)
    n_steps = (max_iter * n) // batch_size
    ewa = ewa_min = None
    no_improvement = 0
    since_reassign = 0
    alpha = min(batch_size * 2.0 / (n + 1), 1.0)
    for step in range(n_steps):
        idx = draws.randint(n, batch_size)
        Xb = X[idx].contiguous()
        labels, d2 = assign_nearest(Xb, centers)
        batch_inertia = float(d2.sum().item()) / batch_size
        # centre update: running mean weighted by the number of samples each centre has seen
        bc_i = torch.bincount(labels, minlength=n_clusters)
        bc = bc_i.to(torch.float64)
        # per-centre sums of the batch rows as a CSR x dense product (rows = centres, entries = the batch members in
        # batch order): sequential accumulation, so the update is reproducible run to run -- an atomic scatter-add is not
        order = torch.argsort(labels, stable=True).to(torch.int32)
        member_ptr = torch.zeros((n_clusters + 1,), dtype=torch.int64, device=dev)
        member_ptr[1:] = torch.cumsum(bc_i, 0)
        members = pipeline.DeviceCSR(member_ptr, order, torch.ones((batch_size,), dtype=torch.float64, device=dev),
                                     (n_clusters, batch_size))
        sums = pipeline.spmm(members, Xb)
        new_counts = counts + bc
        hit = bc > 0
        centers[hit] = (centers[hit] * counts[hit, None] + sums[hit]) / new_counts[hit, None]
        counts = new_counts
        # reassign starved centres to random batch samples
        since_reassign += batch_size
        if bool((counts == 0).any().item()) or since_reassign >= 10 * n_clusters:
            since_reassign = 0
            starved = counts < reassignment_ratio * counts.max()
            ns = int(starved.sum().item())
            if ns > 0.5 * batch_size:
                keep = torch.argsort(counts)[: int(0.5 * batch_size)]
                starved = torch.zeros_like(starved)
                starved[keep] = True
                ns = int(starved.sum().item())
            if ns:
                pick = draws.choice_no_replace(batch_size, ns)
                centers[starved] = Xb[pick]
                counts[starved] = counts[~starved].min() if bool((~starved).any().item()) else 0.0
        # early stopping on the smoothed batch inertia (the first step only measures the initialisation)
        if step == 0:
            continue
        ewa = batch_inertia if ewa is None else ewa * (1 - alpha) + batch_inertia * alpha
        if ewa_min is None or ewa < ewa_min:
            ewa_min, no_improvement = ewa, 0
        else:
            no_improvement += 1
        if max_no_improvement is not None and no_improvement >= max_no_improvement:
            break
    labels, d2 = assign_nearest(X, centers)
    return labels, centers, float(d2.sum().item())


def spectral_clusters(K, P_vals, degree, n_landmark, n_svd, random_state=None):
    """Cluster label of every sample (numpy int32 [N]) from the device-resident kernel: the whole of
    graphs.py:1216-1230 without leaving HBM."""
    _, Vt = randomized_svd_vt(K, degree, n_svd, random_state)
    feats = pipeline.spmm(K, Vt.T.contiguous(), P_vals)              # diff_op . VT^T   [N, n_svd]
    labels, _, _ = minibatch_kmeans(feats, n_landmark, init_size=3 * n_landmark, batch_size=10000,
                                    random_state=random_state)
    return labels.to(torch.int32).cpu().numpy()
