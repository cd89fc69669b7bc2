"""Parity comparator (SURVEY.md Appendix C).

Structure must match exactly except for entries that sit on a discontinuity of the reference's own
definition: |w - thresh| / thresh < 1e-4 (threshold cut) -- those are counted and must be a
vanishing fraction of nnz.  Values on the common structure: |gpu - ref| <= rtol * |ref|, rtol 1e-5
(north_star tolerance for kernel and diff_op values).
"""
import numpy as np
from scipy import sparse

RTOL = 1e-5
SUBNORMAL_ATOL = 2 * 4.9406564584124654e-324


def _coo_keys(M):
    M = sparse.coo_matrix(M)
    return M.row.astype(np.int64) * M.shape[1] + M.col.astype(np.int64), M.data


def _tie_exempt(rows, cols, X, knn_eff, Y=None, metric="euclidean"):
    """True where entry (i, j) sits on a k-th / (k+1)-th neighbour tie (north_star: distances within
    1e-6 relative) in row i -- or in row j for symmetrised in-sample graphs (Y is None).  Cosine ties are
    ties of the Euclidean distance between the rows normalised as sklearn's ``normalize`` does (d_euc^2 = 2 d_cos;
    all-zero rows stay zero)."""
    from sklearn.preprocessing import normalize
    X = np.asarray(X, dtype=np.float64)
    Q = X if Y is None else np.asarray(Y, dtype=np.float64)
    if metric == "cosine":
        Xn = normalize(X)
        Q = Xn if Y is None else normalize(Q)
        X = Xn
    ok = np.zeros(len(rows), dtype=bool)
    cache = {}

    l1 = metric in ("cityblock", "manhattan", "l1")

    def dist(A, b):
        return np.abs(A - b).sum(-1) if l1 else np.sqrt(((A - b) ** 2).sum(-1))

    def kth(i, A):
        key = (i, id(A))
        if key not in cache:
            d = dist(X, A[i])
            cache[key] = np.partition(d, knn_eff - 1)[knn_eff - 1]
        return cache[key]

    for n, (i, j) in enumerate(zip(rows, cols)):
        dij = dist(Q[i], X[j])
        dk = kth(i, Q)
        if abs(dij - dk) <= 1e-6 * max(dk, 1e-300):
            ok[n] = True
        elif Y is None:
            dk = kth(j, X)
            ok[n] = abs(dij - dk) <= 1e-6 * max(dk, 1e-300)
    return ok


def compare_sparse(gpu, ref, rtol=RTOL, thresh=None, max_exempt_frac=1e-5, atol=0.0, what="matrix",
                   tie=None):
    """Returns dict(n_exempt, max_rel). Raises AssertionError on a parity violation.

    tie = dict(X=..., knn=effective neighbour count[, Y=...]) enables the k-th neighbour tie
    exemption for kNN / knn_max cuts."""
    assert gpu.shape == ref.shape, (gpu.shape, ref.shape)
    gpu = sparse.csr_matrix(gpu); ref = sparse.csr_matrix(ref)
    gpu.sum_duplicates(); ref.sum_duplicates()
    kg, vg = _coo_keys(gpu)
    kr, vr = _coo_keys(ref)
    og, orr = np.argsort(kg), np.argsort(kr)
    kg, vg, kr, vr = kg[og], vg[og], kr[orr], vr[orr]
    common, ig, ir = np.intersect1d(kg, kr, assume_unique=True, return_indices=True)
    only_g = np.setdiff1d(np.arange(len(kg)), ig, assume_unique=True)
    only_r = np.setdiff1d(np.arange(len(kr)), ir, assume_unique=True)
    n_exempt = 0
    n_tie = 0
    if (len(only_g) or len(only_r)) and tie is not None:
        ncol = gpu.shape[1]
        keys = np.concatenate([kg[only_g], kr[only_r]])
        ok = _tie_exempt(keys // ncol, keys % ncol, tie["X"], tie["knn"], tie.get("Y"), tie.get("metric", "euclidean"))
        n_tie = int(ok.sum())
        only_g = only_g[~ok[:len(only_g)]]
        only_r = only_r[~ok[len(ok) - len(only_r):]] if len(only_r) else only_r
    if len(only_g) or len(only_r):
        assert thresh is not None and thresh > 0, "{}: structure differs ({} extra, {} missing)".format(
            what, len(only_g), len(only_r))
        stray = np.concatenate([vg[only_g], vr[only_r]])
        bad = np.abs(stray - thresh) / thresh >= 1e-4
        assert not bad.any(), "{}: {} structural differences away from the threshold (e.g. value {})".format(
            what, int(bad.sum()), stray[bad][0])
        n_exempt = len(stray)
        assert n_exempt <= max(1, max_exempt_frac * ref.nnz), "{}: too many threshold-boundary entries ({})".format(
            what, n_exempt)
    a, b = vg[ig], vr[ir]
    err = np.abs(a - b)
    tol = rtol * np.abs(b) + atol
    worst = float((err / np.maximum(np.abs(b), 1e-300)).max()) if len(b) else 0.0
    bad = err > tol
    if bad.any() and tie is not None:
        # a tie decides whether an edge is one- or two-directional, which changes its symmetrised value
        ncol = gpu.shape[1]
        keys = common[bad]
        ok = _tie_exempt(keys // ncol, keys % ncol, tie["X"], tie["knn"], tie.get("Y"), tie.get("metric", "euclidean"))
        n_tie += int(ok.sum())
        bad[np.flatnonzero(bad)[ok]] = False
        worst = float((err[~bad] / np.maximum(np.abs(b[~bad]), 1e-300)).max()) if (~bad).any() else 0.0
    assert not bad.any(), "{}: max relative error {:.3e} exceeds rtol {:g}".format(what, worst, rtol)
    return {"n_exempt": n_exempt + n_tie, "n_tie": n_tie, "max_rel": worst}


def compare_dense(gpu, ref, rtol=RTOL, thresh=None, what="matrix"):
    gpu = np.asarray(gpu); ref = np.asarray(ref)
    assert gpu.shape == ref.shape
    err = np.abs(gpu - ref)
    # float64 subnormals (|v| < 2.2e-308, reached by exp(-(d/bw)^decay) with thresh = 0) carry fewer than 53 bits -- the
    # smallest one a single bit -- so a relative tolerance cannot apply there: two subnormal ulps absolute
    ok = err <= rtol * np.abs(ref) + SUBNORMAL_ATOL
    if thresh:
        # entries zeroed by the threshold on one side only
        edge = (np.abs(np.maximum(gpu, ref) - thresh) / thresh < 1e-4) & ((gpu == 0) | (ref == 0))
        ok |= edge
    worst = float((err[ok] / np.maximum(np.abs(ref[ok]), 1e-300)).max()) if ok.any() else 0.0
    assert ok.all(), "{}: {} entries outside rtol {:g} (max abs err {:.3e})".format(what, int((~ok).sum()), rtol,
                                                                                    float(err[~ok].max()))
    return {"max_rel": worst}
