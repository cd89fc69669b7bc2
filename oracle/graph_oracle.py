"""CPU oracle: numpy / scipy / scikit-learn restatement of graphtools' hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``graphtools_b200/`` may import this
module; only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs do, and there only as the checker or
the timed CPU baseline.

What it restates (all citations relative to /root/reference, graphtools v2.1.0):
the float64, ``NUMBA_AVAILABLE=False`` code path of ``kNNGraph``,
``TraditionalGraph``, ``MNNGraph``, ``LandmarkGraph`` and the ``BaseGraph``
symmetrise / anisotropy / diffusion-operator steps.  The reference delegates its
arithmetic to third-party libraries that are not vendored under /root/reference
(setup.py:6-14 pins only lower bounds): scikit-learn (container: 1.9.0)
``NearestNeighbors`` / ``normalize`` / ``randomized_svd`` / ``MiniBatchKMeans`` /
``euclidean_distances``; scipy (1.18.1) ``pdist`` / ``cdist`` / ``scipy.sparse``;
numpy (2.3.5).  Those same library calls are made here at the same call sites, so
the oracle's numbers ARE the reference's numbers; only the Python glue around them
(ragged per-row lists, per-row loops, LIL block assignment) is re-expressed in
vectorised form.

Parity pin: ``tests/golden/*.npz`` are outputs of the UNMODIFIED reference imported
in the build container (``oracle/make_golden.py``); ``tests/test_oracle_golden.py``
checks every function below against them bit-for-bit.  ``diff_op`` and
``landmark_op`` values are pinned the same way (the reference's own tests never
assert on them, SURVEY.md section 8c).
"""
import numbers
import warnings

import numpy as np
from scipy import sparse
from scipy.spatial.distance import cdist, pdist, squareform
from sklearn.cluster import MiniBatchKMeans
from sklearn.metrics.pairwise import euclidean_distances
from sklearn.neighbors import NearestNeighbors
from sklearn.preprocessing import normalize
from sklearn.utils.extmath import randomized_svd

_EPS = np.finfo(float).eps


# --------------------------------------------------------------------------- kNN
def _alpha_decay(dist, bw, decay):
    """exp(-(d/bw)^decay) with NaN -> 1 (graphs.py:503-507)."""
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        w = np.exp(-np.power(dist / bw, decay))
    return np.where(np.isnan(w), 1.0, w)


def csr_from_neighbors(indices, distances, bandwidth, decay, thresh, shape):
    """graphs.py:450-559 (non-numba branch): weights, threshold, per-row column sort,
    CSR assembly, ``sum_duplicates``.  ``indices`` / ``distances`` are either 2-D
    arrays or ragged lists of 1-D arrays."""
    n_rows = shape[0]
    if isinstance(indices, np.ndarray) and indices.ndim == 2:
        lens = np.full(n_rows, indices.shape[1], dtype=np.int64)
        flat_idx = indices.reshape(-1)
        flat_dist = np.asarray(distances, dtype=np.float64).reshape(-1)
    else:
        lens = np.fromiter((len(r) for r in indices), dtype=np.int64, count=n_rows)
        flat_idx = np.concatenate([np.asarray(r) for r in indices]) if n_rows else np.zeros(0, int)
        flat_dist = (np.concatenate([np.asarray(r, dtype=np.float64) for r in distances])
                     if n_rows else np.zeros(0))
    rows = np.repeat(np.arange(n_rows), lens)
    if isinstance(bandwidth, numbers.Number):
        bw = bandwidth
    else:
        bw = np.asarray(bandwidth, dtype=np.float64)[rows]
    w = _alpha_decay(flat_dist, bw, decay)
    keep = w >= thresh
    rows, cols, w = rows[keep], flat_idx[keep], w[keep]
    order = np.lexsort((cols, rows))
    rows, cols, w = rows[order], cols[order], w[order]
    indptr = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows, minlength=n_rows), out=indptr[1:])
    K = sparse.csr_matrix((w, cols.astype(np.int32), indptr), shape=shape)
    K.sum_duplicates()
    return K


class KnnOracle:
    """State + methods of ``kNNGraph`` that matter for the kernel (graphs.py:562-982)."""

    def __init__(self, data, knn=5, decay=None, knn_max=None, search_multiplier=6,
                 bandwidth=None, bandwidth_scale=1.0, distance="euclidean", thresh=1e-4,
                 n_jobs=-1):
        data = np.asarray(data, dtype=np.float64)
        if decay is not None and thresh < _EPS:           # graphs.py:622-629
            thresh = _EPS
        if knn > data.shape[0] - 2:                        # graphs.py:643-650
            knn = data.shape[0] - 2
        if knn_max is not None and knn_max < knn:          # graphs.py:651-656
            knn_max = knn
        self.data = data
        self.knn, self.decay, self.knn_max = knn, decay, knn_max
        self.search_multiplier = search_multiplier
        self.bandwidth, self.bandwidth_scale = bandwidth, bandwidth_scale
        self.distance, self.thresh, self.n_jobs = distance, thresh, n_jobs
        self._tree = None
        self.passes = []  # (search_knn, rows searched) per kNN pass, for reporting
        # per kernel_to_data call with a decay: dict(todo=rows still to do after the last kNN pass,
        # search_knn=width of the final step, fallback=that step ran on the metric-less brute-force index,
        # branch="kneighbors" | "radius" | None)
        self.schedules = []

    @property
    def tree(self):                                         # graphs.py:748-769
        if self._tree is None:
            self._tree = NearestNeighbors(n_neighbors=self.knn + 1, algorithm="auto",
                                          metric=self.distance, n_jobs=self.n_jobs).fit(self.data)
        return self._tree

    def kernel(self):                                       # graphs.py:771-785
        knn_max = self.knn_max + 1 if self.knn_max else None
        return self.kernel_to_data(self.data, knn=self.knn + 1, knn_max=knn_max)

    def kernel_to_data(self, Y, knn=None, knn_max=None, bandwidth=None, bandwidth_scale=None):
        """graphs.py:819-982."""
        Y = np.asarray(Y, dtype=np.float64)
        n_ref = self.data.shape[0]
        knn = self.knn if knn is None else knn
        bandwidth = self.bandwidth if bandwidth is None else bandwidth
        bandwidth_scale = self.bandwidth_scale if bandwidth_scale is None else bandwidth_scale
        knn = min(knn, n_ref)                               # graphs.py:860-867
        if knn_max is None:
            knn_max = n_ref
        if self.decay is None or self.thresh == 1:          # graphs.py:872-877
            self.passes.append((knn, Y.shape[0]))
            return self.tree.kneighbors_graph(Y, n_neighbors=knn, mode="connectivity")

        tree = self.tree
        mult = self.search_multiplier
        search_knn = min(knn * mult, knn_max)               # graphs.py:882
        dist, ind = tree.kneighbors(Y, n_neighbors=search_knn)
        self.passes.append((search_knn, Y.shape[0]))
        if bandwidth is None:                                # graphs.py:886-897
            bw = np.maximum(dist[:, knn - 1] * bandwidth_scale, _EPS)
        else:
            bw = np.maximum(bandwidth * bandwidth_scale, _EPS)
        scalar_bw = isinstance(bw, numbers.Number)
        radius = bw * np.power(-1 * np.log(self.thresh), 1 / self.decay)   # graphs.py:903-905
        todo = np.flatnonzero(dist.max(axis=1) < radius)    # graphs.py:906-908
        ragged = todo.size > 0
        if ragged:
            dist = list(dist)
            ind = list(ind)
        search_knn = min(search_knn * mult, knn_max)        # graphs.py:916
        while (todo.size > Y.shape[0] // 10 and search_knn < n_ref / 2
               and search_knn < knn_max):                   # graphs.py:917-944
            d_new, i_new = tree.kneighbors(Y[todo], n_neighbors=search_knn)
            self.passes.append((search_knn, todo.size))
            for pos, row in enumerate(todo):
                dist[row], ind[row] = d_new[pos], i_new[pos]
            far = np.fromiter((r.max() for r in dist), dtype=np.float64, count=len(dist))
            todo = np.flatnonzero(far < radius)
            search_knn = min(search_knn * mult, knn_max)
        self.schedules.append(dict(todo=todo.copy(), search_knn=search_knn, fallback=search_knn > n_ref / 2,
                                   branch=(None if todo.size == 0 else
                                           "kneighbors" if search_knn == knn_max else "radius")))
        if search_knn > n_ref / 2:                          # graphs.py:945-948 (no metric!)
            tree = NearestNeighbors(n_neighbors=search_knn, algorithm="brute",
                                    n_jobs=self.n_jobs).fit(self.data)
        if todo.size > 0:                                    # graphs.py:949-976
            if search_knn == knn_max:
                d_new, i_new = tree.kneighbors(Y[todo], n_neighbors=search_knn)
                self.passes.append((search_knn, todo.size))
            else:
                r = radius if scalar_bw else np.max(radius[todo])
                d_new, i_new = tree.radius_neighbors(Y[todo, :], radius=r)
                self.passes.append(("radius", todo.size))
            for pos, row in enumerate(todo):
                dist[row], ind[row] = d_new[pos], i_new[pos]
        if not ragged:
            ind, dist = np.asarray(ind), np.asarray(dist)
        return csr_from_neighbors(ind, dist, bw, self.decay, self.thresh,
                                  (Y.shape[0], n_ref))     # graphs.py:978-981


# ------------------------------------------------------- symmetrise / normalise
def symmetrize(K, kernel_symm="+", theta=None):
    """base.py:557-577 (+ matrix.py:16-29 for min / max)."""
    if kernel_symm == "+":
        return (K + K.T) / 2
    if kernel_symm == "*":
        return K.multiply(K.T) if sparse.issparse(K) else np.multiply(K, K.T)
    if kernel_symm == "mnn":
        if sparse.issparse(K):
            lo, hi = K.minimum(K.T), K.maximum(K.T)
        else:
            lo, hi = np.minimum(K, K.T), np.maximum(K, K.T)
        return theta * lo + (1 - theta) * hi
    if kernel_symm is None:
        return K
    raise NotImplementedError(kernel_symm)


def apply_anisotropy(K, anisotropy):
    """base.py:579-592."""
    if anisotropy == 0:
        return K
    if sparse.issparse(K):
        d = np.array(K.sum(1)).flatten()
        K = K.tocoo()
        K.data = K.data / ((d[K.row] * d[K.col]) ** anisotropy)
        return K.tocsr()
    d = K.sum(1)
    return K / (np.outer(d, d) ** anisotropy)


def finish_kernel(R, kernel_symm="+", theta=None, anisotropy=0):
    """``BaseGraph._build_kernel`` after ``build_kernel`` (base.py:534-555)."""
    return apply_anisotropy(symmetrize(R, kernel_symm, theta), anisotropy)


def diff_op(K):
    """base.py:645."""
    return normalize(K, "l1", axis=1)


def kernel_degree(K):
    """base.py:648-666."""
    s = K.sum(axis=1)
    return np.asarray(s).reshape(-1, 1)


def diff_aff(K):
    """base.py:668-698."""
    deg = kernel_degree(K)
    if sparse.issparse(K):
        n = len(deg)
        D = sparse.csr_matrix((1 / np.sqrt(deg.flatten()), np.arange(n), np.arange(n + 1)))
        return D @ K @ D
    return (K / np.sqrt(deg)) / np.sqrt(deg.T)


# ------------------------------------------------------------------------ exact
def exact_kernel(X, knn=5, decay=40, bandwidth=None, bandwidth_scale=1.0,
                 distance="euclidean", thresh=1e-4):
    """``TraditionalGraph.build_kernel`` for ``precomputed=None`` (graphs.py:1546-1609)."""
    X = np.asarray(X, dtype=np.float64)
    knn = min(knn, X.shape[0] - 2)                          # graphs.py:1413-1420
    pdx = squareform(pdist(X, metric=distance))
    if bandwidth is None:
        bw = np.max(np.partition(pdx, knn + 1, axis=1)[:, :knn + 1], axis=1)
    elif callable(bandwidth):
        bw = bandwidth(pdx)
    else:
        bw = bandwidth
    bw = bw * bandwidth_scale
    pdx = (pdx.T / bw).T
    with np.errstate(invalid="ignore", divide="ignore"):
        K = np.exp(-1 * np.power(pdx, decay))
    K = np.where(np.isnan(K), 1, K)
    K[K < thresh] = 0
    return K


def exact_kernel_to_data(X, Y, knn=5, decay=40, bandwidth=None, bandwidth_scale=1.0,
                         distance="euclidean", thresh=1e-4):
    """``TraditionalGraph.build_kernel_to_data`` float64 branch (graphs.py:1651-1677)."""
    X = np.asarray(X, dtype=np.float64)
    Y = np.asarray(Y, dtype=np.float64)
    pdx = cdist(Y, X, metric=distance)
    if bandwidth is None:
        bw = np.max(np.partition(pdx, knn, axis=1)[:, :knn], axis=1)
    elif callable(bandwidth):
        bw = bandwidth(pdx)
    else:
        bw = bandwidth
    bw = bandwidth_scale * bw
    pdx = (pdx.T / bw).T
    with np.errstate(invalid="ignore", divide="ignore"):
        K = np.exp(-1 * pdx ** decay)
    K = np.where(np.isnan(K), 1, K)
    K[K < thresh] = 0
    return K


# -------------------------------------------------------------------------- MNN
def mnn_kernel(X, sample_idx, knn=5, decay=None, bandwidth=None, thresh=1e-4, beta=1,
               distance="euclidean", n_jobs=-1):
    """``MNNGraph.build_kernel`` (graphs.py:1857-1936) with COO block assembly in place
    of the LIL ``set_submatrix`` (matrix.py:49-51), which densifies every block.  The
    blocks, their values and their placement are the reference's; verified identical to
    ``MNNGraph.K`` before symmetrisation by tests/test_oracle_golden.py.

    Sub-graphs are kNN graphs symmetrised with ``+`` (graphs.py:1883-1896); with
    ``thresh == 0`` and a decay the reference's factory would pick exact sub-graphs
    (api.py:207-209) -- not restated here (out of the configs' range).
    """
    X = np.asarray(X, dtype=np.float64)
    sample_idx = np.asarray(sample_idx)
    if decay is not None and thresh <= 0:
        return _mnn_kernel_dense(X, sample_idx, knn, decay, bandwidth, beta, distance)
    samples = np.unique(sample_idx)
    members = [np.flatnonzero(sample_idx == s) for s in samples]
    subs, within = [], []
    for idx in members:
        g = KnnOracle(X[idx], knn=knn, decay=decay, bandwidth=bandwidth, distance=distance,
                      thresh=thresh, n_jobs=n_jobs)
        Kbb = symmetrize(g.kernel(), "+")
        subs.append(g)
        within.append(Kbb)
    rows, cols, vals = [], [], []
    for i, idx_i in enumerate(members):
        Kii = within[i].tocoo()
        rows.append(idx_i[Kii.row]); cols.append(idx_i[Kii.col]); vals.append(Kii.data)
        within_norm = np.array(np.sum(within[i], 1)).flatten()
        for j, idx_j in enumerate(members):
            if i == j:
                continue
            Kij = subs[j].kernel_to_data(subs[i].data, knn=knn)          # graphs.py:1920
            between_norm = np.array(np.sum(Kij, 1)).flatten()
            with np.errstate(invalid="ignore", divide="ignore"):
                scale = np.minimum(1, within_norm / between_norm) * beta  # graphs.py:1921-1925
            Kij = sparse.coo_matrix(Kij.multiply(scale[:, None]))
            rows.append(idx_i[Kij.row]); cols.append(idx_j[Kij.col]); vals.append(Kij.data)
    n = X.shape[0]
    K = sparse.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))),
                          shape=(n, n)).tocsr()
    K.eliminate_zeros()
    return K


def _mnn_kernel_dense(X, sample_idx, knn, decay, bandwidth, beta, distance):
    """``MNNGraph.build_kernel`` with ``thresh == 0``: the factory picks exact sub-graphs (api.py:207-209), the kernel
    is the dense ndarray of graphs.py:1901-1935."""
    samples = np.unique(sample_idx)
    members = [np.flatnonzero(sample_idx == s) for s in samples]
    n = X.shape[0]
    K = np.zeros((n, n))
    within = []
    for idx in members:
        Kbb = symmetrize(exact_kernel(X[idx], knn=knn, decay=decay, bandwidth=bandwidth, distance=distance, thresh=0),
                         "+")
        within.append(Kbb)
    for i, idx_i in enumerate(members):
        K[np.ix_(idx_i, idx_i)] = within[i]
        within_norm = np.array(np.sum(within[i], 1)).flatten()
        for j, idx_j in enumerate(members):
            if i == j:
                continue
            Kij = exact_kernel_to_data(X[idx_j], X[idx_i], knn=knn, decay=decay, bandwidth=bandwidth,
                                       distance=distance, thresh=0)
            between_norm = np.array(np.sum(Kij, 1)).flatten()
            scale = np.minimum(1, within_norm / between_norm) * beta
            K[np.ix_(idx_i, idx_j)] = Kij * scale[:, None]
    return K


# --------------------------------------------------------------------- landmark
def random_landmark_clusters(X, n_landmark, random_state, distance="euclidean"):
    """graphs.py:1200-1213."""
    X = np.asarray(X, dtype=np.float64)
    n = X.shape[0]
    rng = np.random.default_rng(random_state)
    landmarks = rng.choice(n, n_landmark, replace=False)
    if n > 5000 and distance == "euclidean":
        dist = euclidean_distances(X, X[landmarks])
    else:
        dist = cdist(X, X[landmarks], metric=distance)
    return np.argmin(dist, axis=1)


def spectral_clusters(K, n_landmark, n_svd=100, random_state=None):
    """graphs.py:1216-1230."""
    _, _, VT = randomized_svd(diff_aff(K), n_components=n_svd, random_state=random_state)
    km = MiniBatchKMeans(n_landmark, init_size=3 * n_landmark, n_init=1, batch_size=10000,
                         random_state=random_state)
    return km.fit_predict(diff_op(K).dot(VT.T))


def landmarks_to_data(K, clusters):
    """graphs.py:1169-1182, as one product ``C^T K`` (C = one-hot membership over the
    sorted unique cluster ids).  Summation order per output entry equals the reference's
    ``kernel[clusters == i, :].sum(axis=0)`` for CSR kernels (rows in ascending order)."""
    clusters = np.asarray(clusters)
    uniq, inv = np.unique(clusters, return_inverse=True)
    n = len(clusters)
    if sparse.issparse(K):
        C = sparse.csr_matrix((np.ones(n), (inv, np.arange(n))), shape=(len(uniq), n))
        pmn = (C @ K).tocsr()
        pmn.sort_indices()   # the reference's vstack of dense-row CSRs is column-sorted
        return pmn
    return np.array([np.sum(K[clusters == c, :], axis=0) for c in uniq])


def landmark_operator(K, clusters):
    """graphs.py:1232-1246 -> (landmark_op dense [L,L], transitions [N,L])."""
    pmn = landmarks_to_data(K, clusters)
    pnm = pmn.transpose()
    pmn = normalize(pmn, norm="l1", axis=1)
    pnm = normalize(pnm, norm="l1", axis=1)
    op = pmn.dot(pnm)
    if sparse.issparse(op):
        op = op.toarray()
    return op, pnm


def landmark_extend(Kyx, clusters):
    """graphs.py:1272-1288: aggregate out-of-sample kernel columns by cluster, L1-normalise."""
    clusters = np.asarray(clusters)
    uniq, inv = np.unique(clusters, return_inverse=True)
    n = len(clusters)
    if sparse.issparse(Kyx):
        # ``kernel[:, clusters == c].sum(axis=1)`` is scipy's ``np.add.reduceat`` over each
        # row's entries of that cluster in column order; reproduce exactly that grouping.
        Kc = sparse.csr_matrix(Kyx)
        Kc.sort_indices()
        ny = Kc.shape[0]
        rows = np.repeat(np.arange(ny), np.diff(Kc.indptr))
        lab = inv[Kc.indices]
        order = np.lexsort((Kc.indices, lab, rows))
        r, c, v = rows[order], lab[order], Kc.data[order]
        if v.size:
            first = np.flatnonzero(np.r_[True, (r[1:] != r[:-1]) | (c[1:] != c[:-1])])
            sums = np.add.reduceat(v, first)
            r, c = r[first], c[first]
            nz = sums != 0
            pnm = sparse.csr_matrix((sums[nz], (r[nz], c[nz])), shape=(ny, len(uniq)))
        else:
            pnm = sparse.csr_matrix((ny, len(uniq)))
        pnm.sort_indices()
    else:
        pnm = np.array([np.sum(Kyx[:, clusters == c], axis=1).T for c in uniq]).transpose()
    return normalize(pnm, norm="l1", axis=1)


# ------------------------------------------------------------------ convenience
def knn_graph(X, knn=5, decay=40, thresh=1e-4, knn_max=None, bandwidth=None,
              bandwidth_scale=1.0, kernel_symm="+", theta=None, anisotropy=0,
              search_multiplier=6, distance="euclidean", n_jobs=-1, return_oracle=False):
    """``graphtools.Graph(X, ...)`` kNN path -> (K, P): kernel + diffusion operator."""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        g = KnnOracle(X, knn=knn, decay=decay, knn_max=knn_max, bandwidth=bandwidth,
                      bandwidth_scale=bandwidth_scale, thresh=thresh, distance=distance,
                      search_multiplier=search_multiplier, n_jobs=n_jobs)
        K = finish_kernel(g.kernel(), kernel_symm, theta, anisotropy)
        P = diff_op(K)
    if return_oracle:
        return K, P, g
    return K, P
