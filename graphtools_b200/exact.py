"""TraditionalGraph (exact, dense) on the CUDA engine (reference graphtools/graphs.py:1320-1704).

``precomputed=None`` (the accelerated case): adaptive bandwidths come from the fused kNN pipeline,
then one tiled float64 sweep writes the thresholded, symmetrised alpha-decay kernel and its row sums;
a second sweep scales it into the diffusion operator.  ``precomputed`` inputs carry no distance
computation to accelerate (SURVEY.md section 2): their element-wise kernel function is evaluated with numpy
on the host, mirroring the reference.
"""
import numbers
import warnings

import numpy as np
import torch
from scipy import sparse

from . import dense, pipeline
from .core import DataGraph
from .logging_util import logger as _logger


class TraditionalGraph(DataGraph):
    """Exact alpha-decay graph over all pairs of samples (dense float64 kernel)."""

    def __init__(self, data, knn=5, decay=40, bandwidth=None, bandwidth_scale=1.0, distance="euclidean",
                 n_pca=None, thresh=1e-4, precomputed=None, **kwargs):
        if decay is None and precomputed not in ["affinity", "adjacency"]:
            raise ValueError("`decay` must be provided for a TraditionalGraph. For kNN kernel, use kNNGraph.")
        if precomputed is not None and n_pca not in [None, 0, False]:
            n_pca = None
            warnings.warn("n_pca cannot be given on a precomputed graph. Setting n_pca=None", RuntimeWarning)
        if knn is None and bandwidth is None:
            raise ValueError("Either `knn` or `bandwidth` must be provided.")
        if knn is not None and knn > data.shape[0] - 2:
            warnings.warn("Cannot set knn ({k}) to be greater than  n_samples - 2 ({n}). Setting knn={n}".format(
                k=knn, n=data.shape[0] - 2))
            knn = data.shape[0] - 2
        if precomputed is not None:
            if precomputed not in ["distance", "affinity", "adjacency"]:
                raise ValueError("Precomputed value {} not recognized. Choose from ['distance', 'affinity', "
                                 "'adjacency']".format(precomputed))
            elif data.shape[0] != data.shape[1]:
                raise ValueError("Precomputed {} must be a square matrix. {} was given".format(
                    precomputed, data.shape))
            elif (data < 0).sum() > 0:
                raise ValueError("Precomputed {} should be non-negative".format(precomputed))
        if precomputed is None and distance not in pipeline.METRIC_NAMES:
            raise NotImplementedError(pipeline.unsupported_metric_message(distance))
        self.knn = knn
        self.decay = decay
        self.bandwidth = bandwidth
        self.bandwidth_scale = bandwidth_scale
        self.distance = distance
        self.thresh = thresh
        self.precomputed = precomputed
        super().__init__(data, n_pca=n_pca, **kwargs)

    def get_params(self):
        params = super().get_params()
        params.update({"knn": self.knn, "decay": self.decay, "bandwidth": self.bandwidth,
                       "bandwidth_scale": self.bandwidth_scale, "distance": self.distance,
                       "precomputed": self.precomputed})
        return params

    def set_params(self, **params):
        for name in ("precomputed", "distance", "knn", "decay", "bandwidth", "bandwidth_scale"):
            if name in params and params[name] != getattr(self, name):
                if name == "knn" and self.precomputed is not None:
                    continue
                if name == "decay" and self.precomputed is not None:
                    continue
                raise ValueError("Cannot update {}. Please create a new graph".format(name))
        super().set_params(**params)
        return self

    @property
    def weighted(self):
        """Precomputed graphs: True when K has a non-zero value outside {0.5, 1} (a symmetrised binary adjacency
        holds only those); graphs built from data: ``decay is not None``."""
        if self.precomputed is None:
            return super().weighted
        K = self.K
        vals = K.data if sparse.issparse(K) else K[K != 0]
        return not bool(np.all(np.isin(vals, [0.5, 1.0])))

    # ------------------------------------------------------------------ device side
    def _metric(self):
        return self.distance if self.precomputed is None else "euclidean"

    def _X(self):
        if not hasattr(self, "_dev_X"):
            if sparse.issparse(self.data_nu):
                self.data_nu = self.data_nu.toarray()
            self._dev_X = self._dense_f32(self.data_nu)
        return self._dev_X

    def _degenerate_rows(self, X):
        """Rows of ``X`` from which scipy's distance is NaN (None for metrics without such rows): all-zero rows under
        cosine, constant rows under correlation."""
        return pipeline.degenerate_rows(X, self._metric())

    def _adaptive_bandwidth(self, Xq_op, ref_op, knn_eff):
        """Distance to the knn_eff-th nearest reference point (self counted when in-sample):
        np.partition(pdx, k)[:, :k].max (graphs.py:1583-1587, :1655-1656).

        Degenerate rows (all-zero under cosine, constant under correlation): their distances are NaN in the
        reference, which np.partition sorts last. So the neighbours are searched among the other reference rows, and
        the bandwidth is NaN where the k smallest entries of a row include a NaN: every degenerate query row, and
        every row when fewer than k reference rows are not degenerate."""
        zq, zr = self._degenerate_rows(Xq_op.X), self._degenerate_rows(ref_op.X)
        if zq is None or not bool(zq.any().item() or zr.any().item()):
            _, info = pipeline.knn_kernel(ref_op, Xq_op, knn=knn_eff, decay=max(float(self.decay), 1.0),
                                          thresh=0.5, bandwidth_scale=1.0)
            return info["bandwidth"]
        bw = torch.full((Xq_op.n,), float("nan"), dtype=torch.float64, device=Xq_op.X.device)
        keep_r, keep_q = (~zr).nonzero().flatten(), (~zq).nonzero().flatten()
        if keep_r.shape[0] >= knn_eff and keep_q.shape[0] > 0:
            ref_nz = pipeline.SearchOperand(ref_op.X[keep_r].contiguous(), metric=self._metric())
            qry_nz = pipeline.SearchOperand(Xq_op.X[keep_q].contiguous(), mean=ref_nz.mean, metric=self._metric())
            _, info = pipeline.knn_kernel(ref_nz, qry_nz, knn=knn_eff, decay=max(float(self.decay), 1.0),
                                          thresh=0.5, bandwidth_scale=1.0)
            bw[keep_q] = info["bandwidth"]
        return bw

    def _resolve_bandwidth(self, bandwidth, n_rows, dist_fn, Xq_op, ref_op, knn_eff):
        dev = pipeline._dev()
        if bandwidth is None:
            bw = self._adaptive_bandwidth(Xq_op, ref_op, knn_eff)
        elif callable(bandwidth):
            bw = torch.from_numpy(np.asarray(bandwidth(dist_fn().cpu().numpy()), dtype=np.float64)).to(dev)
        elif isinstance(bandwidth, numbers.Number):
            bw = torch.full((n_rows,), float(bandwidth), dtype=torch.float64, device=dev)
        else:
            bw = torch.from_numpy(np.asarray(bandwidth, dtype=np.float64).reshape(-1)).to(dev)
        return bw

    def build_kernel(self):
        """Raw (unsymmetrised) dense kernel as a CUDA tensor (graphs.py:1514-1610).  ``G.kernel`` does not
        go through here: ``_build_kernel`` fuses the symmetrisation into the same distance sweep."""
        if self.precomputed is not None:
            saved = self.kernel_symm, self.anisotropy
            self.kernel_symm, self.anisotropy = None, 0
            try:
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    return self._build_precomputed()
            finally:
                self.kernel_symm, self.anisotropy = saved
        X = self._X()                    # float32 or float64 as given: distances are evaluated on these rows
        op = pipeline.SearchOperand(X, metric=self._metric())
        bw = self._resolve_bandwidth(self.bandwidth, X.shape[0], lambda: dense.dense_distances(X, X, self._metric()), op, op,
                                     (self.knn or 0) + 1)
        bw = (bw * float(self.bandwidth_scale)).contiguous()
        K, _ = dense.dense_affinity(X, X, bw, None, self.decay, self.thresh, want_rowsum=False, metric=self._metric())
        return K

    def _sparse_route_ok(self):
        """With a positive threshold the exact kernel has the same support as the kNN-graph kernel without
        knn_max (all j with exp(-(d/bw)^decay) >= thresh), so it is built sparse on the tensor-core
        search path and densified once; thresh == 0 or a callable bandwidth need every pair -> dense kernel."""
        if not (self.thresh is not None and self.thresh > 0 and self.decay is not None
                and not callable(self.bandwidth) and self.knn is not None and self.knn + 1 + 8 <= 128):
            return False
        # a degenerate row (all-zero under cosine, constant under correlation) has NaN distances, i.e. affinity 1 to
        # every sample: not sparse
        zero = self._degenerate_rows(self._X())
        return zero is None or not bool(zero.any().item())

    def _build_kernel_via_sparse(self):
        from . import _engine as E
        X = self._X()
        n = X.shape[0]
        op = pipeline.SearchOperand(X, metric=self._metric())
        R, info = pipeline.knn_kernel(op, op, knn=self.knn + 1, knn_max=None, decay=self.decay,
                                      thresh=self.thresh, bandwidth=self.bandwidth,
                                      bandwidth_scale=self.bandwidth_scale)
        self._dev_bandwidth = info["bandwidth"]
        Ks, Pv, degree, flags = pipeline.symmetrize_normalize(R, self.kernel_symm, self.theta,
                                                              float(self.anisotropy))
        if flags & 1:
            warnings.warn("K should be symmetric", RuntimeWarning)
        K = pipeline._empty((n, n), torch.float64)
        E.call("gtb_csr_to_dense", Ks.indptr, Ks.indices, Ks.data, n, n, K)
        P = pipeline._empty((n, n), torch.float64)
        E.call("gtb_csr_to_dense", Ks.indptr, Ks.indices, Pv, n, n, P)
        self._dev_degree, self._dev_P = degree, P
        return K

    def _build_kernel(self):
        if self.precomputed is not None:
            return self._build_precomputed()
        if self._sparse_route_ok():
            with _logger.log_task("affinities"):
                try:
                    return self._build_kernel_via_sparse()
                except pipeline.RowTooLong:
                    # a kernel this wide (fixed bandwidth / small decay: thousands of neighbours inside the support
                    # radius) is not sparse in any useful sense: evaluate every pair with the dense kernel below
                    pass
        with _logger.log_task("affinities"):
            X = self._X()
            n = X.shape[0]
            op = pipeline.SearchOperand(X, metric=self._metric())
            bw = self._resolve_bandwidth(self.bandwidth, n, lambda: dense.dense_distances(X, X, self._metric()), op, op,
                                         (self.knn or 0) + 1)
            bw = (bw * float(self.bandwidth_scale)).contiguous()
            self._dev_bandwidth = bw
            if self.kernel_symm is None:
                K, rowsum = dense.dense_affinity(X, X, bw, None, self.decay, self.thresh, metric=self._metric())
                if float((K - K.T).max().item()) > 1e-5:
                    warnings.warn("K should be symmetric", RuntimeWarning)
            else:
                K, rowsum = dense.dense_affinity(X, X, bw, bw, self.decay, self.thresh, self.kernel_symm, self.theta,
                                                 metric=self._metric())
            if self.anisotropy != 0:
                dense.anisotropy_dense(K, self.anisotropy, rowsum)
                rowsum = dense.rowsum_dense(K)
            self._dev_degree = rowsum
            self._dev_P = dense.row_normalize_dense(K, rowsum)
        return K

    def _build_precomputed(self):
        """Precomputed distance / affinity / adjacency inputs (graphs.py:1532-1544, :1548-1549): no distance
        computation involved; element-wise host evaluation, results handed to the device containers."""
        data = self.data_nu
        dev = pipeline._dev()
        if sparse.issparse(data) and self.precomputed in ("affinity", "adjacency"):
            # sparse precomputed inputs stay sparse, as in the reference (graphs.py:1532-1544, :1597-1607): unit
            # diagonal for adjacencies, threshold, then the shared symmetrise / normalise kernels; K and P come back
            # as scipy CSR (no N x N densification on host or device)
            K = sparse.csr_matrix(data, dtype=np.float64, copy=True)
            if self.precomputed == "adjacency":
                K = K.tolil()
                K.setdiag(1)
                K = K.tocsr()
            K.data[K.data < self.thresh] = 0
            K.eliminate_zeros()
            Ks, Pv, degree, flags = pipeline.symmetrize_normalize(pipeline.csr_from_scipy(K), self.kernel_symm,
                                                                  self.theta, float(self.anisotropy))
            if self.kernel_symm is not None:
                flags &= ~1
            if flags & 1:
                warnings.warn("K should be symmetric", RuntimeWarning)
            if flags & 2:
                warnings.warn("K should have a non-zero diagonal", RuntimeWarning)
            self._dev_degree, self._dev_P = degree, Pv
            return Ks
        if self.precomputed == "distance":
            pdx = data.toarray() if sparse.issparse(data) else np.asarray(data, dtype=np.float64)
            if self.bandwidth is None:
                bw = np.max(np.partition(pdx, self.knn + 1, axis=1)[:, :self.knn + 1], axis=1)
            elif callable(self.bandwidth):
                bw = self.bandwidth(pdx)
            else:
                bw = self.bandwidth
            bw = bw * self.bandwidth_scale
            with np.errstate(invalid="ignore", divide="ignore"):
                K = np.exp(-1 * np.power((pdx.T / bw).T, self.decay))
            K = np.where(np.isnan(K), 1, K)
            K[K < self.thresh] = 0
        else:
            K = data.toarray() if sparse.issparse(data) else np.array(data, dtype=np.float64)
            if self.precomputed == "adjacency":
                np.fill_diagonal(K, 1)
            K[K < self.thresh] = 0
        Kd = torch.from_numpy(np.ascontiguousarray(K, dtype=np.float64)).to(dev)
        Kd = dense.symmetrize_dense(Kd, self.kernel_symm, self.theta).contiguous()
        if self.anisotropy != 0:
            dense.anisotropy_dense(Kd, self.anisotropy)
        if float((Kd - Kd.T).max().item()) > 1e-5:
            warnings.warn("K should be symmetric", RuntimeWarning)
        if bool((torch.diagonal(Kd) == 0).any().item()):
            warnings.warn("K should have a non-zero diagonal", RuntimeWarning)
        self._dev_degree = dense.rowsum_dense(Kd)
        self._dev_P = dense.row_normalize_dense(Kd, self._dev_degree)
        return Kd

    def _kernel_to_data_device(self, Y, knn=None, bandwidth=None, bandwidth_scale=None):
        if knn is None:
            knn = self.knn
        if bandwidth is None:
            bandwidth = self.bandwidth
        if bandwidth_scale is None:
            bandwidth_scale = self.bandwidth_scale
        if self.precomputed is not None:
            raise ValueError("Cannot extend kernel on precomputed graph")
        with _logger.log_task("affinities"):
            Y = self._check_extension_shape(Y)
            X = self._X()
            Yd = self._dense_f32(Y)
            ref = pipeline.SearchOperand(X, metric=self._metric())
            qry = pipeline.SearchOperand(Yd.to(X.dtype), mean=ref.mean, metric=self._metric())
            bw = self._resolve_bandwidth(bandwidth, Yd.shape[0], lambda: dense.dense_distances(Yd, X, self._metric()), qry, ref, knn)
            bw = (bw * float(bandwidth_scale)).contiguous()
            K, _ = dense.dense_affinity(Yd, X, bw, None, self.decay, self.thresh, want_rowsum=False, metric=self._metric())
        return K

    def build_kernel_to_data(self, Y, knn=None, bandwidth=None, bandwidth_scale=None):
        """Dense kernel [n_y, n] from new points to the graph's samples (graphs.py:1612-1678)."""
        return self._kernel_to_data_device(Y, knn, bandwidth, bandwidth_scale).cpu().numpy()
