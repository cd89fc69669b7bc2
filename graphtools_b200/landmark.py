"""LandmarkGraph on the CUDA engine (reference graphtools/graphs.py:985-1317).

Cluster *selection* follows the reference: spectral = scikit-learn ``randomized_svd`` of ``diff_aff`` +
``MiniBatchKMeans`` on the host with the same seeds (SURVEY.md section 8f ranks a GPU version as "next"); random
landmarking = nearest of ``n_landmark`` randomly chosen samples, computed with the fused distance/top-1
kernel.  Everything after the clusters -- ``pnm = K C`` aggregation, both L1 normalisations, the dense
``landmark_op = rownorm(C^T K) rownorm(K C)`` and ``extend_to_data`` -- runs on the GPU (csrc/landmark.cu).
"""
import warnings

import numpy as np
import torch
from scipy import sparse

from . import _engine as E
from . import pipeline
from .core import DataGraph
from .logging_util import logger as _logger


SPECTRAL_AUTO_N = 50_000   # GTB_SPECTRAL=auto: device-side SVD + k-means above this many samples


def aggregate_by_cluster(K, labels_dev, n_label, want_colsum):
    """Row-wise aggregation of DeviceCSR ``K`` by ``labels[col]`` -> (DeviceCSR raw sums, normalised
    values, column sums | None).  Column sums are accumulated in fixed point (csrc/landmark.cu): bit-reproducible."""
    n = K.shape[0]
    cnt = pipeline._empty((n,), torch.int32)
    ws = pipeline._empty((E.lib().gtb_cluster_aggregate_ws_elems(n_label),), torch.int64)
    E.call("gtb_cluster_aggregate_count", K.indptr, K.indices, K.data, n, labels_dev, n_label, cnt, ws)
    outptr = pipeline.exclusive_scan(cnt)
    nnz = int(outptr[-1].item())
    out_idx = pipeline._empty((nnz,), torch.int32)
    out_raw = pipeline._empty((nnz,), torch.float64)
    out_norm = pipeline._empty((nnz,), torch.float64)
    colsum = pipeline._empty((n_label,), torch.float64) if want_colsum else None
    colsum_fx = pipeline._empty((2 * n_label,), torch.int64) if want_colsum else None
    E.call("gtb_cluster_aggregate_fill", K.indptr, K.indices, K.data, n, labels_dev, outptr, out_idx, out_raw,
           out_norm, colsum, colsum_fx, n_label, ws)
    return pipeline.DeviceCSR(outptr, out_idx, out_raw, (n, n_label)), out_norm, colsum


def landmark_operator(pnm, pnm_norm, colsum, n, L):
    """Dense [L, L] operator rownorm(pnm^T) . rownorm(pnm), accumulated in fixed point (order independent)."""
    op = pipeline._empty((L, L), torch.float64)
    op_fx = pipeline._empty((2 * L * L,), torch.int64)
    E.call("gtb_landmark_op", pnm.indptr, pnm.indices, pnm.data, pnm_norm, colsum, n, L, op, op_fx)
    return op


class LandmarkGraph(DataGraph):
    """Adds landmarking to any data graph: cluster the samples, then collapse the kernel into a
    landmark-to-landmark diffusion operator and a sample-to-landmark transition matrix."""

    def __init__(self, data, n_landmark=2000, n_svd=100, random_landmarking=False, **kwargs):
        if n_landmark >= data.shape[0]:
            raise ValueError("n_landmark ({}) >= n_samples ({}). Use kNNGraph instead".format(
                n_landmark, data.shape[0]))
        if (n_svd >= data.shape[0]) and (not random_landmarking):
            warnings.warn("n_svd ({}) >= n_samples ({}) Consider using kNNGraph or lower n_svd".format(
                n_svd, data.shape[0]), RuntimeWarning)
        self.random_landmarking = random_landmarking
        self.n_landmark = n_landmark
        self.n_svd = n_svd
        super().__init__(data, **kwargs)

    def get_params(self):
        params = super().get_params()
        params.update({"n_landmark": self.n_landmark, "n_pca": self.n_pca,
                       "random_landmarking": self.random_landmarking})
        return params

    def set_params(self, **params):
        reset = False
        if "n_landmark" in params and params["n_landmark"] != self.n_landmark:
            self.n_landmark = params["n_landmark"]
            reset = True
        if "n_svd" in params and params["n_svd"] != self.n_svd:
            self.n_svd = params["n_svd"]
            reset = True
        if "random_landmarking" in params and params["random_landmarking"] != self.random_landmarking:
            self.random_landmarking = params["random_landmarking"]
            reset = True
        super().set_params(**params)
        if reset:
            self._reset_landmarks()
        return self

    def _reset_landmarks(self):
        for name in ("_landmark_op", "_transitions", "_clusters", "_dev_labels", "_n_label", "_dev_transitions"):
            if hasattr(self, name):
                delattr(self, name)

    @property
    def landmark_op(self):
        """Landmark diffusion operator, dense float64 [L, L]."""
        if not hasattr(self, "_landmark_op"):
            self.build_landmark_op()
        return self._landmark_op

    @property
    def clusters(self):
        """Cluster assignment of every sample."""
        if not hasattr(self, "_clusters"):
            self.build_landmark_op()
        return self._clusters

    @clusters.setter
    def clusters(self, value):
        self._reset_landmarks()
        self._clusters = np.asarray(value)

    @property
    def transitions(self):
        """Sample-to-landmark transition matrix, CSR [N, L]."""
        if not hasattr(self, "_transitions"):
            self.build_landmark_op()
        return self._transitions

    # ------------------------------------------------------------------ cluster selection
    def _random_landmark_clusters(self):
        n = self.data.shape[0]
        rng = np.random.default_rng(self.random_state)
        landmark_indices = rng.choice(n, self.n_landmark, replace=False)
        data = self.data if not hasattr(self, "data_nu") else self.data_nu
        X = self._dense_f32(data)
        metric = getattr(self, "distance", "euclidean")          # cdist(..., metric=self.distance), graphs.py:1212
        pipeline.reject_constant_rows(X, metric)
        ref = pipeline.SearchOperand(X[torch.from_numpy(landmark_indices).to(X.device)].contiguous(), metric=metric)
        qry = pipeline.SearchOperand(X, mean=ref.mean, metric=metric)
        nearest, _ = pipeline.knn_kernel(ref, qry, knn=1, decay=None)   # exact float64 argmin per sample
        return nearest.indices.cpu().numpy().astype(np.int64)

    def _spectral_impl(self):
        """GTB_SPECTRAL = host | device | auto (default).  ``host`` is the reference's own scikit-learn calls with
        the same seeds (bit-identical clusters; minutes at 1M samples); ``device`` is graphtools_b200/spectral.py
        (same algorithms in HBM, torch random streams); ``auto`` picks the device path for sparse kernels above
        SPECTRAL_AUTO_N samples, where the host path stops being practical."""
        import os
        want = os.environ.get("GTB_SPECTRAL", "auto")
        if want not in ("host", "device", "auto"):
            raise ValueError("GTB_SPECTRAL must be host, device or auto (got %r)" % (want,))
        sparse_kernel = isinstance(getattr(self, "_dev_kernel", None), pipeline.DeviceCSR)
        if want == "auto":
            want = "device" if (sparse_kernel and self.data.shape[0] > SPECTRAL_AUTO_N) else "host"
        if want == "device" and not sparse_kernel:
            raise NotImplementedError("device spectral landmarking needs a sparse (kNN / MNN) kernel")
        return want

    def _spectral_clusters(self):
        if self._spectral_impl() == "device":
            from . import spectral
            with _logger.log_task("SVD + KMeans (device)"):
                K = self._dev_kernel
                if getattr(self, "_dev_P", None) is None:
                    self._dev_P = pipeline.row_normalize(K)
                return spectral.spectral_clusters(K, self._dev_P, self._dev_degree, self.n_landmark, self.n_svd,
                                                  self.random_state)
        from sklearn.cluster import MiniBatchKMeans
        from sklearn.utils.extmath import randomized_svd
        with _logger.log_task("SVD"):
            _, _, VT = randomized_svd(self.diff_aff, n_components=self.n_svd, random_state=self.random_state)
        with _logger.log_task("KMeans"):
            kmeans = MiniBatchKMeans(self.n_landmark, init_size=3 * self.n_landmark, n_init=1, batch_size=10000,
                                     random_state=self.random_state)
            return kmeans.fit_predict(self.diff_op.dot(VT.T))

    # ------------------------------------------------------------------ operator
    def build_landmark_op(self):
        """clusters -> transitions, landmark_op (graphs.py:1187-1246)."""
        with _logger.log_task("landmark operator"):
            self._ensure_built()
            if not hasattr(self, "_clusters"):
                if self.random_landmarking:
                    self._clusters = self._random_landmark_clusters()
                else:
                    self._clusters = self._spectral_clusters()
            K = self._dev_kernel
            uniq, inv = np.unique(self._clusters, return_inverse=True)
            L = len(uniq)
            labels = torch.from_numpy(inv.astype(np.int32)).to(pipeline._dev())
            self._dev_labels, self._n_label = labels, L
            if isinstance(K, pipeline.DeviceCSR):
                # pnm[j, l] = sum_{i in l} K[i, j] (graphs.py:1169-1182): rows of K^T aggregated by the label of the
                # column.  K is symmetric unless kernel_symm=None, where the transpose is formed explicitly.
                Kt = K if self.kernel_symm is not None else pipeline.transpose_csr(K)
                pnm, pnm_norm, colsum = aggregate_by_cluster(Kt, labels, L, want_colsum=True)
                op = landmark_operator(pnm, pnm_norm, colsum, K.shape[0], L)
                self._dev_landmark_op = op
                self._landmark_op = op.cpu().numpy()
                self._transitions = pnm.to_scipy(pnm_norm)
                self._dev_transitions = (pnm, pnm_norm)
            else:
                from .dense import dense_landmark
                self._landmark_op, self._transitions = dense_landmark(K, labels, L)

    def landmark_op_power(self, t, return_device=False):
        """``landmark_op ** t`` (matrix power): the diffusion chain the callers of ``G.landmark_op`` run as
        ``np.linalg.matrix_power(G.landmark_op, t)`` on the operator of graphs.py:1240-1243, here as float64-faithful
        products on the int8 tensor cores (dense.matrix_power, csrc/gemm.cu) without the operator leaving HBM."""
        from .dense import matrix_power
        self.landmark_op  # builds the operator if needed
        op = getattr(self, "_dev_landmark_op", None)
        if op is None:
            op = self._dev_landmark_op = pipeline.to_device(np.ascontiguousarray(self._landmark_op, dtype=np.float64))
        out = matrix_power(op, t)
        return out if return_device else out.cpu().numpy()

    def _extend_to_data_device(self, data, **kwargs):
        """(DeviceCSR [n_y, L], normalised values): out-of-sample kernel aggregated by landmark, in HBM."""
        self.clusters  # make sure labels exist
        if not hasattr(self, "_dev_labels"):
            self.build_landmark_op()
        data = self._check_extension_shape(data)
        Kyx = self._kernel_to_data_device(data, **kwargs)
        if not isinstance(Kyx, pipeline.DeviceCSR):
            from .dense import _dense_to_csr
            Kyx = _dense_to_csr(Kyx)
        agg, agg_norm, _ = aggregate_by_cluster(Kyx, self._dev_labels, self._n_label, want_colsum=False)
        return agg, agg_norm

    def extend_to_data(self, data, **kwargs):
        """Transition matrix from new points to the landmarks (graphs.py:1248-1288)."""
        agg, agg_norm = self._extend_to_data_device(data, **kwargs)
        T = agg.to_scipy(agg_norm)
        return T if isinstance(self._dev_kernel, pipeline.DeviceCSR) else T.toarray()

    def interpolate(self, transform, transitions=None, Y=None):
        """Landmark -> sample interpolation (graphs.py:1290-1317): with neither ``transitions`` nor ``Y`` the
        cached sample-to-landmark transitions are used straight from HBM."""
        if transitions is None and Y is None:
            self.transitions
            dev_t = getattr(self, "_dev_transitions", None)
            if dev_t is not None:
                one_d = np.ndim(transform) == 1
                B = pipeline.to_device(np.asarray(transform, dtype=np.float64).reshape(len(transform), -1))
                out = pipeline.spmm(dev_t[0], B, dev_t[1]).cpu().numpy()
                return out[:, 0] if one_d else out
            transitions = self.transitions
        return super().interpolate(transform, transitions=transitions, Y=Y)
