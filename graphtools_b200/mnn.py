"""MNNGraph on the CUDA engine (reference graphtools/graphs.py:1707-1966).

Per batch: a full kNN graph symmetrised with '+' (device resident).  Per ordered batch pair (b, c):
the out-of-sample kernel from batch b's points to batch c's search operand, rescaled row-wise by
min(1, within / between) * beta.  The blocks are scattered straight into one global CSR staging area
(csrc/sparse.cu block_count / block_fill) -- the reference's LIL ``set_submatrix`` densifies every
block and cannot run at the 4 x 250k size -- then column-sorted, symmetrised with the requested rule
(``mnn`` min/max by default) and normalised by the shared sparse kernels.
"""
import numbers
import warnings

import numpy as np
import torch

from . import _engine as E
from . import pipeline
from .core import DataGraph
from .logging_util import logger as _logger


class MNNGraph(DataGraph):
    """Mutual nearest neighbours graph for batch-structured data."""

    def __init__(self, data, sample_idx, knn=5, beta=1, n_pca=None, decay=None, adaptive_k=None, bandwidth=None,
                 distance="euclidean", thresh=1e-4, n_jobs=1, **kwargs):
        self.beta = beta
        self.sample_idx = sample_idx
        self.samples, self.n_cells = np.unique(self.sample_idx, return_counts=True)
        self.knn = knn
        self.decay = decay
        self.distance = distance
        self.bandwidth = bandwidth
        self.thresh = thresh
        self.n_jobs = n_jobs
        if sample_idx is None:
            raise ValueError("sample_idx must be given. For a graph without batch correction, use kNNGraph.")
        elif len(sample_idx) != data.shape[0]:
            raise ValueError("sample_idx ({}) must be the same length as data ({})".format(
                len(sample_idx), data.shape[0]))
        elif len(self.samples) == 1:
            raise ValueError("sample_idx must contain more than one unique value")
        if adaptive_k is not None:
            warnings.warn("`adaptive_k` has been deprecated. Using fixed knn.", DeprecationWarning)
        super().__init__(data, n_pca=n_pca, **kwargs)

    def _check_symmetrization(self, kernel_symm, theta):
        if (kernel_symm == "theta" or kernel_symm == "mnn") and theta is not None and not isinstance(
                theta, numbers.Number):
            raise TypeError("Expected `theta` as a float. Got {}.".format(type(theta)))
        super()._check_symmetrization(kernel_symm, theta)

    def get_params(self):
        params = super().get_params()
        params.update({"beta": self.beta, "knn": self.knn, "decay": self.decay, "bandwidth": self.bandwidth,
                       "distance": self.distance, "thresh": self.thresh, "n_jobs": self.n_jobs})
        return params

    def set_params(self, **params):
        if "beta" in params and params["beta"] != self.beta:
            raise ValueError("Cannot update beta. Please create a new graph")
        knn_kernel_args = ["knn", "decay", "distance", "thresh", "bandwidth"]
        knn_other_args = ["n_jobs", "random_state", "verbose"]
        for arg in knn_kernel_args:
            if arg in params and params[arg] != getattr(self, arg):
                raise ValueError("Cannot update {}. Please create a new graph".format(arg))
        for arg in knn_other_args:
            if arg in params:
                setattr(self, arg, params[arg])
                for g in getattr(self, "subgraphs", []):
                    g.set_params(**{arg: params[arg]})
        super().set_params(**{k: v for k, v in params.items() if k not in knn_other_args})
        return self

    def build_kernel(self):
        """Assemble the batch-block kernel on the device (graphs.py:1857-1936)."""
        from .factory import Graph
        pipeline.reject_constant_rows(self.data_nu, self.distance)
        dev = pipeline._dev()
        sample_idx = np.asarray(self.sample_idx)
        n = self.data_nu.shape[0]
        with _logger.log_task("subgraphs"):
            self.subgraphs = []
            members = []
            for i, s in enumerate(self.samples):
                idx = np.flatnonzero(sample_idx == s)
                _logger.log_debug("subgraph {}: sample {}, n = {}, knn = {}".format(i, s, len(idx), self.knn))
                g = Graph(self.data_nu[idx], n_pca=None, knn=self.knn, decay=self.decay, bandwidth=self.bandwidth,
                          distance=self.distance, thresh=self.thresh, verbose=self.verbose,
                          random_state=self.random_state, n_jobs=self.n_jobs, kernel_symm="+", initialize=True)
                self.subgraphs.append(g)
                members.append(torch.from_numpy(idx.astype(np.int32)).to(dev))
        if not isinstance(self.subgraphs[0]._dev_kernel, pipeline.DeviceCSR):
            return self._build_kernel_dense(members)
        with _logger.log_task("MNN kernel"):
            rowlen = torch.zeros((n,), dtype=torch.int32, device=dev)
            blocks = []
            for i, gi in enumerate(self.subgraphs):
                Kii = gi._dev_kernel
                blocks.append((Kii, members[i], members[i], None, None))
                for j, gj in enumerate(self.subgraphs):
                    if i == j:
                        continue
                    with _logger.log_task("kernel from sample {} to {}".format(self.samples[i], self.samples[j])):
                        Kij = gj._kernel_to_data_device(gi.data_nu, knn=self.knn)
                        between = pipeline.row_sums(Kij)
                        blocks.append((Kij, members[i], members[j], gi._dev_degree, between))
            for (B, rmap, cmap, within, between) in blocks:
                E.call("gtb_block_count", B.indptr, B.shape[0], rmap, rowlen)
            outptr = pipeline.exclusive_scan(rowlen)
            nnz = int(outptr[-1].item())
            tmp_idx = pipeline._empty((nnz,), torch.int32)
            tmp_val = pipeline._empty((nnz,), torch.float64)
            cursor = torch.zeros((n,), dtype=torch.int32, device=dev)
            for (B, rmap, cmap, within, between) in blocks:
                E.call("gtb_block_fill", B.indptr, B.indices, B.data, B.shape[0], rmap, cmap, within, between,
                       float(self.beta), outptr, cursor, tmp_idx, tmp_val)
            pipeline.sort_rows(outptr, tmp_idx, tmp_val, n)      # blocks land in batch order -> column order
        return pipeline.DeviceCSR(outptr, tmp_idx, tmp_val, (n, n))

    def _build_kernel_dense(self, members):
        """thresh == 0 with a decay: the factory hands back exact (dense) sub-graphs (api.py:207-209) and the
        reference assembles a dense ndarray (graphs.py:1901-1902).  Same blocks, same scaling, dense on the device."""
        n = self.data_nu.shape[0]
        with _logger.log_task("MNN kernel"):
            K = torch.zeros((n, n), dtype=torch.float64, device=pipeline._dev())
            for i, gi in enumerate(self.subgraphs):
                ri = members[i].long()
                K[ri[:, None], ri[None, :]] = gi._dev_kernel
                within = gi._dev_degree
                for j, gj in enumerate(self.subgraphs):
                    if i == j:
                        continue
                    Kij = gj._kernel_to_data_device(gi.data_nu, knn=self.knn)
                    scale = torch.clamp(within / Kij.sum(dim=1), max=1.0) * float(self.beta)   # graphs.py:1921-1925
                    K[ri[:, None], members[j].long()[None, :]] = Kij * scale[:, None]
        return K

    def _kernel_to_data_device(self, Y, theta=None):
        raise NotImplementedError

    def build_kernel_to_data(self, Y, theta=None):
        """Not implemented in the reference either (graphs.py:1938-1966)."""
        raise NotImplementedError
