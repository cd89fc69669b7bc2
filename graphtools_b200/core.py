"""Host-side mirror of graphtools' abstract graph machinery, re-plumbed onto the CUDA engine.

Public surface kept from the reference (citations relative to /root/reference/graphtools):
``Base`` (base.py:25-70), ``Data`` (base.py:72-424), ``BaseGraph`` (base.py:427-988, hot-path part)
and ``DataGraph`` (base.py:1046-1254): same constructor keywords, lazy cached properties
``K``/``kernel``, ``P``/``diff_op``, ``kernel_degree``, ``diff_aff``; same validation messages and
warnings; same result containers (scipy CSR float64/int32 for sparse graphs, ndarray for dense).

What differs: ``build_kernel`` implementations return *device-resident* results
(``pipeline.DeviceCSR`` / CUDA tensors); symmetrisation, anisotropy and the diffusion operator are
computed on the GPU in the same sweep and only materialised as scipy/numpy objects when a property
is read.  There is no CPU compute path.
"""
import abc
import inspect
import numbers
import warnings

import numpy as np
from scipy import sparse

from . import _engine as E
from . import pipeline
from .logging_util import logger as _logger


def _is_dataframe(x):
    try:
        import pandas as pd
        return isinstance(x, pd.DataFrame)
    except ImportError:  # pragma: no cover
        return False


def _is_anndata(x):
    try:
        import anndata
        return isinstance(x, anndata.AnnData)
    except ImportError:
        return False


class Base(object):
    """Keyword-argument sink at the end of the cooperative ``__init__`` chain."""

    def __init__(self):
        super().__init__()

    @classmethod
    def _get_param_names(cls):
        """Names of all constructor keywords of ``cls`` and its bases (used by ``api.Graph``
        to decide which of its arguments a class accepts; reference base.py:33-63)."""
        names = set()
        for klass in cls.__mro__:
            init = klass.__dict__.get("__init__")
            if init is None or klass is object:
                continue
            for p in inspect.signature(init).parameters.values():
                if p.name != "self" and p.kind not in (p.VAR_KEYWORD, p.VAR_POSITIONAL):
                    names.add(p.name)
        return names

    def set_params(self, **kwargs):
        return self


class Data(Base):
    """Data ingestion + optional PCA (host side, unchanged in spirit; reference base.py:72-424).

    PCA is outside the accelerated path (SURVEY.md section 2): it runs with scikit-learn on the host
    exactly as in the reference and its output ``data_nu`` is what the GPU kernels consume.
    """

    def __init__(self, data, n_pca=None, rank_threshold=None, random_state=None, **kwargs):
        if len(data.shape) != 2:
            msg = "Expected 2D array, got {}D array instead (shape: {}.) ".format(len(data.shape), data.shape)
            if len(data.shape) < 2:
                msg += ("\nReshape your data either using array.reshape(-1, 1) "
                        "if your data has a single feature or array.reshape(1, -1) if "
                        "it contains a single sample.")
            raise ValueError(msg)
        n_pca, rank_threshold = self._parse_n_pca_threshold(data, n_pca, rank_threshold)
        if _is_dataframe(data):
            try:
                data = data.sparse.to_coo()
            except AttributeError:
                data = np.array(data)
        elif _is_anndata(data):
            data = data.X
        self.data = data
        self.n_pca = n_pca
        self.rank_threshold = rank_threshold
        self.random_state = random_state
        self.data_nu = self._reduce_data()
        super().__init__(**kwargs)

    def _parse_n_pca_threshold(self, data, n_pca, rank_threshold):
        bad_type = ("n_pca was not an instance of numbers.Number, could not be cast to False, and not None. "
                    "Please supply an integer 0 <= n_pca < min(n_samples,n_features) or None")
        if isinstance(n_pca, str):
            n_pca = n_pca.lower()
            if n_pca != "auto":
                raise ValueError("n_pca must be an integer 0 <= n_pca < min(n_samples,n_features), "
                                 "or in [None, False, True, 'auto'].")
        if isinstance(n_pca, numbers.Number) and not isinstance(n_pca, bool):
            if not float(n_pca).is_integer():
                rounded = np.round(n_pca).astype(int)
                warnings.warn("Cannot perform PCA to fractional {} dimensions. Rounding to {}".format(n_pca, rounded),
                              RuntimeWarning)
                n_pca = rounded
            if n_pca < 0:
                raise ValueError("n_pca cannot be negative. Please supply an integer "
                                 "0 <= n_pca < min(n_samples,n_features) or None")
            elif np.min(data.shape) <= n_pca:
                warnings.warn("Cannot perform PCA to {} dimensions on data with min(n_samples, n_features) = {}"
                              .format(n_pca, np.min(data.shape)), RuntimeWarning)
                n_pca = 0
        if n_pca is True:
            n_pca = "auto"
            _logger.log_info("Estimating n_pca from matrix rank. Supply an integer n_pca for fixed amount.")
        elif n_pca is None or n_pca is False or (isinstance(n_pca, numbers.Number) and n_pca == 0):
            n_pca = None
        if not (n_pca is None or n_pca == "auto" or isinstance(n_pca, numbers.Number)):
            raise ValueError(bad_type)
        if rank_threshold is not None and n_pca != "auto":
            warnings.warn("n_pca = {}, therefore rank_threshold of {} will not be used. To use rank thresholding, "
                          "set n_pca = True".format(n_pca, rank_threshold), RuntimeWarning)
        if n_pca == "auto":
            if isinstance(rank_threshold, str):
                rank_threshold = rank_threshold.lower()
            if rank_threshold is None:
                rank_threshold = "auto"
            ok = (isinstance(rank_threshold, numbers.Number) and rank_threshold > 0) or rank_threshold == "auto"
            if not ok:
                raise ValueError("rank_threshold must be positive float or 'auto'. ")
        return n_pca, rank_threshold

    def _reduce_data(self):
        wants_pca = self.n_pca is not None and (self.n_pca == "auto" or self.n_pca < self.data.shape[1])
        if not wants_pca:
            data_nu = self.data
            if sparse.issparse(data_nu) and not isinstance(
                    data_nu, (sparse.csr_matrix, sparse.csc_matrix, sparse.bsr_matrix)):
                data_nu = data_nu.tocsr()
            return data_nu
        from sklearn.decomposition import PCA, TruncatedSVD
        import os
        impl = os.environ.get("GTB_PCA", "auto")
        if impl not in ("auto", "device", "host"):
            raise ValueError("GTB_PCA must be auto, device or host (got %r)" % (impl,))
        if impl == "auto":
            # the front-end is not part of the accelerated contract: without a GPU (host-side API use with
            # initialize=False) it stays the reference's own scikit-learn call
            import torch
            impl = "device" if torch.cuda.is_available() else "host"
        with _logger.log_task("PCA"):
            k = self.data.shape[1] - 1 if self.n_pca == "auto" else self.n_pca
            if sparse.issparse(self.data):
                if isinstance(self.data, (sparse.coo_matrix, sparse.lil_matrix, sparse.dok_matrix)):
                    self.data = self.data.tocsr()
            dev_nu = None
            if impl == "device":
                # same randomized SVD as sklearn's PCA / TruncatedSVD, in HBM (graphtools_b200/pca.py)
                from . import pca
                if sparse.issparse(self.data):
                    self.data_pca, dev_nu = pca.fit_transform_sparse(self.data, k, self.random_state)
                else:
                    self.data_pca, dev_nu = pca.fit_transform_dense(self.data, k, self.random_state)
            else:
                if sparse.issparse(self.data):
                    self.data_pca = TruncatedSVD(k, random_state=self.random_state)
                else:
                    self.data_pca = PCA(k, svd_solver="randomized", random_state=self.random_state)
                self.data_pca.fit(self.data)
            if self.n_pca == "auto":
                s = self.data_pca.singular_values_
                if self.rank_threshold == "auto":
                    self.rank_threshold = s.max() * np.finfo(self.data.dtype).eps * max(self.data.shape)
                gate = np.where(s >= self.rank_threshold)[0]
                self.n_pca = gate.shape[0]
                if self.n_pca == 0:
                    raise ValueError("Supplied threshold {} was greater than maximum singular value {} "
                                     "for the data matrix".format(self.rank_threshold, s.max()))
                _logger.log_info("Using rank estimate of {} as n_pca".format(self.n_pca))
                op = self.data_pca
                op.components_ = op.components_[gate, :]
                op.explained_variance_ = op.explained_variance_[gate]
                op.explained_variance_ratio_ = op.explained_variance_ratio_[gate]
                op.singular_values_ = op.singular_values_[gate]
                if dev_nu is not None:
                    import torch
                    dev_nu = dev_nu[:, torch.from_numpy(gate).to(dev_nu.device)].contiguous()
            if dev_nu is not None:
                # the reduced data stays in HBM for the graph build; the host copy is the public ``data_nu``
                self._dev_data_nu = dev_nu
                return pipeline.d2h_pinned(dev_nu).numpy()
            return self.data_pca.transform(self.data)

    def get_params(self):
        return {"n_pca": self.n_pca, "random_state": self.random_state}

    def set_params(self, **params):
        if "n_pca" in params and params["n_pca"] != self.n_pca:
            raise ValueError("Cannot update n_pca. Please create a new graph")
        if "random_state" in params:
            self.random_state = params["random_state"]
        super().set_params(**params)
        return self

    def transform(self, Y):
        """Map ``Y`` from the ambient space into the (PCA-)reduced space of ``data_nu``."""
        try:
            return self.data_pca.transform(Y)
        except ValueError:
            raise ValueError("data of shape {0} cannot be transformed to graph built on data of shape {1}. "
                             "Expected shape ({2}, {3})".format(Y.shape, self.data.shape, Y.shape[0],
                                                                self.data.shape[1]))
        except AttributeError:  # no PCA
            try:
                if Y.shape[1] != self.data.shape[1]:
                    raise ValueError
                return Y
            except IndexError:
                raise ValueError("data of shape {0} cannot be transformed to graph built on data of shape {1}. "
                                 "Expected shape ({2}, {3})".format(Y.shape, self.data.shape, Y.shape[0],
                                                                    self.data.shape[1]))
            except ValueError:
                raise ValueError("data of shape {0} cannot be transformed to graph built on data of shape {1}. "
                                 "Expected shape ({2}, {3})".format(Y.shape, self.data.shape, Y.shape[0],
                                                                    self.data.shape[1]))

    def inverse_transform(self, Y, columns=None):
        """Map ``Y`` from the reduced space back to the ambient space (base.py:368-424)."""
        try:
            if not hasattr(self, "data_pca"):
                try:
                    if Y.shape[1] != self.data_nu.shape[1]:
                        raise ValueError
                except IndexError:              # len(Y.shape) < 2
                    raise ValueError
                if columns is None:
                    return Y
                columns = np.array([columns]).flatten()
                return Y[:, columns]
            if columns is None:
                return self.data_pca.inverse_transform(Y)
            columns = np.array([columns]).flatten()
            Y_inv = np.dot(Y, self.data_pca.components_[:, columns])
            if hasattr(self.data_pca, "mean_"):
                Y_inv += self.data_pca.mean_[columns]
            return Y_inv
        except ValueError:
            raise ValueError("data of shape {0} cannot be inverse transformed from graph built on reduced data of "
                             "shape ({1}, {2}). Expected shape ({3}, {2})".format(
                                 Y.shape, self.data_nu.shape[0], self.data_nu.shape[1], Y.shape[0]))


class BaseGraph(Base, metaclass=abc.ABCMeta):
    """Kernel -> symmetrise -> anisotropy -> diffusion operator (reference base.py:427-724).

    Subclasses implement ``build_kernel()`` returning either a ``pipeline.DeviceCSR`` (sparse graphs)
    or a float64 CUDA tensor [N, N] (dense graphs); this class finishes it on the device.
    """

    def __init__(self, kernel_symm="+", theta=None, anisotropy=0, gamma=None, initialize=True, **kwargs):
        if gamma is not None:
            warnings.warn("gamma is deprecated. Setting theta={}".format(gamma), FutureWarning)
            theta = gamma
        for old in ("gamma", "theta"):
            if kernel_symm == old:
                warnings.warn("kernel_symm='{}' is deprecated. Setting kernel_symm='mnn'".format(old), FutureWarning)
                kernel_symm = "mnn"
        self.kernel_symm = kernel_symm
        self.theta = theta
        self._check_symmetrization(kernel_symm, theta)
        if not (isinstance(anisotropy, numbers.Real) and 0 <= anisotropy <= 1):
            raise ValueError("Expected 0 <= anisotropy <= 1. Got {}".format(anisotropy))
        self.anisotropy = anisotropy
        if initialize:
            # build on the device now (as the reference builds K in the constructor, base.py:501-503);
            # the host copy is only materialised when .K / .kernel is read
            _logger.log_debug("Initializing kernel...")
            self._ensure_built()
        else:
            _logger.log_debug("Not initializing kernel.")
        super().__init__(**kwargs)

    def _check_symmetrization(self, kernel_symm, theta):
        if kernel_symm not in ["+", "*", "mnn", None]:
            raise ValueError("kernel_symm '{}' not recognized. Choose from '+', '*', 'mnn', or 'none'."
                             .format(kernel_symm))
        elif kernel_symm != "mnn" and theta is not None:
            warnings.warn("kernel_symm='{}' but theta is not None. Setting kernel_symm='mnn'.".format(kernel_symm))
            self.kernel_symm = kernel_symm = "mnn"
        if kernel_symm == "mnn":
            if theta is None:
                self.theta = theta = 1
                warnings.warn("kernel_symm='mnn' but theta not given. Defaulting to theta={}.".format(self.theta))
            elif not isinstance(theta, numbers.Number) or theta < 0 or theta > 1:
                raise ValueError("theta {} not recognized. Expected a float between 0 and 1".format(theta))

    # ---------------------------------------------------------------- device-side build
    def _build_kernel(self):
        """build -> symmetrise -> anisotropy -> sanity checks, all on the GPU (base.py:534-555)."""
        raw = self.build_kernel()
        if isinstance(raw, pipeline.DeviceCSR):
            K, P, degree, flags = pipeline.symmetrize_normalize(
                raw, self.kernel_symm, self.theta, float(self.anisotropy))
            self._dev_kernel, self._dev_P, self._dev_degree = K, P, degree
            if flags & 1:
                warnings.warn("K should be symmetric", RuntimeWarning)
            if flags & 2:
                warnings.warn("K should have a non-zero diagonal", RuntimeWarning)
            return K
        return self._finish_dense_kernel(raw)

    def _finish_dense_kernel(self, raw):
        """Dense raw kernel (CUDA tensor [N, N]) -> symmetrise, anisotropy, sanity checks, degree, P
        (base.py:534-592, :645 on an ndarray kernel)."""
        import torch
        from . import dense
        K = dense.symmetrize_dense(raw, self.kernel_symm, self.theta).contiguous()
        if self.anisotropy != 0:
            dense.anisotropy_dense(K, self.anisotropy)
        if float((K - K.T).max().item()) > 1e-5:
            warnings.warn("K should be symmetric", RuntimeWarning)
        if bool((torch.diagonal(K) == 0).any().item()):
            warnings.warn("K should have a non-zero diagonal", RuntimeWarning)
        self._dev_degree = dense.rowsum_dense(K)
        self._dev_P = dense.row_normalize_dense(K, self._dev_degree)
        self._dev_kernel = K
        return K

    def _ensure_built(self):
        d = self.__dict__
        if "_dev_kernel" in d or "_dev_shard" in d:
            return
        if "_kernel" in d:
            # host views only (an unpickled graph): put the kernel back into HBM so that every device-side
            # consumer (diffuse, landmark operator, extension, spectral clusters) keeps working
            self._restore_device_state()
            return
        K = self._build_kernel()
        if K is not None:
            self._dev_kernel = K

    def _restore_device_state(self):
        K = self._kernel
        if sparse.issparse(K):
            Kd = pipeline.csr_from_scipy(K)
            self._dev_kernel = Kd
            self._dev_degree = pipeline.row_sums(Kd)
            self._dev_P = pipeline.row_normalize(Kd)
        else:
            import torch
            from . import dense
            Kd = torch.from_numpy(np.ascontiguousarray(K, dtype=np.float64)).to(pipeline._dev())
            self._dev_kernel = Kd
            self._dev_degree = dense.rowsum_dense(Kd)
            self._dev_P = dense.row_normalize_dense(Kd, self._dev_degree)

    def __getattr__(self, name):
        # A row-sharded multi-GPU build keeps only this rank's rows of K / P in HBM (``_dev_shard``); the first
        # consumer that needs the complete device matrices triggers one NCCL all-gather (collective: every rank
        # reaches it, because every rank runs the same program).
        if name in ("_dev_kernel", "_dev_P", "_dev_degree") and "_dev_shard" in self.__dict__:
            self._gather_shards()
            return self.__dict__[name]
        raise AttributeError("'{}' object has no attribute '{}'".format(type(self).__name__, name))

    def _gather_shards(self):
        from . import distributed as gd
        sh = self.__dict__["_dev_shard"]
        heights = [b[1] - b[0] for b in sh["bounds"]]
        full_ptr, full_idx, full_val = gd.allgather_csr_rows(sh["row_len"], sh["indices"], sh["data"], heights,
                                                             pipeline.exclusive_scan)
        nnz_all = gd.allgather_counts(sh["indices"].shape[0], sh["indices"].device)
        n = sh["n"]
        self.__dict__["_dev_kernel"] = pipeline.DeviceCSR(full_ptr, full_idx, full_val, (n, n))
        self.__dict__["_dev_P"] = gd._allgather_padded(sh["P"], nnz_all)
        self.__dict__["_dev_degree"] = gd._allgather_padded(sh["degree"], heights)

    def _materialize_shards(self):
        """Host K and P of a row-sharded build: every rank copies ITS rows device->host into a shared-memory segment
        (parallel PCIe links, parallel first-touch), then all ranks view the complete scipy matrices zero-copy.
        Collective."""
        import torch
        from . import _engine as E
        from . import distributed as gd
        sh = self.__dict__["_dev_shard"]
        bounds, n = sh["bounds"], sh["n"]
        rank = gd.dist.get_rank()
        lo, hi = bounds[rank]
        nnz_all = gd.allgather_counts(sh["indices"].shape[0], sh["indices"].device)
        nnz = int(sum(nnz_all))
        off = int(sum(nnz_all[:rank]))
        from . import hostpool
        specs = [("indptr", n + 1, np.int32), ("indices", nnz, np.int32), ("K", nnz, np.float64),
                 ("P", nnz, np.float64), ("degree", n, np.float64)]
        lay, total = hostpool.layout(specs)
        blk = hostpool.take_shared(total)
        if blk is not None:
            # one recycled page-locked shared segment: every rank DMAs its own shard straight into its slice
            arr = blk.carve(lay)
            m = hi - lo
            if m > 0:
                ip32 = pipeline._empty((m + 1,), torch.int32)
                E.call("gtb_cast_indptr", sh["indptr"], m + 1, ip32)
                ip32 += off
                hostpool.d2h_async(ip32[:m], arr["indptr"][lo:hi])
                hostpool.d2h_async(sh["indices"], arr["indices"][off:off + nnz_all[rank]])
                hostpool.d2h_async(sh["data"], arr["K"][off:off + nnz_all[rank]])
                hostpool.d2h_async(sh["P"], arr["P"][off:off + nnz_all[rank]])
                hostpool.d2h_async(sh["degree"], arr["degree"][lo:hi])
            if rank == 0:
                arr["indptr"][bounds[-1][1]:] = nnz
            torch.cuda.current_stream().synchronize()
            gd.dist.barrier()                                  # every shard has landed
            if rank != 0:
                for a in arr.values():
                    a.flags.writeable = False
            K = sparse.csr_matrix((arr["K"], arr["indices"], arr["indptr"]), shape=(n, n), copy=False)
            P = sparse.csr_matrix((arr["P"], arr["indices"], arr["indptr"]), shape=(n, n), copy=False)
            for M in (K, P):
                M.has_sorted_indices = True
                M.has_canonical_format = True
            self._kernel, self._diff_op = K, P
            self._kernel_degree = arr["degree"].reshape(-1, 1)
            return
        if not gd.SharedResult.available(24 * nnz + 4 * (n + 1)):
            # no room in /dev/shm: assemble on the device, copy the whole matrix on every rank
            self._kernel = self._dev_kernel.to_scipy()
            self._diff_op = self._dev_kernel.to_scipy(self._dev_P)
            self._kernel_degree = self._dev_degree.cpu().numpy().reshape(-1, 1)
            return
        res = gd.SharedResult()
        arr = res.create({"indptr": (n + 1, np.int32), "indices": (nnz, np.int32), "K": (nnz, np.float64),
                          "P": (nnz, np.float64), "degree": (n, np.float64)})
        m = hi - lo
        if m > 0:
            ip32 = pipeline._empty((m + 1,), torch.int32)
            E.call("gtb_cast_indptr", sh["indptr"], m + 1, ip32)
            ip32 += off
            # slice [lo, hi) of the global row pointers; the entry at `hi` is written by the next rank (or below)
            pipeline.d2h_into(ip32[:m], arr["indptr"][lo:hi])
            pipeline.d2h_into(sh["indices"], arr["indices"][off:off + nnz_all[rank]])
            pipeline.d2h_into(sh["data"], arr["K"][off:off + nnz_all[rank]])
            pipeline.d2h_into(sh["P"], arr["P"][off:off + nnz_all[rank]])
            pipeline.d2h_into(sh["degree"], arr["degree"][lo:hi])
        if rank == 0:
            arr["indptr"][bounds[-1][1]:] = nnz            # rows past the last non-empty shard, and the end marker
        torch.cuda.current_stream().synchronize()
        arr = res.finish(arr)
        K = sparse.csr_matrix((arr["K"], arr["indices"], arr["indptr"]), shape=(n, n), copy=False)
        P = sparse.csr_matrix((arr["P"], arr["indices"], arr["indptr"]), shape=(n, n), copy=False)
        for M in (K, P):
            M.has_sorted_indices = True
            M.has_canonical_format = True
        self._kernel, self._diff_op = K, P
        self._kernel_degree = arr["degree"].reshape(-1, 1)

    def symmetrize_kernel(self, K):
        """Host-callable symmetrisation of an arbitrary scipy / numpy kernel on the GPU."""
        from .hostops import symmetrize_host_matrix
        return symmetrize_host_matrix(K, self.kernel_symm, self.theta)

    def apply_anisotropy(self, K):
        if self.anisotropy == 0:
            return K
        from .hostops import anisotropy_host_matrix
        return anisotropy_host_matrix(K, self.anisotropy)

    def get_params(self):
        return {"kernel_symm": self.kernel_symm, "theta": self.theta, "anisotropy": self.anisotropy}

    def set_params(self, **params):
        for name in ("theta", "anisotropy", "kernel_symm"):
            if name in params and params[name] != getattr(self, name):
                raise ValueError("Cannot update {}. Please create a new graph".format(name))
        super().set_params(**params)
        return self

    # ---------------------------------------------------------------- cached host views
    @property
    def K(self):
        """Kernel matrix (scipy CSR or ndarray), materialised from HBM on first access."""
        if "_kernel" not in self.__dict__:
            self._ensure_built()
            if "_dev_shard" in self.__dict__ and "_dev_kernel" not in self.__dict__:
                self._materialize_shards()
            else:
                self._kernel = self._materialize(self._dev_kernel)
        return self._kernel

    @property
    def kernel(self):
        return self.K

    @property
    def P(self):
        """Diffusion operator = row-L1-normalised kernel (base.py:629-646)."""
        if "_diff_op" not in self.__dict__:
            self._ensure_built()
            if "_dev_shard" in self.__dict__ and "_dev_kernel" not in self.__dict__:
                self._materialize_shards()
                return self._diff_op
            K = self._dev_kernel
            if isinstance(K, pipeline.DeviceCSR):
                if getattr(self, "_dev_P", None) is None:
                    self._dev_P = pipeline.row_normalize(K)
                self._diff_op = K.to_scipy(self._dev_P)
            else:
                self._diff_op = self._dev_P.cpu().numpy()
        return self._diff_op

    @property
    def diff_op(self):
        return self.P

    @property
    def kernel_degree(self):
        """Row sums of the kernel, shape [N, 1] (base.py:648-666)."""
        if "_kernel_degree" not in self.__dict__:
            self._ensure_built()
            self._kernel_degree = self._dev_degree.cpu().numpy().reshape(-1, 1)
        return self._kernel_degree

    @property
    def diff_aff(self):
        """Symmetric diffusion affinity D^-1/2 K D^-1/2 (base.py:668-698)."""
        self._ensure_built()
        Kd = getattr(self, "_dev_kernel", None)
        if isinstance(Kd, pipeline.DeviceCSR):
            # K_ij / (d_i d_j)^(1/2) on the device: the anisotropy kernel with alpha = 1/2 on a copy of the values
            from . import _engine as E
            vals = Kd.data.clone()
            E.call("gtb_anisotropy", Kd.indptr, Kd.indices, vals, self._dev_degree, 0.5, Kd.shape[0])
            return Kd.to_scipy(vals)
        deg = self.kernel_degree
        K = self.kernel
        if sparse.issparse(K):
            n = len(deg)
            D = sparse.csr_matrix((1 / np.sqrt(deg.flatten()), np.arange(n), np.arange(n + 1)))
            return D @ K @ D
        return (K / np.sqrt(deg)) / np.sqrt(deg.T)

    def diffuse(self, signal, t=1, return_device=False):
        """``P^t . signal`` by ``t`` repeated products with the device-resident diffusion operator -- what the
        callers (MAGIC-style imputation) do with ``G.diff_op`` on the host, without materialising P there.
        Each product is bit-identical to ``G.diff_op.dot(x)``."""
        import torch
        self._ensure_built()
        K = self._dev_kernel
        one_d = np.ndim(signal) == 1
        if isinstance(signal, torch.Tensor):
            x = signal.to(device=pipeline._dev(), dtype=torch.float64).reshape(signal.shape[0], -1).contiguous()
        else:
            x = pipeline.to_device(np.asarray(signal, dtype=np.float64).reshape(len(signal), -1))
        if isinstance(K, pipeline.DeviceCSR):
            if getattr(self, "_dev_P", None) is None:
                self._dev_P = pipeline.row_normalize(K)
            for _ in range(int(t)):
                x = pipeline.spmm(K, x, self._dev_P)
        else:
            from . import dense
            if self._dev_P.shape[1] <= E.lib().gtb_gemm_max_k():
                # dense graph: float64-faithful products on the int8 tensor cores; P is sliced once for all t steps
                Pd = dense.slice_operand(self._dev_P.contiguous(), False)
                for _ in range(int(t)):
                    x = dense.gemm_digits(Pd, dense.slice_operand(x, True), self._dev_P.shape[0], x.shape[1])
            else:
                for _ in range(int(t)):
                    x = torch.matmul(self._dev_P, x)
        if return_device:
            return x[:, 0] if one_d else x
        x = x.cpu().numpy()
        return x[:, 0] if one_d else x

    @property
    def weighted(self):
        """True when the kernel holds affinities (``decay is not None``) rather than a binary adjacency."""
        return getattr(self, "decay", None) is not None

    def shortest_path(self, method="auto", distance=None):
        """Length of the shortest path between every pair of vertices (reference base.py:934-988), float64 [N, N].

        ``distance`` sets the edge lengths on every stored entry of K: "constant" (K_ij itself; unweighted graphs),
        "data" (Euclidean distance between the rows of ``data_nu``; unweighted graphs) or "affinity" (-log K_ij;
        weighted graphs); None picks "data" for unweighted and "affinity" for weighted graphs.  Paths are directed
        along K's rows; the result is then averaged with its transpose, pairs at distance 0 (duplicate points) or
        without a path get inf, and the diagonal is 0.  ``method`` is checked against scipy's names ("auto", "FW",
        "D", "BF", "J"); every method yields the float64 fixpoint of the edge relaxations, which is bit-identical
        to scipy's Dijkstra (FW rounds differently, within 1e-12 relative).  Negative lengths (affinities above 1,
        possible with anisotropy > 0) raise NotImplementedError.  Runs on the device (csrc/paths.cu)."""
        from . import paths
        return paths.shortest_path(self, method=method, distance=distance)

    @staticmethod
    def _materialize(dev):
        if isinstance(dev, pipeline.DeviceCSR):
            return dev.to_scipy()
        return dev.cpu().numpy()

    @abc.abstractmethod
    def build_kernel(self):
        """Build the raw (unsymmetrised) kernel on the device."""
        raise NotImplementedError

    def __getstate__(self):
        # device handles do not pickle: materialise the host views first (base.py:887-902 contract)
        state = dict(self.__dict__)
        if any(k.startswith("_dev_") for k in state):
            self.K, self.P, self.kernel_degree
            state = dict(self.__dict__)
        for k in [k for k in state if k.startswith("_dev_") or k in ("_ref_operand", "_knn_tree")]:
            del state[k]
        return state

    def to_pickle(self, path):
        import pickle
        with open(path, "wb") as f:
            pickle.dump(self, f, protocol=pickle.HIGHEST_PROTOCOL)


class DataGraph(Data, BaseGraph, metaclass=abc.ABCMeta):
    """Graph built from a data matrix (reference base.py:1046-1254)."""

    def __init__(self, data, verbose=True, n_jobs=1, **kwargs):
        self.n_jobs = n_jobs
        self.verbose = verbose
        _logger.set_level(verbose)
        super().__init__(data, **kwargs)

    def get_params(self):
        params = Data.get_params(self)
        params.update(BaseGraph.get_params(self))
        return params

    @abc.abstractmethod
    def build_kernel_to_data(self, Y):
        raise NotImplementedError

    def _check_extension_shape(self, Y):
        if len(Y.shape) != 2:
            raise ValueError("Expected a 2D matrix. Y has shape {}".format(Y.shape))
        if not Y.shape[1] == self.data_nu.shape[1]:
            if Y.shape[1] == self.data.shape[1]:
                Y = self.transform(Y)
            else:
                if self.data.shape[1] != self.data_nu.shape[1]:
                    msg = "Y must be of shape either (n, {}) or (n, {})".format(self.data.shape[1],
                                                                                 self.data_nu.shape[1])
                else:
                    msg = "Y must be of shape (n, {})".format(self.data.shape[1])
                raise ValueError(msg)
        return Y

    def _extend_to_data_device(self, Y):
        """Out-of-sample transition matrix kept in HBM: (DeviceCSR, normalised values) for sparse graphs,
        a float64 CUDA tensor for dense graphs."""
        Y = self._check_extension_shape(Y)
        dev = self._kernel_to_data_device(Y)
        if isinstance(dev, pipeline.DeviceCSR):
            return dev, pipeline.row_normalize(dev)
        from .dense import row_normalize_dense
        return row_normalize_dense(dev), None

    def extend_to_data(self, Y):
        """Transition matrix from new points ``Y`` to the graph's samples (base.py:1166-1193):
        out-of-sample kernel, L1-row-normalised on the device."""
        T, vals = self._extend_to_data_device(Y)
        if vals is not None:
            return T.to_scipy(vals)
        return T.cpu().numpy()

    def interpolate(self, transform, transitions=None, Y=None):
        """``transitions.dot(transform)`` (base.py:1195-1229) as a device-resident chain: the out-of-sample
        kernel, its normalisation and the sparse x dense product (csrc/spmm.cu) never leave HBM; only the
        interpolated [n_y, f] array is copied back.  A caller-supplied ``transitions`` (scipy / ndarray) is
        uploaded and multiplied the same way; the product is bit-identical to scipy's."""
        import torch
        if transitions is None:
            if Y is None:
                raise ValueError("Either `transitions` or `Y` must be provided.")
            T, vals = self._extend_to_data_device(Y)
        elif sparse.issparse(transitions):
            T, vals = pipeline.csr_from_scipy(transitions), None
        else:
            T, vals = pipeline.to_device(np.asarray(transitions, dtype=np.float64)), None
        one_d = np.ndim(transform) == 1
        B = pipeline.to_device(np.asarray(transform, dtype=np.float64).reshape(len(transform), -1))
        if isinstance(T, pipeline.DeviceCSR):
            out = pipeline.spmm(T, B, vals)
        else:
            out = torch.matmul(T, B)          # dense transitions (exact graphs): plain library GEMM
        out = out.cpu().numpy()
        return out[:, 0] if one_d else out

    def set_params(self, **params):
        if "n_jobs" in params:
            self.n_jobs = params["n_jobs"]
        if "verbose" in params:
            self.verbose = params["verbose"]
            _logger.set_level(self.verbose)
        super().set_params(**params)
        return self

    # helper shared by the sparse graph types -------------------------------------------------
    def _dense_f32(self, A):
        """Densify (scipy sparse -> ndarray) and hand to the device: float64 inputs stay float64 (exact
        distances are evaluated on them), everything else becomes float32."""
        import torch
        if A is getattr(self, "data_nu", None) and getattr(self, "_dev_data_nu", None) is not None:
            return self._dev_data_nu
        if isinstance(A, torch.Tensor):
            return pipeline.to_device(A)
        if sparse.issparse(A):
            A = A.toarray()
        return pipeline.to_device(np.asarray(A))
