"""kNNGraph on the CUDA engine (reference graphtools/graphs.py:562-982).

Constructor arguments, validation, warnings and ``get_params``/``set_params`` follow the reference;
``build_kernel`` / ``build_kernel_to_data`` run the fused distance/top-k + float64 refine pipeline
(pipeline.knn_kernel) instead of sklearn ``NearestNeighbors`` + the Python CSR loop.
"""
import warnings

import numpy as np
from scipy import sparse

from . import pipeline
from .core import DataGraph
from .logging_util import logger as _logger


def search_schedule(count_ge, nq, n_ref, knn, knn_max, search_multiplier):
    """Replay of the reference's search escalation (graphs.py:882-948) from neighbour counts.

    ``count_ge(s)`` is the number of query rows (all ``nq`` of them, over every rank) with at least ``s`` reference
    points strictly inside their kernel radius.  The reference searches ``s`` neighbours per row and keeps a row to do
    when all ``s`` lie inside the radius, i.e. exactly when its count is >= s; whether it searches wider follows from
    the number of such rows.  Returns ``(s_todo, search_knn, n_todo)``: after the last kNN pass the rows with a count
    >= ``s_todo`` are still to do (``n_todo`` of them), and ``search_knn`` is the width of the step that finishes
    them.  When ``search_knn > n_ref / 2`` the reference finishes those rows on a new brute-force search built without
    its ``metric`` argument, i.e. with Euclidean distances."""
    knn = min(knn, n_ref)
    knn_max = n_ref if knn_max is None else knn_max
    s = min(knn * search_multiplier, knn_max)
    s_todo, n_todo = s, count_ge(s)
    s_next = min(s * search_multiplier, knn_max)
    while n_todo > nq // 10 and s_next < n_ref / 2 and s_next < knn_max and s_next > s_todo:
        s_todo, n_todo = s_next, count_ge(s_next)
        s_next = min(s_next * search_multiplier, knn_max)
    return s_todo, s_next, n_todo


def _schedule_widths(n_ref, knn, knn_max, search_multiplier):
    """Every search width ``search_schedule`` can ask ``count_ge`` about, in order."""
    knn = min(knn, n_ref)
    knn_max = n_ref if knn_max is None else knn_max
    s = min(knn * search_multiplier, knn_max)
    widths = [s]
    s = min(s * search_multiplier, knn_max)
    while s < n_ref / 2 and s < knn_max and s > widths[-1]:
        widths.append(s)
        s = min(s * search_multiplier, knn_max)
    return widths


def _splice_rows(R, rows, R2):
    """DeviceCSR ``R`` with its rows ``rows`` (int64 device tensor) replaced by the rows of ``R2``, in that order.
    Rows of both matrices are sorted by column, so a stable sort of all entries by row keeps them sorted."""
    import torch
    n = R.shape[0]
    dev = R.indices.device
    lens = R.indptr[1:] - R.indptr[:-1]
    lens2 = R2.indptr[1:] - R2.indptr[:-1]
    replaced = torch.zeros((n,), dtype=torch.bool, device=dev)
    replaced[rows] = True
    row_of = torch.repeat_interleave(torch.arange(n, device=dev), lens)
    keep = ~replaced[row_of]
    all_rows = torch.cat([row_of[keep], torch.repeat_interleave(rows, lens2)])
    order = torch.argsort(all_rows, stable=True)
    idx = torch.cat([R.indices[keep], R2.indices])[order].contiguous()
    val = torch.cat([R.data[keep], R2.data])[order].contiguous()
    new_lens = lens.clone()
    new_lens[rows] = lens2
    indptr = torch.zeros((n + 1,), dtype=torch.int64, device=dev)
    torch.cumsum(new_lens, dim=0, out=indptr[1:])
    return pipeline.DeviceCSR(indptr, idx, val, R.shape)


def _zero_distance_pairs(X, rows, metric):
    """{(j, i)}: every sample j < i at distance exactly 0 from row i, for each i in ``rows`` (the rows with more than one
    zero-distance candidate) -- the pairs the reference names from its neighbour indices (graphs.py:787-817).  Under
    correlation these include affine copies a x + b (a > 0), which are not equal rows."""
    import torch
    from . import dense
    D = dense.dense_distances(X[torch.from_numpy(rows).to(X.device)], X, metric)
    return {(int(j), int(rows[r])) for r, j in (D == 0).nonzero().cpu().tolist() if j < rows[r]}


class kNNGraph(DataGraph):
    """K nearest neighbours graph, optionally with alpha-decay affinities."""

    def __init__(self, data, knn=5, decay=None, knn_max=None, search_multiplier=6, bandwidth=None,
                 bandwidth_scale=1.0, distance="euclidean", thresh=1e-4, n_pca=None, **kwargs):
        if decay is not None:
            if thresh <= 0 and knn_max is None:
                raise ValueError("Cannot instantiate a kNNGraph with `decay=None`, "
                                 "`thresh=0` and `knn_max=None`. Use a TraditionalGraph instead.")
            elif thresh < np.finfo(float).eps:
                thresh = np.finfo(float).eps
        if callable(bandwidth):
            raise NotImplementedError("Callable bandwidth is only supported by"
                                      " graphtools.graphs.TraditionalGraph.")
        if knn is None and bandwidth is None:
            raise ValueError("Either `knn` or `bandwidth` must be provided.")
        elif knn is None and bandwidth is not None:
            knn = 5  # the implementation needs some knn value
        if decay is None and bandwidth is not None:
            warnings.warn("`bandwidth` is not used when `decay=None`.", UserWarning)
        if knn > data.shape[0] - 2:
            warnings.warn("Cannot set knn ({k}) to be greater than "
                          "n_samples - 2 ({n}). Setting knn={n}".format(k=knn, n=data.shape[0] - 2))
            knn = data.shape[0] - 2
        if knn_max is not None and knn_max < knn:
            warnings.warn("Cannot set knn_max ({knn_max}) to be less than "
                          "knn ({knn}). Setting knn_max={knn}".format(knn=knn, knn_max=knn_max))
            knn_max = knn
        if n_pca in [None, 0, False] and data.shape[1] > 500:
            warnings.warn("Building a kNNGraph on data of shape {} is "
                          "expensive. Consider setting n_pca.".format(data.shape), UserWarning)
        if distance not in pipeline.METRIC_NAMES:
            raise NotImplementedError(pipeline.unsupported_metric_message(distance))
        self.knn = knn
        self.knn_max = knn_max
        self.search_multiplier = search_multiplier
        self.decay = decay
        self.bandwidth = bandwidth
        self.bandwidth_scale = bandwidth_scale
        self.distance = distance
        self.thresh = thresh
        super().__init__(data, n_pca=n_pca, **kwargs)

    def get_params(self):
        params = super().get_params()
        params.update({"knn": self.knn, "decay": self.decay, "bandwidth": self.bandwidth,
                       "bandwidth_scale": self.bandwidth_scale, "knn_max": self.knn_max,
                       "distance": self.distance, "thresh": self.thresh, "n_jobs": self.n_jobs,
                       "random_state": self.random_state, "verbose": self.verbose})
        return params

    def set_params(self, **params):
        if "knn" in params and params["knn"] != self.knn:
            raise ValueError("Cannot update knn. Please create a new graph")
        # the reference compares knn_max with self.knn (graphs.py:721); kept as is
        if "knn_max" in params and params["knn_max"] != self.knn:
            raise ValueError("Cannot update knn_max. Please create a new graph")
        for name in ("decay", "bandwidth", "bandwidth_scale", "distance"):
            if name in params and params[name] != getattr(self, name):
                raise ValueError("Cannot update {}. Please create a new graph".format(name))
        if "thresh" in params and params["thresh"] != self.thresh and self.decay != 0:
            raise ValueError("Cannot update thresh. Please create a new graph")
        if "n_jobs" in params:
            self.n_jobs = params["n_jobs"]
        if "random_state" in params:
            self.random_state = params["random_state"]
        if "verbose" in params:
            self.verbose = params["verbose"]
        super().set_params(**params)
        return self

    # ------------------------------------------------------------------ device side
    @property
    def knn_tree(self):
        """The fitted search structure: the device-resident search operand of ``data_nu``
        (centred k-major copy + norms).  Stands in for the reference's sklearn NearestNeighbors
        (graphs.py:748-769)."""
        if "_ref_operand" not in self.__dict__:
            rows = self._reference_rows()
            pipeline.reject_constant_rows(rows, self.distance)
            self._ref_operand = pipeline.SearchOperand(rows, metric=self.distance)
        return self._ref_operand

    def _reference_rows(self):
        """``data_nu`` in HBM.  One process per GPU: every rank uploads its own row block of the host array and the
        blocks are assembled by an NCCL all-gather (SURVEY section 8e, collective 1) instead of every rank copying all
        of X across its PCIe link."""
        import torch
        from . import distributed as gd
        A = self.data_nu
        host_dense = isinstance(A, np.ndarray) or (isinstance(A, torch.Tensor) and not A.is_cuda)
        if (gd.active() and host_dense and getattr(self, "_dev_data_nu", None) is None
                and A.shape[0] >= gd.MIN_ROWS_PER_RANK * gd.world_size()):
            is64 = (A.dtype == np.float64) if isinstance(A, np.ndarray) else (A.dtype == torch.float64)
            return gd.upload_sharded(A, torch.float64 if is64 else torch.float32, pipeline._dev())
        return self._dense_f32(A)

    def build_kernel(self):
        """Raw in-sample kernel: every sample queried against all samples with knn+1 neighbours
        (self included), graphs.py:771-785."""
        knn_max = self.knn_max + 1 if self.knn_max else None
        from . import distributed as gd
        with _logger.log_task("KNN search"):
            ref = self.knn_tree
            if gd.active() and np.ndim(self.bandwidth) == 0:
                return self._build_kernel_sharded(ref, knn_max)
            R, info = self._kernel_device(ref, ref, knn=self.knn + 1, knn_max=knn_max,
                                          bandwidth=self.bandwidth, bandwidth_scale=self.bandwidth_scale)
        self._check_duplicates(info, ref, ref)
        self._dev_bandwidth = info["bandwidth"]
        return R

    def _local_raw_rows(self, ref, knn_max, Xq=None, knn=None, bandwidth=None, bandwidth_scale=None):
        """(bounds, indptr, row_len int32 [m], indices, data, info) of this rank's raw kernel rows [lo, hi) of the
        query set ``Xq`` (default: the reference set itself, i.e. the in-sample build)."""
        import torch
        import torch.distributed as dist
        from . import distributed as gd
        world, rank = dist.get_world_size(), dist.get_rank()
        Xq = ref.X if Xq is None else Xq
        knn = self.knn + 1 if knn is None else knn
        bandwidth = self.bandwidth if bandwidth is None else bandwidth
        bandwidth_scale = self.bandwidth_scale if bandwidth_scale is None else bandwidth_scale
        bounds = [gd.shard_bounds(Xq.shape[0], world, r) for r in range(world)]
        lo, hi = bounds[rank]
        dev = ref.X.device
        if hi > lo:
            qry = pipeline.SearchOperand(Xq[lo:hi], mean=ref.mean, metric=ref.metric)
            Rl, info = self._kernel_device(qry, ref, knn=knn, knn_max=knn_max, bandwidth=bandwidth,
                                           bandwidth_scale=bandwidth_scale, nq_total=Xq.shape[0])
            return (bounds, Rl.indptr, (Rl.indptr[1:] - Rl.indptr[:-1]).to(torch.int32), Rl.indices, Rl.data,
                    info)
        z = torch.zeros((0,), dtype=torch.int32, device=dev)
        if ref.metric != "euclidean" and not (self.decay is None or self.thresh == 1):
            self._fallback_plan(z, ref.n, knn, knn_max, Xq.shape[0])      # the other ranks' replay is collective
        return (bounds, torch.zeros((1,), dtype=torch.int64, device=dev), z, z,
                torch.zeros((0,), dtype=torch.float64, device=dev), {"nzero": z, "bandwidth": None})

    def _build_kernel_sharded(self, ref, knn_max):
        """One process per GPU, raw kernel only (used when the symmetrisation cannot be sharded): this rank
        builds the rows of its contiguous query shard against the replicated reference set, the raw CSR
        shards are all-gathered (NCCL) and every rank continues with the complete matrix."""
        from . import distributed as gd
        bounds, _, row_len, idx, val, _ = self._local_raw_rows(ref, knn_max)
        n = ref.n
        indptr, idx, val = gd.allgather_csr_rows(row_len, idx, val, [b[1] - b[0] for b in bounds],
                                                 pipeline.exclusive_scan)
        return pipeline.DeviceCSR(indptr, idx, val, (n, n))

    def _build_kernel(self):
        """Sharded build when torch.distributed is initialised (SURVEY section 8e): rows are sharded, every raw edge
        (i, j, w) is routed to the owner of column j with one NCCL all-to-all of packed records (bucketed by kernels,
        csrc/symm.cu route_count / route_fill), each rank turns what it received into the rows of the transposed matrix
        (records_count / scan / records_scatter / csr_sort_rows), merges them with its raw rows and normalises its
        shard with the same kernel as the single-GPU build (sym_merge) -- bit-identical for any rank count.  The
        result stays row-sharded in HBM (``_dev_shard``); the complete K / P are assembled on demand
        (core.BaseGraph._gather_shards on the device, _materialize_shards on the host)."""
        from . import distributed as gd
        sharded = (gd.active() and np.ndim(self.bandwidth) == 0 and self.anisotropy == 0
                   and self.kernel_symm in ("+", "*", "mnn"))
        if not sharded:
            return super()._build_kernel()
        import torch
        import torch.distributed as dist
        from . import _engine as E
        knn_max = self.knn_max + 1 if self.knn_max else None
        ref = self.knn_tree
        n = ref.n
        with _logger.log_task("KNN search"):
            bounds, indptr_a, row_len, idx, val, info = self._local_raw_rows(ref, knn_max)
        rank = dist.get_rank()
        lo, hi = bounds[rank]
        m = hi - lo
        dev = idx.device
        rec = gd.exchange_edges(indptr_a, idx, val, lo, bounds)
        mode = pipeline.SYM_MODES[self.kernel_symm]
        theta = 0.0 if self.theta is None else float(self.theta)
        flags = pipeline._zeros((1,), torch.int32)
        if m > 0:
            k = rec.shape[0]
            cnt = pipeline._empty((m,), torch.int32)
            E.call("gtb_records_count", rec, k, lo, cnt, m)
            ptr_t = pipeline.exclusive_scan(cnt)
            t_rec = pipeline._empty((k, 2), torch.int64)
            E.call("gtb_records_scatter", rec, k, lo, pipeline.cursor32(ptr_t), t_rec)
            outptr, k_idx, k_val, p_val, deg, newlen = pipeline.merge_with_transpose(
                indptr_a, idx, val, ptr_t, t_rec, m, lo, mode, theta, want_p=True, flags=flags)
        else:
            newlen = torch.zeros((0,), dtype=torch.int32, device=dev)
            outptr = torch.zeros((1,), dtype=torch.int64, device=dev)
            k_idx = torch.zeros((0,), dtype=torch.int32, device=dev)
            k_val = p_val = deg = torch.zeros((0,), dtype=torch.float64, device=dev)
        self._dev_shard = {"bounds": bounds, "n": n, "lo": lo, "hi": hi, "indptr": outptr, "row_len": newlen,
                           "indices": k_idx, "data": k_val, "P": p_val, "degree": deg, "flags": flags}
        if info.get("bandwidth") is not None:
            self._dev_bandwidth_shard = info["bandwidth"]
        pipeline._STATS.update(nnz_sym_local=int(k_idx.shape[0]))
        return None

    def _kernel_device(self, qry, ref, knn, knn_max, bandwidth, bandwidth_scale, nq_total=None):
        """Raw kernel rows of ``qry`` against ``ref``.  ``nq_total``: the query rows are this rank's shard of that
        many rows (the search schedule is then replayed on counts summed over the ranks)."""
        if self.decay is None or self.thresh == 1:
            return pipeline.knn_kernel(ref, qry, knn=knn, knn_max=None, decay=None)
        R, info = pipeline.knn_kernel(ref, qry, knn=knn, knn_max=knn_max, decay=self.decay,
                                      thresh=self.thresh, bandwidth=bandwidth, bandwidth_scale=bandwidth_scale)
        if ref.metric != "euclidean":
            R = self._euclidean_fallback(R, info, qry, ref, knn, knn_max, nq_total)
        return R, info

    def _fallback_plan(self, row_len, n_ref, knn, knn_max, nq_total):
        """(s_todo, search_knn, n_todo) of ``search_schedule`` from the raw row lengths of this rank's query rows
        (the number of reference points inside each row's radius, capped at knn_max); the counts are summed over
        the ranks when ``nq_total`` is given.  Collective in that case: every rank calls it, also with no rows."""
        import torch
        widths = _schedule_widths(n_ref, knn, knn_max, self.search_multiplier)
        ge = torch.stack([(row_len >= s).sum() for s in widths]).to(torch.int64)
        if nq_total is not None:
            import torch.distributed as dist
            dist.all_reduce(ge)
        at = dict(zip(widths, ge.tolist()))
        nq = row_len.shape[0] if nq_total is None else nq_total
        return search_schedule(at.__getitem__, nq, n_ref, knn, knn_max, self.search_multiplier)

    def _euclidean_fallback(self, R, info, qry, ref, knn, knn_max, nq_total=None):
        """Reference quirk H9 (graphs.py:945-948): when its search escalates beyond N/2 neighbours, the rows still
        to do are searched on a brute-force index built WITHOUT ``metric=``.  Their kernel rows then hold Euclidean
        distances divided by the metric's own bandwidth: the radius search, or the ``knn_max`` nearest when the
        search width has reached knn_max.  The schedule is replayed from the metric rows' lengths and those rows
        are rebuilt on a Euclidean operand of the same data."""
        row_len = R.indptr[1:] - R.indptr[:-1]
        s_todo, s_final, n_todo = self._fallback_plan(row_len, ref.n, knn, knn_max, nq_total)
        if not (s_final > ref.n / 2 and n_todo > 0):
            return R
        rows = (row_len >= s_todo).nonzero().flatten()
        main_stats = dict(pipeline._STATS, euclidean_fallback_rows=int(n_todo))
        if rows.shape[0] == 0:
            pipeline._STATS.update(main_stats)
            return R
        if getattr(self, "_euclid_ref", None) is None or self._euclid_ref[0] is not ref:
            self._euclid_ref = (ref, pipeline.SearchOperand(ref.X, metric="euclidean"))
        eref = self._euclid_ref[1]
        sub = pipeline.SearchOperand(qry.X[rows].contiguous(), mean=eref.mean, metric="euclidean")
        bw = info["bandwidth"][rows].cpu().numpy()
        kmax = ref.n if knn_max is None else knn_max
        R2, _ = pipeline.knn_kernel(eref, sub, knn=knn, knn_max=kmax if s_final == kmax else None,
                                    decay=self.decay, thresh=self.thresh, bandwidth=bw, bandwidth_scale=1.0)
        pipeline._STATS.clear()
        pipeline._STATS.update(main_stats)           # stats() describes the metric search, plus the rebuilt rows
        return _splice_rows(R, rows, R2)

    def _check_duplicates(self, info, qry, ref):
        """Warn about zero distances between distinct samples (graphs.py:787-817)."""
        if self.decay is None or self.thresh == 1:
            return
        nzero = info["nzero"]
        n_dup_rows = int((nzero > 1).sum().item())
        if n_dup_rows == 0:
            return
        total = int((nzero - 1).clamp(min=0).sum().item())
        pairs = None
        if total < 20 and qry is ref:
            rows = (nzero > 1).nonzero().flatten().cpu().numpy()
            if ref.metric in ("sqeuclidean", "correlation"):
                pairs = _zero_distance_pairs(ref.X, rows, ref.metric) or None
            else:
                Xh = ref.X.cpu().numpy()
                pairs = set()
                for i in rows:
                    same = np.flatnonzero((Xh == Xh[i]).all(axis=1))
                    for j in same:
                        if j < i:
                            pairs.add((int(j), int(i)))
        if pairs is not None:
            names = ", ".join("{} and {}".format(a, b) for a, b in sorted(pairs))
            warnings.warn("Detected zero distance between samples {}. Consider removing duplicates to avoid "
                          "errors in downstream processing.".format(names), RuntimeWarning)
        else:
            warnings.warn("Detected zero distance between {} pairs of samples. Consider removing duplicates to "
                          "avoid errors in downstream processing.".format(total // 2), RuntimeWarning)

    def _kernel_to_data_device(self, Y, knn=None, knn_max=None, bandwidth=None, bandwidth_scale=None):
        if knn is None:
            knn = self.knn
        if bandwidth is None:
            bandwidth = self.bandwidth
        if bandwidth_scale is None:
            bandwidth_scale = self.bandwidth_scale
        if knn > self.data.shape[0]:
            warnings.warn("Cannot set knn ({k}) to be greater than "
                          "n_samples ({n}). Setting knn={n}".format(k=knn, n=self.data_nu.shape[0]))
            knn = self.data_nu.shape[0]
        Y = self._check_extension_shape(Y)
        ref = self.knn_tree
        from . import distributed as gd
        with _logger.log_task("KNN search"):
            Yd = self._dense_f32(Y).to(ref.X.dtype)
            pipeline.reject_constant_rows(Yd, ref.metric)
            if gd.active() and np.ndim(bandwidth) == 0 and Yd.shape[0] >= gd.MIN_ROWS_PER_RANK * gd.world_size():
                return self._kernel_to_data_sharded(Yd, ref, knn, knn_max, bandwidth, bandwidth_scale)
            qry = pipeline.SearchOperand(Yd, mean=ref.mean, metric=ref.metric)
            R, info = self._kernel_device(qry, ref, knn=knn, knn_max=knn_max, bandwidth=bandwidth,
                                          bandwidth_scale=bandwidth_scale)
        self._check_duplicates(info, qry, ref)
        return R

    def _kernel_to_data_sharded(self, Yd, ref, knn, knn_max, bandwidth, bandwidth_scale):
        """Out-of-sample kernel with the query rows sharded over the ranks (SURVEY section 8e: MNN cross-batch blocks,
        ``extend_to_data``): each rank searches its contiguous block of ``Y`` against the replicated reference
        set, the CSR row shards are all-gathered (NCCL) and every rank returns the complete [n_y, n] matrix --
        bit-identical to the single-GPU result because every row still sees the whole reference set."""
        from . import distributed as gd
        bounds, _, row_len, idx, val, info = self._local_raw_rows(ref, knn_max, Xq=Yd, knn=knn, bandwidth=bandwidth,
                                                                  bandwidth_scale=bandwidth_scale)
        heights = [b[1] - b[0] for b in bounds]
        indptr, idx, val = gd.allgather_csr_rows(row_len, idx, val, heights, pipeline.exclusive_scan)
        if not (self.decay is None or self.thresh == 1):
            nzero = gd._allgather_padded(info["nzero"], heights)
            self._check_duplicates({"nzero": nzero}, None, ref)
        return pipeline.DeviceCSR(indptr, idx, val, (Yd.shape[0], ref.n))

    def build_kernel_to_data(self, Y, knn=None, knn_max=None, bandwidth=None, bandwidth_scale=None):
        """Kernel from new points ``Y`` to ``self.data`` as scipy CSR [n_y, n] (graphs.py:819-982)."""
        return self._kernel_to_data_device(Y, knn, knn_max, bandwidth, bandwidth_scale).to_scipy()
