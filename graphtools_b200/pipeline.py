"""Device pipeline: the order in which the C-ABI kernels are chained for one graph build.

search operand -> fused distance/top-S -> float64 refine + certification -> (radius pass for
uncertified rows) -> CSR emission -> symmetrise -> row-normalise.

Everything stays in HBM as torch tensors; the two host synchronisations per kernel build are the
reads of `number of uncertified rows` and `nnz` (sizes of the next allocations).
"""
import math
from collections import namedtuple
from typing import NamedTuple

import numpy as np
import torch

from . import _engine as E

SYM_MODES = {"+": 0, "*": 1, "mnn": 2, None: 3}
METRIC_ALIASES = {"manhattan": "cityblock", "l1": "cityblock", "l2": "euclidean"}
METRIC_CODE = {"euclidean": 0, "cosine": 1, "cityblock": 2, "sqeuclidean": 3, "correlation": 4}
METRIC_NAMES = tuple(METRIC_CODE) + ("manhattan", "l1")      # the ``distance`` values graphs accept
AUTO_TC = "tch1"         # tensor-core flavour picked by impl="auto": "tch1" (fp16, one product, seeded), "tch" (fp16x2), "tc16" (bf16x3) or "tc" (3xTF32)
BALL_CAP = 8192          # longest radius-pass row handled by refine_ball (shared-memory sort)
_STATS = {}


class RowTooLong(NotImplementedError):
    """A row has more neighbours inside the kernel radius than the radius-pass refine handles (BALL_CAP)."""


def unsupported_metric_message(distance):
    return ("graphtools_b200 accelerates the euclidean, cosine and cityblock metrics, and sqeuclidean and correlation "
            "(got distance={!r})".format(distance))


def degenerate_rows(X, metric):
    """Rows on which ``metric`` has no value (scipy's distances from them are NaN): all-zero rows under cosine, constant
    rows (max == min, whose centred row is zero) under correlation; None for the other metrics.  ``X``: torch tensor
    or numpy array [n, d] (also a scipy sparse matrix under correlation); the mask is a bool tensor or numpy array."""
    if metric == "cosine":
        return (X == 0).all(1)
    if metric == "correlation":
        if isinstance(X, torch.Tensor):
            return X.amax(dim=1) == X.amin(dim=1)
        hi, lo = X.max(axis=1), X.min(axis=1)
        if not isinstance(X, np.ndarray):                   # scipy sparse: matrices of shape [n, 1]
            hi, lo = hi.toarray(), lo.toarray()
        return np.asarray(hi == lo).reshape(-1)
    return None


def reject_constant_rows(X, metric):
    """Searches under correlation (kNN, MNN and landmark graphs, out-of-sample kernels) raise ValueError on constant
    rows before any work: the reference's neighbours of such a row are in undefined order, and its symmetrised kernel
    spreads their NaN distances into other rows.  (Exact graphs accept them: their affinity is 1.)"""
    if metric != "correlation":
        return
    n = int(degenerate_rows(X, metric).sum())
    if n:
        raise ValueError(
            "{} of {} rows are constant: their correlation distance to every row is undefined (the row minus its mean "
            "is zero). Remove them, or use graphtype='exact', which gives them affinity 1 to every "
            "sample.".format(n, X.shape[0]))


def stats():
    """Counters of the last kernel build (rows sent to the radius pass, passes, nnz)."""
    return dict(_STATS)


def _dev():
    return torch.device("cuda", torch.cuda.current_device())


def _empty(shape, dtype):
    return torch.empty(shape, dtype=dtype, device=_dev())


def _zeros(shape, dtype):
    return torch.zeros(shape, dtype=dtype, device=_dev())


def to_device_f32(X):
    """Host array / tensor -> contiguous float32 CUDA tensor."""
    E.require_cuda()
    if isinstance(X, torch.Tensor):
        return X.to(device=_dev(), dtype=torch.float32).contiguous()
    X = np.ascontiguousarray(np.asarray(X), dtype=np.float32)
    t = torch.from_numpy(X)
    return t.to(_dev(), non_blocking=False)


def to_device(X):
    """Host array / tensor -> contiguous CUDA tensor that keeps float64 inputs in float64 (the exact
    distances are then evaluated on the original float64 rows, e.g. PCA output); everything else becomes
    float32."""
    E.require_cuda()
    if isinstance(X, torch.Tensor):
        dt = torch.float64 if X.dtype == torch.float64 else torch.float32
        return X.to(device=_dev(), dtype=dt).contiguous()
    X = np.asarray(X)
    dt = np.float64 if X.dtype == np.float64 else np.float32
    return torch.from_numpy(np.ascontiguousarray(X, dtype=dt)).to(_dev())


_D2H_CHUNK = 32 << 20      # bytes per staging buffer
_D2H_RING = 3
_d2h_state = {}


def _d2h_ring():
    """Page-locked staging ring, a side stream and a small thread pool, created once per process: the result
    arrays (K / P values, indices: ~350 MB at 1M samples) are handed to the caller, so they must live in ordinary
    pageable memory, but a direct pageable cudaMemcpy runs at ~2.6 GB/s (first-touch page faults serialised with
    the copy)."""
    if not _d2h_state:
        from concurrent.futures import ThreadPoolExecutor
        _d2h_state["bufs"] = [torch.empty((_D2H_CHUNK,), dtype=torch.uint8, pin_memory=True) for _ in range(_D2H_RING)]
        _d2h_state["stream"] = torch.cuda.Stream()
        _d2h_state["pool"] = ThreadPoolExecutor(max_workers=4)
    return _d2h_state["bufs"], _d2h_state["stream"], _d2h_state["pool"]


def d2h_into(t, dst_array):
    """Device tensor -> an existing host numpy array of the same size and dtype (e.g. a slice of a shared-memory
    segment), through the pinned staging ring."""
    assert dst_array.nbytes == t.numel() * t.element_size(), (dst_array.nbytes, t.numel(), t.element_size())
    if t.numel() == 0:
        return
    d2h_pinned(t, dst_array.reshape(-1).view(np.uint8))


def d2h_pinned(t, dst=None):
    """Device->host copy into a fresh pageable tensor (or into ``dst``, a uint8 numpy view of the destination).
    Large tensors go through the pinned staging ring in 32 MB chunks: the DMA of chunk i+1 overlaps the host-side
    copy of chunk i, which four threads perform in parallel (so the first-touch page faults of the destination are
    taken in parallel too)."""
    nbytes = t.numel() * t.element_size()
    if nbytes < (8 << 20) or not t.is_cuda:
        if dst is None:
            return t.cpu()
        dst[:] = t.contiguous().view(-1).view(torch.uint8).cpu().numpy()
        return None
    bufs, side, pool = _d2h_ring()
    src = t.contiguous().view(-1).view(torch.uint8)
    out = None
    if dst is None:
        out = torch.empty(t.shape, dtype=t.dtype)
        dst = out.view(-1).view(torch.uint8).numpy()
    side.wait_stream(torch.cuda.current_stream())
    chunks = [(off, min(_D2H_CHUNK, nbytes - off)) for off in range(0, nbytes, _D2H_CHUNK)]
    events = [None] * len(chunks)
    pending = [[] for _ in range(_D2H_RING)]           # host copies still reading staging buffer r

    def issue(i):
        off, n = chunks[i]
        r = i % _D2H_RING
        for f in pending[r]:
            f.result()
        pending[r] = []
        with torch.cuda.stream(side):
            bufs[r][:n].copy_(src[off:off + n], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(side)
        events[i] = ev

    def drain(i):
        off, n = chunks[i]
        r = i % _D2H_RING
        events[i].synchronize()
        hb = bufs[r].numpy()
        step = (n + 3) // 4
        for a in range(0, n, step):
            b = min(n, a + step)
            pending[r].append(pool.submit(np.copyto, dst[off + a:off + b], hb[a:b]))

    for i in range(min(_D2H_RING - 1, len(chunks))):
        issue(i)
    for i in range(len(chunks)):
        if i + _D2H_RING - 1 < len(chunks):
            issue(i + _D2H_RING - 1)
        drain(i)
    for r in range(_D2H_RING):
        for f in pending[r]:
            f.result()
    t.record_stream(side)
    return out


class SearchOperand:
    """k-major centred copy of a point set + squared norms (csrc/prep.cu)."""

    def __init__(self, X, mean=None, metric="euclidean"):
        """X: the ORIGINAL rows on the device, float32 or float64 (kept for the exact distances).  The search
        copy is always float32: float64 inputs are centred in float64 first and rounded once, so the
        rounding error of the fast pass stays relative to the centred magnitudes (same bound E).

        metric="cosine": the search copy is built from the row-normalised data (normalised and centred in float64,
        rounded once), on which squared Euclidean distance = 2 x cosine distance; the exact stage evaluates
        1 - x.y / (|x||y|) on the original rows.  All-zero rows stay zero, as in sklearn's ``normalize``; their
        search distance to a normalised row is 1 (to another zero row 0), below the 2 x 1 of their exact cosine
        distance, so the certification bounds stay conservative for them.

        metric="correlation": as cosine, after subtracting each row's own mean in float64 (scipy centres every row
        by its np.mean before its cosine routine): row-centred, normalised, column-centred, rounded once.  ``X``
        keeps the original rows, which the exact stage and the reference's Euclidean fallback read.

        metric="sqeuclidean": the Euclidean operand, unchanged; the exact stage squares the Euclidean distance."""
        n, d = X.shape
        self.X, self.n, self.d = X, n, d
        self.metric = metric
        self.is64 = X.dtype == torch.float64
        self.n_pad = (n + 127) // 128 * 128
        self.d_pad = (d + 7) // 8 * 8
        metric = METRIC_ALIASES.get(metric, metric)
        self.metric = metric
        if metric not in METRIC_CODE:
            raise NotImplementedError("metric {!r} is not supported by the CUDA search".format(metric))
        if metric == "cityblock":
            # |x - y| is translation invariant and has no GEMM form: the search copy is the float32 data itself,
            # NOT centred, so that the float32 accumulation of sum |x - y| stays accurate relative to the distance
            # (float64 inputs are rounded once; that rounding enters the certification bound through the L1 norms)
            self.Xs = X.to(torch.float32).contiguous() if self.is64 else X
            self._kmean = None
            mean = torch.zeros((d,), dtype=torch.float32, device=X.device) if mean is None else mean
        elif self.is64 or metric in ("cosine", "correlation"):
            rows = X.to(torch.float64)
            if metric == "correlation":
                rows = rows - rows.mean(dim=1, keepdim=True)
            if metric in ("cosine", "correlation"):
                norms = rows.norm(dim=1, keepdim=True)
                rows = rows / torch.where(norms > 0, norms, torch.ones_like(norms))
            if mean is None:
                mean = rows.mean(dim=0)
            self.Xs = (rows - mean.to(torch.float64)).to(torch.float32).contiguous()
            self._kmean = None                       # already centred
            del rows
        else:
            if mean is None:
                ws = _empty((E.lib().gtb_col_mean_ws_doubles(d),), torch.float64)
                mean = _empty((d,), torch.float32)
                E.call("gtb_col_mean", X, n, d, ws, mean)
            self.Xs = X
            self._kmean = mean.to(torch.float32)
        self.mean = mean
        self._simt = None
        self._tc = {}
        self._n2_tc = None
        self._maxnorm = None
        self._maxnorm_host = None
        self._perm = None

    # -- CUDA-core operand: k-major [d_pad][n_pad] + norms
    def simt(self):
        if self._simt is None:
            XT = _empty((self.d_pad, self.n_pad), torch.float32)
            n2 = _empty((self.n_pad,), torch.float32)
            mx = _empty((1,), torch.float32)
            E.call("gtb_prepare_operand", self.Xs, self.n, self.d, self._kmean, XT, self.n_pad, self.d_pad, n2, mx)
            self._simt = (XT, n2)
            if self._maxnorm is None:
                self._maxnorm = mx
        return self._simt

    @property
    def XT(self):
        return self.simt()[0]

    @property
    def n2(self):
        return self.simt()[1]

    # -- tensor-core operand: row-major [n_pad][Kp] hi/lo pair for one role (0 query, 1 reference) in the layout of
    #    one flavour's dtype code (TC_FLAVOURS)
    def kp(self, dtype=0):
        return TC_FLAVOURS[dtype].kp(self.d)

    def l1_norms(self):
        """(per-row L1 norms float32 [n], max) of the search copy -- bound on its rounding for float64 inputs."""
        if getattr(self, "_l1", None) is None:
            n1 = self.Xs.abs().sum(dim=1, dtype=torch.float64)
            self._l1 = (n1.to(torch.float32).contiguous(), float(n1.max().item()))
        return self._l1

    def tc(self, role, dtype=0, scale=1.0):
        """(hi, lo, norm2) of one role; dtype 0 = tf32 pairs in float32, 1 = bfloat16 pairs, 2 = float16 pairs of the
        data scaled by ``scale`` (norm2 stays unscaled); 3 = the float16 pairs of dtype 2."""
        dtype = TC_FLAVOURS[dtype].operand
        key = (role, dtype, float(scale))
        if key not in self._tc:
            Kp = self.kp(dtype)
            st = (torch.float32, torch.bfloat16, torch.float16)[dtype]
            hi = _empty((self.n_pad, Kp), st)
            lo = _empty((self.n_pad, Kp), st)
            if getattr(self, "_n2_tc", None) is not None:
                # the norms are on hand (norm_max, or the other role): split only
                n2 = self._n2_tc
                E.call("gtb_split_operand_tc", self.Xs, self.n, self.d, self._kmean, role, hi, lo, self.n_pad, Kp,
                       dtype, float(scale), n2)
            else:
                n2 = _empty((self.n_pad,), torch.float32)
                mx = _empty((1,), torch.float32)
                E.call("gtb_prepare_operand_tc", self.Xs, self.n, self.d, self._kmean, role, hi, lo, self.n_pad, Kp,
                       dtype, float(scale), n2, mx)
                self._n2_tc = n2
                if self._maxnorm is None:
                    self._maxnorm = mx
            self._tc[key] = (hi, lo, n2)
        return self._tc[key]

    def norm_max(self):
        """max squared norm of the centred rows WITHOUT building an operand (the fp16 flavour needs it to choose its
        scale before the split); one pass over X and one host read."""
        if self._maxnorm_host is None and self._maxnorm is None:
            n2 = _empty((self.n_pad,), torch.float32)
            mx = _empty((1,), torch.float32)
            E.call("gtb_row_norms", self.Xs, self.n, self.d, self._kmean, self.n_pad, n2, mx)
            self._maxnorm = mx
            self._n2_tc = n2
        return self.maxnorm

    def locality_order(self):
        """perm (int32 [n]): the rows grouped by nearest of ORDER_PIVOTS pivot rows, stable (csrc/order.cu) -- consecutive
        rows of the order lie close together, so a 128-row tile of them covers one region of the data."""
        if self._perm is None:
            P = min(ORDER_PIVOTS, self.n)
            cell = _empty((self.n,), torch.int32)
            E.call("gtb_order_assign", self.Xs, self.n, self.d, P, cell)
            ws = _empty((E.lib().gtb_order_ws_elems(self.n, P),), torch.int32)
            self._perm = _empty((self.n,), torch.int32)
            E.call("gtb_order_sort", cell, self.n, P, ws, self._perm)
        return self._perm

    def geometry(self, rows):
        """(centroids float64 [d][g], radii float64 [g]) of the groups of ``rows`` consecutive rows of the locality order,
        over ``X`` (the rows the exact stage reads); g = n_pad / rows rounded up, radius -1 for a group without rows."""
        g = -(-self.n_pad // rows)
        cent = _empty((self.d, g), torch.float64)
        rad = _empty((g,), torch.float64)
        E.call("gtb_tile_geometry", self.X, self.n, self.d, int(self.is64), self.locality_order(), rows, g, cent, rad)
        return cent, rad

    @property
    def maxnorm(self):
        if self._maxnorm_host is None:
            if self._maxnorm is None:
                self.simt()
            self._maxnorm_host = float(self._maxnorm.item())
        return self._maxnorm_host


_NP_OF = {torch.int32: np.int32, torch.int64: np.int64, torch.float64: np.float64, torch.float32: np.float32}


def _d2h_pooled(named):
    """[(name, device tensor)] -> {name: numpy array} carved out of ONE recycled page-locked block (hostpool.py) and
    filled by DMA -- no staging copy, no first-touch page faults after the first build.  None when the pool is off,
    full, or the arrays are small (the plain path is as good)."""
    from . import hostpool
    if not all(t.is_cuda for _, t in named) or sum(t.numel() * t.element_size() for _, t in named) < (8 << 20):
        return None
    lay, total = hostpool.layout([(nm, t.numel(), _NP_OF[t.dtype]) for nm, t in named])
    blk = hostpool.take_local(total)
    if blk is None:
        return None
    out = blk.carve(lay)
    for nm, t in named:
        hostpool.d2h_async(t, out[nm])
    torch.cuda.current_stream().synchronize()
    return out


class DeviceCSR:
    """CSR in HBM: int64 indptr [n+1], int32 indices, float64 data."""

    def __init__(self, indptr, indices, data, shape):
        self.indptr, self.indices, self.data, self.shape = indptr, indices, data, tuple(shape)

    @property
    def nnz(self):
        return int(self.indices.shape[0])

    def _host_structure(self):
        """(indices, indptr int32) as numpy arrays, copied device->host once through pinned buffers and
        shared by every scipy view of this matrix (K, P, transitions...)."""
        if getattr(self, "_host_struct", None) is None:
            n1 = self.indptr.shape[0]
            ip32 = _empty((n1,), torch.int32)
            E.call("gtb_cast_indptr", self.indptr, n1, ip32)
            got = _d2h_pooled([("indices", self.indices), ("indptr", ip32)])
            if got is not None:
                self._host_struct = (got["indices"], got["indptr"])
            else:
                idx_h, ip_h = d2h_pinned(self.indices), d2h_pinned(ip32)
                torch.cuda.current_stream().synchronize()
                self._host_struct = (idx_h.numpy(), ip_h.numpy())
        return self._host_struct

    def to_scipy(self, data=None):
        from scipy import sparse
        src = self.data if data is None else data
        got = _d2h_pooled([("vals", src)])
        vals = got["vals"] if got is not None else d2h_pinned(src).numpy()
        indices, indptr = self._host_structure()
        torch.cuda.current_stream().synchronize()
        M = sparse.csr_matrix((vals, indices, indptr), shape=self.shape)
        M.has_sorted_indices = True
        M.has_canonical_format = True
        return M


def exclusive_scan(counts):
    n = counts.shape[0]
    out = _empty((n + 1,), torch.int64)
    ws = _empty((E.lib().gtb_scan_ws_elems(n),), torch.int64)
    E.call("gtb_exclusive_scan", counts, n, out, ws)
    return out


def choose_S(knn_eff, binary):
    """Candidate-list length of the fused top-k: the reference's first search is
    knn * search_multiplier = 36 wide (graphs.py:882); we keep a little more so that the
    certification margin rarely sends a row to the radius pass."""
    need = knn_eff + (4 if binary else 8)
    for S in ((16, 32, 48, 64, 128) if binary else (48, 64, 128)):
        if need <= S:
            return S
    raise NotImplementedError(
        "knn={} needs a candidate list longer than 128; not supported by the fused top-k yet".format(knn_eff))


def default_impl():
    """GTB_SEARCH_IMPL = tc (3xTF32 tensor cores) | tc16 (bf16x3 tensor cores) | tch (fp16x2 tensor cores: two
    products, wider certified bound) | tch1 (fp16, ONE product, seeded thresholds, lists of 64) | simt (fp32 CUDA
    cores) | auto (default: tensor cores whenever the operand fits)."""
    import os
    return os.environ.get("GTB_SEARCH_IMPL", "auto")


def eps_rel_tc(d):
    """Same bound for the 3xTF32 tensor-core pass: dropped lo*lo terms and the tf32 rounding of the lo
    parts contribute 3 * 2^-22, float32 accumulation in the tensor core at most Kp * 2^-23 (truncation);
    doubled."""
    return 4.0 * (d + 16) * 2.0 ** -24


def eps_rel_tc16(d):
    """bf16x3 (hi*hi + hi*lo + lo*hi, 16 mantissa bits kept): dropped terms <= (2^-16 + 2^-18) |a||b| per
    product, sum |a||b| <= 2 (|x~|^2 + max|y~|^2); float32 accumulation as for tf32."""
    return 2.0 * (2.0 ** -16 + 2.0 ** -18) + 2.0 * (d + 32) * 2.0 ** -24


def eps_rel_l1(d):
    """Cityblock pass: float32 subtraction and accumulation of d terms |x_k - y_k| -- relative error of the
    DISTANCE at most (d + 1) * 2^-24 (all terms non-negative, no cancellation), doubled."""
    return 2.0 * (d + 2) * 2.0 ** -24


def eps_rel_tch(d):
    """fp16x2 (A_hi B_hi + A_hi B_lo on float16 pairs): the dropped query low part is <= 2^-11 |a| per element, so
    the dropped product is <= 2^-11 sum |a||b| <= 2^-11 |x~| |2 y~| <= 2^-11 (|x~|^2 + |y~|^2); the reference operand
    keeps 22 bits (2^-22, twice for the two parts), float32 accumulation as for the other flavours, 1e-6 covers fp16
    subnormals of the low parts at the chosen scale."""
    return 2.0 ** -11 + 2.0 ** -20 + 2.0 * (d + 32) * 2.0 ** -24 + 1e-6


def fp16_scale(maxnorm):
    """Power of two s with s^2 * maxnorm <= gtb_tc_fp16_maxnorm(): scaled data fits float16 with headroom."""
    limit = float(E.lib().gtb_tc_fp16_maxnorm())
    if not (maxnorm > 0):
        return 1.0
    return 2.0 ** math.floor(0.5 * math.log2(limit / maxnorm))


def eps_rel_tch1(d):
    """fp16x1 (A_hi B_hi only, float16): both operands are rounded to 11 bits, |delta(2 x.y)| <= 2 (2 u + u^2)
    sum |x_k||y_k| <= 2^-10 (1 + 2^-12) (|x~|^2 + |y~|^2) with u = 2^-11; |y|^2 keeps 22 bits (hi + spare-column low
    part); float32 accumulation and fp16 subnormals as for fp16x2."""
    return 2.0 ** -10 + 2.0 ** -20 + 2.0 * (d + 32) * 2.0 ** -24 + 1e-6


def eps_rel_simt(d):
    """Relative bound on |approx d^2 - exact d^2| / (|x~|^2 + |y~|^2) for the fp32 CUDA-core pass:
    (d + 11) * 2^-24 from a standard rounding analysis (dot product, norms, centring), doubled."""
    return 2.0 * (d + 16) * 2.0 ** -24


class TcFlavour(NamedTuple):
    """One tensor-core search flavour (csrc/search_tc.cu).  Its operand rows are whole 32-byte k-steps (SWIZZLE_128B
    blocks plus SWIZZLE_32B tail blocks) holding the d centred features, the |y|^2 column and ``spare`` more.
    (Padding bf16 rows to whole 128-byte blocks was measured slower: 699 vs 682 ms at d = 100 -- the extra MMAs cost
    more than the tail blocks.)"""
    name: str
    dtype: int          # dtype code of the C ABI
    step: int           # elements per k-step: 8 tf32, 16 bf16 / fp16
    spare: int          # float16 operands keep one more column: the low part of |y|^2
    max_steps: int      # k-steps of the resident query tile (the fp16x2 flavour streams longer rows in chunks)
    list_cap: int       # candidates per row: 2 lists x 32, one list of 64 for the one-product flavour
    eps_rel: object     # relative bound of its squared distances (certification)
    fp16: bool          # operands are the data scaled by fp16_scale, in float16
    operand: int        # dtype code of the operands it reads and of its radius pass

    def kp(self, d):
        return (d + 1 + self.spare + self.step - 1) // self.step * self.step

    def fits(self, d):
        return self.kp(d) // self.step <= self.max_steps


TC_FLAVOURS = (                                               # indexed by dtype code
    TcFlavour("tc", 0, 8, 0, 13, 32, eps_rel_tc, False, 0),           # 3xTF32
    TcFlavour("tc16", 1, 16, 0, 8, 32, eps_rel_tc16, False, 1),       # bf16x3
    TcFlavour("tch", 2, 16, 1, 32, 32, eps_rel_tch, True, 2),         # fp16x2: two products
    TcFlavour("tch1", 3, 16, 1, 8, 64, eps_rel_tch1, True, 2),        # fp16, one product: reads the fp16x2 operands
)
FLAVOURS = {f.name: f for f in TC_FLAVOURS}
# GTB_SEARCH_IMPL is a preference: a flavour that cannot take the shape (feature count beyond the resident query tile,
# knn beyond the candidate lists) hands over to the next one
FALLBACK = {"auto": (AUTO_TC, "tch", "tc16", "tc", "simt"), "tc": ("tc", "tc16", "simt"), "tc16": ("tc16", "tc", "simt"),
            "tch": ("tch", "tc16", "tc", "simt"), "tch1": ("tch1", "tch", "tc16", "tc", "simt"), "simt": ("simt",)}
TC_CLUSTER = 2           # CTAs per cluster sharing each reference tile by TMA multicast
SEED_STRIDE = 16         # the seed sweep of the one-product flavour visits every 16th reference tile
ORDER_PIVOTS = 256       # cells of the locality order of the pruned sweep
PRUNE_MAX_VISITED = 0.5  # the pruned sweep runs when its tile lists hold at most this share of all (unit, tile) pairs
SearchPlan = namedtuple("SearchPlan", "impl ls qtiles S ntau seeded")


def plan_search(want, d, n_pad, metric, knn, kmax, binary):
    """Flavour and list shapes of a kNN search: ``want`` = GTB_SEARCH_IMPL, ``d`` features, ``n_pad`` padded
    reference rows, ``knn`` / ``kmax`` (0 = none) neighbours per row, ``binary`` = no decay.  Returns a SearchPlan:
    the flavour (a key of FLAVOURS, or "simt"), entries per candidate list ``ls`` and query tiles per CTA ``qtiles``
    (tensor cores; None for simt), candidates per row ``S``, thresholds per row ``ntau``, and whether a seed sweep
    sets the starting thresholds."""
    # a strided sample needs enough tiles to carry the order statistic: 32 sampled tiles at least
    seedable = n_pad // 128 >= 32 * SEED_STRIDE
    if metric == "cityblock":
        impl = "simt"                                     # |x - y| has no GEMM form: CUDA-core L1 kernel only
    elif want not in FALLBACK:
        raise ValueError("GTB_SEARCH_IMPL must be auto, tc, tc16, tch, tch1 or simt (got %r)" % (want,))
    else:
        # auto: the one-product flavour pays off only with seeded thresholds (cold, its list of 64 costs more than the
        # second product saves: C3 at 50k x 50 6.7 ms against 2.5 ms) -- unless the longer list is what knn needs
        impl = next(c for c in FALLBACK[want] if c == "simt" or (
            FLAVOURS[c].fits(d) and knn + 8 <= FLAVOURS[c].list_cap
            and not (c == "tch1" and want == "auto" and not seedable and knn + 8 <= 32)))
    if impl == "simt":
        S = choose_S(knn, binary)
        return SearchPlan(impl, None, None, S, 1, False)
    f = FLAVOURS[impl]
    if f.dtype == 3:
        ls, qtiles = 32, 2                                # one product: one list of 64 per row, always two tiles
    else:
        # short lists (16) halve the selection work of the sweep when the neighbourhood asked for is small -- rows
        # whose kernel support is wider fail certification and are finished by the radius pass.  The fp16x2 flavour
        # with rows of 8 k-steps runs two query tiles per CTA and keeps ONE list of 32 per row.  knn_max neighbours
        # must fit the lists as well.
        two_tiles = f.dtype == 2 and f.kp(d) <= 128
        ls = 16 if max(knn, kmax) + 8 <= (32 if two_tiles else 16) else 32
        qtiles = 2 if two_tiles and ls == 16 else 1
    return SearchPlan(impl, ls, qtiles, 2 * ls, 2, f.dtype == 3 and seedable)


def prunable(plan, metric):
    """Whether a search tries the pruned sweep (tile lists over locality-ordered operands): the seeded one-product
    flavour under a metric whose exact stage reads the rows the tile geometry is computed from.  (Cosine and correlation
    search a normalised copy whose rounding the bound does not cover.)"""
    return plan.impl == "tch1" and plan.seeded and metric in ("euclidean", "sqeuclidean")


def use_tile_lists(visited, total):
    """The pruned sweep, or the plain seeded sweep when the lists visit more than PRUNE_MAX_VISITED of all (unit, tile)
    pairs (isotropic data, no region holds a unit's neighbourhood): the listed sweep gives up the grid-wide pacing that
    lets every reference tile be read from DRAM once."""
    return 0 < total and visited <= PRUNE_MAX_VISITED * total


def unit_bounds(seed, qn2, eps_rel, maxnorm, s2, unit_rows, n_units):
    """T_U (float64 [n_units]): per unit of ``unit_rows`` consecutive query rows, the largest seed + E of its rows in data
    units -- ``seed`` [nq, >= 1] the sweep's starting thresholds (scaled squared distances, slot 0), ``qn2`` [nq] the
    rows' squared norms, E = eps_rel (qn2 + maxnorm) the certified rounding bound of the sweep, widened by 2^-20
    (qn2 + maxnorm) for the float32 rounding of threshold - |x|^2 in the sweep.  A reference point at exact squared
    distance >= T_U from a row of the unit has approximate distance >= the row's seed, so the sweep would never admit
    it: skipping it leaves the candidate lists as they were.  Units without rows: -inf."""
    t = seed[:, 0].to(torch.float64) / s2 + (eps_rel + 2.0 ** -20) * (qn2.to(torch.float64) + maxnorm)
    out = torch.full((n_units * unit_rows,), -math.inf, dtype=torch.float64, device=seed.device)
    out[:t.shape[0]] = t
    return out.view(n_units, unit_rows).amax(dim=1)


def _tile_lists(qry, ref, seed, q_n2, eps_rel, s2, unit_rows):
    """Reference tile lists of the query units (csrc/order.cu) over the locality orders of both operands.  Returns
    (visited, total, lists) with lists = (unit_ptr, unit_tiles, unit_order) or None when use_tile_lists declines."""
    nt = ref.n_pad // 128
    n_units = -(-qry.n_pad // unit_rows)
    rc, rr = ref.geometry(128)
    uc, ur = qry.geometry(unit_rows)
    pq = qry.locality_order().long()
    ub = unit_bounds(seed.index_select(0, pq), q_n2[:qry.n].index_select(0, pq), eps_rel, ref.maxnorm, s2, unit_rows,
                     n_units)
    keep = _empty((n_units, nt), torch.uint8)
    count = _empty((n_units,), torch.int32)
    E.call("gtb_tile_lists_count", uc, ur, ub, n_units, rc, rr, nt, ref.d, keep, count)
    ptr = exclusive_scan(count)
    visited, total = int(ptr[-1].item()), n_units * nt
    if not use_tile_lists(visited, total):
        return visited, total, None
    tiles = _empty((max(visited, 1),), torch.int32)
    E.call("gtb_tile_lists_fill", keep, n_units, nt, ptr, tiles)
    order = torch.argsort(count, descending=True, stable=True).to(torch.int32)   # longest lists first
    return visited, total, (ptr, tiles, order)


def _permuted_rows(t, perm, n):
    """Rows of ``t`` [n_pad, ...] in the locality order; padding rows stay in place."""
    idx = torch.cat([perm.long(), torch.arange(n, t.shape[0], device=t.device)])
    return t.index_select(0, idx)


def _sweep_tc(plan, qry, ref):
    """Tensor-core sweep: (candidates, tau, query norms, eps_rel, fp16 scale)."""
    f = FLAVOURS[plan.impl]
    nq = qry.n
    # grid-wide pacing of the TMA producers: one caller-owned device word per launch (no library state)
    pace = _empty((1,), torch.int32)
    scale = fp16_scale(max(qry.norm_max(), ref.norm_max())) if f.fp16 else 1.0
    q_hi, q_lo, q_n2 = qry.tc(0, f.dtype, scale)
    r_hi, r_lo, _ = ref.tc(1, f.dtype, scale)
    Kp = ref.kp(f.dtype)
    cand = _empty((nq, plan.S), torch.int32)
    tau = _empty((nq, plan.ntau), torch.float32)
    scratch = _empty((E.lib().gtb_tc_scratch_bytes(qry.n_pad),), torch.uint8)
    s2 = scale * scale
    qn2_s = q_n2 * s2 if f.fp16 else q_n2
    if f.dtype == 3:
        seed = None
        if plan.seeded:
            # threshold seeds: the 8th smallest tile minimum over every stride-th reference tile (6 % of the tensor
            # work of a sweep, no selection work); it sits near the (8 stride)-th smallest distance overall, so the
            # full sweep starts with a threshold that admits ~8 stride points per row instead of climbing down from
            # +inf (64 ln(N / 64) threshold updates)
            seed = _empty((nq, plan.ntau), torch.float32)
            E.call("gtb_knn_seed_tc", q_hi, qn2_s, nq, qry.n_pad, r_hi, ref.n, ref.n_pad, Kp, TC_CLUSTER, SEED_STRIDE,
                   seed, pace)
        lists = None
        _STATS.update(tile_pairs_visited=None)
        if prunable(plan, ref.metric):
            # pruned sweep: both operands in locality order, every unit (the TC_CLUSTER x 2 query tiles of one cluster
            # round) sweeps only the reference tiles its seeds can reach; the lists come back in original row ids
            visited, total, lists = _tile_lists(qry, ref, seed, q_n2, f.eps_rel(ref.d), s2, TC_CLUSTER * plan.qtiles * 128)
            _STATS.update(tile_pairs_visited=visited / total)
        _STATS.update(tile_lists=lists is not None)
        if lists is None:
            E.call("gtb_knn_topk_tc_seeded", q_hi, q_lo, qn2_s, nq, qry.n_pad, r_hi, r_lo, ref.n, ref.n_pad, Kp,
                   f.dtype, plan.ls, TC_CLUSTER, plan.qtiles, seed, 1, cand, scratch, tau, pace)
        else:
            perm_q, perm_r = qry.locality_order(), ref.locality_order()
            pq_hi = _permuted_rows(q_hi, perm_q, nq)
            pr_hi = _permuted_rows(r_hi, perm_r, ref.n)
            cand_p = _empty((nq, plan.S), torch.int32)
            tau_p = _empty((nq, plan.ntau), torch.float32)
            # (the one-product flavour reads the hi arrays only)
            E.call("gtb_knn_topk_tc_seeded", pq_hi, pq_hi, _permuted_rows(qn2_s, perm_q, nq), nq, qry.n_pad, pr_hi,
                   pr_hi, ref.n, ref.n_pad, Kp, f.dtype, plan.ls, TC_CLUSTER, plan.qtiles,
                   seed.index_select(0, perm_q.long()), 1, cand_p, scratch, tau_p, None, *lists)
            E.call("gtb_unpermute_candidates", cand_p, tau_p, nq, plan.S, plan.ntau, perm_q, perm_r, cand, tau)
    else:
        E.call("gtb_knn_topk_tc", q_hi, q_lo, qn2_s, nq, qry.n_pad, r_hi, r_lo, ref.n, ref.n_pad, Kp, f.dtype, plan.ls,
               TC_CLUSTER, plan.qtiles, cand, scratch, tau, pace)
    if f.fp16:
        tau = tau / s2                                   # scaled squared distances -> data units (inf stays inf)
    return cand, tau, q_n2, f.eps_rel(ref.d), scale


def _sweep_simt(plan, qry, ref):
    """CUDA-core sweep: (candidates, tau, query norms, eps_rel, 1.0)."""
    nq = qry.n
    tau = _empty((nq,), torch.float32)
    cand = _empty((nq, plan.S), torch.int32)
    if ref.metric == "cityblock":
        q_n2 = qry.l1_norms()[0] if ref.is64 else None       # float32 inputs: the search copy is exact
        E.call("gtb_knn_topk_simt_l1", qry.XT, nq, qry.n_pad, ref.XT, ref.n, ref.n_pad, ref.d_pad, plan.S, cand, tau)
        return cand, tau, q_n2, eps_rel_l1(ref.d), 1.0
    E.call("gtb_knn_topk_simt", qry.XT, qry.n2, nq, qry.n_pad, ref.XT, ref.n2, ref.n, ref.n_pad, ref.d_pad, plan.S,
           cand, tau)
    return cand, tau, qry.n2, eps_rel_simt(ref.d), 1.0


def _radius_pass(plan, qry, ref, scale, todo_rows, lim2, status, n_keep, bw_out, nzero, x64, kern):
    """Rows the refine could not certify: every reference point inside the row's radius ``lim2``, refined in float64
    and merged into ``n_keep`` / ``bw_out`` / ``nzero``.  Returns the rows' segments (ptr, idx, val, n_keep)."""
    nr, d = ref.n, ref.d
    nt = todo_rows.shape[0]
    nt_pad = (nt + 127) // 128 * 128
    lim_t = _zeros((nt_pad,), torch.float32)
    lim_t[:nt] = lim2[todo_rows.long()]
    f = FLAVOURS.get(plan.impl)
    if f:
        # the radius rows form their own (small) query operand; build it from the gathered rows
        sub = SearchOperand(qry.X[todo_rows.long()].contiguous(), mean=ref.mean, metric=ref.metric)
        s_hi, s_lo, s_n2 = sub.tc(0, f.dtype, scale)
        r_hi, r_lo, _ = ref.tc(1, f.dtype, scale)
        if f.fp16:
            s_n2 = s_n2 * (scale * scale)
            lim_t = lim_t * (scale * scale)
        pace = _empty((1,), torch.int32)
    else:
        QT = _empty((ref.d_pad, nt_pad), torch.float32)
        qn2 = _empty((nt_pad,), torch.float32)
        E.call("gtb_gather_operand", qry.XT, qry.n_pad, qry.n2, todo_rows, nt, QT, nt_pad, ref.d_pad, qn2)
    capacity = max(1 << 20, nt * 4 * plan.S)
    while True:
        pairs = _empty((capacity, 2), torch.int32)
        counter = _zeros((1,), torch.int64)
        rowcnt = _zeros((nt_pad,), torch.int32)
        if f:
            # (the one-product flavour hands its uncertified rows to the two-product sweep on the same operands)
            E.call("gtb_knn_radius_tc", s_hi, s_lo, s_n2, lim_t, nt, nt_pad, r_hi, r_lo, nr, ref.n_pad, ref.kp(f.dtype),
                   f.operand, TC_CLUSTER, pairs, capacity, counter, rowcnt, pace)
        elif ref.metric == "cityblock":
            E.call("gtb_knn_radius_simt_l1", QT, lim_t, nt, nt_pad, ref.XT, nr, ref.n_pad, ref.d_pad, pairs,
                   capacity, counter, rowcnt)
        else:
            E.call("gtb_knn_radius_simt", QT, qn2, lim_t, nt, nt_pad, ref.XT, ref.n2, nr, ref.n_pad, ref.d_pad,
                   pairs, capacity, counter, rowcnt)
        npairs = int(counter.item())
        if npairs <= capacity:
            break
        capacity = npairs
    _STATS.update(radius_pairs=npairs)
    seg_ptr = exclusive_scan(rowcnt[:nt].contiguous())
    seg_idx = _empty((max(npairs, 1),), torch.int32)
    seg_val = _empty((max(npairs, 1),), torch.float64)
    cursor = _empty((nt,), torch.int32)
    E.call("gtb_scatter_pairs", pairs, npairs, seg_ptr, cursor, nt, seg_idx)
    n_keep_t = _empty((nt,), torch.int32)
    overflow = _empty((1,), torch.int32)
    longest = int(rowcnt.max().item())
    cap = 64
    while cap < longest:
        cap *= 2
    if cap > BALL_CAP:
        raise RowTooLong(
            "a row has {} neighbours inside the kernel radius; the sparse kNN pipeline handles rows of up to {} "
            "(a kernel this dense calls for graphtype='exact', which evaluates every pair)".format(longest, BALL_CAP))
    E.call("gtb_refine_ball", qry.X, todo_rows, status, nt, ref.X, d, x64, seg_ptr, seg_idx, seg_val, *kern, n_keep_t,
           n_keep, bw_out, nzero, overflow, cap)
    return seg_ptr, seg_idx, seg_val, n_keep_t


def knn_kernel(ref, qry=None, *, knn, knn_max=None, decay=40, thresh=1e-4, bandwidth=None, bandwidth_scale=1.0):
    """Raw (unsymmetrised) kNN / alpha-decay kernel from the rows of ``qry`` (default ``ref``) to ``ref`` as DeviceCSR.

    Semantics = reference ``kNNGraph.build_kernel_to_data`` (graphs.py:819-982) with the float64
    path: ``knn`` is the effective neighbour count (callers pass knn+1 for the self-including
    in-sample build), ``knn_max`` likewise.  Returns (csr, info) with info['bandwidth'] (device),
    info['nzero'] (zero-distance candidates per row, for duplicate warnings).
    """
    E.require_cuda()
    qry = ref if qry is None else qry
    nq, nr, d = qry.n, ref.n, ref.d
    if qry.is64 != ref.is64 or qry.metric != ref.metric:
        raise ValueError("query and reference operands must have the same dtype and metric")
    x64 = int(ref.is64) | (METRIC_CODE[ref.metric] << 1)            # x_kind of the refine entry points
    binary = decay is None
    knn = int(min(knn, nr))
    kmax = 0 if knn_max is None else int(knn_max)
    if kmax >= nr:
        kmax = 0
    plan = plan_search(default_impl(), d, ref.n_pad, ref.metric, knn, kmax, binary)
    sweep = _sweep_simt if plan.impl == "simt" else _sweep_tc
    cand, tau, q_n2, eps_rel, scale = sweep(plan, qry, ref)

    # bandwidth argument
    bw_mode, bw_fixed = 0, None
    if not binary and bandwidth is not None:
        if np.ndim(bandwidth) == 0:
            bw_mode, bw_fixed = 1, torch.tensor([float(bandwidth)], dtype=torch.float64, device=_dev())
        else:
            bw_arr = np.asarray(bandwidth, dtype=np.float64).reshape(-1)
            if bw_arr.shape[0] != nq:
                raise ValueError("bandwidth must be a scalar or have one entry per row ({}), got {}".format(
                    nq, bw_arr.shape[0]))
            bw_mode, bw_fixed = 2, torch.from_numpy(bw_arr).to(_dev())
    # kernel parameters, in the order both refine entry points take them
    kern = (knn, kmax, -1.0 if binary else float(decay), 1.0 if binary else float(thresh), bw_fixed, bw_mode,
            float(bandwidth_scale))

    S = plan.S
    st_idx = _empty((nq, S), torch.int32)
    st_val = _empty((nq, S), torch.float64)
    n_keep = _empty((nq,), torch.int32)
    bw_out = _empty((nq,), torch.float64)
    lim2 = _empty((nq,), torch.float32)
    status = _empty((nq,), torch.int32)
    nzero = _empty((nq,), torch.int32)
    maxnorm = (ref.l1_norms()[1] if ref.is64 else 0.0) if ref.metric == "cityblock" else ref.maxnorm
    E.call("gtb_refine_topk", qry.X, nq, ref.X, d, x64, cand, S, S, tau, plan.ntau, q_n2, maxnorm, eps_rel, *kern,
           st_idx, st_val, n_keep, bw_out, lim2, status, nzero)

    todo_rows = _empty((nq,), torch.int32)
    count = _empty((1,), torch.int32)
    E.call("gtb_compact_todo", status, nq, todo_rows, count)
    nt = int(count.item())                       # host sync #1
    _STATS.update(rows=nq, radius_rows=nt, S=S, radius_pairs=0, impl=plan.impl, euclidean_fallback_rows=0)

    seg = (None,) * 4
    if nt > 0:
        todo_rows = todo_rows[:nt].contiguous()
        seg = _radius_pass(plan, qry, ref, scale, todo_rows, lim2, status, n_keep, bw_out, nzero, x64, kern)

    indptr = exclusive_scan(n_keep)
    nnz = int(indptr[-1].item())                 # host sync #2
    out_idx = _empty((nnz,), torch.int32)
    out_val = _empty((nnz,), torch.float64)
    E.call("gtb_csr_gather", st_idx, st_val, n_keep, status, indptr, nq, S, todo_rows if nt else None, nt, *seg,
           out_idx, out_val)
    _STATS.update(nnz_raw=nnz)
    csr = DeviceCSR(indptr, out_idx, out_val, (nq, nr))
    return csr, {"bandwidth": bw_out, "nzero": nzero}


def sort_rows(ptr, idx, val, n):
    """Order every row of a CSR by column, in place (csrc/symm.cu: tiered segmented sort)."""
    if n == 0 or idx.shape[0] == 0:
        return
    E.call("gtb_csr_sort_rows", ptr, idx, val, n, _empty((1,), torch.int32))


def cursor32(ptr):
    """32-bit copy of the first n entries of a row-pointer array: the per-row scatter cursors."""
    n = ptr.shape[0] - 1
    cur = _empty((max(n, 1),), torch.int32)
    if n:
        E.call("gtb_cast_indptr", ptr, n, cur)
    return cur


def transpose_records(R, sort_min_total=None, pa=None):
    """Rows of R^T as 16-byte edge records {int32 i, int32 j, float64 w} (csrc/symm.cu): histogram of the columns ->
    scan -> scatter (one atomic + one 16-byte store per edge).  Rows come out in arrival order; rows whose length plus
    the matching row of ``pa`` exceeds ``sort_min_total`` are then ordered by column (None: no sort, 0: every row).
    Returns (ptr_t int64 [n_cols + 1], records [nnz, 2] int64)."""
    n_rows, n_cols = R.shape
    cnt = _empty((n_cols,), torch.int32)
    E.call("gtb_transpose_count", R.indices, R.nnz, 0, cnt, n_cols)
    ptr_t = exclusive_scan(cnt)
    rec = _empty((R.nnz, 2), torch.int64)
    if R.nnz:
        E.call("gtb_transpose_scatter", R.indptr, R.indices, R.data, n_rows, 0, 0, cursor32(ptr_t), rec)
        if sort_min_total is not None:
            sort_records(ptr_t, rec, n_cols, pa, sort_min_total)
    return ptr_t, rec


def sort_records(ptr_t, rec, n, pa=None, min_total=0):
    if n and rec.shape[0]:
        E.call("gtb_rec_sort_rows", ptr_t, rec, n, pa, int(min_total), _empty((1,), torch.int32))


def transpose_csr(R):
    """R^T as a DeviceCSR with column-sorted rows."""
    ptr_t, rec = transpose_records(R, sort_min_total=0)
    idx = rec.view(torch.int32).view(-1, 4)[:, 0].contiguous()
    val = rec.view(torch.float64).view(-1, 2)[:, 1].contiguous()
    return DeviceCSR(ptr_t, idx, val, (R.shape[1], R.shape[0]))


def merge_with_transpose(A_ptr, A_idx, A_val, T_ptr, T_rec, n_rows, row0, mode, theta, want_p=True, flags=None):
    """sym(A, T) row by row (csrc/symm.cu sym_merge): returns (outptr, k_idx, k_val, p_val | None, degree, newlen).
    ``T_rec``: record rows of the transposed matrix in any order (long rows are sorted in place by the count call)."""
    newlen = _empty((n_rows,), torch.int32)
    worklist = _empty((n_rows + 1,), torch.int32)        # rows too long for the register path, sorted inside the call
    E.call("gtb_sym_merge_count", A_ptr, A_idx, A_val, T_ptr, T_rec, n_rows, mode, theta, newlen, worklist)
    outptr = exclusive_scan(newlen)
    nnz = int(outptr[-1].item())
    k_idx = _empty((nnz,), torch.int32)
    k_val = _empty((nnz,), torch.float64)
    p_val = _empty((nnz,), torch.float64) if want_p else None
    degree = _empty((n_rows,), torch.float64)
    E.call("gtb_sym_merge_fill", A_ptr, A_idx, A_val, T_ptr, T_rec, n_rows, row0, mode, theta, outptr,
           k_idx, k_val, p_val, degree, flags)
    return outptr, k_idx, k_val, p_val, degree, newlen


def symmetrize_normalize(R, kernel_symm="+", theta=None, anisotropy=0.0, want_p=True):
    """``BaseGraph._build_kernel`` post-processing (base.py:534-592) + ``P`` (base.py:645).

    Returns (K DeviceCSR, P values tensor | None, degree tensor, flags int) where flags bit 0 =
    asymmetric beyond 1e-5 (only evaluated for kernel_symm=None), bit 1 = a row has no diagonal.
    """
    n = R.shape[0]
    square = R.shape[0] == R.shape[1]
    mode = SYM_MODES[kernel_symm]
    flags = _zeros((1,), torch.int32)
    if mode != 3 and not square:
        raise ValueError("symmetrisation needs a square kernel")
    if mode == 3:
        if square:
            E.call("gtb_asym_check", R.indptr, R.indices, R.data, n, flags)
        K = R
        P = _empty((R.nnz,), torch.float64) if want_p else None
        degree = _empty((n,), torch.float64)
        E.call("gtb_row_finalize", K.indptr, K.indices, K.data, n, P, degree, flags, int(square))
    else:
        th = 0.0 if theta is None else float(theta)
        ptr_t, rec = transpose_records(R)                # arrival order: the merge sorts the (few) long rows itself
        outptr, k_idx, k_val, P, degree, _ = merge_with_transpose(
            R.indptr, R.indices, R.data, ptr_t, rec, n, 0, mode, th,
            want_p=want_p and anisotropy == 0, flags=flags)
        K = DeviceCSR(outptr, k_idx, k_val, R.shape)
    if anisotropy != 0:
        E.call("gtb_anisotropy", K.indptr, K.indices, K.data, degree, float(anisotropy), n)
        P = _empty((K.nnz,), torch.float64) if want_p else None
        E.call("gtb_row_finalize", K.indptr, K.indices, K.data, n, P, degree, flags, 0)
    _STATS.update(nnz_sym=K.nnz)
    return K, P, degree, int(flags.item())


def row_normalize(K):
    """sklearn ``normalize(K, 'l1', axis=1)`` on a DeviceCSR -> values tensor."""
    P = _empty((K.nnz,), torch.float64)
    flags = _zeros((1,), torch.int32)
    if K.shape[0]:
        E.call("gtb_row_finalize", K.indptr, K.indices, K.data, K.shape[0], P, None, flags, 0)
    return P


def row_sums(K):
    """Row L1 sums of a DeviceCSR (``np.sum(K, 1)`` for the non-negative kernels of this package)."""
    deg = _empty((K.shape[0],), torch.float64)
    flags = _zeros((1,), torch.int32)
    E.call("gtb_row_finalize", K.indptr, K.indices, K.data, K.shape[0], None, deg, flags, 0)
    return deg


def csr_from_scipy(M):
    """scipy sparse -> DeviceCSR (canonical CSR: sorted columns, duplicates summed)."""
    from scipy import sparse
    M = sparse.csr_matrix(M, dtype=np.float64)
    if not M.has_canonical_format:
        M = M.copy()
        M.sum_duplicates()
    dev = _dev()
    return DeviceCSR(torch.from_numpy(M.indptr.astype(np.int64)).to(dev),
                     torch.from_numpy(M.indices.astype(np.int32)).to(dev),
                     torch.from_numpy(np.ascontiguousarray(M.data)).to(dev), M.shape)


def spmm(A, B, vals=None):
    """``A.dot(B)`` on the device (csrc/spmm.cu): A = DeviceCSR (``vals`` substitutes its values, e.g. the
    diffusion operator sharing K's structure), B = float64 CUDA tensor [n_cols, f] (row-major, any row
    stride).  Accumulation order and rounding are scipy's, so the result is bit-identical to the host product
    the reference computes (base.py:1229)."""
    if B.dim() != 2 or B.shape[0] != A.shape[1]:
        raise ValueError("shapes {} and {} not aligned".format(A.shape, tuple(B.shape)))
    if B.dtype != torch.float64 or B.stride(1) != 1:
        B = B.to(torch.float64).contiguous()
    f = B.shape[1]
    out = _empty((A.shape[0], f), torch.float64)
    if A.shape[0] == 0 or f == 0:
        return out
    E.call("gtb_spmm_csr", A.indptr, A.indices, A.data if vals is None else vals, A.shape[0], B, B.stride(0), f,
           out, f)
    return out
