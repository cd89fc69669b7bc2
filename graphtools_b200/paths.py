"""Geodesic distances along the graph: ``BaseGraph.shortest_path`` (reference base.py:934-988) on the device.

The reference wrapper, restated (the error texts and the ``weighted`` rule are written from the graphtools >= 1.5
behaviour, not pinned against a copy of v2.1.0)::

    distance None  -> "data" if not G.weighted else "affinity"
    "constant"     -> edge length K_ij                                   (unweighted graphs)
    "data"         -> |data_nu_i - data_nu_j|_2 on every stored entry of K (unweighted graphs)
    "affinity"     -> -log(K_ij)                                         (weighted graphs)
    D = scipy.sparse.csgraph.shortest_path(lengths, method=method)       # directed
    D = (D + D.T) / 2;  D[D == 0] = inf;  D[diag] = 0

Here every step after the kernel build runs in HBM (csrc/paths.cu): edge lengths, connected components, batched
multi-source traversal, the transpose-average and the two quirks; only the finished [N, N] float64 matrix is
copied to the host.  The traversal computes the fixpoint of float64 relaxations, which is bit-identical to
``method="D"`` (see DESIGN.md section 2b); ``method`` is validated as scipy does but selects nothing.
"""
import numpy as np
import torch
from scipy import sparse

from . import _engine as E
from . import pipeline
from .logging_util import logger as _logger

BATCH = 256                     # sources per traversal launch (8 chunks of 32 lanes)
DISTANCES = {"constant": 0, "data": 1, "affinity": 2}
METHODS = ("auto", "FW", "D", "BF", "J")
_STATS = {}


def stats():
    """Counters of the last call: n, nnz, components, batches, and the (source, edge) pairs the traversal covers."""
    return dict(_STATS)


def default_distance(G):
    if not G.weighted:
        _logger.log_info("Using ambient data distances.")
        return "data"
    _logger.log_info("Using negative log affinity distances.")
    return "affinity"


def check_distance(G, distance):
    if distance in ("data", "constant") and G.weighted:
        raise NotImplementedError("Graph shortest path with constant or data distance only implemented for "
                                  "unweighted graphs. For weighted graphs, use `distance='affinity'`.")
    if distance == "affinity" and not G.weighted:
        raise ValueError("Graph shortest path with affinity distance only valid for weighted graphs. For unweighted "
                         "graphs, use `distance='constant'` or `distance='data'`.")
    if distance not in DISTANCES:
        raise ValueError("Expected `distance` in ['constant', 'data', 'affinity']. Got {}".format(distance))


def _host_available_bytes():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return None


def _check_memory(n, nnz):
    result = 8 * n * n
    avail = _host_available_bytes()
    if avail is not None and result > avail:
        raise MemoryError("shortest_path: the {0} x {0} float64 result needs {1:.1f} GB of host memory, {2:.1f} GB "
                          "are available".format(n, result / 1e9, avail / 1e9))
    work = result + 8 * n * BATCH + E.lib().gtb_sp_ws_bytes(n, BATCH) + 12 * nnz + 16 * n
    free, _ = torch.cuda.mem_get_info()
    free += torch.cuda.memory_reserved() - torch.cuda.memory_allocated()
    if work > free:
        raise MemoryError("shortest_path: the {0} x {0} result and its working set need {1:.1f} GB of device memory, "
                          "{2:.1f} GB are free".format(n, work / 1e9, free / 1e9))


def dense_to_csr(K):
    """Present entries of a dense float64 CUDA tensor as a DeviceCSR (what ``csr_matrix(K)`` stores)."""
    n_rows, n_cols = K.shape
    cnt = pipeline._empty((n_rows,), torch.int32)
    E.call("gtb_dense_to_csr_count", K, n_rows, n_cols, cnt)
    indptr = pipeline.exclusive_scan(cnt)
    nnz = int(indptr[-1].item())
    idx = pipeline._empty((nnz,), torch.int32)
    val = pipeline._empty((nnz,), torch.float64)
    if nnz:
        E.call("gtb_dense_to_csr_fill", K, n_rows, n_cols, indptr, idx, val)
    return pipeline.DeviceCSR(indptr, idx, val, (n_rows, n_cols))


def _data_rows(G):
    """data_nu in HBM in the dtype numpy computes the reference's distances in: float32 stays float32, everything
    else is float64."""
    dev = G.__dict__.get("_dev_data_nu")
    if dev is not None and dev.dtype in (torch.float32, torch.float64):
        return dev.contiguous()
    X = G.data_nu
    if sparse.issparse(X):
        X = X.toarray()
    X = np.asarray(X)
    X = np.ascontiguousarray(X, dtype=np.float32 if X.dtype == np.float32 else np.float64)
    return torch.from_numpy(X).to(pipeline._dev())


def shortest_path(G, method="auto", distance=None):
    if distance is None:
        distance = default_distance(G)
    check_distance(G, distance)
    if method not in METHODS:
        raise ValueError("unrecognized method '{}'".format(method))
    G._ensure_built()
    K = G._dev_kernel
    if not isinstance(K, pipeline.DeviceCSR):
        K = dense_to_csr(K.contiguous())
    n, nnz = K.shape[0], K.nnz
    _check_memory(n, nnz)

    lengths = pipeline._empty((nnz,), torch.float64)
    flags = pipeline._zeros((1,), torch.int32)
    X, d, x_f64 = None, 0, 0
    if distance == "data":
        X = _data_rows(G)
        d, x_f64 = X.shape[1], int(X.dtype == torch.float64)
    if nnz:
        E.call("gtb_sp_lengths", K.indptr, K.indices, K.data, n, X, d, x_f64, DISTANCES[distance], lengths, flags)
    if int(flags.item()) & 1:
        raise NotImplementedError("Graph shortest path with negative edge lengths (-log of affinities above 1, e.g. "
                                  "from anisotropy > 0) is not implemented")

    labels = pipeline._empty((n,), torch.int32)
    E.call("gtb_sp_components", K.indptr, K.indices, n, labels)
    lab = labels.cpu().numpy()
    # sources sorted by component: the lanes of a traversal launch then mostly share one component
    order = np.argsort(lab, kind="stable").astype(np.int32)
    rowlen = np.diff(K.indptr.cpu().numpy())
    comp_edges = np.bincount(lab, weights=rowlen, minlength=n)
    comp_size = np.bincount(lab, minlength=n)

    D = pipeline._empty((n, n), torch.float64)
    dist = pipeline._empty((n, BATCH), torch.float64)
    ws = pipeline._empty((E.lib().gtb_sp_ws_bytes(n, BATCH),), torch.uint8)
    src_all = torch.from_numpy(order).to(pipeline._dev())
    for s0 in range(0, n, BATCH):
        nb = min(BATCH, n - s0)
        src = src_all[s0:s0 + nb]
        E.call("gtb_sp_traverse", K.indptr, K.indices, lengths, n, src, nb, BATCH, dist, ws)
        E.call("gtb_sp_store_rows", dist, BATCH, n, src, nb, D, n)
    E.call("gtb_sp_finish", D, n)
    _STATS.clear()
    _STATS.update(n=n, nnz=nnz, components=int(np.count_nonzero(comp_size)), batches=-(-n // BATCH),
                  source_edges=int(np.dot(comp_size, comp_edges)), distance=distance)

    got = pipeline._d2h_pooled([("D", D)])
    if got is not None:
        return got["D"].reshape(n, n)
    out = pipeline.d2h_pinned(D).numpy()
    torch.cuda.current_stream().synchronize()
    return out
