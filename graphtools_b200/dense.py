"""Dense (exact-graph) device operations: thin wrappers over csrc/dense.cu."""
import numpy as np
import torch

from . import _engine as E
from . import pipeline

SYM = {"+": 0, "*": 1, "mnn": 2, None: 3}
METRIC = {"euclidean": 0, "cosine": 1, "cityblock": 2, "manhattan": 2, "l1": 2, "sqeuclidean": 3, "correlation": 4}


def _same_dtype(Xq, Xr):
    """Both operands in the precision of the data as given: float64 when either is (scipy's pdist / cdist work on
    the float64 values the reference holds), else float32."""
    is64 = Xq.dtype == torch.float64 or Xr.dtype == torch.float64
    dt = torch.float64 if is64 else torch.float32
    return Xq.to(dt).contiguous(), Xr.to(dt).contiguous(), int(is64)


def _row_centred(X):
    """float64 copy of X minus each row's mean, scipy's correlation arithmetic (``XA - XA.mean(axis=1)``, then its
    cosine routine).  Constant rows are set to exactly zero, so that their distances are NaN whatever the rounding of
    their mean: the degenerate rows of ``pipeline.degenerate_rows``."""
    X = X.to(torch.float64)
    C = X - X.mean(dim=1, keepdim=True)
    C[pipeline.degenerate_rows(X, "correlation")] = 0.0
    return C.contiguous()


def _operands(Xq, Xr, metric):
    """(Xq, Xr, is64, metric code) for gtb_dense_kernel: correlation runs the cosine branch on row-centred float64
    copies (8 n d bytes each, small beside the n^2 output)."""
    Xq, Xr, is64 = _same_dtype(Xq, Xr)
    if metric != "correlation":
        return Xq, Xr, is64, METRIC[metric]
    Cq = _row_centred(Xq)
    return Cq, (Cq if Xr is Xq else _row_centred(Xr)), 1, METRIC["cosine"]


def dense_affinity(Xq, Xr, bw_q, bw_r, decay, thresh, symm=None, theta=None, want_rowsum=True, metric="euclidean"):
    """[nq, nr] float64 thresholded alpha-decay affinities; symmetrised in the same sweep when
    ``bw_r`` is given (square problems)."""
    Xq, Xr, is64, code = _operands(Xq, Xr, metric)
    nq, d = Xq.shape
    nr = Xr.shape[0]
    out = pipeline._empty((nq, nr), torch.float64)
    rowsum = pipeline._empty((nq,), torch.float64) if want_rowsum else None
    what = 2 if bw_r is not None else 1
    E.call("gtb_dense_kernel", Xq, nq, Xr, nr, d, is64, what, code, bw_q, bw_r, float(decay), float(thresh),
           SYM[symm], 0.0 if theta is None else float(theta), out, rowsum)
    return out, rowsum


def dense_distances(Xq, Xr, metric="euclidean"):
    Xq, Xr, is64, code = _operands(Xq, Xr, metric)
    nq, d = Xq.shape
    nr = Xr.shape[0]
    out = pipeline._empty((nq, nr), torch.float64)
    E.call("gtb_dense_kernel", Xq, nq, Xr, nr, d, is64, 0, code, None, None, 0.0, 0.0, 3, 0.0, out, None)
    return out


def rowsum_dense(K):
    s = pipeline._empty((K.shape[0],), torch.float64)
    E.call("gtb_dense_rowsum", K, K.shape[0], K.shape[1], s)
    return s


def row_normalize_dense(K, rowsum=None):
    if rowsum is None:
        rowsum = rowsum_dense(K)
    out = pipeline._empty(tuple(K.shape), torch.float64)
    E.call("gtb_dense_row_scale", K, rowsum, K.shape[0], K.shape[1], out)
    return out


def anisotropy_dense(K, alpha, deg=None):
    if deg is None:
        deg = rowsum_dense(K)
    newsum = pipeline._empty((K.shape[0],), torch.float64)
    E.call("gtb_dense_anisotropy", K, deg, float(alpha), K.shape[0], newsum)
    return K


def symmetrize_dense(K, kernel_symm, theta):
    """Dense symmetrisation of an arbitrary square matrix already in HBM (host-callable helper).
    The exact-graph build does not use this: it fuses the rule into the distance tile."""
    if kernel_symm == "+":
        return (K + K.T) / 2
    if kernel_symm == "*":
        return K * K.T
    if kernel_symm == "mnn":
        return theta * torch.minimum(K, K.T) + (1 - theta) * torch.maximum(K, K.T)
    return K


def _dense_to_csr(K):
    """Dense [n, m] device matrix -> DeviceCSR of its non-zeros (used to feed the landmark kernels)."""
    nz = K != 0
    counts = nz.sum(dim=1, dtype=torch.int32)
    indptr = pipeline.exclusive_scan(counts.contiguous())
    cols = nz.nonzero()[:, 1].to(torch.int32).contiguous()
    return pipeline.DeviceCSR(indptr, cols, K[nz].contiguous(), tuple(K.shape))


def _one_hot(labels, L):
    C = torch.zeros((labels.shape[0], L), dtype=torch.float64, device=labels.device)
    C[torch.arange(labels.shape[0], device=labels.device), labels.long()] = 1.0
    return C


def dense_landmark(K, labels, L):
    """Landmark operator of a DENSE kernel (graphs.py:1169-1246 on an ndarray K): two plain float64 library GEMMs --
    pmn = C^T K, op = rownorm(pmn) rownorm(pmn^T).  (Going through the sparse aggregation kernels would turn every
    row of the n x n matrix into a "hub row".)  Plumbing, not a hot path: dense graphs are the small-n case."""
    C = _one_hot(labels, L)
    pmn = C.T @ K                                   # [L, n]: sum of the kernel rows of each cluster
    pnm = pmn.T.contiguous()                        # [n, L]
    rs_m = pmn.abs().sum(1, keepdim=True)
    rs_n = pnm.abs().sum(1, keepdim=True)
    pmn_n = torch.where(rs_m != 0, pmn / rs_m, pmn)
    pnm_n = torch.where(rs_n != 0, pnm / rs_n, pnm)
    op = pmn_n @ pnm_n
    return op.cpu().numpy(), pnm_n.cpu().numpy()


def dense_landmark_extend(Kyx, labels, L):
    """rownorm(Kyx C) for a dense out-of-sample kernel (graphs.py:1272-1288)."""
    agg = Kyx @ _one_hot(labels, L)
    rs = agg.abs().sum(1, keepdim=True)
    return torch.where(rs != 0, agg / rs, agg).cpu().numpy()


# ---------------------------------------------------------------------- float64-faithful products on the int8 tensor cores
GEMM_SLICES = 7          # digit planes per operand: 54 significant bits below the row / column maximum


def _pad128(n):
    return (int(n) + 127) // 128 * 128


def slice_operand(X, transposed=False, slices=GEMM_SLICES):
    """Digit planes of a float64 device matrix for gtb_gemm_i8: the rows of X (left operand) or, with
    ``transposed``, its columns (right operand).  Returns (int8 [slices, R_pad, K_pad], scale [R])."""
    assert X.dtype == torch.float64 and X.dim() == 2 and X.stride(1) == 1
    if transposed:
        K, R = X.shape
    else:
        R, K = X.shape
    R_pad, K_pad = _pad128(R), _pad128(K)
    dig = pipeline._empty((slices, R_pad, K_pad), torch.int8)
    scale = pipeline._empty((R,), torch.float64)
    E.call("gtb_slice_f64", X, R, K, X.stride(0), int(bool(transposed)), slices, R_pad, K_pad, dig, scale)
    return dig, scale


def gemm_digits(a, b, M, N, row_bytes=None):
    """C [M, N] float64 = A . B from the digit planes ``a = slice_operand(A)`` and ``b = slice_operand(B, True)``."""
    import os
    (ad, sa), (bd, sb) = a, b
    S, M_pad, K_pad = ad.shape
    assert bd.shape[0] == S and bd.shape[2] == K_pad
    if K_pad > E.lib().gtb_gemm_max_k():
        raise ValueError("inner dimension {} exceeds the exact int32 accumulation range ({})".format(
            K_pad, E.lib().gtb_gemm_max_k()))
    rb = int(os.environ.get("GTB_GEMM_ROW_BYTES", "64")) if row_bytes is None else int(row_bytes)
    C = pipeline._empty((M, N), torch.float64)
    E.call("gtb_gemm_i8", ad, bd, S, M, N, K_pad, M_pad, bd.shape[1], sa, sb, C, N, rb)
    return C


def gemm_f64(A, B, slices=GEMM_SLICES, row_bytes=None):
    """A @ B for float64 device matrices: exact int32 accumulation of base-256 digit products on the tensor cores
    (csrc/gemm.cu), combined in float64 -- error below that of a float64 dot product of the same length."""
    A = A.contiguous() if A.stride(1) != 1 else A
    B = B.contiguous() if B.stride(1) != 1 else B
    assert A.shape[1] == B.shape[0], (tuple(A.shape), tuple(B.shape))
    return gemm_digits(slice_operand(A, False, slices), slice_operand(B, True, slices), A.shape[0], B.shape[1],
                       row_bytes)


def matrix_power(M, t, slices=GEMM_SLICES):
    """M^t for a square float64 device matrix with numpy's multiplication schedule (np.linalg.matrix_power: binary
    decomposition of t, squarings of z, products result @ z) -- what the callers of ``G.landmark_op`` /
    a dense ``G.diff_op`` run on the host.  Every product is gemm_f64; z^2 slices z once per operand role."""
    t = int(t)
    if M.dim() != 2 or M.shape[0] != M.shape[1]:
        raise ValueError("matrix_power needs a square matrix")
    if t < 0:
        raise ValueError("negative powers are not supported on the device")
    n = M.shape[0]
    if t == 0:
        return torch.eye(n, dtype=torch.float64, device=M.device)
    M = M.to(torch.float64).contiguous()
    if t == 1:
        return M.clone()
    if t == 2:
        return gemm_f64(M, M, slices)
    if t == 3:
        return gemm_f64(gemm_f64(M, M, slices), M, slices)
    z = result = None
    while t > 0:
        if z is None:
            z = M
        else:
            z = gemm_f64(z, z, slices)
        t, bit = divmod(t, 2)
        if bit:
            result = z if result is None else gemm_f64(result, z, slices)
    return result
