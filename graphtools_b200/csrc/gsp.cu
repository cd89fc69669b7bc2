// Graph Laplacian of a kernel matrix on the device (graph signal processing, graphtools_b200/gsp.py): pygsp's
// Graph.compute_laplacian on W = K with its diagonal removed.
//
//   dw_i = sum of the off-diagonal stored values of row i, added sequentially in column order (from +0.0);
//   combinatorial  L_ij = -W_ij,                L_ii = dw_i;
//   normalized     L_ij = -((s_i W_ij) s_j),    L_ii = 1,   s_i = 1 / sqrt(dw_i) (both correctly rounded);
//   a vertex with dw_i = 0 gets s_i = 0 and a stored L_ii = 0 under both types.
//
// L stores K's off-diagonal pattern plus exactly one diagonal entry per row, also where K stores none.  Two passes:
// count writes dw and the row lengths of L, gtb_exclusive_scan turns those into L's row pointers, and fill writes the
// column-sorted rows (the normalized fill reads dw_j of the neighbours, which is why dw comes first).
#include "common.cuh"
#include "gtb200.h"

namespace {

constexpr int GSP_THREADS = 256;

// one thread per row: the sequential sum fixes the rounding order
__global__ void laplacian_count_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx,
                                       const double* __restrict__ val, int64_t n, double* __restrict__ dw,
                                       int32_t* __restrict__ len) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  const int64_t p0 = indptr[row], p1 = indptr[row + 1];
  double acc = 0.0;
  int has_diag = 0;
  for (int64_t p = p0; p < p1; ++p) {
    if (idx[p] == row) has_diag = 1;
    else acc = __dadd_rn(acc, val[p]);
  }
  dw[row] = acc;
  len[row] = (int32_t)(p1 - p0 - has_diag + 1);
}

__device__ __forceinline__ double inv_sqrt_degree(double d) {
  return d == 0.0 ? 0.0 : __ddiv_rn(1.0, __dsqrt_rn(d));
}

// one warp per row, lanes striding over its entries.  An off-diagonal entry at position p of K's row moves one
// place right in L when its column lies past the diagonal and K stores no diagonal entry; the diagonal goes where
// the first column >= row sits, or last when there is none.
__global__ void laplacian_fill_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx,
                                      const double* __restrict__ val, int64_t n, const double* __restrict__ dw,
                                      const int64_t* __restrict__ lptr, int normalized, int32_t* __restrict__ lidx,
                                      double* __restrict__ lval) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (GSP_THREADS / 32) + (threadIdx.x >> 5);
  if (row >= n) return;
  const int64_t p0 = indptr[row], p1 = indptr[row + 1], q0 = lptr[row], q1 = lptr[row + 1];
  const int shift = (q1 - q0 == p1 - p0 + 1) ? 1 : 0;       // 1: K stores no diagonal entry in this row
  const double d = dw[row];
  const double si = normalized ? inv_sqrt_degree(d) : 0.0;
  for (int64_t p = p0 + lane; p < p1; p += 32) {
    const int32_t j = idx[p];
    if (j >= row && (p == p0 || idx[p - 1] < row)) {         // the diagonal's slot
      lidx[q0 + (p - p0)] = (int32_t)row;
      lval[q0 + (p - p0)] = normalized ? (d == 0.0 ? 0.0 : 1.0) : d;
    }
    if (j == row) continue;
    const int64_t q = q0 + (p - p0) + (j > row ? shift : 0);
    lidx[q] = j;
    lval[q] = normalized ? -__dmul_rn(__dmul_rn(si, val[p]), inv_sqrt_degree(dw[j])) : -val[p];
  }
  if (lane == 0 && (p1 == p0 || idx[p1 - 1] < row)) {       // no column >= row: the diagonal closes the row
    lidx[q1 - 1] = (int32_t)row;
    lval[q1 - 1] = normalized ? (d == 0.0 ? 0.0 : 1.0) : d;
  }
}

}  // namespace

extern "C" int gtb_laplacian_count(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n,
                                   double* dw, int32_t* len, void* stream) {
  GTB_CHECK_ARG(n > 0, "bad shape");
  laplacian_count_kernel<<<(unsigned)gtb_cdiv(n, GSP_THREADS), GSP_THREADS, 0, (cudaStream_t)stream>>>(
      indptr, idx, val, n, dw, len);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_laplacian_fill(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n,
                                  const double* dw, const int64_t* lptr, int lap_type, int32_t* lidx, double* lval,
                                  void* stream) {
  GTB_CHECK_ARG(n > 0, "bad shape");
  GTB_CHECK_ARG(lap_type == 0 || lap_type == 1, "lap_type must be 0 (combinatorial) or 1 (normalized)");
  laplacian_fill_kernel<<<(unsigned)gtb_cdiv(n, GSP_THREADS / 32), GSP_THREADS, 0, (cudaStream_t)stream>>>(
      indptr, idx, val, n, dw, lptr, lap_type, lidx, lval);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}
