// CSR (float64) x dense (float64, row-major) product on the device: out = A . B.
//
// Replaces scipy's csr_matvecs behind `transitions.dot(transform)` (reference graphtools/base.py:1229),
// the repeated `diff_op.dot(X)` of the callers (MAGIC-style diffusion) and the two sparse products per power
// iteration of sklearn randomized_svd(diff_aff) (graphs.py:1217).  HBM / gather bound: every stored entry pulls
// one f-wide row of B (8f bytes, coalesced), so algorithmic bytes = nnz (12 + 8f) + 8 n_rows f.
//
// Arithmetic contract: each output element is accumulated in stored (column-sorted) order with a separate
// multiply and add (no FMA contraction) -- the order and rounding of scipy's axpy loop, so results are
// bit-identical to `A.dot(B)` on the host.
//
// Layout: one warp per output row; lane l owns columns {2l, 2l+1} of every 64-column chunk (double2 loads:
// 512 contiguous bytes per warp and chunk).  Entries are consumed four at a time so that four independent row
// gathers are in flight per warp.
//
// The same body, instantiated with the Chebyshev epilogue, is the filter step of the diffusion-map eigensolver
// (eigen.py): out = (alpha (A . Y) + beta Y) + gamma Z, each product and sum rounded separately, i.e. numpy's
// `alpha*S + beta*Y + gamma*Z` after scipy's S = A.dot(Y).  At the solver's block widths (16-32 columns) a whole
// warp per row would leave most lanes idle, so that entry point gives each row the smallest power-of-two group of
// LPR lanes that covers its columns two per lane, and packs 32 / LPR rows into a warp.  Algorithmic bytes per call:
// nnz (12 + 8b) + 8 N (3b + 1) -- CSR, row gathers, the own rows of Y and Z, the write, indptr.
//
// A second epilogue on top of that one is the step of a Chebyshev filter bank (gsp.py, pygsp's cheby_op): after
// out = (alpha (A . Y) + beta Y) + gamma Z it adds coef[a] * out into each of F accumulators R_a, every product and
// sum rounded separately (numpy's `r += c * out`), while the thread still holds the out values in registers, so T_k
// is not read back from HBM.  Algorithmic bytes per call: nnz (12 + 8f) + 8 N (f (3 + 2F) + 1).
#include "common.cuh"
#include "gtb200.h"

namespace {

constexpr int SPMM_WARPS = 8;
constexpr int SPMM_UNROLL = 4;

// NCH = chunks of 2 LPR columns held in registers by one pass of a row's LPR-lane group (f <= 2 LPR NCH handled in
// one sweep over the row).  CHEB adds the epilogue (alpha s + beta B[row]) + gamma Z[row]; B is then square-indexed
// (Y) and Z may alias out: every element of Z is read only by the thread that writes that element of out.  ACC
// (with CHEB) adds R[a][row] += coef[a] * out[row] for the F blocks of R (block stride ldrb, leading dimension ldr).
// The ACC parameters come last so that the other instantiations keep their parameter offsets (and their SASS).
template <int NCH, int LPR, bool CHEB, bool ACC = false>
__global__ void __launch_bounds__(SPMM_WARPS * 32)
spmm_csr_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx, const double* __restrict__ val,
                int64_t n_rows, const double* __restrict__ B, int64_t ldb, int f, int col0, double* out,
                int64_t ldo, double alpha, double beta, double gamma, const double* Z, int64_t ldz,
                const double* coef = nullptr, int F = 0, double* R = nullptr, int64_t ldr = 0, int64_t ldrb = 0) {
  static_assert(CHEB || !ACC, "the accumulation epilogue follows the Chebyshev one");
  constexpr int CW = 2 * LPR;                      // columns per chunk
  const int lane = threadIdx.x & (LPR - 1);
  const int64_t row = (int64_t)blockIdx.x * (SPMM_WARPS * 32 / LPR) + (threadIdx.x / LPR);
  if (row >= n_rows) return;
  const int64_t p0 = indptr[row], p1 = indptr[row + 1];
  double ax[NCH], ay[NCH];
  bool okx[NCH], oky[NCH];
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    ax[c] = 0.0; ay[c] = 0.0;
    const int k = col0 + c * CW + 2 * lane;
    okx[c] = k < f; oky[c] = k + 1 < f;
  }
  const bool vec = ((ldb & 1) == 0) && ((reinterpret_cast<uintptr_t>(B) & 15) == 0);
  for (int64_t p = p0; p < p1; p += SPMM_UNROLL) {
    double a[SPMM_UNROLL];
    const double* src[SPMM_UNROLL];
#pragma unroll
    for (int u = 0; u < SPMM_UNROLL; ++u) {
      const bool in = p + u < p1;
      a[u] = in ? val[p + u] : 0.0;
      src[u] = B + (int64_t)(in ? idx[p + u] : 0) * ldb + col0 + 2 * lane;
    }
    double bx[SPMM_UNROLL][NCH], by[SPMM_UNROLL][NCH];
#pragma unroll
    for (int u = 0; u < SPMM_UNROLL; ++u) {
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        bx[u][c] = 0.0; by[u][c] = 0.0;
        if (p + u < p1) {
          if (vec && oky[c]) {
            const double2 t = *reinterpret_cast<const double2*>(src[u] + c * CW);
            bx[u][c] = t.x; by[u][c] = t.y;
          } else {
            if (okx[c]) bx[u][c] = src[u][c * CW];
            if (oky[c]) by[u][c] = src[u][c * CW + 1];
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < SPMM_UNROLL; ++u) {
      if (p + u < p1) {
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          ax[c] = __dadd_rn(ax[c], __dmul_rn(a[u], bx[u][c]));
          ay[c] = __dadd_rn(ay[c], __dmul_rn(a[u], by[u][c]));
        }
      }
    }
  }
  double* o = out + row * ldo + col0 + 2 * lane;
  // ACC: the first accumulator's coefficient and elements are loaded together with the epilogue's Y and Z (after the
  // gathers, where registers are free), each later one while the previous one is stored
  double rc = 0.0, rx[NCH], ry[NCH];
  if constexpr (ACC) {
    rc = coef[0];
    const double* r = R + row * ldr + col0 + 2 * lane;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      rx[c] = okx[c] ? r[c * CW] : 0.0;
      ry[c] = oky[c] ? r[c * CW + 1] : 0.0;
    }
  }
  if constexpr (CHEB) {
    const double* y = B + row * ldb + col0 + 2 * lane;
    const double* z = Z + row * ldz + col0 + 2 * lane;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      if (okx[c])
        ax[c] = __dadd_rn(__dadd_rn(__dmul_rn(alpha, ax[c]), __dmul_rn(beta, y[c * CW])), __dmul_rn(gamma, z[c * CW]));
      if (oky[c])
        ay[c] = __dadd_rn(__dadd_rn(__dmul_rn(alpha, ay[c]), __dmul_rn(beta, y[c * CW + 1])),
                          __dmul_rn(gamma, z[c * CW + 1]));
    }
  }
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    if (okx[c]) o[c * CW] = ax[c];
    if (oky[c]) o[c * CW + 1] = ay[c];
  }
  if constexpr (ACC) {
    for (int a = 0; a < F; ++a) {
      double* r = R + a * ldrb + row * ldr + col0 + 2 * lane;
      double nc = 0.0, nx[NCH], ny[NCH];
      if (a + 1 < F) {
        nc = coef[a + 1];
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          nx[c] = okx[c] ? r[ldrb + c * CW] : 0.0;
          ny[c] = oky[c] ? r[ldrb + c * CW + 1] : 0.0;
        }
      }
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        if (okx[c]) r[c * CW] = __dadd_rn(rx[c], __dmul_rn(rc, ax[c]));
        if (oky[c]) r[c * CW + 1] = __dadd_rn(ry[c], __dmul_rn(rc, ay[c]));
        rx[c] = nx[c]; ry[c] = ny[c];
      }
      rc = nc;
    }
  }
}

template <int LPR>
void launch_cheb(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n, const double* Y, int64_t ldy,
                 int f, double alpha, double beta, double gamma, const double* Z, int64_t ldz, double* out,
                 int64_t ldo, cudaStream_t st) {
  const unsigned grid = (unsigned)gtb_cdiv(n, SPMM_WARPS * 32 / LPR);
  spmm_csr_kernel<1, LPR, true><<<grid, SPMM_WARPS * 32, 0, st>>>(indptr, idx, val, n, Y, ldy, f, 0, out, ldo, alpha,
                                                                 beta, gamma, Z, ldz);
}

template <int LPR>
void launch_cheb_acc(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n, const double* Y,
                     int64_t ldy, int f, double alpha, double beta, double gamma, const double* Z, int64_t ldz,
                     double* out, int64_t ldo, const double* coef, int F, double* R, int64_t ldr, int64_t ldrb,
                     cudaStream_t st) {
  const unsigned grid = (unsigned)gtb_cdiv(n, SPMM_WARPS * 32 / LPR);
  spmm_csr_kernel<1, LPR, true, true><<<grid, SPMM_WARPS * 32, 0, st>>>(indptr, idx, val, n, Y, ldy, f, 0, out, ldo,
                                                                       alpha, beta, gamma, Z, ldz, coef, F, R, ldr,
                                                                       ldrb);
}

// out[i][k] *= s[i]  /  out[i][k] = in[i][k] * s[i]   (row scaling used around the SpMM for D^-1/2 K D^-1/2 products)
__global__ void row_scale_kernel(const double* __restrict__ in, const double* __restrict__ s, int64_t n, int f,
                                 int power_neg_half, double* __restrict__ out) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n * f) return;
  const int64_t r = e / f;
  double w = s[r];
  if (power_neg_half) w = 1.0 / sqrt(w);
  out[e] = in[e] * w;
}

}  // namespace

extern "C" int gtb_spmm_csr(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n_rows,
                            const double* B, int64_t ldb, int f, double* out, int64_t ldo, void* stream) {
  GTB_CHECK_ARG(n_rows > 0 && f > 0 && ldb >= f && ldo >= f, "bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)gtb_cdiv(n_rows, SPMM_WARPS);
  for (int col0 = 0; col0 < f; col0 += 128) {
    if (f - col0 > 64)
      spmm_csr_kernel<2, 32, false><<<grid, SPMM_WARPS * 32, 0, st>>>(indptr, idx, val, n_rows, B, ldb, f, col0, out,
                                                                     ldo, 0.0, 0.0, 0.0, nullptr, 0);
    else
      spmm_csr_kernel<1, 32, false><<<grid, SPMM_WARPS * 32, 0, st>>>(indptr, idx, val, n_rows, B, ldb, f, col0, out,
                                                                     ldo, 0.0, 0.0, 0.0, nullptr, 0);
    GTB_CHECK_LAUNCH();
  }
  return GTB_OK;
}

extern "C" int gtb_spmm_cheb(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n,
                             const double* Y, int64_t ldy, int f, double alpha, double beta, double gamma,
                             const double* Z, int64_t ldz, double* out, int64_t ldo, void* stream) {
  GTB_CHECK_ARG(n > 0 && f > 0 && ldy >= f && ldz >= f && ldo >= f, "bad shape");
  GTB_CHECK_ARG(Y != nullptr && Z != nullptr && out != nullptr, "null operand");
  // out overlapping Y would overwrite rows other threads still gather.  out may be Z itself (same pointer, same
  // leading dimension: every element of Z is then read only by the thread that writes it); any other overlap with
  // Z would let one thread's write land on an element another thread still reads.
  const uintptr_t o0 = reinterpret_cast<uintptr_t>(out), o1 = o0 + (uintptr_t)(((n - 1) * ldo + f) * sizeof(double));
  const uintptr_t y0 = reinterpret_cast<uintptr_t>(Y), y1 = y0 + (uintptr_t)(((n - 1) * ldy + f) * sizeof(double));
  const uintptr_t z0 = reinterpret_cast<uintptr_t>(Z), z1 = z0 + (uintptr_t)(((n - 1) * ldz + f) * sizeof(double));
  GTB_CHECK_ARG(o1 <= y0 || y1 <= o0, "out must not overlap Y");
  GTB_CHECK_ARG((o0 == z0 && ldo == ldz) || o1 <= z0 || z1 <= o0, "out must be Z itself or not overlap it");
  cudaStream_t st = (cudaStream_t)stream;
  if (f > 64) {
    const unsigned grid = (unsigned)gtb_cdiv(n, SPMM_WARPS);
    for (int col0 = 0; col0 < f; col0 += 128) {
      if (f - col0 > 64)
        spmm_csr_kernel<2, 32, true><<<grid, SPMM_WARPS * 32, 0, st>>>(indptr, idx, val, n, Y, ldy, f, col0, out, ldo,
                                                                      alpha, beta, gamma, Z, ldz);
      else
        spmm_csr_kernel<1, 32, true><<<grid, SPMM_WARPS * 32, 0, st>>>(indptr, idx, val, n, Y, ldy, f, col0, out, ldo,
                                                                      alpha, beta, gamma, Z, ldz);
      GTB_CHECK_LAUNCH();
    }
    return GTB_OK;
  }
  const int lanes = (f + 1) / 2;                 // smallest power-of-two group with at least ceil(f / 2) lanes
  if (lanes <= 1)       launch_cheb<1>(indptr, idx, val, n, Y, ldy, f, alpha, beta, gamma, Z, ldz, out, ldo, st);
  else if (lanes <= 2)  launch_cheb<2>(indptr, idx, val, n, Y, ldy, f, alpha, beta, gamma, Z, ldz, out, ldo, st);
  else if (lanes <= 4)  launch_cheb<4>(indptr, idx, val, n, Y, ldy, f, alpha, beta, gamma, Z, ldz, out, ldo, st);
  else if (lanes <= 8)  launch_cheb<8>(indptr, idx, val, n, Y, ldy, f, alpha, beta, gamma, Z, ldz, out, ldo, st);
  else if (lanes <= 16) launch_cheb<16>(indptr, idx, val, n, Y, ldy, f, alpha, beta, gamma, Z, ldz, out, ldo, st);
  else                  launch_cheb<32>(indptr, idx, val, n, Y, ldy, f, alpha, beta, gamma, Z, ldz, out, ldo, st);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_spmm_cheb_acc(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n,
                                 const double* Y, int64_t ldy, int f, double alpha, double beta, double gamma,
                                 const double* Z, int64_t ldz, double* out, int64_t ldo, const double* coef, int F,
                                 double* R, int64_t ldr, int64_t ldrb, void* stream) {
  GTB_CHECK_ARG(n > 0 && f > 0 && ldy >= f && ldz >= f && ldo >= f && F > 0 && ldr >= f, "bad shape");
  GTB_CHECK_ARG(F == 1 || ldrb >= (n - 1) * ldr + f, "the blocks of R overlap each other");
  GTB_CHECK_ARG(Y != nullptr && Z != nullptr && out != nullptr && coef != nullptr && R != nullptr, "null operand");
  // the aliasing rules of gtb_spmm_cheb, and R apart from everything: every thread reads coef, Y rows are gathered
  // by many threads, and an R element sharing storage with Z or out would be read or written twice
  const uintptr_t o0 = reinterpret_cast<uintptr_t>(out), o1 = o0 + (uintptr_t)(((n - 1) * ldo + f) * sizeof(double));
  const uintptr_t y0 = reinterpret_cast<uintptr_t>(Y), y1 = y0 + (uintptr_t)(((n - 1) * ldy + f) * sizeof(double));
  const uintptr_t z0 = reinterpret_cast<uintptr_t>(Z), z1 = z0 + (uintptr_t)(((n - 1) * ldz + f) * sizeof(double));
  const uintptr_t r0 = reinterpret_cast<uintptr_t>(R),
                  r1 = r0 + (uintptr_t)(((F - 1) * ldrb + (n - 1) * ldr + f) * sizeof(double));
  const uintptr_t c0 = reinterpret_cast<uintptr_t>(coef), c1 = c0 + (uintptr_t)F * sizeof(double);
  GTB_CHECK_ARG(o1 <= y0 || y1 <= o0, "out must not overlap Y");
  GTB_CHECK_ARG((o0 == z0 && ldo == ldz) || o1 <= z0 || z1 <= o0, "out must be Z itself or not overlap it");
  GTB_CHECK_ARG((r1 <= y0 || y1 <= r0) && (r1 <= z0 || z1 <= r0) && (r1 <= o0 || o1 <= r0),
                "R must not overlap Y, Z or out");
  GTB_CHECK_ARG((c1 <= r0 || r1 <= c0) && (c1 <= o0 || o1 <= c0), "coef must not overlap R or out");
  cudaStream_t st = (cudaStream_t)stream;
  if (f > 64) {
    const unsigned grid = (unsigned)gtb_cdiv(n, SPMM_WARPS);
    for (int col0 = 0; col0 < f; col0 += 128) {
      if (f - col0 > 64)
        spmm_csr_kernel<2, 32, true, true><<<grid, SPMM_WARPS * 32, 0, st>>>(
            indptr, idx, val, n, Y, ldy, f, col0, out, ldo, alpha, beta, gamma, Z, ldz, coef, F, R, ldr, ldrb);
      else
        spmm_csr_kernel<1, 32, true, true><<<grid, SPMM_WARPS * 32, 0, st>>>(
            indptr, idx, val, n, Y, ldy, f, col0, out, ldo, alpha, beta, gamma, Z, ldz, coef, F, R, ldr, ldrb);
      GTB_CHECK_LAUNCH();
    }
    return GTB_OK;
  }
  const int lanes = (f + 1) / 2;
#define GTB_ACC_ARGS indptr, idx, val, n, Y, ldy, f, alpha, beta, gamma, Z, ldz, out, ldo, coef, F, R, ldr, ldrb, st
  if (lanes <= 1)       launch_cheb_acc<1>(GTB_ACC_ARGS);
  else if (lanes <= 2)  launch_cheb_acc<2>(GTB_ACC_ARGS);
  else if (lanes <= 4)  launch_cheb_acc<4>(GTB_ACC_ARGS);
  else if (lanes <= 8)  launch_cheb_acc<8>(GTB_ACC_ARGS);
  else if (lanes <= 16) launch_cheb_acc<16>(GTB_ACC_ARGS);
  else                  launch_cheb_acc<32>(GTB_ACC_ARGS);
#undef GTB_ACC_ARGS
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_row_scale(const double* in, const double* s, int64_t n, int f, int power_neg_half, double* out,
                             void* stream) {
  GTB_CHECK_ARG(n > 0 && f > 0, "bad shape");
  row_scale_kernel<<<(unsigned)gtb_cdiv(n * f, 256), 256, 0, (cudaStream_t)stream>>>(in, s, n, f, power_neg_half, out);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}
