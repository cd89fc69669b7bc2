// Locality order and reference tile lists for the pruned one-product top-k sweep (search_tc.cu, listed mode).
//
// 1. gtb_order_assign / gtb_order_sort: every row goes to the nearest of P pivots (every floor(n/P)-th row; float32,
//    pivots in shared memory), and a stable counting sort by pivot gives the permutation `perm` (position -> row).
//    Any permutation is correct; only how well 128-row tiles of the permuted rows cover one region depends on it.
// 2. gtb_tile_geometry: per group of `rows` consecutive permuted rows (a reference tile, or the query rows of one
//    sweep unit) the float64 centroid c and the radius r = max |x - c| (rounded up) of the rows the exact stage reads.
// 3. gtb_tile_lists_count / gtb_tile_lists_fill: reference tile R stays in the list of unit U unless the lower bound
//    LB = (|c_U - c_R| - r_U - r_R)^2 of every distance between their rows reaches the unit's bound T_U; the lists are
//    CSR (count -> exclusive scan -> fill), ascending tile id.
// 4. gtb_unpermute_candidates: candidate lists and thresholds of the permuted sweep back to original row ids.
#include "common.cuh"
#include "gtb200.h"

namespace {

constexpr int ORD_DMAX = 128;           // features the pruned path handles (the one-product sweep takes d <= 126)
constexpr int ORD_ASSIGN_THREADS = 128;
constexpr int ORD_CHUNK = 1024;         // rows per block of the counting sort
constexpr int LIST_UNITS = 8;           // units per block of the list count

// cell[r] = argmin_p |x_r - x_{p * pstride}|^2 (as |p|^2 - 2 x.p; the first pivot wins ties)
__global__ void __launch_bounds__(ORD_ASSIGN_THREADS) order_assign_kernel(const float* __restrict__ X, int64_t n, int d,
                                                                          int P, int64_t pstride,
                                                                          int32_t* __restrict__ cell) {
  extern __shared__ float4 piv4[];
  const int d4 = (d + 3) / 4;                                // float4 per pivot
  float* piv = reinterpret_cast<float*>(piv4);
  float* pn = piv + (size_t)P * d4 * 4;
  for (int i = threadIdx.x; i < P * d4 * 4; i += blockDim.x) {
    const int pv = i / (d4 * 4), k = i - pv * d4 * 4;
    piv[i] = k < d ? X[(int64_t)pv * pstride * d + k] : 0.f;
  }
  __syncthreads();
  for (int pv = threadIdx.x; pv < P; pv += blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < d4 * 4; ++k) s = fmaf(piv[pv * d4 * 4 + k], piv[pv * d4 * 4 + k], s);
    pn[pv] = s;
  }
  __syncthreads();
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  float x[ORD_DMAX];
#pragma unroll
  for (int k = 0; k < ORD_DMAX; ++k) x[k] = k < d ? X[r * d + k] : 0.f;
  float best = gtb_inf_f();
  int bi = 0;
  for (int pv = 0; pv < P; ++pv) {
    const float4* pp = piv4 + pv * d4;
    float a0 = 0.f, a1 = 0.f;
#pragma unroll
    for (int k4 = 0; k4 < ORD_DMAX / 4; ++k4) {
      if (k4 < d4) {
        const float4 q = pp[k4];
        a0 = fmaf(x[4 * k4], q.x, a0);
        a1 = fmaf(x[4 * k4 + 1], q.y, a1);
        a0 = fmaf(x[4 * k4 + 2], q.z, a0);
        a1 = fmaf(x[4 * k4 + 3], q.w, a1);
      }
    }
    const float s = pn[pv] - 2.f * (a0 + a1);
    if (s < best) { best = s; bi = pv; }
  }
  cell[r] = bi;
}

// counts[c][p] = rows of chunk c in cell p
__global__ void order_count_kernel(const int32_t* __restrict__ cell, int64_t n, int P, int32_t* __restrict__ counts) {
  extern __shared__ int32_t hist[];
  for (int p = threadIdx.x; p < P; p += blockDim.x) hist[p] = 0;
  __syncthreads();
  const int64_t r0 = (int64_t)blockIdx.x * ORD_CHUNK;
  for (int64_t r = r0 + threadIdx.x; r < n && r < r0 + ORD_CHUNK; r += blockDim.x) atomicAdd(&hist[cell[r]], 1);
  __syncthreads();
  for (int p = threadIdx.x; p < P; p += blockDim.x) counts[(int64_t)blockIdx.x * P + p] = hist[p];
}

// one warp per cell: counts[c][p] -> rows of cell p in chunks before c; total[p] = rows of cell p
__global__ void order_cellscan_kernel(int32_t* __restrict__ counts, int64_t nchunks, int P, int32_t* __restrict__ total) {
  const int lane = threadIdx.x & 31;
  const int p = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (p >= P) return;
  int run = 0;
  for (int64_t c0 = 0; c0 < nchunks; c0 += 32) {
    const int64_t c = c0 + lane;
    const int v = c < nchunks ? counts[c * P + p] : 0;
    int inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, inc, off);
      if (lane >= off) inc += o;
    }
    if (c < nchunks) counts[c * P + p] = run + inc - v;
    run += __shfl_sync(0xffffffffu, inc, 31);
  }
  if (lane == 0) total[p] = run;
}

// one warp per chunk, rows in order: equal cells within 32 rows are ranked by lane (match_any), so the sort is stable
__global__ void __launch_bounds__(32) order_fill_kernel(const int32_t* __restrict__ cell, int64_t n, int P,
                                                        const int32_t* __restrict__ counts,
                                                        const int32_t* __restrict__ total, int32_t* __restrict__ perm) {
  extern __shared__ int64_t off[];
  const int lane = threadIdx.x;
  int64_t run = 0;                                           // exclusive scan of the cell totals
  for (int p0 = 0; p0 < P; p0 += 32) {
    const int p = p0 + lane;
    const int64_t v = p < P ? total[p] : 0;
    int64_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t u = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += u;
    }
    if (p < P) off[p] = run + inc - v + counts[(int64_t)blockIdx.x * P + p];
    run += __shfl_sync(0xffffffffu, inc, 31);
  }
  __syncwarp();
  const int64_t r0 = (int64_t)blockIdx.x * ORD_CHUNK;
  for (int64_t rb = r0; rb < n && rb < r0 + ORD_CHUNK; rb += 32) {
    const int64_t r = rb + lane;
    const bool ok = r < n;
    const int c = ok ? cell[r] : -1 - lane;                  // rows past n: a cell of their own
    const unsigned peers = __match_any_sync(0xffffffffu, c);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    if (ok) perm[off[c] + rank] = (int32_t)r;
    __syncwarp();
    if (ok && rank == 0) off[c] += __popc(peers);
    __syncwarp();
  }
}

// one warp per group g of rows [g * rows, min(n, (g + 1) * rows)) of the permuted order; lane owns columns lane + 32 j
template <typename T>
__global__ void tile_geometry_kernel(const T* __restrict__ X, int64_t n, int d, const int32_t* __restrict__ perm,
                                     int64_t rows, int64_t ngroups, double* __restrict__ cent, double* __restrict__ rad) {
  constexpr int J = ORD_DMAX / 32;
  const int lane = threadIdx.x & 31;
  const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (g >= ngroups) return;
  const int64_t r0 = g * rows, r1 = (r0 + rows < n) ? r0 + rows : n;
  double c[J];
#pragma unroll
  for (int j = 0; j < J; ++j) c[j] = 0.0;
#pragma unroll 8
  for (int64_t r = r0; r < r1; ++r) {
    const T* xr = X + (int64_t)perm[r] * d;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int k = lane + 32 * j;
      if (k < d) c[j] += (double)xr[k];
    }
  }
  const double inv = r1 > r0 ? 1.0 / (double)(r1 - r0) : 0.0;
#pragma unroll
  for (int j = 0; j < J; ++j) c[j] *= inv;
  double m = 0.0;
#pragma unroll 8
  for (int64_t r = r0; r < r1; ++r) {
    const T* xr = X + (int64_t)perm[r] * d;
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int k = lane + 32 * j;
      if (k < d) {
        const double v = (double)xr[k] - c[j];
        s = fma(v, v, s);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    m = fmax(m, s);
  }
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int k = lane + 32 * j;
    if (k < d) cent[(int64_t)k * ngroups + g] = c[j];
  }
  if (lane == 0) rad[g] = r1 > r0 ? __dsqrt_ru(m) : -1.0;     // -1: a group without rows
}

// keep[u][t] = 1 unless tile t provably holds no row under unit u's bound; count[u] += kept tiles.
// Outward rounding: the radii are enlarged and the centre distance shrunk by 1e-12 relative, the squared gap by 1e-12
// -- far beyond the float64 rounding of these sums of <= 128 terms.
__global__ void tile_lists_count_kernel(const double* __restrict__ uc, const double* __restrict__ ur,
                                        const double* __restrict__ ub, int64_t nu, const double* __restrict__ rc,
                                        const double* __restrict__ rr, int64_t nt, int d, uint8_t* __restrict__ keep,
                                        int32_t* __restrict__ count) {
  __shared__ double cu[LIST_UNITS][ORD_DMAX];
  const int64_t u0 = (int64_t)blockIdx.y * LIST_UNITS;
  for (int i = threadIdx.x; i < LIST_UNITS * d; i += blockDim.x) {
    const int u = i / d, k = i - u * d;
    cu[u][k] = (u0 + u < nu) ? uc[(int64_t)k * nu + u0 + u] : 0.0;
  }
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double s[LIST_UNITS];
#pragma unroll
  for (int u = 0; u < LIST_UNITS; ++u) s[u] = 0.0;
  if (t < nt) {
    for (int k = 0; k < d; ++k) {
      const double y = rc[(int64_t)k * nt + t];
#pragma unroll
      for (int u = 0; u < LIST_UNITS; ++u) {
        const double v = cu[u][k] - y;
        s[u] = fma(v, v, s[u]);
      }
    }
  }
  const double rt = t < nt ? rr[t] * (1.0 + 1e-12) : 0.0;
#pragma unroll
  for (int u = 0; u < LIST_UNITS; ++u) {
    const int64_t uu = u0 + u;
    bool k = false;
    if (t < nt && uu < nu && ur[uu] >= 0.0) {
      const double gap = sqrt(s[u]) * (1.0 - 1e-12) - ur[uu] * (1.0 + 1e-12) - rt;
      k = !(gap > 0.0 && gap * gap * (1.0 - 1e-12) >= ub[uu]);
    }
    if (t < nt && uu < nu) keep[uu * nt + t] = k ? 1 : 0;
    const unsigned b = __ballot_sync(0xffffffffu, k);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(&count[uu], __popc(b));
  }
}

// one block per unit: the kept tiles in ascending order at tiles[ptr[u] ..)
__global__ void __launch_bounds__(256) tile_lists_fill_kernel(const uint8_t* __restrict__ keep, int64_t nt,
                                                              const int64_t* __restrict__ ptr,
                                                              int32_t* __restrict__ tiles) {
  __shared__ int wsum[8];
  const int64_t u = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t run = ptr[u];
  for (int64_t t0 = 0; t0 < nt; t0 += 256) {
    const int64_t t = t0 + threadIdx.x;
    const bool k = t < nt && keep[u * nt + t];
    const unsigned b = __ballot_sync(0xffffffffu, k);
    if (lane == 0) wsum[warp] = __popc(b);
    __syncthreads();
    int before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      before += (w < warp) ? wsum[w] : 0;
      all += wsum[w];
    }
    if (k) tiles[run + before + __popc(b & ((1u << lane) - 1u))] = (int32_t)t;
    run += all;
    __syncthreads();
  }
}

// row perm_q[i] of the output = row i of the permuted sweep, its candidates mapped through perm_r
__global__ void unpermute_kernel(const int32_t* __restrict__ cand_p, const float* __restrict__ tau_p, int64_t nq, int S,
                                 int ntau, const int32_t* __restrict__ perm_q, const int32_t* __restrict__ perm_r,
                                 int32_t* __restrict__ cand, float* __restrict__ tau) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nq * S) return;
  const int64_t i = e / S;
  const int s = (int)(e - i * S);
  const int64_t o = perm_q[i];
  const int32_t c = cand_p[e];
  cand[o * S + s] = c >= 0 ? perm_r[c] : c;
  if (s < ntau) tau[o * ntau + s] = tau_p[i * ntau + s];
}

}  // namespace

extern "C" int gtb_order_assign(const float* X, int64_t n, int d, int P, int32_t* cell, void* stream) {
  GTB_CHECK_ARG(n > 0 && d > 0 && d <= ORD_DMAX, "bad shape (d <= 128)");
  GTB_CHECK_ARG(P >= 1 && P <= 512 && P <= n, "pivot count must be in [1, min(512, n)]");
  const size_t smem = ((size_t)P * ((d + 3) / 4) * 4 + P) * sizeof(float);
  GTB_CUDA(cudaFuncSetAttribute(order_assign_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  order_assign_kernel<<<(unsigned)gtb_cdiv(n, ORD_ASSIGN_THREADS), ORD_ASSIGN_THREADS, smem, (cudaStream_t)stream>>>(
      X, n, d, P, n / P, cell);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int64_t gtb_order_ws_elems(int64_t n, int P) { return gtb_cdiv(n, ORD_CHUNK) * P + P; }

extern "C" int gtb_order_sort(const int32_t* cell, int64_t n, int P, int32_t* ws, int32_t* perm, void* stream) {
  GTB_CHECK_ARG(n > 0 && P >= 1 && P <= 512, "bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t nchunks = gtb_cdiv(n, ORD_CHUNK);
  int32_t* counts = ws;
  int32_t* total = ws + nchunks * P;
  order_count_kernel<<<(unsigned)nchunks, 256, P * sizeof(int32_t), st>>>(cell, n, P, counts);
  GTB_CHECK_LAUNCH();
  order_cellscan_kernel<<<(unsigned)gtb_cdiv(P, 8), 256, 0, st>>>(counts, nchunks, P, total);
  GTB_CHECK_LAUNCH();
  order_fill_kernel<<<(unsigned)nchunks, 32, P * sizeof(int64_t), st>>>(cell, n, P, counts, total, perm);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_tile_geometry(const void* X, int64_t n, int d, int x64, const int32_t* perm, int64_t rows,
                                 int64_t ngroups, double* cent, double* rad, void* stream) {
  GTB_CHECK_ARG(n > 0 && d > 0 && d <= ORD_DMAX && rows > 0 && ngroups > 0, "bad shape (d <= 128)");
  const unsigned grid = (unsigned)gtb_cdiv(ngroups * 32, 256);
  if (x64)
    tile_geometry_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>((const double*)X, n, d, perm, rows, ngroups,
                                                                         cent, rad);
  else
    tile_geometry_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)X, n, d, perm, rows, ngroups,
                                                                        cent, rad);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_tile_lists_count(const double* uc, const double* ur, const double* ub, int64_t nu, const double* rc,
                                    const double* rr, int64_t nt, int d, uint8_t* keep, int32_t* count, void* stream) {
  GTB_CHECK_ARG(nu > 0 && nt > 0 && d > 0 && d <= ORD_DMAX, "bad shape (d <= 128)");
  GTB_CHECK_ARG(gtb_cdiv(nu, LIST_UNITS) < 65536, "too many units");
  cudaStream_t st = (cudaStream_t)stream;
  GTB_CUDA(cudaMemsetAsync(count, 0, nu * sizeof(int32_t), st));
  tile_lists_count_kernel<<<dim3((unsigned)gtb_cdiv(nt, 256), (unsigned)gtb_cdiv(nu, LIST_UNITS)), 256, 0, st>>>(
      uc, ur, ub, nu, rc, rr, nt, d, keep, count);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_tile_lists_fill(const uint8_t* keep, int64_t nu, int64_t nt, const int64_t* ptr, int32_t* tiles,
                                   void* stream) {
  GTB_CHECK_ARG(nu > 0 && nt > 0, "bad shape");
  tile_lists_fill_kernel<<<(unsigned)nu, 256, 0, (cudaStream_t)stream>>>(keep, nt, ptr, tiles);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_unpermute_candidates(const int32_t* cand_p, const float* tau_p, int64_t nq, int S, int ntau,
                                        const int32_t* perm_q, const int32_t* perm_r, int32_t* cand, float* tau,
                                        void* stream) {
  GTB_CHECK_ARG(nq > 0 && S > 0 && ntau >= 1 && ntau <= S, "bad shape");
  unpermute_kernel<<<(unsigned)gtb_cdiv(nq * S, 256), 256, 0, (cudaStream_t)stream>>>(cand_p, tau_p, nq, S, ntau,
                                                                                      perm_q, perm_r, cand, tau);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}
