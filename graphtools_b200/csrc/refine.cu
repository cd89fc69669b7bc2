// K3: float64 re-evaluation of the selected candidates, bandwidth, certification of the
// candidate set, alpha-decay affinities and per-row column-sorted staging for CSR emission.
//
// Replaces (reference graphtools/graphs.py): bandwidth / radius / update-set logic :886-911, the
// per-row Python loop of _build_csr_from_neighbors :450-559, and the "is the row finished?" test
// that drives the x6 escalation loop :917-976.  Instead of escalating the neighbour count, each
// row is *certified*: every reference point NOT among the S candidates has approximate squared
// distance >= tau (top-k epilogue invariant) and therefore exact squared distance >= tau - E,
// E = eps_rel * (|x~|^2 + max|y~|^2) bounding the error of the fast pass.  A row is complete when
// its kernel support radius r = bw * (-ln thresh)^(1/decay) (or its knn_max-th neighbour) lies
// inside that certified radius; otherwise it is sent to the radius pass with an inflated limit.
//
// All distances that reach the output are float64 direct differences sum((x-y)^2) of the
// ORIGINAL float32 rows (SURVEY.md H1).
#include "common.cuh"
#include "gtb200.h"
#include <float.h>

namespace {

struct RowParams {
  const void* Xq; const void* Xr; int d;   // original rows, float32 or float64 (template T of the kernels)
  int knn; int64_t kmax;       // kmax = INT64_MAX when knn_max is None
  double decay;                // < 0: binary kNN (decay=None)
  double thresh; double rfac;  // rfac = (-ln thresh)^(1/decay)
  const double* bw_fixed; int bw_mode;  // 0 adaptive (k-th neighbour), 1 scalar, 2 per-row
  double bw_scale; double bw_floor;     // bw_floor = eps (np.finfo(float).eps)
  int metric;                           // 0 euclidean, 1 cosine (1 - x.y / (|x||y|), sklearn cosine_distances),
                                        // 2 cityblock (sum |x - y|, sklearn manhattan_distances),
                                        // 3 sqeuclidean (sum (x - y)^2), 4 correlation (cosine of the row-centred rows)
};

// metrics whose exact stage evaluates the Euclidean sum s = sum (x - y)^2 on the fast gather paths below
__host__ __device__ __forceinline__ bool euclidean_sum(int metric) { return metric == 0 || metric == 3; }

// exact squared distance between query row xq and reference row xr, cooperatively by one warp
// (float32 rows made of whole, 16-byte aligned float4s are read as float4 -- the same element-to-lane assignment and
// summation order as the gather loop of refine_topk_kernel, so both refine stages return identical bits)
template <typename T>
__device__ __forceinline__ double warp_dist2(const T* __restrict__ xq, const T* __restrict__ xr, int d, int lane) {
  double s = 0.0;
  bool vec = false;
  if constexpr (sizeof(T) == 4) {
    vec = ((d & 3) == 0) && (((reinterpret_cast<uintptr_t>(xq) | reinterpret_cast<uintptr_t>(xr)) & 15) == 0);
  }
  if (vec) {
    if constexpr (sizeof(T) == 4) {
      const float4* q4 = reinterpret_cast<const float4*>(xq);
      const float4* r4 = reinterpret_cast<const float4*>(xr);
      for (int kv = lane; kv < (d >> 2); kv += 32) {
        const float4 q = q4[kv], r = r4[kv];
        double df = (double)q.x - (double)r.x; s = fma(df, df, s);
        df = (double)q.y - (double)r.y; s = fma(df, df, s);
        df = (double)q.z - (double)r.z; s = fma(df, df, s);
        df = (double)q.w - (double)r.w; s = fma(df, df, s);
      }
    }
  } else {
    for (int k = lane; k < d; k += 32) {
      double df = (double)xq[k] - (double)xr[k];
      s = fma(df, df, s);
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  return s;
}

// Cosine metric.  The fast pass runs on the row-normalised copies, where |x^ - y^|^2 = 2 (1 - cos) = 2 d_cos: same
// ordering, and the certification arithmetic below converts between the metric's own units (in which key[] holds the
// SQUARED exact distance, so sqrt(key) is the distance for both metrics) and search-space squared distances.
// Cityblock: the fast pass accumulates sum |x - y| itself, so the search-space value IS the distance.
// Correlation: cosine of the row-centred rows, searched like cosine on the centred, row-normalised copies.
// Sqeuclidean: the fast pass is the Euclidean one and key = s^2 for the Euclidean sum s (the distance), so
// sqrt(key) == s exactly (binary64, no overflow or underflow) is both the distance and its search-space value.
__device__ __forceinline__ double search2_of_key(double key, int metric) {
  return metric == 0 ? key : ((metric == 1 || metric == 4) ? 2.0 * sqrt(key) : sqrt(key));
}
__device__ __forceinline__ double search2_of_radius(double r, int metric) {
  return metric == 0 ? r * r : ((metric == 1 || metric == 4) ? 2.0 * r : r);
}
// inverse of search2_of_radius (rounded: callers widen the result)
__device__ __forceinline__ double radius_of_search2(double s2, int metric) {
  return metric == 0 ? sqrt(s2) : ((metric == 1 || metric == 4) ? 0.5 * s2 : s2);
}

// squared cosine distance between two rows of the ORIGINAL data, float64, one warp.  An all-zero row is at
// distance 1 from every row, itself included: sklearn's normalize leaves it at zero, so its dot products are 0.
template <typename T>
__device__ __forceinline__ double warp_cos2(const T* __restrict__ xq, const T* __restrict__ xr, int d, int lane) {
  double dot = 0.0, nx = 0.0, ny = 0.0;
  for (int k = lane; k < d; k += 32) {
    const double a = (double)xq[k], b = (double)xr[k];
    dot = fma(a, b, dot); nx = fma(a, a, nx); ny = fma(b, b, ny);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    dot += __shfl_xor_sync(0xffffffffu, dot, off);
    nx += __shfl_xor_sync(0xffffffffu, nx, off);
    ny += __shfl_xor_sync(0xffffffffu, ny, off);
  }
  if (nx == 0.0 || ny == 0.0) return 1.0;
  double dc = 1.0 - dot / (sqrt(nx) * sqrt(ny));
  dc = fmin(fmax(dc, 0.0), 2.0);          // np.clip(S, 0, 2) in sklearn cosine_distances
  return dc * dc;
}

// float64 mean of one row of the ORIGINAL data, one warp (scipy's correlation centres each row by its np.mean)
template <typename T>
__device__ __forceinline__ double warp_mean(const T* __restrict__ x, int d, int lane) {
  double s = 0.0;
  for (int k = lane; k < d; k += 32) s += (double)x[k];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  return s / d;
}

// squared correlation distance between query row xq (row mean mq) and reference row xr of the ORIGINAL data, float64,
// one warp: the mean of xr first, then the centred dot product and norms on a second pass over the row (now in L1).
// A constant row (centred row zero) is rejected by the host before any search; like an all-zero cosine row it would
// be at distance 1 from every row.  Not inlined: inlined, it raises refine_ball_kernel<float> from 48 to 58 registers
// for every metric, the Euclidean one included.
template <typename T>
__device__ __noinline__ double warp_corr2(const T* __restrict__ xq, double mq, const T* __restrict__ xr, int d,
                                             int lane) {
  const double mr = warp_mean<T>(xr, d, lane);
  double dot = 0.0, nx = 0.0, ny = 0.0;
  for (int k = lane; k < d; k += 32) {
    const double a = (double)xq[k] - mq, b = (double)xr[k] - mr;
    dot = fma(a, b, dot); nx = fma(a, a, nx); ny = fma(b, b, ny);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    dot += __shfl_xor_sync(0xffffffffu, dot, off);
    nx += __shfl_xor_sync(0xffffffffu, nx, off);
    ny += __shfl_xor_sync(0xffffffffu, ny, off);
  }
  if (nx == 0.0 || ny == 0.0) return 1.0;
  double dc = 1.0 - dot / (sqrt(nx) * sqrt(ny));
  dc = fmin(fmax(dc, 0.0), 2.0);
  return dc * dc;
}

// squared cityblock distance between two rows of the ORIGINAL data, float64, one warp
template <typename T>
__device__ __forceinline__ double warp_l1sq(const T* __restrict__ xq, const T* __restrict__ xr, int d, int lane) {
  double s = 0.0;
  for (int k = lane; k < d; k += 32) s += fabs((double)xq[k] - (double)xr[k]);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  return s * s;
}

// cosine, cityblock, correlation (mq: the query row's mean, read by correlation only)
template <typename T>
__device__ __forceinline__ double warp_metric2(const T* xq, double mq, const T* xr, int d, int lane, int metric) {
  if (metric == 4) return warp_corr2<T>(xq, mq, xr, d, lane);
  return metric == 1 ? warp_cos2<T>(xq, xr, d, lane) : warp_l1sq<T>(xq, xr, d, lane);
}

// The radius pass of a row the candidate list cannot finish.  Every reference point whose exact distance is <= the
// returned radius must reach the row's ball.  dk: the knn-th distance, or an upper bound on it; bw: the row's bandwidth
// (from dk when bw_mode == 0); bw_cert: bw is the row's true bandwidth -- otherwise bw is only an upper bound and the
// ball must also hold the true knn nearest (radius >= dk), from which refine_ball_kernel recomputes it; dkmax: an upper
// bound on the kmax-th distance (+inf: none), beyond which no neighbour is kept.
__device__ __forceinline__ double collect_radius(const RowParams& rp, double dk, double bw, bool bw_cert, double dkmax) {
  if (rp.decay < 0) return dk;
  const double r = bw * rp.rfac;
  return fmin(bw_cert ? r : fmax(r, dk), dkmax);
}
// Collect limit in search units, rounded up: search2 of the radius widened by 1e-6 (rounding of the radius itself), plus
// the sweep's rounding bound E at the row (cityblock: plus its relative error at the radius).
__device__ __forceinline__ float collect_limit(double r_search, int metric, double E, double eps_rel) {
  double l2 = search2_of_radius(r_search, metric) * (1.0 + 1e-6) + E;
  if (metric == 2) l2 += 2.0 * eps_rel * r_search;     // relative error at the radius, not at tau
  return __double2float_ru(l2);
}

__device__ __forceinline__ int next_pow2(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

// Shared tail of both refine kernels.  On entry key[0..npow2) holds exact squared distances sorted
// ascending by (d2, idx) with +inf padding, idx[] the reference indices, n_cand the valid count and
// bw the row's bandwidth (already final).  Keeps the leading entries with affinity >= thresh among
// the first min(n_cand, kmax), converts them to (column, weight) sorted by column in key[]/idx[].
// Returns n_keep (uniform across the group).  scratch = one int in shared memory.
template <int NT, typename SyncT>
__device__ int finalize_sorted_row(double* key, int32_t* idx, int n_cand, double bw, const RowParams& rp,
                                   int tid, int* scratch, SyncT sync) {
  int64_t m64 = rp.kmax < (int64_t)n_cand ? rp.kmax : (int64_t)n_cand;
  int m = (int)m64;
  if (rp.decay < 0) {
    // binary kNN: the knn nearest, weight 1 (graphs.py:872-877)
    int keep = rp.knn < m ? rp.knn : m;
    for (int t = tid; t < keep; t += NT) key[t] = 1.0;
    if (tid == 0) *scratch = keep;
  } else {
    if (tid == 0) *scratch = m;
    sync();
    // first position whose affinity drops below thresh
    for (int t = tid; t < m; t += NT) {
      double w = gtb_affinity(sqrt(key[t]), bw, rp.decay);
      if (w >= rp.thresh) key[t] = w;
      else atomicMin(scratch, t);
    }
  }
  sync();
  int n_keep = *scratch;
  sync();
  int np2 = next_pow2(n_keep < 2 ? 2 : n_keep);
  for (int t = n_keep + tid; t < np2; t += NT) { idx[t] = 0x7fffffff; key[t] = 0.0; }
  sync();
  GTB_BITONIC_SORT(idx, key, np2, tid, NT, sync, int32_t, double);
  return n_keep;
}

// Reduce eight per-lane partial sums acc[0..7] across the warp with a halving exchange: at offsets 16, 8, 4 every lane
// keeps half of its accumulators and hands the other half to its partner (4 + 2 + 1 exchanges), then two butterfly
// steps finish the single value left per lane -- 9 shuffles instead of 40.  Every partial sum is formed from the same
// pairs as in the plain butterfly of warp_dist2 (a + b == b + a), so the bits agree.  Lane l ends with the sum of
// candidate u = 4*bit4 + 2*bit3 + bit2 of l; lanes with l % 4 == 0 store key[] / idx[].  Uses acc, j, c0, S, lane,
// key, idx, n_cand of the enclosing scope.
#define GTB_REDUCE8_AND_STORE() do { \
        double h4[4], h2[2], h1; \
        { \
          const bool up = (lane & 16) != 0; \
    _Pragma("unroll") \
          for (int u = 0; u < 4; ++u) { \
            const double keep = up ? acc[u + 4] : acc[u]; \
            const double give = up ? acc[u] : acc[u + 4]; \
            h4[u] = keep + __shfl_xor_sync(0xffffffffu, give, 16); \
          } \
        } \
        { \
          const bool up = (lane & 8) != 0; \
    _Pragma("unroll") \
          for (int u = 0; u < 2; ++u) { \
            const double keep = up ? h4[u + 2] : h4[u]; \
            const double give = up ? h4[u] : h4[u + 2]; \
            h2[u] = keep + __shfl_xor_sync(0xffffffffu, give, 8); \
          } \
        } \
        { \
          const bool up = (lane & 4) != 0; \
          const double keep = up ? h2[1] : h2[0]; \
          const double give = up ? h2[0] : h2[1]; \
          h1 = keep + __shfl_xor_sync(0xffffffffu, give, 4); \
        } \
        h1 += __shfl_xor_sync(0xffffffffu, h1, 2); \
        h1 += __shfl_xor_sync(0xffffffffu, h1, 1); \
        const int myu = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1); \
        int myj = j[0]; \
    _Pragma("unroll") \
        for (int u = 1; u < 8; ++u) myj = (myu == u) ? j[u] : myj; \
    _Pragma("unroll") \
        for (int u = 0; u < 8; ++u) n_cand += (c0 + u < S && j[u] >= 0) ? 1 : 0; \
        if ((lane & 3) == 0 && c0 + myu < S) { \
          key[c0 + myu] = (myj >= 0) ? h1 : DBL_MAX * 2.0; \
          idx[c0 + myu] = (myj >= 0) ? myj : 0x7fffffff; \
        } \
  } while (0)

// ------------------------------------------------------------------ stage 1: warp per row
constexpr int R1_WARPS = 4;
constexpr int R1_CAP = 128;  // max candidates per row handled by the warp kernel

struct Refine1Params {
  RowParams rp;
  int64_t nq; int S; int cand_stride; int ntau;
  const int32_t* cand_idx; const float* tau; const float* qn2; float maxrn2; double eps_rel;
  int32_t* st_idx; double* st_val; int32_t* n_keep; double* bw_out; float* lim2_out;
  int32_t* status; int32_t* nzero;
  int staged;                  // 1: candidate rows are staged through shared memory with cp.async (Euclidean sum,
                               // float32, d % 4 == 0, d <= 128)
};

template <typename T>
__global__ void __launch_bounds__(R1_WARPS * 32, 6) refine_topk_kernel(Refine1Params p) {
  __shared__ double key_s[R1_WARPS][R1_CAP];
  __shared__ int32_t idx_s[R1_WARPS][R1_CAP];
  __shared__ int scratch_s[R1_WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * R1_WARPS + warp;
  if (row >= p.nq) return;  // whole warp exits together
  double* key = key_s[warp];
  int32_t* idx = idx_s[warp];
  const RowParams& rp = p.rp;
  const int S = p.S;
  const int np2 = next_pow2(S);
  auto sync = [] { __syncwarp(); };

  // 1. exact distances
  const T* xq = reinterpret_cast<const T*>(rp.Xq) + row * rp.d;
  const T* Xr = reinterpret_cast<const T*>(rp.Xr);
  int n_cand = 0;
  bool vec = false;
  const bool l2sum = euclidean_sum(rp.metric);
  if (!l2sum) {
    const double mq = (rp.metric == 4) ? warp_mean<T>(xq, rp.d, lane) : 0.0;
    for (int c0 = 0; c0 < S; ++c0) {
      const int j = p.cand_idx[row * p.cand_stride + c0];
      const double v = (j >= 0) ? warp_metric2<T>(xq, mq, Xr + (int64_t)j * rp.d, rp.d, lane, rp.metric) : DBL_MAX * 2.0;
      if (j >= 0) ++n_cand;
      if (lane == 0) { key[c0] = v; idx[c0] = (j >= 0) ? j : 0x7fffffff; }
    }
  } else
  if constexpr (sizeof(T) == 4) {
    vec = ((rp.d & 3) == 0) && (((reinterpret_cast<uintptr_t>(rp.Xq) | reinterpret_cast<uintptr_t>(rp.Xr)) & 15) == 0);
  }
  if (!l2sum) {
    // done above
  } else if (p.staged && sizeof(T) == 4) {
    if constexpr (sizeof(T) == 4) {
      // Candidate rows stream through a two-deep shared-memory ring of eight rows per warp with cp.async (L2 -> smem,
      // no registers held while in flight): sixteen 400-byte row gathers per warp are outstanding while the previous
      // eight are reduced -- the gathers are latency-bound (~2 us under load), so bytes in flight set the rate.
      // Lane l copies and later reads float4 l of every row, so no cross-lane visibility is needed.
      extern __shared__ __align__(16) float stage_all[];
      const int nv = rp.d >> 2;                                  // <= 32
      float* stage = stage_all + (size_t)warp * (2 * 8 * rp.d);
      const float4* Xr4 = reinterpret_cast<const float4*>(Xr);
      const int ngroups = (S + 7) >> 3;
      const bool on = lane < nv;
      auto issue = [&](int g) {
        float* dst = stage + (g & 1) * 8 * rp.d;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int c = g * 8 + u;
          const int jj = (c < S) ? p.cand_idx[row * p.cand_stride + c] : -1;
          if (on) {
            const float4* src = Xr4 + (int64_t)(jj >= 0 ? jj : 0) * nv + lane;
            const uint32_t d32 = (uint32_t)__cvta_generic_to_shared(dst + u * rp.d + lane * 4);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d32), "l"(src) : "memory");
          }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
      };
      issue(0);
      if (ngroups > 1) issue(1);
      float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
      if (on) q = reinterpret_cast<const float4*>(xq)[lane];
      for (int g = 0; g < ngroups; ++g) {
        if (g + 1 < ngroups) asm volatile("cp.async.wait_group 1;" ::: "memory");
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
        const int c0 = g * 8;
        const float* src = stage + (g & 1) * 8 * rp.d + lane * 4;
        int j[8];
        double acc[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          j[u] = (c0 + u < S) ? p.cand_idx[row * p.cand_stride + c0 + u] : -1;  // uniform loads
          acc[u] = 0.0;
          if (on) {
            const float4 r = *reinterpret_cast<const float4*>(src + u * rp.d);
            double df = (double)q.x - (double)r.x; acc[u] = fma(df, df, acc[u]);
            df = (double)q.y - (double)r.y; acc[u] = fma(df, df, acc[u]);
            df = (double)q.z - (double)r.z; acc[u] = fma(df, df, acc[u]);
            df = (double)q.w - (double)r.w; acc[u] = fma(df, df, acc[u]);
          }
        }
        if (g + 2 < ngroups) issue(g + 2);       // this lane has consumed its part of ring slot g & 1
        GTB_REDUCE8_AND_STORE();
      }
    }
  } else if (vec) {
    if constexpr (sizeof(T) == 4) {
      // float32 rows of whole float4s: one 16-byte load per lane covers a 400-byte row with 25 lanes, and eight
      // candidate rows are gathered per pass -- the gathers are latency-bound, so bytes in flight are what counts
      const int nv = rp.d >> 2;
      const float4* xq4 = reinterpret_cast<const float4*>(xq);
      const float4* Xr4 = reinterpret_cast<const float4*>(Xr);
      for (int c0 = 0; c0 < S; c0 += 8) {
        int j[8];
        double acc[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          acc[u] = 0.0;
          j[u] = (c0 + u < S) ? p.cand_idx[row * p.cand_stride + c0 + u] : -1;  // uniform loads
        }
        for (int kv = lane; kv < nv; kv += 32) {
          const float4 q = xq4[kv];
          float4 r[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            r[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j[u] >= 0) r[u] = Xr4[(int64_t)j[u] * nv + kv];
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            if (j[u] >= 0) {
              double df = (double)q.x - (double)r[u].x; acc[u] = fma(df, df, acc[u]);
              df = (double)q.y - (double)r[u].y; acc[u] = fma(df, df, acc[u]);
              df = (double)q.z - (double)r[u].z; acc[u] = fma(df, df, acc[u]);
              df = (double)q.w - (double)r[u].w; acc[u] = fma(df, df, acc[u]);
            }
          }
        }
        GTB_REDUCE8_AND_STORE();
      }
    }
  } else {
  // four candidates in flight per pass: the row gathers are latency-bound, not bandwidth-bound
  for (int c0 = 0; c0 < S; c0 += 4) {
    int j[4];
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int u = 0; u < 4; ++u) j[u] = (c0 + u < S) ? p.cand_idx[row * p.cand_stride + c0 + u] : -1;  // uniform loads
    for (int k = lane; k < rp.d; k += 32) {
      const double q = (double)xq[k];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (j[u] >= 0) {
          const double df = q - (double)Xr[(int64_t)j[u] * rp.d + k];
          acc[u] = fma(df, df, acc[u]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) acc[u] += __shfl_xor_sync(0xffffffffu, acc[u], off);
      if (c0 + u < S) {
        if (j[u] >= 0) ++n_cand;
        if (lane == 0) {
          key[c0 + u] = (j[u] >= 0) ? acc[u] : DBL_MAX * 2.0;  // +inf for empty slots
          idx[c0 + u] = (j[u] >= 0) ? j[u] : 0x7fffffff;
        }
      }
    }
  }
  }
  if (rp.metric == 3) {
    // sqeuclidean: key = s^2 of the Euclidean sum s (see search2_of_key); +inf padding stays +inf
    __syncwarp();
    for (int t = lane; t < S; t += 32) key[t] = key[t] * key[t];
  }
  // 2. sort by (d2, idx); 3. zero-distance count (duplicate detection, graphs.py:787-817)
  const bool small = S <= 32;            // one candidate per lane: both sorts of the row run in registers
  double mk = DBL_MAX * 2.0;
  int32_t mi = 0x7fffffff;
  int nz = 0;
  if (small) {
    __syncwarp();
    if (lane < S) { mk = key[lane]; mi = idx[lane]; }
    warp_sort32<double, int32_t>(mk, mi, lane);
    __syncwarp();
    key[lane] = mk; idx[lane] = mi;      // the certification below reads order statistics by position
    __syncwarp();
    nz = __popc(__ballot_sync(0xffffffffu, lane < n_cand && mk == 0.0));
  } else {
    for (int t = S + lane; t < np2; t += 32) { key[t] = DBL_MAX * 2.0; idx[t] = 0x7fffffff; }
    __syncwarp();
    GTB_BITONIC_SORT(key, idx, np2, lane, 32, sync, double, int32_t);
    for (int t = lane; t < n_cand; t += 32) nz += (key[t] == 0.0);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) nz += __shfl_xor_sync(0xffffffffu, nz, off);
  }

  // 4. bandwidth + certification
  float tau = p.tau[row * p.ntau];
  for (int t = 1; t < p.ntau; ++t) tau = fminf(tau, p.tau[row * p.ntau + t]);  // lists of disjoint reference subsets
  const bool all_found = isinf(tau);  // list never filled: every reference is a candidate
  // euclidean / cosine: absolute bound relative to the squared norms of the centred rows; cityblock: the float32
  // accumulation of |x - y| is accurate RELATIVE to the distance (eps_rel * tau), plus the rounding of float64
  // inputs to the float32 search copy (2^-23 of the rows' L1 norms; qn2 is NULL for float32 inputs)
  const double E = (rp.metric == 2)
                       ? p.eps_rel * fabs((double)tau) + (p.qn2 ? ((double)p.qn2[row] + (double)p.maxrn2) * 0x1p-23 : 0.0)
                       : p.eps_rel * ((double)p.qn2[row] + (double)p.maxrn2);
  const double rho2 = (double)tau - E;  // exact d2 of every non-candidate is >= rho2
  double bw = 0.0, dk = 0.0;
  bool done, bw_cert = true;
  if (rp.decay < 0) {
    double dk2 = key[rp.knn - 1];
    done = all_found || search2_of_key(dk2, rp.metric) < rho2;
    dk = sqrt(dk2);
  } else {
    if (rp.bw_mode == 0) {
      double dk2 = key[rp.knn - 1];
      dk = sqrt(dk2);
      bw = fmax(dk * rp.bw_scale, rp.bw_floor);
      bw_cert = all_found || search2_of_key(dk2, rp.metric) < rho2;
    } else {
      bw = fmax((rp.bw_mode == 1 ? rp.bw_fixed[0] : rp.bw_fixed[row]) * rp.bw_scale, rp.bw_floor);
    }
    double r = bw * rp.rfac;
    bool ball_cert = all_found || search2_of_radius(r, rp.metric) < rho2;
    bool kmax_cert = (rp.kmax <= (int64_t)n_cand) && search2_of_key(key[rp.kmax - 1], rp.metric) < rho2;
    done = bw_cert && (ball_cert || kmax_cert);
  }
  const double dkmax = (rp.decay >= 0 && rp.kmax <= (int64_t)n_cand) ? sqrt(key[rp.kmax - 1]) : DBL_MAX * 2.0;
  const double r_search = collect_radius(rp, dk, bw, bw_cert, dkmax);
  if (lane == 0) {
    p.bw_out[row] = bw;
    p.status[row] = done ? 1 : (bw_cert ? 0 : 2);
    p.nzero[row] = nz;
    if (!done) {
      p.lim2_out[row] = collect_limit(r_search, rp.metric, E, p.eps_rel);
      p.n_keep[row] = 0;
    } else {
      p.lim2_out[row] = 0.f;
    }
  }
  if (!done) return;
  __syncwarp();
  // 5. affinities, threshold, column sort, staging
  if (small) {
    // lane t holds the t-th nearest candidate: keep the leading entries with affinity >= thresh among the first
    // min(n_cand, kmax) (finalize_sorted_row's rule), then order the survivors by column in registers
    const int64_t m64 = rp.kmax < (int64_t)n_cand ? rp.kmax : (int64_t)n_cand;
    const int m = (int)m64;
    double w = 0.0;
    int n_keep;
    if (rp.decay < 0) {
      n_keep = rp.knn < m ? rp.knn : m;            // binary kNN: the knn nearest, weight 1 (graphs.py:872-877)
      w = 1.0;
    } else {
      const bool inm = lane < m;
      if (inm) w = gtb_affinity(sqrt(mk), bw, rp.decay);
      const unsigned fail = __ballot_sync(0xffffffffu, inm && !(w >= rp.thresh));
      n_keep = fail ? (__ffs(fail) - 1) : m;
    }
    int32_t ci = (lane < n_keep) ? mi : 0x7fffffff;
    warp_sort32<int32_t, double>(ci, w, lane);
    if (lane < n_keep) {
      p.st_idx[row * S + lane] = ci;
      p.st_val[row * S + lane] = w;
    }
    if (lane == 0) p.n_keep[row] = n_keep;
    return;
  }
  int n_keep = finalize_sorted_row<32>(key, idx, n_cand, bw, rp, lane, &scratch_s[warp], sync);
  for (int t = lane; t < n_keep; t += 32) {
    p.st_idx[row * S + t] = idx[t];
    p.st_val[row * S + t] = key[t];
  }
  if (lane == 0) p.n_keep[row] = n_keep;
}

// ------------------------------------------------------------------ stage 2: block per row
constexpr int R2_THREADS = 256;

struct Refine2Params {
  RowParams rp;
  const int32_t* todo_rows; const int32_t* status; int64_t nt;
  const int64_t* seg_ptr; int32_t* seg_idx; double* seg_val;
  int32_t* n_keep_t; double* bw_out; int32_t* nzero; int32_t* overflow; int cap;
};

template <typename T>
__global__ void __launch_bounds__(R2_THREADS) refine_ball_kernel(Refine2Params p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* key = reinterpret_cast<double*>(smem_raw);               // [cap]
  int32_t* idx = reinterpret_cast<int32_t*>(key + p.cap);          // [cap]
  __shared__ int scratch;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t t_row = blockIdx.x;
  const int64_t row = p.todo_rows[t_row];
  const int64_t p0 = p.seg_ptr[t_row], p1 = p.seg_ptr[t_row + 1];
  const int64_t L64 = p1 - p0;
  const RowParams& rp = p.rp;
  auto sync = [] { __syncthreads(); };
  if (L64 > p.cap) {
    if (tid == 0) { atomicMax(p.overflow, (int)(L64 > 0x7fffffff ? 0x7fffffff : L64)); p.n_keep_t[t_row] = 0; }
    return;
  }
  const int L = (int)L64;
  const int np2 = next_pow2(L < 2 ? 2 : L);
  const T* xq = reinterpret_cast<const T*>(rp.Xq) + row * rp.d;
  const T* Xr = reinterpret_cast<const T*>(rp.Xr);
  const double mq = (rp.metric == 4) ? warp_mean<T>(xq, rp.d, lane) : 0.0;
  for (int c = warp; c < L; c += R2_THREADS / 32) {
    int j = p.seg_idx[p0 + c];
    double d2 = euclidean_sum(rp.metric) ? warp_dist2<T>(xq, Xr + (int64_t)j * rp.d, rp.d, lane)
                                         : warp_metric2<T>(xq, mq, Xr + (int64_t)j * rp.d, rp.d, lane, rp.metric);
    if (rp.metric == 3) d2 *= d2;                                  // sqeuclidean: key = s^2, as in stage 1
    if (lane == 0) { key[c] = d2; idx[c] = j; }
  }
  for (int t = L + tid; t < np2; t += R2_THREADS) { key[t] = DBL_MAX * 2.0; idx[t] = 0x7fffffff; }
  __syncthreads();
  GTB_BITONIC_SORT(key, idx, np2, tid, R2_THREADS, sync, double, int32_t);

  if (warp == 0) {
    int nz = 0;
    for (int t = lane; t < L; t += 32) nz += (key[t] == 0.0);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) nz += __shfl_xor_sync(0xffffffffu, nz, off);
    if (lane == 0) p.nzero[row] = nz;
  }
  double bw = 0.0;
  if (rp.decay >= 0) {
    if (rp.bw_mode == 0) {
      if (p.status[row] == 2) {
        // the search ball (radius >= k-th candidate distance) holds the true k nearest
        int kk = rp.knn - 1 < L ? rp.knn - 1 : L - 1;
        bw = fmax(sqrt(key[kk < 0 ? 0 : kk]) * rp.bw_scale, rp.bw_floor);
      } else {
        bw = p.bw_out[row];  // certified in stage 1
      }
    } else {
      bw = fmax((rp.bw_mode == 1 ? rp.bw_fixed[0] : rp.bw_fixed[row]) * rp.bw_scale, rp.bw_floor);
    }
  }
  __syncthreads();
  int n_keep = finalize_sorted_row<R2_THREADS>(key, idx, L, bw, rp, tid, &scratch, sync);
  for (int t = tid; t < n_keep; t += R2_THREADS) {
    p.seg_idx[p0 + t] = idx[t];
    p.seg_val[p0 + t] = key[t];
  }
  if (tid == 0) { p.n_keep_t[t_row] = n_keep; p.bw_out[row] = bw; }
}

// segment scatter: pairs (slot, col) -> seg_idx[seg_ptr[slot] + cursor[slot]++]
__global__ void scatter_pairs_kernel(const int2* __restrict__ pairs, int64_t npairs,
                                     const int64_t* __restrict__ seg_ptr, int32_t* __restrict__ cursor,
                                     int32_t* __restrict__ seg_idx) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npairs) return;
  int2 pr = pairs[i];
  int pos = atomicAdd(cursor + pr.x, 1);
  seg_idx[seg_ptr[pr.x] + pos] = pr.y;
}

__global__ void scatter_counts_kernel(const int32_t* __restrict__ todo_rows, const int32_t* __restrict__ n_keep_t,
                                      int64_t nt, int32_t* __restrict__ n_keep) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nt) n_keep[todo_rows[t]] = n_keep_t[t];
}

// CSR gather from the stage-1 staging area [nq][S]
__global__ void csr_gather1_kernel(const int32_t* __restrict__ st_idx, const double* __restrict__ st_val,
                                   const int32_t* __restrict__ n_keep, const int32_t* __restrict__ status,
                                   const int64_t* __restrict__ indptr, int64_t nq, int S,
                                   int32_t* __restrict__ out_idx, double* __restrict__ out_val) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq * S) return;
  int64_t row = i / S;
  int t = (int)(i - row * S);
  if (status[row] == 1 && t < n_keep[row]) {
    int64_t o = indptr[row] + t;
    out_idx[o] = st_idx[i];
    out_val[o] = st_val[i];
  }
}

__global__ void csr_gather2_kernel(const int32_t* __restrict__ todo_rows, const int64_t* __restrict__ seg_ptr,
                                   const int32_t* __restrict__ seg_idx, const double* __restrict__ seg_val,
                                   const int32_t* __restrict__ n_keep_t, const int64_t* __restrict__ indptr,
                                   int32_t* __restrict__ out_idx, double* __restrict__ out_val) {
  int64_t t_row = blockIdx.x;
  int64_t row = todo_rows[t_row];
  int64_t src = seg_ptr[t_row], dst = indptr[row];
  int n = n_keep_t[t_row];
  for (int t = threadIdx.x; t < n; t += blockDim.x) {
    out_idx[dst + t] = seg_idx[src + t];
    out_val[dst + t] = seg_val[src + t];
  }
}

// stream compaction of rows with status == 0 (order is irrelevant to the result)
__global__ void compact_todo_kernel(const int32_t* __restrict__ status, int64_t nq, int32_t* __restrict__ todo_rows,
                                    int32_t* __restrict__ count) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool todo = (i < nq) && status[i] != 1;
  unsigned m = __ballot_sync(0xffffffffu, todo);
  if (!m) return;
  int lane = threadIdx.x & 31;
  int base = 0;
  if (lane == 0) base = atomicAdd(count, __popc(m));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (todo) todo_rows[base + __popc(m & ((1u << lane) - 1))] = (int32_t)i;
}

// ------------------------------------------------------------------ bound selection from the count sweeps
// Histograms of the approximate squared distances w (search units, the float32 values the sweep computes) from
// gtb_knn_count_tc / gtb_knn_count_simt.  Coarse bin b < 63 holds w < 2^(elo + b - 126) (bin b > 0: w >= 2^(elo + b -
// 127)), bin 63 everything above; the fine histogram splits the octave [t/2, t) below the coarse crossing edge t into
// 16 sub-bins, bin 0 = everything under t/2.  Every edge is a power of two or a power of two times (1 + j/16): exact in
// float32 and float64, so "count at edge" means exactly c(e) = #{w < e}.
//
// Why the bound holds: if c(e) >= k, then k reference points have w < e, hence exact squared distance < e + E (E the
// sweep's rounding bound at the row, plus the float32 rounding of w = (|y|^2 - 2 x.y) + |x|^2), so the exact k-th
// smallest squared distance is <= U = e + E.  A count that misses a point only moves the crossing up and U with it.
// U bounds the knn-th distance from above exactly as the k-th candidate of an uncertified list does (status 2), so
// collect_radius / collect_limit give the row's collect limit by the refine's own rule.
struct BoundParams {
  RowParams rp;
  const uint32_t* coarse; const uint32_t* fine; int64_t nq; int elo, margin; float s2;
  const float* qn2; float maxrn2; double eps_rel; int64_t nr;
  float* top; float* lim2; int32_t* ball_lo; int32_t* ball_hi;
};

__device__ __forceinline__ float coarse_edge(int elo, int b) {     // upper edge of coarse bin b (+inf for bin 63)
  return b >= 63 ? gtb_inf_f() : __uint_as_float((uint32_t)(elo + b + 1) << 23);
}

// first bin whose cumulative count reaches k (nb when none), cumulative counts before it and at it
__device__ __forceinline__ int crossing(const uint32_t* h, int nb, int64_t k, int64_t* before) {
  int64_t c = 0;
  for (int b = 0; b < nb; ++b) {
    if (c + h[b] >= k) { *before = c; return b; }
    c += h[b];
  }
  *before = c;
  return nb;
}

__global__ void count_bound_kernel(BoundParams p) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.nq) return;
  const RowParams& rp = p.rp;
  const int metric = rp.metric;
  const double nrm = p.qn2 ? (double)p.qn2[i] + (double)p.maxrn2 : 0.0;
  if (p.coarse == nullptr) {
    // fixed bandwidth: the kernel support alone (status 0 of the refine), no count needed
    const double bw = fmax((rp.bw_mode == 1 ? rp.bw_fixed[0] : rp.bw_fixed[i]) * rp.bw_scale, rp.bw_floor);
    const double r = collect_radius(rp, 0.0, bw, true, DBL_MAX * 2.0);
    const double E = metric == 2 ? nrm * 0x1p-23 : p.eps_rel * nrm;
    p.lim2[i] = collect_limit(r, metric, E, p.eps_rel);
    return;
  }
  const uint32_t* hc = p.coarse + i * 64;
  int64_t before = 0;
  const int bc = crossing(hc, 64, rp.knn, &before);
  const float t = bc < 64 ? coarse_edge(p.elo, bc) : gtb_inf_f();
  if (p.fine == nullptr) { p.top[i] = t; return; }
  if (!(t < gtb_inf_f())) {
    // fewer than k points under the window's top (fewer than k reference rows): every point is in the ball
    p.lim2[i] = gtb_inf_f();
    p.ball_lo[i] = (int32_t)p.nr; p.ball_hi[i] = (int32_t)p.nr;
    return;
  }
  // fine crossing of k (and of kmax <= k): upper edge of the first sub-bin reaching it; t itself when the fine counts
  // fall short (the coarse count at t already reaches k)
  const uint32_t* hf = p.fine + i * 17;
  auto fine_edge = [&](int64_t k) -> double {
    int64_t c0 = 0;
    const int b = crossing(hf, 17, k, &c0);
    return b == 0 ? 0.5 * (double)t : (b < 17 ? 0.5 * (double)t * (1.0 + b / 16.0) : (double)t);
  };
  // search units -> data units (s2 is a power of two), plus the rounding bound
  auto upper = [&](double e) {
    e /= p.s2;
    return metric == 2 ? e * (1.0 + p.eps_rel) + nrm * 0x1p-23 : e + (p.eps_rel + 0x1p-20) * nrm;
  };
  const double ek = fine_edge(rp.knn);
  const double dk = radius_of_search2(upper(ek), metric);
  const double bw = rp.decay >= 0 ? fmax(dk * rp.bw_scale, rp.bw_floor) : 0.0;
  const double dkmax = (rp.decay >= 0 && rp.kmax <= (int64_t)rp.knn)
                           ? radius_of_search2(upper(fine_edge(rp.kmax)), metric) : DBL_MAX * 2.0;
  const double r = collect_radius(rp, dk, bw, false, dkmax);
  const double E = metric == 2 ? p.eps_rel * ek / p.s2 + nrm * 0x1p-23 : p.eps_rel * nrm;
  const float l2 = collect_limit(r, metric, E, p.eps_rel);
  p.lim2[i] = l2;
  // ball size: every point with w under the lower edge of the limit's bin is in the ball, every point of the ball has w
  // under its upper edge.  Coarse counts are complete below the crossing + margin octaves (the sweep's top edge never
  // fell below it); above, only the lower bound is known (ball_hi = -1).
  const float ls = l2 * p.s2;
  int64_t lo, hi = -1;
  if (ls < 0.5f * t) {
    lo = 0;
    hi = hf[0];
  } else if (ls < t) {
    const int j = (int)((__float_as_uint(ls) >> 19) & 15u);          // sub-bin of the limit
    lo = hf[0];
    for (int b = 0; b < j; ++b) lo += hf[1 + b];
    hi = lo + hf[1 + j];
  } else {
    const int e = (int)(__float_as_uint(ls) >> 23);
    const int bl = min(max(e - p.elo, 0), 63);
    const int bmax = bc + p.margin - 1;                  // last coarse bin counted in full
    int64_t c = 0;
    lo = 0;
    for (int b = 0; b <= min(bl, bmax); ++b) {
      if (b < bl) lo = c + hc[b];
      c += hc[b];
    }
    if (bl <= bmax && bl < 63) hi = c;
  }
  p.ball_lo[i] = (int32_t)(lo < p.nr ? lo : p.nr);
  p.ball_hi[i] = hi < 0 ? -1 : (int32_t)(hi < p.nr ? hi : p.nr);
}

RowParams make_row_params(const void* Xq, const void* Xr, int d, int knn, int64_t kmax, double decay,
                          double thresh, const double* bw_fixed, int bw_mode, double bw_scale, int metric) {
  RowParams rp;
  rp.metric = metric;
  rp.Xq = Xq; rp.Xr = Xr; rp.d = d; rp.knn = knn; rp.kmax = kmax <= 0 ? INT64_MAX : kmax;
  rp.decay = decay; rp.thresh = thresh;
  rp.rfac = decay >= 0 ? pow(-log(thresh), 1.0 / decay) : 0.0;
  rp.bw_fixed = bw_fixed; rp.bw_mode = bw_mode; rp.bw_scale = bw_scale; rp.bw_floor = DBL_EPSILON;
  return rp;
}

}  // namespace

extern "C" int gtb_refine_topk(const void* Xq, int64_t nq, const void* Xr, int d, int x_kind,
                               const int32_t* cand_idx,
                               int S, int cand_stride, const float* tau, int ntau, const float* qn2, float maxrn2, double eps_rel,
                               int knn, int64_t kmax, double decay, double thresh, const double* bw_fixed,
                               int bw_mode, double bw_scale, int32_t* st_idx, double* st_val, int32_t* n_keep,
                               double* bw_out, float* lim2_out, int32_t* status, int32_t* nzero, void* stream) {
  GTB_CHECK_ARG(nq > 0 && S > 0 && S <= R1_CAP, "S out of range");
  GTB_CHECK_ARG(knn >= 1 && knn <= S, "knn must be in [1, S]");
  GTB_CHECK_ARG(decay < 0 || (thresh > 0 && thresh <= 1), "thresh must be in (0, 1]");
  GTB_CHECK_ARG(x_kind >= 0 && x_kind <= 9, "x_kind: bit 0 = float64 rows, bits 1-3 = metric (0 euclidean, 1 cosine, 2 cityblock, 3 sqeuclidean, 4 correlation)");
  const int x_is_f64 = x_kind & 1;
  Refine1Params p;
  p.rp = make_row_params(Xq, Xr, d, knn, kmax, decay, thresh, bw_fixed, bw_mode, bw_scale, x_kind >> 1);
  GTB_CHECK_ARG(cand_stride >= S, "cand_stride must be >= S");
  p.nq = nq; p.S = S; p.cand_stride = cand_stride; p.ntau = ntau < 1 ? 1 : ntau; p.cand_idx = cand_idx; p.tau = tau; p.qn2 = qn2; p.maxrn2 = maxrn2; p.eps_rel = eps_rel;
  p.st_idx = st_idx; p.st_val = st_val; p.n_keep = n_keep; p.bw_out = bw_out; p.lim2_out = lim2_out;
  p.status = status; p.nzero = nzero;
  // float32 rows of whole, 16-byte aligned float4s no longer than one warp-wide load: stage the gathers through smem
  p.staged = (!x_is_f64 && euclidean_sum(x_kind >> 1) && (d & 3) == 0 && d <= 128 &&
              (((uintptr_t)Xq | (uintptr_t)Xr) & 15) == 0) ? 1 : 0;
  const size_t smem = p.staged ? (size_t)R1_WARPS * 2 * 8 * d * sizeof(float) : 0;
  if (x_is_f64)
    refine_topk_kernel<double><<<(unsigned)gtb_cdiv(nq, R1_WARPS), R1_WARPS * 32, 0, (cudaStream_t)stream>>>(p);
  else
    refine_topk_kernel<float><<<(unsigned)gtb_cdiv(nq, R1_WARPS), R1_WARPS * 32, smem, (cudaStream_t)stream>>>(p);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_compact_todo(const int32_t* status, int64_t nq, int32_t* todo_rows, int32_t* count, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  GTB_CUDA(cudaMemsetAsync(count, 0, sizeof(int32_t), st));
  compact_todo_kernel<<<(unsigned)gtb_cdiv(nq, 256), 256, 0, st>>>(status, nq, todo_rows, count);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_scatter_pairs(const int32_t* pairs, int64_t npairs, const int64_t* seg_ptr, int32_t* cursor,
                                 int64_t nt, int32_t* seg_idx, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  GTB_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int32_t) * nt, st));
  if (npairs > 0) {
    scatter_pairs_kernel<<<(unsigned)gtb_cdiv(npairs, 256), 256, 0, st>>>(
        reinterpret_cast<const int2*>(pairs), npairs, seg_ptr, cursor, seg_idx);
    GTB_CHECK_LAUNCH();
  }
  return GTB_OK;
}

extern "C" int gtb_refine_ball(const void* Xq, const int32_t* todo_rows, const int32_t* status, int64_t nt,
                               const void* Xr, int d, int x_kind,
                               const int64_t* seg_ptr, int32_t* seg_idx, double* seg_val, int knn, int64_t kmax,
                               double decay, double thresh, const double* bw_fixed, int bw_mode, double bw_scale,
                               int32_t* n_keep_t, int32_t* n_keep, double* bw_out, int32_t* nzero,
                               int32_t* overflow, int cap, void* stream) {
  GTB_CHECK_ARG(nt > 0, "no rows");
  GTB_CHECK_ARG(cap >= 2 && (cap & (cap - 1)) == 0 && cap <= 8192, "cap must be a power of two <= 8192");
  cudaStream_t st = (cudaStream_t)stream;
  GTB_CHECK_ARG(x_kind >= 0 && x_kind <= 9, "x_kind: bit 0 = float64 rows, bits 1-3 = metric (0 euclidean, 1 cosine, 2 cityblock, 3 sqeuclidean, 4 correlation)");
  const int x_is_f64 = x_kind & 1;
  Refine2Params p;
  p.rp = make_row_params(Xq, Xr, d, knn, kmax, decay, thresh, bw_fixed, bw_mode, bw_scale, x_kind >> 1);
  p.todo_rows = todo_rows; p.status = status; p.nt = nt; p.seg_ptr = seg_ptr; p.seg_idx = seg_idx; p.seg_val = seg_val;
  p.n_keep_t = n_keep_t; p.bw_out = bw_out; p.nzero = nzero; p.overflow = overflow; p.cap = cap;
  size_t smem = (size_t)cap * 12;
  GTB_CUDA(cudaMemsetAsync(overflow, 0, sizeof(int32_t), st));
  if (x_is_f64) {
    GTB_CUDA(cudaFuncSetAttribute(refine_ball_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    refine_ball_kernel<double><<<(unsigned)nt, R2_THREADS, smem, st>>>(p);
  } else {
    GTB_CUDA(cudaFuncSetAttribute(refine_ball_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    refine_ball_kernel<float><<<(unsigned)nt, R2_THREADS, smem, st>>>(p);
  }
  GTB_CHECK_LAUNCH();
  scatter_counts_kernel<<<(unsigned)gtb_cdiv(nt, 256), 256, 0, st>>>(todo_rows, n_keep_t, nt, n_keep);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_csr_gather(const int32_t* st_idx, const double* st_val, const int32_t* n_keep,
                              const int32_t* status, const int64_t* indptr, int64_t nq, int S,
                              const int32_t* todo_rows, int64_t nt, const int64_t* seg_ptr,
                              const int32_t* seg_idx, const double* seg_val, const int32_t* n_keep_t,
                              int32_t* out_idx, double* out_val, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (st_idx) {
    csr_gather1_kernel<<<(unsigned)gtb_cdiv(nq * S, 256), 256, 0, st>>>(st_idx, st_val, n_keep, status, indptr, nq, S,
                                                                      out_idx, out_val);
    GTB_CHECK_LAUNCH();
  }
  if (nt > 0) {
    csr_gather2_kernel<<<(unsigned)nt, 128, 0, st>>>(todo_rows, seg_ptr, seg_idx, seg_val, n_keep_t, indptr,
                                                     out_idx, out_val);
    GTB_CHECK_LAUNCH();
  }
  return GTB_OK;
}

extern "C" int gtb_knn_count_bound(const uint32_t* coarse, const uint32_t* fine, int64_t nq, int64_t nr, int elo,
                                   int margin, float s2, const float* qn2, float maxrn2, double eps_rel, int x_kind,
                                   int knn, int64_t kmax, double decay, double thresh, const double* bw_fixed,
                                   int bw_mode, double bw_scale, float* top, float* lim2, int32_t* ball_lo,
                                   int32_t* ball_hi, void* stream) {
  GTB_CHECK_ARG(nq > 0 && nr > 0 && knn >= 1 && s2 > 0.f, "bad shape");
  GTB_CHECK_ARG(x_kind >= 0 && x_kind <= 9, "x_kind: bit 0 = float64 rows, bits 1-3 = metric");
  GTB_CHECK_ARG(coarse != nullptr || (bw_mode != 0 && decay >= 0 && lim2),
                "without a coarse histogram: a fixed bandwidth (bw_mode 1 or 2) and lim2");
  GTB_CHECK_ARG(coarse == nullptr || fine != nullptr || top, "coarse only: top is required");
  GTB_CHECK_ARG(coarse == nullptr || fine == nullptr || (lim2 && ball_lo && ball_hi), "lim2, ball_lo, ball_hi required");
  GTB_CHECK_ARG(elo >= 1 && elo + 64 <= 254 && margin >= 1, "1 <= elo <= 190, margin >= 1");
  GTB_CHECK_ARG(decay < 0 || (thresh > 0 && thresh <= 1), "thresh must be in (0, 1]");
  BoundParams p;
  p.rp = make_row_params(nullptr, nullptr, 0, knn, kmax, decay, thresh, bw_fixed, bw_mode, bw_scale, x_kind >> 1);
  p.coarse = coarse; p.fine = fine; p.nq = nq; p.nr = nr; p.elo = elo; p.margin = margin; p.s2 = s2;
  p.qn2 = qn2; p.maxrn2 = maxrn2; p.eps_rel = eps_rel;
  p.top = top; p.lim2 = lim2; p.ball_lo = ball_lo; p.ball_hi = ball_hi;
  count_bound_kernel<<<(unsigned)gtb_cdiv(nq, 256), 256, 0, (cudaStream_t)stream>>>(p);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}
