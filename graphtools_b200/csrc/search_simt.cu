// K1/K2 (CUDA-core variant): tiled pairwise squared distance |x|^2+|y|^2-2xy in fp32 with the
// per-query selection fused into the tile epilogue; the N x N distance matrix is never written.
//
//   * TOPK epilogue  : per query row keep the S smallest approximate distances (candidate set
//                      for the float64 re-evaluation) and tau = S-th smallest approximate d^2.
//                      Replaces sklearn ArgKmin behind knn_tree.kneighbors (reference
//                      graphtools/graphs.py:883, :922, :957).
//   * RADIUS epilogue: append every (query, ref) pair with approximate d^2 <= lim2[query].
//                      Replaces knn_tree.radius_neighbors (graphs.py:966-973) and the x6
//                      escalation loop (graphs.py:916-944): one pass returns the whole ball.
//   * COUNT epilogue : per query row, a histogram of the float32 bits of the approximate d^2 under the row's top edge
//                      (the histogram count sweep of csrc/search_tc.cu on the CUDA cores: cityblock, d > 510).
//
// Operands are the k-major centred search operands built by prep.cu.  CTA = 128 queries x
// 128 refs x KC=8, 256 threads; warp w owns query rows 16w..16w+15 (all 128 columns), lane l owns
// columns 4l..4l+3, so a row's running top-S list is private to one warp (no locks).  4-stage
// cp.async ring over the flattened (ref tile, k chunk) sequence.
#include "common.cuh"
#include "gtb200.h"
#include <type_traits>

namespace {

constexpr int TM = 128, TN = 128, KC = 8, NST = 4, NTHREADS = 256;

__device__ __forceinline__ void cp_async16_ca(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async16_cg(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

struct SearchParams {
  const float* QT; const float* qn2; int64_t nq; int64_t nq_pad;
  const float* RT; const float* rn2; int64_t nr; int64_t nr_pad;
  int d_pad;
  // top-k
  int32_t* cand_idx; float* tau;
  // radius
  const float* lim2; int2* pairs; unsigned long long capacity; unsigned long long* counter;
  int32_t* rowcnt;
};
// count sweeps (contract of gtb_knn_count_tc): hist [nq_pad][count_bins], top = fine-pass top edges (NULL: coarse pass).
// A separate type, so that the top-k and radius kernels keep their parameter block.
struct CountParams : SearchParams {
  uint32_t* hist; const float* top; int count_k, count_margin, count_elo, count_bins;
};

// L1 = true: cityblock metric.  The tile accumulates sum_k |x_k - y_k| directly (two FADDs per pair and feature
// instead of one FFMA; there is no GEMM form of the L1 distance), the norms are not used, and padding columns are
// masked by index (their zero rows would otherwise be at a finite distance).
template <int S, bool RADIUS, bool L1, bool COUNT = false>
__global__ void __launch_bounds__(NTHREADS, (S <= 64 ? 2 : 1))
search_simt_kernel(std::conditional_t<COUNT, CountParams, SearchParams> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* As = reinterpret_cast<float*>(smem_raw);                 // [NST][KC][TM]
  float* Bs = As + NST * KC * TM;                                  // [NST][KC][TN]
  float* thr_s = Bs + NST * KC * TN;                               // [TM]  primed threshold
  float* nx_s = thr_s + TM;                                        // [TM]
  float* list_d = nx_s + TM;                                       // [TM][S]  (TOPK only)
  int32_t* list_i = reinterpret_cast<int32_t*>(list_d + (RADIUS ? 0 : TM * S));  // [TM][S]
  uint32_t* hist_s = reinterpret_cast<uint32_t*>(list_d);          // [count_bins][TM]  (COUNT only)

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t q0 = (int64_t)blockIdx.x * TM;
  const int nk = p.d_pad / KC;
  const int64_t ntiles = p.nr_pad / TN;
  const int64_t nchunks = ntiles * nk;

  // per-row state
  if (tid < TM) {
    int64_t q = q0 + tid;
    float nx = (q < p.nq && !L1) ? p.qn2[q] : 0.f;
    nx_s[tid] = nx;
    if constexpr (COUNT) {
      // fine pass: the octave top from the coarse pass (rows without one are not counted); coarse: no edge yet
      const float t = (q < p.nq && p.top) ? p.top[q] : gtb_inf_f();
      thr_s[tid] = (q < p.nq && (!p.top || t < gtb_inf_f())) ? t - nx : -gtb_inf_f();
    } else {
    if (RADIUS) thr_s[tid] = (q < p.nq) ? (p.lim2[q] - nx) : -gtb_inf_f();
    else thr_s[tid] = (q < p.nq) ? gtb_inf_f() : -gtb_inf_f();
    }
  }
  if constexpr (COUNT) {
    for (int i = tid; i < p.count_bins * TM; i += NTHREADS) hist_s[i] = 0u;
  }
  if (!RADIUS) {
    for (int i = tid; i < TM * S; i += NTHREADS) { list_d[i] = gtb_inf_f(); list_i[i] = -1; }
  }
  __syncthreads();

  // loader: thread -> (k row kk, float4 column x4) of the A and B chunk
  const int ld_kk = tid >> 5, ld_x4 = tid & 31;
  auto issue = [&](int64_t c) {
    if (c < nchunks) {
      int st = (int)(c % NST);
      int64_t tile = c / nk;
      int kc = (int)(c - tile * nk);
      int64_t k = (int64_t)kc * KC + ld_kk;
      cp_async16_ca(As + (st * KC + ld_kk) * TM + ld_x4 * 4, p.QT + k * p.nq_pad + q0 + ld_x4 * 4);
      cp_async16_cg(Bs + (st * KC + ld_kk) * TN + ld_x4 * 4, p.RT + k * p.nr_pad + tile * TN + ld_x4 * 4);
    }
    cp_async_commit();
  };

  float acc[16][4];
#pragma unroll
  for (int i = 0; i < 16; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

#pragma unroll
  for (int s = 0; s < NST - 1; ++s) issue(s);

  float4 ny = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t c = 0; c < nchunks; ++c) {
    cp_async_wait<NST - 2>();
    __syncthreads();
    issue(c + NST - 1);
    const int st = (int)(c % NST);
    const int64_t tile = c / nk;
    const int kc = (int)(c - tile * nk);
    const bool last = (kc == nk - 1);
    if (last && !L1) ny = __ldg(reinterpret_cast<const float4*>(p.rn2 + tile * TN) + lane);
    const float* a_base = As + st * KC * TM + warp * 16;
    const float* b_base = Bs + st * KC * TN + lane * 4;
#pragma unroll
    for (int kk = 0; kk < KC; ++kk) {
      float a[16];
      const float4* ap = reinterpret_cast<const float4*>(a_base + kk * TM);
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        float4 t = ap[v];
        a[4 * v] = t.x; a[4 * v + 1] = t.y; a[4 * v + 2] = t.z; a[4 * v + 3] = t.w;
      }
      float4 b = *reinterpret_cast<const float4*>(b_base + kk * TN);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        if (L1) {
          acc[i][0] += fabsf(a[i] - b.x);
          acc[i][1] += fabsf(a[i] - b.y);
          acc[i][2] += fabsf(a[i] - b.z);
          acc[i][3] += fabsf(a[i] - b.w);
        } else {
          acc[i][0] = fmaf(a[i], b.x, acc[i][0]);
          acc[i][1] = fmaf(a[i], b.y, acc[i][1]);
          acc[i][2] = fmaf(a[i], b.z, acc[i][2]);
          acc[i][3] = fmaf(a[i], b.w, acc[i][3]);
        }
      }
    }
    if (!last) continue;

    // ---- tile epilogue: acc holds x.y for rows 16w..16w+15 x cols 4l..4l+3 of this ref tile
    const int32_t colbase = (int32_t)(tile * TN) + lane * 4;
    const float nyv[4] = {ny.x, ny.y, ny.z, ny.w};
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int r = warp * 16 + i;
      float t = thr_s[r];
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (L1) v[j] = (colbase + j < p.nr) ? acc[i][j] : gtb_inf_f();
        else v[j] = fmaf(-2.f, acc[i][j], nyv[j]);
        acc[i][j] = 0.f;
      }
      if constexpr (COUNT) {
        bool mine = false;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (L1 && colbase + j >= p.nr) v[j] = gtb_inf_f();
          mine |= v[j] < t;
        }
        if (__ballot_sync(0xffffffffu, mine)) {
          const float nx = nx_s[r];
          const int eo = p.top ? (int)(__float_as_uint(p.top[q0 + r]) >> 23) - 1 : 0;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (v[j] < t) {
              // bins of csrc/search_tc.cu (COUNT mode)
              const uint32_t bits = __float_as_uint(v[j] + nx);
              const int e = (int)bits >> 23;
              int bin;
              if (!p.top) bin = min(max(e - p.count_elo, 0), 63);
              else bin = (e < eo) ? 0 : (e == eo ? 1 + (int)((bits >> 19) & 15u) : -1);
              if (bin >= 0) atomicAdd(hist_s + bin * TM + r, 1u);
            }
          }
          if (!p.top) {
            // coarse top edge: count_margin octaves above the first bin whose cumulative count reaches k (the warp
            // owns row r: two bins per lane, warp-inclusive scan)
            __syncwarp();
            const uint32_t c0 = hist_s[(2 * lane) * TM + r], c1 = hist_s[(2 * lane + 1) * TM + r];
            uint32_t incl = c0 + c1;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
              const uint32_t o = __shfl_up_sync(0xffffffffu, incl, off);
              if (lane >= off) incl += o;
            }
            const uint32_t k = (uint32_t)p.count_k;
            const unsigned m0 = __ballot_sync(0xffffffffu, incl - c1 >= k), m1 = __ballot_sync(0xffffffffu, incl >= k);
            // first bin b with cumulative count >= k: 2l (m0) or 2l + 1 (m1 only)
            const int b = m1 ? ((m0 && (__ffs(m0) <= __ffs(m1))) ? 2 * (__ffs(m0) - 1) : 2 * (__ffs(m1) - 1) + 1) : 64;
            const int tb = b + p.count_margin;
            if (b < 63 && tb < 63) t = fminf(t, __uint_as_float((uint32_t)(p.count_elo + tb + 1) << 23) - nx);
            if (lane == 0) thr_s[r] = t;
            __syncwarp();
          }
        }
      } else {
      if (RADIUS) {
        int cnt = (v[0] <= t) + (v[1] <= t) + (v[2] <= t) + (v[3] <= t);
        unsigned any = __ballot_sync(0xffffffffu, cnt > 0);
        if (any) {
          // warp-exclusive scan of cnt
          int incl = cnt;
#pragma unroll
          for (int off = 1; off < 32; off <<= 1) {
            int o = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += o;
          }
          int total = __shfl_sync(0xffffffffu, incl, 31);
          unsigned long long base = 0;
          if (lane == 0) {
            base = atomicAdd(p.counter, (unsigned long long)total);
            atomicAdd(p.rowcnt + (q0 + r), total);
          }
          base = __shfl_sync(0xffffffffu, base, 0);
          unsigned long long pos = base + (unsigned long long)(incl - cnt);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (v[j] <= t) {
              if (pos < p.capacity) p.pairs[pos] = make_int2((int)(q0 + r), colbase + j);
              ++pos;
            }
          }
        }
      } else {
        bool mine = (v[0] < t) | (v[1] < t) | (v[2] < t) | (v[3] < t);
        if (__ballot_sync(0xffffffffu, mine)) {
          float* ld = list_d + r * S;
          int32_t* li = list_i + r * S;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            unsigned m = __ballot_sync(0xffffffffu, v[j] < t);
            while (m) {
              int src = __ffs(m) - 1;
              m &= m - 1;
              float val = __shfl_sync(0xffffffffu, v[j], src);
              if (val < t) {  // uniform across the warp (t is warp-uniform)
                // arg-max of the row's list (ties -> lowest slot)
                float best = -gtb_inf_f();
                int slot = 0x7fffffff;
                for (int s = lane; s < S; s += 32) {
                  float e = ld[s];
                  if (e > best) { best = e; slot = s; }
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                  float ob = __shfl_xor_sync(0xffffffffu, best, off);
                  int os = __shfl_xor_sync(0xffffffffu, slot, off);
                  if (ob > best || (ob == best && os < slot)) { best = ob; slot = os; }
                }
                if (lane == 0) { ld[slot] = val; li[slot] = colbase - lane * 4 + src * 4 + j; }
                __syncwarp();
                float nb = -gtb_inf_f();
                for (int s = lane; s < S; s += 32) nb = fmaxf(nb, ld[s]);
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) nb = fmaxf(nb, __shfl_xor_sync(0xffffffffu, nb, off));
                t = nb;
              }
            }
          }
          if (lane == 0) thr_s[r] = t;
          __syncwarp();
        }
      }
      }
    }
  }
  cp_async_wait<0>();

  if constexpr (COUNT) {
    // each CTA sweeps every reference tile for its own query rows: its counts are the rows' histograms
    __syncthreads();
    for (int i = tid; i < p.count_bins * TM; i += NTHREADS) {
      const int b = i / TM, r = i - b * TM;
      if (q0 + r < p.nq) p.hist[(q0 + r) * p.count_bins + b] = hist_s[i];
    }
  } else {
  if (!RADIUS) {
    __syncwarp();
    // write candidate lists (slot order is arbitrary; the refine stage sorts by exact distance)
#pragma unroll 1
    for (int i = 0; i < 16; ++i) {
      const int r = warp * 16 + i;
      const int64_t q = q0 + r;
      if (q >= p.nq) continue;
      for (int s = lane; s < S; s += 32) p.cand_idx[q * S + s] = list_i[r * S + s];
      if (lane == 0) p.tau[q] = thr_s[r] + nx_s[r];
    }
  }
  }
}

template <int S, bool RADIUS, bool L1 = false, bool COUNT = false, typename P = SearchParams>
int launch(const P& p, cudaStream_t st) {
  size_t smem = sizeof(float) * (NST * KC * (TM + TN) + 2 * TM) + (RADIUS ? 0 : (size_t)TM * S * 8) +
                (COUNT ? (size_t)64 * TM * sizeof(uint32_t) : 0);
  auto kern = search_simt_kernel<S, RADIUS, L1, COUNT>;
  GTB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)(p.nq_pad / TM), NTHREADS, smem, st>>>(p);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

}  // namespace

extern "C" int gtb_knn_topk_simt(const float* QT, const float* qn2, int64_t nq, int64_t nq_pad,
                                 const float* RT, const float* rn2, int64_t nr, int64_t nr_pad,
                                 int d_pad, int S, int32_t* cand_idx, float* tau, void* stream) {
  GTB_CHECK_ARG(nq > 0 && nr > 0 && nq_pad % TM == 0 && nr_pad % TN == 0 && d_pad % KC == 0, "bad shape");
  SearchParams p{};
  p.QT = QT; p.qn2 = qn2; p.nq = nq; p.nq_pad = nq_pad; p.RT = RT; p.rn2 = rn2; p.nr = nr;
  p.nr_pad = nr_pad; p.d_pad = d_pad; p.cand_idx = cand_idx; p.tau = tau;
  cudaStream_t st = (cudaStream_t)stream;
  switch (S) {
    case 16: return launch<16, false>(p, st);
    case 32: return launch<32, false>(p, st);
    case 48: return launch<48, false>(p, st);
    case 64: return launch<64, false>(p, st);
    case 128: return launch<128, false>(p, st);
    default: gtb_set_error("gtb_knn_topk: S must be one of 16,32,48,64,128 (got %d)", S); return GTB_ERR_ARG;
  }
}

extern "C" int gtb_knn_radius_simt(const float* QT, const float* qn2, const float* lim2, int64_t nq,
                                   int64_t nq_pad, const float* RT, const float* rn2, int64_t nr,
                                   int64_t nr_pad, int d_pad, int32_t* pairs, int64_t capacity,
                                   unsigned long long* counter, int32_t* rowcnt, void* stream) {
  GTB_CHECK_ARG(nq > 0 && nr > 0 && nq_pad % TM == 0 && nr_pad % TN == 0 && d_pad % KC == 0, "bad shape");
  SearchParams p{};
  p.QT = QT; p.qn2 = qn2; p.nq = nq; p.nq_pad = nq_pad; p.RT = RT; p.rn2 = rn2; p.nr = nr;
  p.nr_pad = nr_pad; p.d_pad = d_pad; p.lim2 = lim2; p.pairs = reinterpret_cast<int2*>(pairs);
  p.capacity = (unsigned long long)capacity; p.counter = counter; p.rowcnt = rowcnt;
  return launch<16, true>(p, (cudaStream_t)stream);
}

// cityblock (L1) variants: same operands (k-major rows, NOT centred -- |x - y| is translation invariant and the
// uncentred float32 copy keeps the rounding error relative to the distance itself), approximate distance
// sum_k |x_k - y_k| in float32; tau / lim hold distances, not squared distances.  Replaces sklearn's brute-force
// manhattan search behind knn_tree for distance="cityblock" (graphs.py:763-768).
extern "C" int gtb_knn_topk_simt_l1(const float* QT, int64_t nq, int64_t nq_pad, const float* RT, int64_t nr,
                                    int64_t nr_pad, int d_pad, int S, int32_t* cand_idx, float* tau, void* stream) {
  GTB_CHECK_ARG(nq > 0 && nr > 0 && nq_pad % TM == 0 && nr_pad % TN == 0 && d_pad % KC == 0, "bad shape");
  SearchParams p{};
  p.QT = QT; p.nq = nq; p.nq_pad = nq_pad; p.RT = RT; p.nr = nr;
  p.nr_pad = nr_pad; p.d_pad = d_pad; p.cand_idx = cand_idx; p.tau = tau;
  cudaStream_t st = (cudaStream_t)stream;
  switch (S) {
    case 16: return launch<16, false, true>(p, st);
    case 32: return launch<32, false, true>(p, st);
    case 48: return launch<48, false, true>(p, st);
    case 64: return launch<64, false, true>(p, st);
    case 128: return launch<128, false, true>(p, st);
    default: gtb_set_error("gtb_knn_topk: S must be one of 16,32,48,64,128 (got %d)", S); return GTB_ERR_ARG;
  }
}

extern "C" int gtb_knn_radius_simt_l1(const float* QT, const float* lim, int64_t nq, int64_t nq_pad, const float* RT,
                                      int64_t nr, int64_t nr_pad, int d_pad, int32_t* pairs, int64_t capacity,
                                      unsigned long long* counter, int32_t* rowcnt, void* stream) {
  GTB_CHECK_ARG(nq > 0 && nr > 0 && nq_pad % TM == 0 && nr_pad % TN == 0 && d_pad % KC == 0, "bad shape");
  SearchParams p{};
  p.QT = QT; p.nq = nq; p.nq_pad = nq_pad; p.RT = RT; p.nr = nr;
  p.nr_pad = nr_pad; p.d_pad = d_pad; p.lim2 = lim; p.pairs = reinterpret_cast<int2*>(pairs);
  p.capacity = (unsigned long long)capacity; p.counter = counter; p.rowcnt = rowcnt;
  return launch<16, true, true>(p, (cudaStream_t)stream);
}

// Histogram count sweeps on the CUDA cores: the contract of gtb_knn_count_tc (bins, top, k, margin, elo) on the operands
// of gtb_knn_radius_simt (qn2 / rn2 non-NULL) or gtb_knn_radius_simt_l1 (qn2 = rn2 = NULL: cityblock distances).
extern "C" int gtb_knn_count_simt(const float* QT, const float* qn2, const float* top, int64_t nq, int64_t nq_pad,
                                  const float* RT, const float* rn2, int64_t nr, int64_t nr_pad, int d_pad, int k,
                                  int margin, int elo, uint32_t* hist, void* stream) {
  GTB_CHECK_ARG(nq > 0 && nr > 0 && nq_pad % TM == 0 && nr_pad % TN == 0 && d_pad % KC == 0, "bad shape");
  GTB_CHECK_ARG(k >= 1 && margin >= 1 && elo >= 1 && elo + 64 <= 254, "k >= 1, margin >= 1, 1 <= elo <= 190");
  GTB_CHECK_ARG((qn2 == nullptr) == (rn2 == nullptr), "qn2 and rn2: both (squared distances) or neither (cityblock)");
  CountParams p{};
  p.QT = QT; p.qn2 = qn2; p.nq = nq; p.nq_pad = nq_pad; p.RT = RT; p.rn2 = rn2; p.nr = nr;
  p.nr_pad = nr_pad; p.d_pad = d_pad; p.hist = hist; p.top = top; p.count_k = k; p.count_margin = margin;
  p.count_elo = elo; p.count_bins = top ? 17 : 64;
  cudaStream_t st = (cudaStream_t)stream;
  GTB_CUDA(cudaMemsetAsync(hist, 0, sizeof(uint32_t) * nq_pad * p.count_bins, st));
  return qn2 ? launch<16, true, false, true, CountParams>(p, st) : launch<16, true, true, true, CountParams>(p, st);
}
