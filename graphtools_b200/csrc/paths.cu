// All-pairs shortest paths on the kernel graph (K10): replaces scipy.sparse.csgraph.shortest_path behind
// BaseGraph.shortest_path (reference graphtools/base.py:934-988).
//
// Pipeline per call (graphtools_b200/paths.py): dense K -> CSR (present entries, as csr_matrix(K)) -> edge lengths ->
// weakly connected components -> batches of up to 256 sources, sources sorted by component -> per batch: one
// persistent traversal kernel on a [N][B] distance block, then a tiled transpose that writes the block into the
// sources' rows of the [N][N] result -> one in-place finishing pass (D + D^T) / 2, 0 -> inf, zero diagonal.
//
// Arithmetic contract.  Lengths are non-negative (checked before any traversal), so float64 addition is monotone:
// a <= b implies fl(a + w) <= fl(b + w), and fl(a + w) >= a.  Under that condition every label-correcting
// relaxation dist[v] = min(dist[v], fl(dist[u] + w_uv)) run to its fixpoint -- Dijkstra, Bellman-Ford, or the
// frontier relaxation below -- ends at the same number: the minimum over paths of the left-to-right float64 sum
// from the source.  The traversal is therefore bit-identical to scipy's method="D" (and "BF" / "J", which reduce to
// the same relaxations for non-negative lengths) whatever order the relaxations happen in, and bit-reproducible.
#include <cooperative_groups.h>

#include "common.cuh"
#include "gtb200.h"

namespace cg = cooperative_groups;

namespace {

constexpr int SP_THREADS = 256;
constexpr int SP_MAX_BATCH = 1024;

// ------------------------------------------------------------------------------------------- double-double log
// Correctly rounded natural logarithm: log(x) = e ln2 + 2 atanh(f), f = (m - 1) / (m + 1), m in [sqrt(1/2), sqrt(2)),
// evaluated in double-double (~2^-104 relative) and rounded once.  CUDA's log() is within 1 ulp, and numpy's log is
// platform-dependent (SVML on AVX-512 hosts, libm elsewhere); a correctly rounded value is the one both can be
// checked against.
struct dd { double hi, lo; };

__device__ __forceinline__ dd dd_two_sum(double a, double b) {
  const double s = __dadd_rn(a, b);
  const double bb = __dsub_rn(s, a);
  const double e = __dadd_rn(__dsub_rn(a, __dsub_rn(s, bb)), __dsub_rn(b, bb));
  return {s, e};
}
__device__ __forceinline__ dd dd_fast_two_sum(double a, double b) {
  const double s = __dadd_rn(a, b);
  return {s, __dsub_rn(b, __dsub_rn(s, a))};
}
__device__ __forceinline__ dd dd_add(dd a, dd b) {
  dd s = dd_two_sum(a.hi, b.hi);
  const dd t = dd_two_sum(a.lo, b.lo);
  s = dd_fast_two_sum(s.hi, __dadd_rn(s.lo, t.hi));
  return dd_fast_two_sum(s.hi, __dadd_rn(s.lo, t.lo));
}
__device__ __forceinline__ dd dd_mul(dd a, dd b) {
  const double p = __dmul_rn(a.hi, b.hi);
  double e = __fma_rn(a.hi, b.hi, -p);
  e = __fma_rn(a.hi, b.lo, e);
  e = __fma_rn(a.lo, b.hi, e);
  return dd_fast_two_sum(p, e);
}
__device__ __forceinline__ dd dd_div(dd a, dd b) {
  const double q1 = __ddiv_rn(a.hi, b.hi);
  dd r = dd_add(a, dd_mul({-q1, 0.0}, b));
  const double q2 = __ddiv_rn(r.hi, b.hi);
  r = dd_add(r, dd_mul({-q2, 0.0}, b));
  const double q3 = __ddiv_rn(r.hi, b.hi);
  return dd_add(dd_fast_two_sum(q1, q2), {q3, 0.0});
}

__device__ double log_cr(double x) {
  // x >= 0 and finite (K values of a built graph); -log(0) = inf, as numpy gives for a stored zero
  if (x == 0.0) return -__longlong_as_double(0x7ff0000000000000LL);
  int e = 0;
  double m = frexp(x, &e);                    // x = m 2^e, m in [0.5, 1)
  m = __dmul_rn(m, 2.0); e -= 1;              // m in [1, 2)
  if (m > 1.4142135623730951) { m = __dmul_rn(m, 0.5); e += 1; }
  const dd num = {__dsub_rn(m, 1.0), 0.0};    // exact (Sterbenz)
  const dd f = dd_div(num, dd_two_sum(m, 1.0));
  const dd s = dd_mul(f, f);
  // P(s) = sum_k s^k / (2k + 1); |s| < 0.0295, 23 terms reach 2^-110
  dd p = dd_div({1.0, 0.0}, {45.0, 0.0});
#pragma unroll 1
  for (int k = 21; k >= 0; --k) p = dd_add(dd_mul(p, s), dd_div({1.0, 0.0}, {(double)(2 * k + 1), 0.0}));
  dd r = dd_mul(f, p);
  r = {__dmul_rn(r.hi, 2.0), __dmul_rn(r.lo, 2.0)};
  const dd ln2 = {6.93147180559945286227e-01, 2.31904681384629955842e-17};
  const dd el = dd_mul({(double)e, 0.0}, ln2);
  r = dd_add(el, r);
  return __dadd_rn(r.hi, r.lo);
}

// numpy's pairwise summation (np.sum over a contiguous row of length n, any n), so that the "data" lengths equal
// np.sqrt(np.sum((a - b) ** 2, axis=1)) bit for bit in the dtype of data_nu.  Blocks of <= 128 elements use eight
// interleaved accumulators; longer runs are split at n/2 rounded down to a multiple of 8 (iteratively, no recursion).
// separate multiply and add (no FMA contraction): numpy squares and sums with plain IEEE operations
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }

template <typename T>
__device__ T sqdist_block(const T* a, const T* b, int n) {
  auto sq = [&](int i) { const T t = a[i] - b[i]; return mul_rn(t, t); };
  if (n < 8) {
    T r = T(-0.0);
    for (int i = 0; i < n; ++i) r = add_rn(r, sq(i));
    return r;
  }
  T r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = sq(j);
  int i = 8;
  for (; i < n - (n % 8); i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = add_rn(r[j], sq(i + j));
  }
  T res = add_rn(add_rn(add_rn(r[0], r[1]), add_rn(r[2], r[3])), add_rn(add_rn(r[4], r[5]), add_rn(r[6], r[7])));
  for (; i < n; ++i) res = add_rn(res, sq(i));
  return res;
}

template <typename T>
__device__ T sqdist_pairwise(const T* a, const T* b, int n) {
  if (n <= 128) return sqdist_block(a, b, n);
  // explicit stack of (offset, length, partial) for the recursion sum(left) + sum(right)
  int off[24], len[24], state[24];
  T part[24];
  int top = 0;
  off[0] = 0; len[0] = n; state[0] = 0;
  T ret = T(0);
  while (top >= 0) {
    const int o = off[top], l = len[top];
    if (l <= 128) {
      ret = sqdist_block(a + o, b + o, l);
      --top;
    } else {
      int h = l / 2; h -= h % 8;
      if (state[top] == 0) {                  // descend left
        state[top] = 1;
        ++top; off[top] = o; len[top] = h; state[top] = 0;
        continue;
      }
      if (state[top] == 1) {                  // left done, descend right
        part[top] = ret; state[top] = 2;
        ++top; off[top] = o + h; len[top] = l - h; state[top] = 0;
        continue;
      }
      ret = add_rn(part[top], ret);
      --top;
    }
  }
  return ret;
}

// mode 0 constant: w = K_ij; 1 data: |x_i - x_j|_2 (T = float or double); 2 affinity: -log(K_ij)
template <typename T>
__global__ void __launch_bounds__(256) lengths_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx,
                                                      const double* __restrict__ val, int64_t n, const T* __restrict__ X,
                                                      int d, int mode, double* __restrict__ len, int32_t* flags) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const int lane = threadIdx.x & 31;
  bool bad = false;
  for (int64_t p = indptr[row] + lane; p < indptr[row + 1]; p += 32) {
    double w;
    if (mode == 0) {
      w = val[p];
    } else if (mode == 1) {
      w = (double)sqrt(sqdist_pairwise<T>(X + row * d, X + (int64_t)idx[p] * d, d));
    } else {
      w = -log_cr(val[p]);
    }
    bad |= !(w >= 0.0);                       // negative or NaN
    len[p] = __dadd_rn(w, 0.0);               // -0 -> +0: the traversal orders lengths by their bit patterns
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(flags, 1);
}

// ------------------------------------------------------------------------------------------- components
// Weakly connected components by lock-free union-find (hook the larger root under the smaller by CAS, find with
// path halving): parent[v] = smallest vertex of v's component after compress.
__device__ __forceinline__ int32_t uf_find(int32_t* parent, int32_t v) {
  int32_t p = __ldcg(parent + v);
  while (p != v) {
    const int32_t gp = __ldcg(parent + p);
    if (gp != p) atomicCAS(parent + v, p, gp);   // path halving (only ever lowers a parent)
    v = p;
    p = gp;
  }
  return v;
}

__global__ void cc_init_kernel(int32_t* parent, int64_t n) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) parent[v] = (int32_t)v;
}

__global__ void cc_hook_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx, int64_t n,
                               int32_t* parent) {
  const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= n) return;
  for (int64_t p = indptr[u]; p < indptr[u + 1]; ++p) {
    int32_t a = (int32_t)u, b = idx[p];
    while (true) {
      a = uf_find(parent, a);
      b = uf_find(parent, b);
      if (a == b) break;
      if (a < b) { const int32_t t = a; a = b; b = t; }
      if (atomicCAS(parent + a, a, b) == a) break;   // a was still a root: hooked
    }
  }
}

__global__ void cc_compress_kernel(int32_t* parent, int64_t n) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) parent[v] = uf_find(parent, (int32_t)v);
}

// ------------------------------------------------------------------------------------------- traversal
// Distance block dist[v][b] (row stride ldb = 32 * nch) for the nb sources src[b].  Work items are (vertex, 32-source
// chunk) slots with a 32-bit mask of the chunk's sources whose distance to the vertex dropped in the last round.  One
// warp per item: lanes are sources, so an edge (index + length, 12 bytes) is read once per 32 sources and each lane's
// relaxation is a coalesced 8-byte atomicMin on the bit pattern (non-negative doubles order like their bits).
// Rounds are separated by grid-wide barriers of one persistent cooperative kernel; the loop ends when a round
// lowers nothing.
__global__ void __launch_bounds__(SP_THREADS) sp_traverse_kernel(
    const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx, const double* __restrict__ len, int64_t n,
    const int32_t* __restrict__ src, int nb, double* dist, int nch, uint32_t* mask0, uint32_t* mask1, int32_t* list0,
    int32_t* list1, int32_t* cnt) {
  cg::grid_group grid = cg::this_grid();
  const int64_t tid = grid.thread_rank(), nth = grid.size();
  const int64_t ldb = (int64_t)nch * 32;
  const double inf = __longlong_as_double(0x7ff0000000000000LL);
  for (int64_t e = tid; e < n * ldb; e += nth) dist[e] = inf;
  for (int64_t e = tid; e < n * nch; e += nth) { mask0[e] = 0u; mask1[e] = 0u; }
  if (tid < 2) cnt[tid] = 0;
  grid.sync();
  for (int64_t b = tid; b < nb; b += nth) {
    const int64_t v = src[b];
    dist[v * ldb + b] = 0.0;
    const int32_t slot = (int32_t)(v * nch + (b >> 5));
    if (atomicOr(mask0 + slot, 1u << (b & 31)) == 0u) list0[atomicAdd(cnt, 1)] = slot;
  }
  grid.sync();
  const int lane = threadIdx.x & 31;
  const int64_t warp = tid >> 5, nwarps = nth >> 5;
  int cur = 0;
  while (true) {
    const int count = *(volatile int32_t*)(cnt + cur);
    if (count == 0) break;
    uint32_t* cm = cur ? mask1 : mask0;
    uint32_t* nm = cur ? mask0 : mask1;
    const int32_t* cl = cur ? list1 : list0;
    int32_t* nl = cur ? list0 : list1;
    int32_t* ncnt = cnt + (cur ^ 1);
    for (int64_t it = warp; it < count; it += nwarps) {
      const int32_t slot = __ldcg(cl + it);
      const uint32_t m = __ldcg(cm + slot);
      const int64_t u = slot / nch;
      const int c = slot - (int32_t)(u * nch);
      const bool act = (m >> lane) & 1u;
      const int64_t col = (int64_t)c * 32 + lane;
      const double du = act ? __ldcg(dist + u * ldb + col) : inf;
      const int64_t p1 = indptr[u + 1];
      for (int64_t p = indptr[u]; p < p1; ++p) {
        const int32_t v = idx[p];
        const double nd = __dadd_rn(du, len[p]);
        bool lowered = false;
        if (act) {
          unsigned long long* a = reinterpret_cast<unsigned long long*>(dist + (int64_t)v * ldb + col);
          if (nd < __longlong_as_double((long long)__ldcg(a))) {
            const unsigned long long old = atomicMin(a, (unsigned long long)__double_as_longlong(nd));
            lowered = nd < __longlong_as_double((long long)old);
          }
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, lowered);
        if (bal != 0u && lane == __ffs(bal) - 1) {
          const int32_t ns = (int32_t)((int64_t)v * nch + c);
          if (atomicOr(nm + ns, bal) == 0u) nl[atomicAdd(ncnt, 1)] = ns;
        }
      }
      if (lane == 0) cm[slot] = 0u;
    }
    grid.sync();
    if (tid == 0) cnt[cur] = 0;
    cur ^= 1;
    grid.sync();
  }
}

// out[src[b]][v] = dist[v][b]: 32 x 32 tiles through shared memory (reads along b, writes along v coalesced)
__global__ void sp_store_rows_kernel(const double* __restrict__ dist, int64_t ldb, int64_t n,
                                     const int32_t* __restrict__ src, int nb, double* __restrict__ out, int64_t ldo) {
  __shared__ double tile[32][33];
  const int64_t v0 = (int64_t)blockIdx.x * 32;
  const int b0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int64_t v = v0 + r;
    const int b = b0 + threadIdx.x;
    if (v < n && b < nb) tile[r][threadIdx.x] = dist[v * ldb + b];
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int b = b0 + r;
    const int64_t v = v0 + threadIdx.x;
    if (b < nb && v < n) out[(int64_t)src[b] * ldo + v] = tile[threadIdx.x][r];
  }
}

// In place on D[n][n]: D_ij = D_ji = (D_ij + D_ji) / 2, then 0 -> inf off the diagonal and 0 on it.  One block per
// pair of 32 x 32 tiles (ti <= tj); (a + b) / 2 is commutative, so the result is bitwise symmetric.
__device__ __forceinline__ double sp_finish_value(double a, double b, bool diag) {
  const double s = __ddiv_rn(__dadd_rn(a, b), 2.0);
  if (diag) return 0.0;
  return s == 0.0 ? __longlong_as_double(0x7ff0000000000000LL) : s;
}

__global__ void sp_finish_kernel(double* D, int64_t n) {
  const int ti = blockIdx.y, tj = blockIdx.x;
  if (ti > tj) return;
  __shared__ double A[32][33], B[32][33];
  const int64_t i0 = (int64_t)ti * 32, j0 = (int64_t)tj * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int c = threadIdx.x;
    if (i0 + r < n && j0 + c < n) A[r][c] = D[(i0 + r) * n + j0 + c];
    if (j0 + r < n && i0 + c < n) B[r][c] = D[(j0 + r) * n + i0 + c];
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int c = threadIdx.x;
    const int64_t i = i0 + r, j = j0 + c;
    if (i < n && j < n) D[i * n + j] = sp_finish_value(A[r][c], B[c][r], i == j);
    if (ti != tj && j0 + r < n && i0 + c < n) D[(j0 + r) * n + i0 + c] = sp_finish_value(B[r][c], A[c][r], false);
  }
}

// ------------------------------------------------------------------------------------------- dense -> CSR
// Present (non-zero) entries of a dense float64 matrix, column-sorted, as csr_matrix(K) stores them: one warp per
// row, ballot + popcount give each lane its output position.
__global__ void dense_nnz_kernel(const double* __restrict__ K, int64_t n_rows, int64_t n_cols, int32_t* cnt) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int lane = threadIdx.x & 31;
  int c = 0;
  for (int64_t j0 = 0; j0 < n_cols; j0 += 32) {
    const bool nz = j0 + lane < n_cols && K[row * n_cols + j0 + lane] != 0.0;
    c += __popc(__ballot_sync(0xffffffffu, nz));
  }
  if (lane == 0) cnt[row] = c;
}

__global__ void dense_fill_kernel(const double* __restrict__ K, int64_t n_rows, int64_t n_cols,
                                  const int64_t* __restrict__ indptr, int32_t* __restrict__ idx,
                                  double* __restrict__ val) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int lane = threadIdx.x & 31;
  int64_t pos = indptr[row];
  for (int64_t j0 = 0; j0 < n_cols; j0 += 32) {
    const int64_t j = j0 + lane;
    const double x = j < n_cols ? K[row * n_cols + j] : 0.0;
    const uint32_t bal = __ballot_sync(0xffffffffu, x != 0.0);
    if (x != 0.0) {
      const int64_t q = pos + __popc(bal & ((1u << lane) - 1u));
      idx[q] = (int32_t)j;
      val[q] = x;
    }
    pos += __popc(bal);
  }
}

}  // namespace

extern "C" int gtb_dense_to_csr_count(const double* K, int64_t n_rows, int64_t n_cols, int32_t* cnt, void* stream) {
  GTB_CHECK_ARG(n_rows > 0 && n_cols > 0, "bad shape");
  dense_nnz_kernel<<<(unsigned)gtb_cdiv(n_rows, 8), 256, 0, (cudaStream_t)stream>>>(K, n_rows, n_cols, cnt);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_dense_to_csr_fill(const double* K, int64_t n_rows, int64_t n_cols, const int64_t* indptr,
                                     int32_t* idx, double* val, void* stream) {
  GTB_CHECK_ARG(n_rows > 0 && n_cols > 0, "bad shape");
  dense_fill_kernel<<<(unsigned)gtb_cdiv(n_rows, 8), 256, 0, (cudaStream_t)stream>>>(K, n_rows, n_cols, indptr, idx,
                                                                                       val);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_sp_lengths(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n, const void* X,
                              int d, int x_is_f64, int mode, double* len, int32_t* flags, void* stream) {
  GTB_CHECK_ARG(n > 0 && mode >= 0 && mode <= 2, "bad shape or mode");
  GTB_CHECK_ARG(mode != 1 || (X != nullptr && d > 0), "data lengths need the data rows");
  const unsigned grid = (unsigned)gtb_cdiv(n, 8);
  cudaStream_t st = (cudaStream_t)stream;
  if (x_is_f64)
    lengths_kernel<double><<<grid, 256, 0, st>>>(indptr, idx, val, n, (const double*)X, d, mode, len, flags);
  else
    lengths_kernel<float><<<grid, 256, 0, st>>>(indptr, idx, val, n, (const float*)X, d, mode, len, flags);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_sp_components(const int64_t* indptr, const int32_t* idx, int64_t n, int32_t* label, void* stream) {
  GTB_CHECK_ARG(n > 0 && n < INT32_MAX, "bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)gtb_cdiv(n, 256);
  cc_init_kernel<<<grid, 256, 0, st>>>(label, n);
  cc_hook_kernel<<<grid, 256, 0, st>>>(indptr, idx, n, label);
  cc_compress_kernel<<<grid, 256, 0, st>>>(label, n);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int64_t gtb_sp_ws_bytes(int64_t n, int batch) {
  const int64_t nch = (batch + 31) / 32;
  return 16 * n * nch + 64;
}

extern "C" int gtb_sp_traverse(const int64_t* indptr, const int32_t* idx, const double* len, int64_t n,
                               const int32_t* src, int nb, int batch, double* dist, void* ws, void* stream) {
  GTB_CHECK_ARG(n > 0 && n < INT32_MAX / ((batch + 31) / 32 + 1), "bad shape");
  GTB_CHECK_ARG(nb > 0 && nb <= batch && batch % 32 == 0 && batch <= SP_MAX_BATCH, "bad batch");
  int nch = batch / 32;
  uint32_t* mask0 = (uint32_t*)ws;
  uint32_t* mask1 = mask0 + n * nch;
  int32_t* list0 = (int32_t*)(mask1 + n * nch);
  int32_t* list1 = list0 + n * nch;
  int32_t* cnt = list1 + n * nch;
  int dev = 0, sms = 0, per_sm = 0;
  GTB_CUDA(cudaGetDevice(&dev));
  GTB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  GTB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sp_traverse_kernel, SP_THREADS, 0));
  GTB_CHECK_ARG(per_sm > 0, "traversal kernel does not fit on an SM");
  void* args[] = {(void*)&indptr, (void*)&idx, (void*)&len, (void*)&n, (void*)&src, (void*)&nb, (void*)&dist,
                  (void*)&nch, (void*)&mask0, (void*)&mask1, (void*)&list0, (void*)&list1, (void*)&cnt};
  GTB_CUDA(cudaLaunchCooperativeKernel((const void*)sp_traverse_kernel, dim3(sms * per_sm), dim3(SP_THREADS), args, 0,
                                       (cudaStream_t)stream));
  return GTB_OK;
}

extern "C" int gtb_sp_store_rows(const double* dist, int batch, int64_t n, const int32_t* src, int nb, double* out,
                                 int64_t ldo, void* stream) {
  GTB_CHECK_ARG(n > 0 && nb > 0 && nb <= batch && ldo >= n, "bad shape");
  sp_store_rows_kernel<<<dim3((unsigned)gtb_cdiv(n, 32), (unsigned)gtb_cdiv(nb, 32)), dim3(32, 8), 0,
                         (cudaStream_t)stream>>>(dist, batch, n, src, nb, out, ldo);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_sp_finish(double* D, int64_t n, void* stream) {
  GTB_CHECK_ARG(n > 0, "bad shape");
  const unsigned t = (unsigned)gtb_cdiv(n, 32);
  sp_finish_kernel<<<dim3(t, t), dim3(32, 8), 0, (cudaStream_t)stream>>>(D, n);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}
