// K1/K2 (tensor-core variant): pairwise squared distances on the 5th-gen tensor cores with the
// per-query selection fused into the TMEM epilogue -- the N x N matrix never leaves the SM.
//
//   d~2(i,j) - |x_i|^2  =  |y_j|^2 - 2 x_i.y_j  =  sum_k A[i,k] * B[j,k]
//       A (query role) = [ x~_1 .. x~_d , 1 , 0.. ]        B (ref role) = [ -2y~_1 .. -2y~_d , |y~|^2 , 0.. ]
//
// Every float32 operand value v is split v = hi + lo and the tile is accumulated into a float32 TMEM accumulator, in one
// of three flavours (template FMT):
//   0  3xTF32  hi = tf32(v), lo = tf32(v - hi), kind::tf32, 8 elements per 32-byte k-step, A_hi.B_hi + A_hi.B_lo + A_lo.B_hi
//   1  bf16x3  hi = bf16(v), lo = bf16(v - hi), kind::f16, 16 per k-step, the same three products (>= 16 mantissa bits)
//   2  fp16x2  hi = fp16(s v), lo = fp16(s v - hi) with a power-of-two scale s that brings the data into fp16 range;
//              TWO products A_hi.B_hi + A_hi.B_lo: the reference operand keeps 22 bits, the query operand 11, so the
//              dropped term A_lo.B is bounded by 2^-11 sum|a||b| -- two thirds of the tensor work of the other flavours
//              for a wider (but still certified) rounding bound.
//   3  fp16x1  the same float16 hi arrays, ONE product A_hi.B_hi (the low part of |y|^2 rides in a spare K column, so
//              only the rounding of the coordinates remains: 2^-10 (|x|^2 + |y|^2)) -- half the tensor work again.
//              Top-k only, two query tiles per CTA, one list of 64 per row; the per-row threshold can be SEEDED from
//              a sweep over every tile_stride-th reference tile, which removes most of the threshold-update hits.
// All of them are only used to SELECT candidates; every value that reaches the output is re-evaluated in float64 by
// refine.cu, and rows whose candidate list cannot be certified against the flavour's bound take the radius pass.
//
// CTA = 128 query rows (UMMA M=128, cta_group::1), persistent: cluster c sweeps the whole reference set once per
// round for its next pair of query tiles.  The query tile (A_hi, A_lo) lives in TENSOR MEMORY for the whole sweep
// (tcgen05.st by the epilogue warps; the MMA reads A from TMEM, so shared-memory bandwidth is spent on B only);
// reference tiles of 128 rows (B_hi, B_lo) stream through a 3-stage (bf16) / 2-stage (tf32) TMA ring, multicast to
// the CTAs of the cluster; a ring of three (bf16) / two (tf32) 128-column TMEM accumulators lets the epilogue of
// tile t overlap the MMAs of tiles t+1, t+2.  Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM
// alloc), warps 2-9 = two epilogue groups of four (tcgen05.ld 32x32b: thread == query row), alternating tiles.
// Shared-memory B tiles are K-major: SWIZZLE_128B blocks of four k-steps, then SWIZZLE_32B tail blocks.
//
// Epilogue, TOPK mode: each thread keeps a running threshold; per 32-column batch a 3-input-min tree and one
// ballot decide whether any row of the warp has a value under its threshold.  Hits are appended to the row's
// 96-slot candidate buffer in global memory (L2 resident) -- rows served one at a time by the whole warp, or by
// per-lane predicated stores when many rows hit; a buffer that nears capacity is compacted to its LS smallest by
// a warp-cooperative quickselect on 64-bit ordered keys (ballots and popcounts only) and the threshold tightens.
// RADIUS mode: values under the row's limit are appended to the global pair list.
//
// Replaces sklearn ArgKmin / RadiusNeighbors behind knn_tree.kneighbors / radius_neighbors
// (reference graphtools/graphs.py:883, :922, :957, :966).
#include "common.cuh"
#include "gtb200.h"
#include "tc_ptx.cuh"
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace {

#ifndef GTB_TC_CAP
#define GTB_TC_CAP 96
#endif
#ifndef GTB_TC_HYBRID
#define GTB_TC_HYBRID 4     // hot rows per batch from which the append switches to per-lane predicated stores (0 = never)
#endif
constexpr int TC_M = 128, TC_N = 128, TC_CAP = GTB_TC_CAP, TC_S = 32, TC_GROUPS = 2, TC_THREADS = 64 + 128 * TC_GROUPS;
static_assert(TC_CAP % 32 == 0 && TC_CAP >= TC_S + 64 && TC_CAP <= 128, "candidate buffer: TC_S kept + two batches of 32");
constexpr float TC_BIG = 1e29f;       // "no threshold yet"; padded reference rows carry |y|^2 = 1e30
constexpr float TC_PAD_NORM = 1e30f;
// fp16 operands: the scaled data keeps |y|^2 <= 2^13, so every real value |y|^2 - 2 x.y stays below 3 * 2^13 < TC_BIG_H,
// and padded reference rows (|y|^2 = TC_PAD_NORM_H, the rest zero) never pass the initial threshold
constexpr float TC_BIG_H = 50000.f;
constexpr float TC_PAD_NORM_H = 60000.f;
constexpr float TC_H_MAXNORM = 8192.f;
constexpr int64_t TC_SPLIT_ROWS_MAX = 40 * 4 * 128;   // rows of a piece launch: at most half of the (<= 80) clusters x 4 tiles
#ifndef GTB_TC_SEED_K
#define GTB_TC_SEED_K 8
#endif
constexpr int TC_SEED_K = GTB_TC_SEED_K;   // SEED mode: order statistic of the sampled tile minima that becomes the threshold

using namespace gtbptx;

struct TcParams {
  int64_t nq, nq_pad, nr, nr_pad;
  int nks;                                                 // 32-byte k-steps per operand row
  int64_t nrounds;
  int64_t n_qclusters, tiles_per_split;                    // RADIUS with few query tiles: the reference range is split over CTAs
  unsigned int* sync_ctr;                                  // grid-wide pacing counter (zeroed per launch)
  int64_t tile_stride;                                     // TOPK: sweep every tile_stride-th reference tile (1 = all)
  const float* seed_tau;                                   // TOPK: optional per-row initial threshold, layout of `tau`
  // TOPK, one-product flavour: a last round with work for at most half of the clusters runs as a SECOND launch of
  // split_k pieces of the reference range per cluster-unit (the static n_qclusters / tiles_per_split mapping of the
  // RADIUS launches); the piece lists land in piece_buf / piece_meta (piece-major, split_rows rows from split_row0)
  // and merge_pieces_kernel builds the rows.  split_k = 0: ordinary launch.  q_unit0: first cluster-unit of the launch.
  int64_t q_unit0, split_k, split_row0, split_rows;
  uint2* piece_buf; uint2* piece_meta;
  // TOPK, listed (gtb_knn_topk_tc_seeded with tile lists): unit u = the CL x QT query tiles one cluster sweeps in a round,
  // rows [u * CL * QT * 128, ...); it visits the reference tiles unit_tiles[unit_ptr[u] .. unit_ptr[u + 1]) only.  Round r
  // of cluster c takes slot r * n_clusters + c (c mirrored in odd rounds) of unit_order, longest list first.
  const int64_t* unit_ptr; const int32_t* unit_tiles; const int32_t* unit_order; int64_t n_units;
  const float* qn2;
  int32_t* cand_idx; uint2* cand_buf; float* tau;          // TOPK: out [nq][2*TC_S], scratch [nq_pad][2][TC_CAP], tau [nq][2]
  const float* lim2; int2* pairs; unsigned long long capacity; unsigned long long* counter; int32_t* rowcnt;
};

// ---------------------------------------------------------------- warp-cooperative compaction
// order-preserving map float -> uint32 (and back): a < b  <=>  f2ord(a) < f2ord(b)
__device__ __forceinline__ uint32_t f2ord(uint32_t bits) {
  return bits ^ ((uint32_t)((int32_t)bits >> 31) | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u ^ 0x80000000u) : ~u);
}

// Compact one candidate buffer (<= TC_CAP (value, index) pairs owned by one row): keep the LS smallest and
// return the LS-th smallest value (the row's new threshold), uniform across the warp.
//
// Selection instead of sorting: every pair becomes one unique 64-bit key (ordered value bits : index), held
// TC_CAP/32 per lane; a warp-cooperative quickselect narrows (lo, hi) around the LS-th smallest key with one
// pivot per step -- 64-bit compares, ballots and popcounts only, no data movement and no divergent branches
// (the register bitonic sort this replaces compiled to ~100 shuffle stages of branchy compare-swaps, ~10k cycles
// per call).  The survivors are written back in ballot-prefix order.
template <int LS, int CAP>
__device__ __noinline__ float compact_row(uint2* buf, int cnt, int lane) {
  constexpr int NSLOT = CAP / 32;
  constexpr unsigned long long NONE = ~0ull;
  uint2 t[NSLOT];
  unsigned long long key[NSLOT];
#pragma unroll
  for (int i = 0; i < NSLOT; ++i) {
    const int e = i * 32 + lane;
    t[i] = make_uint2(0u, 0u);
    key[i] = NONE;
    if (e < cnt) {
      t[i] = buf[e];
      key[i] = ((unsigned long long)f2ord(t[i].x) << 32) | (unsigned long long)t[i].y;
    }
  }
  unsigned long long lo = 0ull, hi = NONE, T = NONE;    // the LS-th smallest key lies strictly inside (lo, hi)
  for (int iter = 0; iter < CAP + 1; ++iter) {
    // pivot = an element still inside the interval; slot and end of the lane scan rotate with the step so that no
    // arrival order of the buffer is systematically bad
    unsigned m[NSLOT];
#pragma unroll
    for (int i = 0; i < NSLOT; ++i) m[i] = __ballot_sync(0xffffffffu, key[i] > lo && key[i] < hi);
    unsigned long long cand = 0ull;
    unsigned mm = 0u;
#pragma unroll
    for (int i = 0; i < NSLOT; ++i) {
      const int sl = (i + iter) % NSLOT;                 // iter is warp-uniform; first non-empty slot in rotated order
      unsigned long long ks = key[0];
      unsigned ms = m[0];
#pragma unroll
      for (int q = 1; q < NSLOT; ++q) { if (sl == q) { ks = key[q]; ms = m[q]; } }   // static indexing only
      if (mm == 0u && ms != 0u) { cand = ks; mm = ms; }
    }
    if (mm == 0u) break;                                  // cannot happen while cnt >= LS
    const int src = (iter & 2) ? (31 - __clz(mm)) : (__ffs(mm) - 1);
    const unsigned long long pv = __shfl_sync(0xffffffffu, cand, src);
    int c = 0;
#pragma unroll
    for (int i = 0; i < NSLOT; ++i) c += __popc(__ballot_sync(0xffffffffu, key[i] < pv));
    if (c == LS - 1) { T = pv; break; }
    if (c >= LS) hi = pv; else lo = pv;
  }
  int base = 0;
  const unsigned lt = (1u << lane) - 1u;
#pragma unroll
  for (int i = 0; i < NSLOT; ++i) {
    const bool keep = key[i] <= T;
    const unsigned km = __ballot_sync(0xffffffffu, keep);
    if (keep) buf[base + __popc(km & lt)] = t[i];
    base += __popc(km);
  }
  return ord2f((uint32_t)(T >> 32));
}

// minimum of 32 accumulator values as a balanced tree of 3-input minima (depth 4)
__device__ __forceinline__ float tmin32(const uint32_t (&r)[32]) {
  float b[11];
#pragma unroll
  for (int i = 0; i < 10; ++i)
    b[i] = fminf(fminf(__uint_as_float(r[3 * i]), __uint_as_float(r[3 * i + 1])), __uint_as_float(r[3 * i + 2]));
  b[10] = fminf(__uint_as_float(r[30]), __uint_as_float(r[31]));
  const float c0 = fminf(fminf(b[0], b[1]), b[2]), c1 = fminf(fminf(b[3], b[4]), b[5]);
  const float c2 = fminf(fminf(b[6], b[7]), b[8]), c3 = fminf(b[9], b[10]);
  return fminf(fminf(fminf(c0, c1), c2), c3);
}

// ---------------------------------------------------------------- the kernel
// TMEM column map (512 columns allocated): [0, 8*nks) A_hi, [8*nks, 16*nks) A_lo, then the accumulator
// ring [ACC0 + a*TC_N, +TC_N): tf32 (nks <= 13) ACC0 = 256, 2 accumulators; bf16 (nks <= 8) ACC0 = 128, 3.
constexpr int TC_SYNC_EVERY = 128;   // tiles between grid-wide pacing points of the TMA producers

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float4& a, const float4& b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(__float_as_uint(a.x)), "r"(__float_as_uint(a.y)), "r"(__float_as_uint(a.z)),
               "r"(__float_as_uint(a.w)), "r"(__float_as_uint(b.x)), "r"(__float_as_uint(b.y)),
               "r"(__float_as_uint(b.z)), "r"(__float_as_uint(b.w))
               : "memory");
}
// CL = thread-block cluster size: the CL CTAs of a cluster sweep the same reference tiles for CL different
// query tiles; each loads 1/CL of every B stage and TMA-multicasts it to all of them, so the L2 -> SM
// traffic per output drops by CL.  A stage is recycled once every CTA's MMAs have retired (commit
// multicast to all empty barriers).
// Predicated forms: issued from warp-uniform control flow with the election folded into the instruction
// predicate, so there is no divergent region (BSSY/BSYNC) around the MMAs at all.
__device__ __forceinline__ void tc_mma_ts_pred(bool bf16, uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc,
                                               uint32_t idesc, uint32_t accumulate, uint32_t leader) {
  if (bf16) {
    asm volatile(
        "{\n .reg .pred p, q;\n setp.ne.b32 p, %4, 0;\n setp.ne.b32 q, %5, 0;\n"
        " @q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
  } else {
    asm volatile(
        "{\n .reg .pred p, q;\n setp.ne.b32 p, %4, 0;\n setp.ne.b32 q, %5, 0;\n"
        " @q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
  }
}
__device__ __forceinline__ void tc_commit_pred(uint32_t bar, uint32_t leader) {
  asm volatile(
      "{\n .reg .pred q;\n setp.ne.b32 q, %1, 0;\n"
      " @q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n}"
      ::"r"(bar), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tc_commit_mc_pred(uint32_t bar, uint16_t mask, uint32_t leader) {
  asm volatile(
      "{\n .reg .pred q;\n setp.ne.b32 q, %2, 0;\n"
      " @q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n}"
      ::"r"(bar), "h"(mask), "r"(leader)
      : "memory");
}

// FMT 0: operands are tf32 hi/lo float32 pairs (3xTF32, kind::tf32, 8 elements per 32-byte k-step);
// FMT 1: bfloat16 hi/lo pairs (bf16x3, kind::f16, 16 elements per k-step, twice the MMA rate);
// FMT 2: float16 hi/lo pairs, two products (fp16x2, kind::f16).
// QT: query tiles per CTA.  QT = 1: the two epilogue groups alternate over the reference tiles of ONE query tile (two
// candidate lists of LS per row, over disjoint halves of the reference set).  QT = 2 (fp16x2 only: its query operand
// needs a single 64-column TMEM slice per tile): every reference stage is multiplied against TWO resident query tiles,
// epilogue group g owning query tile g and ONE list of 2 LS entries per row -- each byte streamed from L2 feeds twice
// the tensor work.  (The L2 -> SM path, ~6300 B/clk chip-wide, is what bounds a single-tile sweep once the MMA work
// drops to two products: 57 KB per stage and SM = 1340 clk against 896 clk of MMAs.)
// PIECE: the second launch of a split top-k sweep (own instantiation: the ordinary sweep sits exactly at the register
// budget ptxas grants this kernel, and one more live value in its epilogue costs 13 % of the sweep)
// LISTED: the pruned one-product top-k sweep -- every unit sweeps its own list of reference tiles (TcParams::unit_ptr);
// no grid-wide pacing (the units do not stream the same tiles) and no split last round
// WIDE: operand rows longer than 8 k-steps (129 .. 512 float16 elements, i.e. d up to 510): the query tile still
// lives in TMEM (hi parts only: 8 columns per k-step, up to 256 columns beside two accumulators), the reference tiles
// stream in CHUNKS of 8 k-steps -- a stage is one (tile, chunk) pair and the accumulator collects all chunks of a tile.
template <int MODE, int CL, int FMT, int LS, int QT, bool PIECE = false, bool WIDE = false,   // MODE 0 = TOPK, 1 = RADIUS,
          bool LISTED = false>                                                                   // 2 = SEED
__global__ void __launch_bounds__(TC_THREADS, 1)
search_tc_kernel(const __grid_constant__ CUtensorMap mBh, const __grid_constant__ CUtensorMap mBht,
                 const __grid_constant__ CUtensorMap mBl, const __grid_constant__ CUtensorMap mBlt,
                 const void* __restrict__ q_hi_v, const void* __restrict__ q_lo_v, TcParams p) {
  extern __shared__ unsigned char smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  unsigned char* gbase = smem_raw + (base - raw);

  constexpr bool BF16 = FMT != 0;                            // 2-byte operand elements (bf16 or fp16): kind::f16
  constexpr int NPROD = (FMT == 3) ? 1 : (FMT == 2) ? 2 : 3;  // (A_hi,B_hi)[, (A_hi,B_lo)[, (A_lo,B_hi)]]
  constexpr int NPART = (FMT == 3) ? 1 : 2;                  // operand arrays streamed per stage (hi[, lo])
  constexpr float BIG = (FMT >= 2) ? TC_BIG_H : TC_BIG;
  constexpr int EPK = BF16 ? 16 : 8;                         // elements per 32-byte k-step
  static_assert(QT == 1 || (QT == 2 && FMT >= 2 && MODE != 1), "two query tiles per CTA: fp16 top-k / seed only");
  static_assert(MODE != 2 || (FMT == 3 && QT == 2), "seed sweeps use the one-product flavour");
  static_assert(FMT != 3 || QT == 2, "the one-product flavour runs two query tiles per CTA");
  static_assert(!WIDE || (FMT == 2 && QT == 1 && !PIECE), "wide operand rows: fp16x2, one query tile per CTA");
  static_assert(!LISTED || (MODE == 0 && FMT == 3 && !PIECE && !WIDE), "tile lists: one-product top-k sweep");
  constexpr int LSO = (QT == 2) ? 2 * LS : LS;               // entries of one output list
  // candidate buffer of one list: a row owns TC_GROUPS * TC_CAP slots of scratch; the single long list of QT == 2 may
  // use all of them (fewer compactions between the seeded threshold and the final selection)
  constexpr int CAP = (LSO > 32) ? TC_GROUPS * TC_CAP : TC_CAP;
  static_assert(CAP >= LSO + 64, "room for a list and two batches of 32");
  // burst append (per-lane predicated stores when >= GTB_TC_HYBRID rows of a batch hit): pays off while thresholds
  // are still falling from +inf; the one-product sweep over all tiles starts from seeded thresholds, where bursts do
  // not occur and the extra code only costs instruction-cache misses (188.7 vs 204.3 ms at 1M) -- compiled out there
  constexpr bool HYB = !(FMT == 3 && LS == 32);
  const int nks = p.nks;                                     // 32-byte k-steps per operand row
  const int nfull = nks / 4, ntail = nks % 4;                // SWIZZLE_128B blocks (4 k-steps) + SWIZZLE_32B tail blocks
  const int a_lo_col = nks * 8;                              // TMEM column of A_lo (A_hi at 0)
  const int nch = WIDE ? (nks + 7) / 8 : 1;                  // chunks of 8 k-steps per reference tile (WIDE)
  const uint32_t sizeB = (uint32_t)TC_N * (WIDE ? 8 : nks) * 32;   // one part (hi or lo) of one stage
  const char* q_hi = reinterpret_cast<const char*>(q_hi_v);
  const char* q_lo = reinterpret_cast<const char*>(q_lo_v);
  // shared-memory ring of NS reference stages (3 fit for bf16 operands, 2 for tf32); the two TMEM
  // accumulators form an independent 2-deep ring
  constexpr int NS = BF16 ? (NPART == 1 ? 4 : 3) : 2;
  // TMEM accumulator ring: bf16 query tiles need only 2 x 64 columns, leaving room for three 128-column
  // accumulators (the MMA warp can run two tiles ahead of a busy epilogue group); tf32 has room for two.
  constexpr int NA = (BF16 && !WIDE) ? 3 : 2;
  constexpr int ACC0 = (BF16 && !WIDE) ? 128 : 256;
  const uint32_t B0 = base;                                  // stage s, part q at B0 + (NPART*s+q)*sizeB
  const uint32_t bar0 = B0 + NPART * NS * sizeB;
  const uint32_t bar_a = bar0, full_b = bar0 + 8, empty_b = bar0 + 40, tm_full = bar0 + 72, tm_empty = bar0 + 104;
  const uint32_t round_done = bar0 + 136;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gbase + (bar0 - base) + 144);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Persistent CTAs: cluster c sweeps the whole reference set once per ROUND for the query tiles
  // (c + round * n_clusters) * CL + rank.  All resident CTAs therefore stream the same reference tiles
  // at the same time (one DRAM read per round instead of one per CTA), and odd rounds sweep backwards so
  // the tail of the previous sweep is still in L2.
  // RADIUS launches with fewer query tiles than SMs run one round and split the reference range instead
  // (cluster c = query cluster c % n_qclusters, tile range c / n_qclusters): the output is an append list,
  // so the pieces need no merge.
  const int64_t n_clusters = gridDim.x / CL;
  const int64_t cluster_id = blockIdx.x / CL;
  const int64_t nrounds = p.nrounds;
  const int64_t qcluster = cluster_id % p.n_qclusters;
  const int64_t tile0 = (cluster_id / p.n_qclusters) * p.tiles_per_split;
  const int64_t tstride = (MODE != 1) ? p.tile_stride : 1;
  const int64_t tiles_left = (p.nr_pad / TC_N + tstride - 1) / tstride - tile0;
  const int64_t ntiles = tiles_left < p.tiles_per_split ? tiles_left : p.tiles_per_split;
  // LISTED: the unit of a round (slots past the last unit are padding units: rows beyond nq_pad, no tiles) and its list
  auto unit_of = [&](int64_t round) -> int64_t {
    const int64_t slot = round * n_clusters + ((round & 1) ? (n_clusters - 1 - qcluster) : qcluster);
    return slot < p.n_units ? (int64_t)p.unit_order[slot] : slot;
  };
  auto list_lo = [&](int64_t u) -> int64_t { return u < p.n_units ? p.unit_ptr[u] : 0; };
  auto list_len = [&](int64_t u) -> int64_t { return u < p.n_units ? p.unit_ptr[u + 1] - p.unit_ptr[u] : 0; };
  // first query row of (round, query tile qt of this CTA)
  auto q0_of = [&](int64_t round, int qt) {
    const int64_t u = LISTED ? unit_of(round) : (PIECE ? p.q_unit0 : 0) + qcluster + round * n_clusters;
    return ((u * CL + (blockIdx.x % CL)) * QT + qt) * TC_M;
  };
  static_assert(!PIECE || (MODE == 0 && FMT == 3), "piece launches belong to the one-product top-k sweep");
  auto btile = [&](int64_t round, int64_t t) { return (tile0 + ((round & 1) ? (ntiles - 1 - t) : t)) * tstride; };
  const uint32_t crank = (CL > 1) ? cluster_ctarank() : 0u;
  constexpr uint16_t cmask = (uint16_t)((1u << CL) - 1u);
  constexpr int ROWS = TC_N / CL;                            // rows of each B block this CTA loads

  if (threadIdx.x == 0) {
    mbar_init(bar_a, 4 * QT);
    mbar_init(round_done, 1);
    for (int s = 0; s < NS; ++s) {
      mbar_init(full_b + 8 * s, 1);
      mbar_init(empty_b + 8 * s, CL);
    }
    for (int s = 0; s < NA; ++s) {
      mbar_init(tm_full + 8 * s, 1);
      mbar_init(tm_empty + 8 * s, 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();               // peers' barriers are initialised before any remote signal
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 && WIDE) {
    // ===================== TMA producer, chunked rows =====================
    if (lane == 0) {
      int64_t it = 0, sit = 0;                     // running tile / stage counters across rounds
      for (int64_t round = 0; round < nrounds; ++round) {
        for (int64_t t = 0; t < ntiles; ++t, ++it) {
          if (p.sync_ctr != nullptr && (it % TC_SYNC_EVERY) == 0) {
            const unsigned int target = (unsigned int)(it / TC_SYNC_EVERY + 1) * gridDim.x;
            atomicAdd(p.sync_ctr, 1u);
            for (int polls = 0; polls < (1 << 16); ++polls) {
              unsigned int seen;
              asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(p.sync_ctr) : "memory");
              if (seen >= target) break;
              __nanosleep(64);
            }
          }
          const int row0 = (int)(btile(round, t) * TC_N) + (int)crank * ROWS;
          for (int c = 0; c < nch; ++c, ++sit) {
            const int s = (int)(sit % NS);
            const uint32_t ph = (uint32_t)((sit / NS) & 1);
            const int nk = (nks - 8 * c) < 8 ? (nks - 8 * c) : 8;      // k-steps of this chunk
            const int nf = nk / 4, nt2 = nk % 4;
            mbar_wait(empty_b + 8 * s, ph ^ 1);
            mbar_arrive_expect_tx(full_b + 8 * s, (uint32_t)(NPART * TC_N * nk * 32));
            for (int part = 0; part < NPART; ++part) {
              const CUtensorMap* mm = part ? &mBl : &mBh;
              const CUtensorMap* mt = part ? &mBlt : &mBht;
              const uint32_t dst = B0 + (NPART * s + part) * sizeB;
              for (int b = 0; b < nf; ++b) {
                const uint32_t d = dst + b * (TC_N * 128) + crank * (ROWS * 128);
                if (CL > 1) tma_load_2d_mc(d, mm, full_b + 8 * s, (c * 8 + b * 4) * EPK, row0, cmask);
                else tma_load_2d(d, mm, full_b + 8 * s, (c * 8 + b * 4) * EPK, row0);
              }
              for (int t2 = 0; t2 < nt2; ++t2) {
                const uint32_t d = dst + nf * (TC_N * 128) + t2 * (TC_N * 32) + crank * (ROWS * 32);
                if (CL > 1) tma_load_2d_mc(d, mt, full_b + 8 * s, (c * 8 + nf * 4 + t2) * EPK, row0, cmask);
                else tma_load_2d(d, mt, full_b + 8 * s, (c * 8 + nf * 4 + t2) * EPK, row0);
              }
            }
          }
        }
      }
    }
  } else if (warp == 1 && WIDE) {
    // ===================== MMA issuer, chunked rows =====================
    const bool leader = elect_one();
    const uint32_t lead = leader ? 1u : 0u;
    constexpr uint32_t fmt = (FMT == 0) ? 2u : (FMT == 1 ? 1u : 0u);
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(TC_N >> 3) << 17) |
                           ((uint32_t)(TC_M >> 4) << 24);
    const uint64_t bd_main0 = make_desc(B0, 1024, 2);
    const uint32_t part_off = sizeB >> 4, stage_off = (NPART * sizeB) >> 4;
    int64_t it = 0, sit = 0;
    for (int64_t round = 0; round < nrounds; ++round) {
      mbar_wait(bar_a, (uint32_t)(round & 1));
      tc_fence_after();
      for (int64_t tile = 0; tile < ntiles; ++tile, ++it) {
        const int ac_i = (int)(it % NA);
        const uint32_t aph = (uint32_t)((it / NA) & 1);
        mbar_wait(tm_empty + 8 * ac_i, aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(ACC0 + ac_i * TC_N);
        uint32_t accum = 0;
#pragma unroll 1
        for (int c = 0; c < nch; ++c, ++sit) {
          const int s = (int)(sit % NS);
          const uint32_t ph = (uint32_t)((sit / NS) & 1);
          const int nk = (nks - 8 * c) < 8 ? (nks - 8 * c) : 8;
          const int nf = nk / 4, nt2 = nk % 4;
          mbar_wait(full_b + 8 * s, ph);
          tc_fence_after();
          const uint64_t bd_tail0 = make_desc(B0 + nf * (TC_N * 128), 256, 6);
#pragma unroll 1
          for (int prod = 0; prod < NPROD; ++prod) {   // (A_hi,B_hi), (A_hi,B_lo)
            uint32_t ac = tmem_base + (uint32_t)(c * 64);
            const uint64_t boff = (uint64_t)(s * stage_off + ((prod == 1) ? part_off : 0u));
            uint64_t bd = bd_main0 + boff;
#pragma unroll 1
            for (int blk = 0; blk < nf; ++blk) {
#pragma unroll
              for (int sub = 0; sub < 4; ++sub) {
                tc_mma_ts_pred(BF16, d_tmem, ac + sub * 8, bd + sub * 2, idesc, accum, lead);
                accum = 1;
              }
              bd += (TC_N * 128) >> 4;
              ac += 32;
            }
            bd = bd_tail0 + boff;
#pragma unroll 1
            for (int t = 0; t < nt2; ++t) {
              tc_mma_ts_pred(BF16, d_tmem, ac, bd, idesc, accum, lead);
              accum = 1;
              bd += (TC_N * 32) >> 4;
              ac += 8;
            }
          }
          if (CL > 1) tc_commit_mc_pred(empty_b + 8 * s, cmask, lead);
          else tc_commit_pred(empty_b + 8 * s, lead);
        }
        tc_commit_pred(tm_full + 8 * ac_i, lead);
      }
      tc_commit_pred(round_done, lead);
    }
  } else if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int64_t it = 0;                              // running stage counter across rounds
      for (int64_t round = 0; round < nrounds; ++round) {
        int64_t nt = ntiles, lo = 0;
        if (LISTED) { const int64_t u = unit_of(round); lo = list_lo(u); nt = list_len(u); }
        for (int64_t t = 0; t < nt; ++t, ++it) {
          const int s = (int)(it % NS);
          const uint32_t ph = (uint32_t)((it / NS) & 1);
          if (p.sync_ctr != nullptr && (it % TC_SYNC_EVERY) == 0) {
            // Pace the reference stream grid-wide: all producers enter tile `it` together, so one DRAM read
            // of a reference tile serves every SM out of L2 (without this the 74 clusters drift apart by more
            // than the 126 MB L2 window and each streams the operand from DRAM on its own: 2.1 TB instead of
            // 44 GB per sweep set).  Performance only -- the wait is bounded, never a correctness dependency.
            const unsigned int target = (unsigned int)(it / TC_SYNC_EVERY + 1) * gridDim.x;
            atomicAdd(p.sync_ctr, 1u);
            for (int polls = 0; polls < (1 << 16); ++polls) {
              unsigned int seen;
              asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(p.sync_ctr) : "memory");
              if (seen >= target) break;
              __nanosleep(64);
            }
          }
          mbar_wait(empty_b + 8 * s, ph ^ 1);      // every CTA of the cluster has consumed this stage
          mbar_arrive_expect_tx(full_b + 8 * s, NPART * sizeB);
          const int64_t tile = LISTED ? (int64_t)p.unit_tiles[lo + t] : btile(round, t);
          const int row0 = (int)(tile * TC_N) + (int)crank * ROWS;
          for (int part = 0; part < NPART; ++part) {
            const CUtensorMap* mm = part ? &mBl : &mBh;
            const CUtensorMap* mt = part ? &mBlt : &mBht;
            const uint32_t dst = B0 + (NPART * s + part) * sizeB;
            for (int b = 0; b < nfull; ++b) {
              const uint32_t d = dst + b * (TC_N * 128) + crank * (ROWS * 128);
              if (CL > 1) tma_load_2d_mc(d, mm, full_b + 8 * s, b * 4 * EPK, row0, cmask);
              else tma_load_2d(d, mm, full_b + 8 * s, b * 4 * EPK, row0);
            }
            for (int t2 = 0; t2 < ntail; ++t2) {
              const uint32_t d = dst + nfull * (TC_N * 128) + t2 * (TC_N * 32) + crank * (ROWS * 32);
              if (CL > 1) tma_load_2d_mc(d, mt, full_b + 8 * s, (nfull * 4 + t2) * EPK, row0, cmask);
              else tma_load_2d(d, mt, full_b + 8 * s, (nfull * 4 + t2) * EPK, row0);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The whole warp runs this loop in uniform control flow so that every MMA operand (descriptors,
    // TMEM addresses) is computed on the uniform datapath; only the tcgen05 instructions themselves
    // are predicated on the elected lane.  (Issuing from inside an `if (lane == 0)` region costs ~18
    // SASS instructions per MMA -- R2UR + an ELECT loop -- and left the tensor pipe 3/4 idle.)
    const bool leader = elect_one();
    // instruction descriptor: D=f32, A=B=tf32 (2, kind::tf32) / bf16 (1) / f16 (0, both kind::f16), K-major, N=TC_N, M=128
    constexpr uint32_t fmt = (FMT == 0) ? 2u : (FMT == 1 ? 1u : 0u);
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(TC_N >> 3) << 17) |
                           ((uint32_t)(TC_M >> 4) << 24);
    const uint64_t bd_main0 = make_desc(B0, 1024, 2);                          // stage 0, hi part, block 0
    const uint64_t bd_tail0 = make_desc(B0 + nfull * (TC_N * 128), 256, 6);    // stage 0, hi part, first tail block
    const uint32_t part_off = sizeB >> 4, stage_off = (NPART * sizeB) >> 4;     // in descriptor address units (16 B)
    int64_t it = 0;
    for (int64_t round = 0; round < nrounds; ++round) {
    mbar_wait(bar_a, (uint32_t)(round & 1));   // this round's A rows stored to TMEM by the epilogue warps
    tc_fence_after();
    const int64_t nt = LISTED ? list_len(unit_of(round)) : ntiles;
    for (int64_t tile = 0; tile < nt; ++tile, ++it) {
      const int s = (int)(it % NS);            // shared-memory stage
      const uint32_t ph = (uint32_t)((it / NS) & 1);
      mbar_wait(full_b + 8 * s, ph);
      const uint32_t lead = leader ? 1u : 0u;
#pragma unroll 1
      for (int qt = 0; qt < QT; ++qt) {
      const int64_t ait = it * QT + qt;        // running accumulator index
      const int ac_i = (int)(ait % NA);        // TMEM accumulator
      const uint32_t aph = (uint32_t)((ait / NA) & 1);
      mbar_wait(tm_empty + 8 * ac_i, aph ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(ACC0 + ac_i * TC_N);
      uint32_t accum = 0;
#pragma unroll 1
      for (int prod = 0; prod < NPROD; ++prod) {   // (A_hi,B_hi), (A_hi,B_lo), (A_lo,B_hi)
        uint32_t ac = tmem_base + (uint32_t)((prod == 2) ? a_lo_col : 0) + (uint32_t)(qt * 64);
        const uint64_t boff = (uint64_t)(s * stage_off + ((prod == 1) ? part_off : 0u));
        uint64_t bd = bd_main0 + boff;
#pragma unroll 1
        for (int blk = 0; blk < nfull; ++blk) {
#pragma unroll
          for (int sub = 0; sub < 4; ++sub) {
            tc_mma_ts_pred(BF16, d_tmem, ac + sub * 8, bd + sub * 2, idesc, accum, lead);
            accum = 1;
          }
          bd += (TC_N * 128) >> 4;
          ac += 32;
        }
        bd = bd_tail0 + boff;
#pragma unroll 1
        for (int t = 0; t < ntail; ++t) {
          tc_mma_ts_pred(BF16, d_tmem, ac, bd, idesc, accum, lead);
          accum = 1;
          bd += (TC_N * 32) >> 4;
          ac += 8;
        }
      }
      tc_commit_pred(tm_full + 8 * ac_i, lead);   // accumulator ready for the epilogue
      }
      // smem stage free once these MMAs retire -- signalled to every CTA that multicasts into it
      if (CL > 1) tc_commit_mc_pred(empty_b + 8 * s, cmask, lead);
      else tc_commit_pred(empty_b + 8 * s, lead);
    }
    tc_commit_pred(round_done, leader ? 1u : 0u);   // every MMA that reads this round's A has retired
    }
  } else {
    // ===================== epilogue warps =====================
    // Two groups of four warps: group g owns accumulator g, i.e. the reference tiles with tile % 2 == g,
    // and keeps its own per-row threshold and candidate buffer (no state shared between groups; two
    // epilogue warps per SM sub-partition hide each other's latencies).  The refine stage merges the two
    // lists; every non-candidate of group g has approximate d2 >= tau[row][g].
    const int quad = warp & 3;                       // TMEM lane quadrant this warp may access
    const int grp = (warp - 2) >> 2;                 // 0 or 1
    float* xpose = reinterpret_cast<float*>(gbase + (bar0 - base) + 256) + (warp - 2) * 32;   // 128-byte slot per warp
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16);
    // QT == 2: group g owns query tile g of this CTA (its A slice at TMEM columns [64 g, 64 g + 8 nks)), sees every
    // reference tile and keeps ONE candidate list of 2 LS entries per row.
    const int my_qt = (QT == 2) ? grp : 0;
    const int lgrp = (QT == 2) ? 0 : grp;            // list index inside a row's candidate storage
    const uint32_t a_col0 = (uint32_t)(my_qt * 64);
    int64_t it_run = 0;                              // LISTED: tiles of the earlier rounds (lists differ in length)
    for (int64_t round = 0; round < nrounds; ++round) {
    int64_t nt = ntiles, lo = 0;
    if (LISTED) { const int64_t u = unit_of(round); lo = list_lo(u); nt = list_len(u); }
    const int64_t q0 = q0_of(round, my_qt);
    const int64_t gq = q0 + row;
    const bool valid = gq < p.nq;

    if (grp == 0 || QT == 2) {
      if (round > 0) { mbar_wait(round_done, (uint32_t)((round - 1) & 1)); tc_fence_after(); }
      // ---- stage the query tile into TMEM: thread == row, one column per K element
      const bool in_pad = gq < p.nq_pad;             // cluster padding CTAs carry all-zero query rows
      const float4* rh = reinterpret_cast<const float4*>(q_hi + (in_pad ? gq : 0) * (int64_t)(nks * 32));
      const float4* rl = reinterpret_cast<const float4*>(q_lo + (in_pad ? gq : 0) * (int64_t)(nks * 32));
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int ks = 0; ks < nks; ++ks) {
        tmem_st8(lane_addr + a_col0 + (uint32_t)(ks * 8), in_pad ? rh[2 * ks] : z4, in_pad ? rh[2 * ks + 1] : z4);
        if (NPROD == 3)
          tmem_st8(lane_addr + (uint32_t)(a_lo_col + ks * 8), in_pad ? rl[2 * ks] : z4, in_pad ? rl[2 * ks + 1] : z4);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_a);
    }

    const float nx = valid ? p.qn2[gq] : 0.f;
    float thr;
    if (MODE == 0) {
      thr = valid ? BIG : -gtb_inf_f();
      if (valid && p.seed_tau != nullptr) {
        // seeded threshold: every reference point under it is appended, the buffer compacts as usual when it fills
        const float t0 = p.seed_tau[gq * TC_GROUPS] - nx;
        if (t0 < BIG) thr = t0;
      }
    } else if (MODE == 1) {
      // capped at BIG: every real value stays below it and every padded reference row above it, so a radius wider
      // than the data (a kernel support beyond all points) cannot admit padded columns j >= nr
      thr = valid ? fminf(p.lim2[gq] - nx, BIG) : -gtb_inf_f();
    } else {
      thr = 0.f;
    }
    // SEED mode: the TC_SEED_K smallest TILE MINIMA of the row, ascending, in registers.  Distinct tiles hold distinct
    // points, so the k-th smallest tile minimum bounds the k-th smallest value from above (and equals it unless two of
    // the k smallest share a tile) -- a threshold estimate that needs no candidate buffer, no hit servicing and no
    // divergent code: one min tree and one 8-deep insertion network per tile.
    float best[TC_SEED_K];
#pragma unroll
    for (int i = 0; i < TC_SEED_K; ++i) best[i] = BIG;
    int cnt = 0;
    // this thread's candidate buffer: uniform base + per-thread offset (rows past nq never append)
    const int64_t boff = valid ? (gq * TC_GROUPS + lgrp) * TC_CAP : 0;     // (CAP > TC_CAP only with lgrp == 0)
    uint2* wbuf = p.cand_buf + (q0 + quad * 32) * TC_GROUPS * TC_CAP;   // warp-uniform: first row of this quadrant
    uint2* mybuf = p.cand_buf + boff;                                     // this row's buffer (never written when !valid)
    if (PIECE) {
      // piece launch: this cluster's piece of the reference range has its own buffers (piece-major, same row stride)
      uint2* pb = p.piece_buf + ((cluster_id / p.n_qclusters) * p.split_rows - p.split_row0) * (TC_GROUPS * TC_CAP);
      wbuf = pb + (q0 + quad * 32) * TC_GROUPS * TC_CAP;
      mybuf = pb + boff;
    }

    // this group's tiles.  QT == 1: running iteration index it = round * ntiles + t with it % 2 == grp; QT == 2:
    // every tile, accumulator index 2 it + grp
    const int64_t it0 = LISTED ? it_run : round * ntiles;
    if (LISTED) it_run += nt;
    for (int64_t t = (QT == 2) ? 0 : ((grp + (it0 & 1)) & 1); t < nt; t += (QT == 2 ? 1 : TC_GROUPS)) {
      const int64_t it = it0 + t;
      const int64_t tile = LISTED ? (int64_t)p.unit_tiles[lo + t] : btile(round, t);
      const int64_t ait = (QT == 2) ? (it * 2 + grp) : it;
      const int s = (int)(ait % NA);                   // accumulator of this iteration
      const uint32_t ph = (uint32_t)((ait / NA) & 1);
      mbar_wait(tm_full + 8 * s, ph);
      tc_fence_after();
      // drain the whole accumulator into registers, hand it back to the MMA warp, THEN select: the
      // accumulator is held for four back-to-back tcgen05.ld only, never across the selection work
      uint32_t r0[32], r1[32], r2[32], r3[32];
      __syncwarp();
      const uint32_t acc_addr = lane_addr + (uint32_t)(ACC0 + s * TC_N);
      tmem_ld32_nowait(acc_addr, r0);
      tmem_ld32_nowait(acc_addr + 32, r1);
      tmem_ld32_nowait(acc_addr + 64, r2);
      tmem_ld32_nowait(acc_addr + 96, r3);
      tmem_wait_ld(r0, r1, r2, r3);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tm_empty + 8 * s);
#ifdef GTB_EXP_NOSELECT
      continue;                                   // experiment build: the sweep without any selection work (DESIGN.md section 4)
#endif
      if (MODE == 2) {
        float v = fminf(fminf(tmin32(r0), tmin32(r1)), fminf(tmin32(r2), tmin32(r3)));
#pragma unroll
        for (int i = 0; i < TC_SEED_K; ++i) {      // sorted insertion: best[] stays ascending, v carries the evicted value
          const float lo = fminf(best[i], v);
          v = fmaxf(best[i], v);
          best[i] = lo;
        }
        continue;
      }
      // Selection.  The minima of the four 32-column batches first -- balanced 3-input trees, four independent
      // chains (a running fminf is a 31-deep dependent chain per batch, and the latency of this stretch is what decides
      // how much hit servicing the accumulator ring can absorb before the MMA warp stalls) -- then one ballot per
      // batch.  A tile in which no row has a qualifying column, the common case, ends at ONE warp-uniform branch.
      const float bm0 = tmin32(r0), bm1 = tmin32(r1), bm2 = tmin32(r2), bm3 = tmin32(r3);
      unsigned h0 = __ballot_sync(0xffffffffu, (MODE == 0) ? (bm0 < thr) : (bm0 <= thr));
      unsigned h1 = __ballot_sync(0xffffffffu, (MODE == 0) ? (bm1 < thr) : (bm1 <= thr));
      unsigned h2 = __ballot_sync(0xffffffffu, (MODE == 0) ? (bm2 < thr) : (bm2 <= thr));
      unsigned h3 = __ballot_sync(0xffffffffu, (MODE == 0) ? (bm3 < thr) : (bm3 <= thr));
#ifdef GTB_EXP_NOSERVICE
      h0 = h1 = h2 = h3 = 0;
#endif
      if ((h0 | h1 | h2 | h3) == 0u) continue;
#pragma unroll
      for (int part = 0; part < TC_N / 32; ++part) {
        // (a compaction in an earlier batch of this tile may have tightened thr since the ballot: the pass test below
        // uses the current threshold, a stale hot bit only costs an empty service)
        unsigned hot = part == 0 ? h0 : part == 1 ? h1 : part == 2 ? h2 : h3;
        if (hot == 0u) continue;
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j)
          v[j] = __uint_as_float(part == 0 ? r0[j] : part == 1 ? r1[j] : part == 2 ? r2[j] : r3[j]);
        const int32_t col0 = (int32_t)(tile * TC_N) + part * 32;
        if (MODE == 0) {
#if GTB_TC_HYBRID > 0
          // Burst regime (round start: most rows hit in every batch): every lane appends its own hits to its own
          // row buffer with predicated stores behind one warp-uniform branch -- a fixed ~130 issue slots instead
          // of ~350 cycles per hot row.  With few hot rows the cooperative path below is cheaper.
          if (HYB && __popc(hot) >= GTB_TC_HYBRID) {
            uint2* wp = mybuf + cnt;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              asm volatile(
                  "{\n .reg .pred p;\n setp.lt.f32 p, %1, %2;\n @p st.global.v2.b32 [%0], {%3, %4};\n"
                  " @p add.u64 %0, %0, 8;\n}"
                  : "+l"(wp)
                  : "f"(v[j]), "f"(thr), "r"(__float_as_uint(v[j])), "r"(col0 + j)
                  : "memory");
            }
            cnt = (int)(wp - mybuf);
            hot = 0;
          }
#endif
        }
        while (hot) {
          const int L = __ffs(hot) - 1;
          hot &= hot - 1;
          if (lane == L) {
            float4* dst4 = reinterpret_cast<float4*>(xpose);
#pragma unroll
            for (int j = 0; j < 8; ++j) dst4[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
          __syncwarp();
          const float x = xpose[lane];
          const float tL = __shfl_sync(0xffffffffu, thr, L);
          const bool pass = (MODE == 0) ? (x < tL) : (x <= tL);
          const unsigned pm = __ballot_sync(0xffffffffu, pass);
          const int npass = __popc(pm);
          const int rank = __popc(pm & ((1u << lane) - 1u));
          if (MODE == 0) {
            const int cL = __shfl_sync(0xffffffffu, cnt, L);
            if (pass) wbuf[(L * TC_GROUPS + lgrp) * TC_CAP + cL + rank] = make_uint2(__float_as_uint(x), (uint32_t)(col0 + lane));
            if (lane == L) cnt += npass;
          } else {
            unsigned long long basepos = 0;
            if (lane == L) {
              basepos = atomicAdd(p.counter, (unsigned long long)npass);
              atomicAdd(p.rowcnt + gq, npass);
            }
            basepos = __shfl_sync(0xffffffffu, basepos, L);
            if (pass && basepos + (unsigned long long)rank < p.capacity)
              p.pairs[basepos + rank] = make_int2((int)(q0 + quad * 32 + L), col0 + lane);
          }
          __syncwarp();
        }
        if (MODE == 0) {
          // keep >= 32 free slots for the next batch
          unsigned need = __ballot_sync(0xffffffffu, cnt > CAP - 32);
          while (need) {
            const int owner = __ffs(need) - 1;
            need &= need - 1;
            const int ocnt = __shfl_sync(0xffffffffu, cnt, owner);
            __syncwarp();
            const float nt = compact_row<LSO, CAP>(wbuf + (owner * TC_GROUPS + lgrp) * TC_CAP, ocnt, lane);
            __syncwarp();
            if (lane == owner) { thr = nt; cnt = LSO; }
          }
        }
      }
    }

    if (MODE == 2) {
      if (valid) {
        const float tv = (best[TC_SEED_K - 1] >= BIG) ? gtb_inf_f() : best[TC_SEED_K - 1] + nx;
        p.tau[gq * TC_GROUPS] = tv;
        p.tau[gq * TC_GROUPS + 1] = tv;
      }
    }
    if (MODE == 0) {
      // final compaction of every buffer still holding more than a list's worth of candidates
      unsigned need = __ballot_sync(0xffffffffu, cnt > LSO);
      while (need) {
        const int owner = __ffs(need) - 1;
        need &= need - 1;
        const int ocnt = __shfl_sync(0xffffffffu, cnt, owner);
        __syncwarp();
        const float nt = compact_row<LSO, CAP>(wbuf + (owner * TC_GROUPS + lgrp) * TC_CAP, ocnt, lane);
        __syncwarp();
        if (lane == owner) { thr = nt; cnt = LSO; }
      }
      __syncwarp();
      if (valid) {
        // QT == 1: two lists of LS per row (one per group) with their own thresholds; QT == 2: one list of 2 LS,
        // the second threshold slot repeats the first (the refine takes the minimum)
        // a list that never filled keeps its initial threshold: +inf unseeded, the seed otherwise (every point under
        // the seed IS in the list)
        const float tv = (thr >= BIG) ? gtb_inf_f() : thr + nx;
        if (PIECE) {
          // piece launch: count and threshold of this piece's list; merge_pieces_kernel builds the row
          p.piece_meta[(cluster_id / p.n_qclusters) * p.split_rows + (gq - p.split_row0)] =
              make_uint2((uint32_t)cnt, __float_as_uint(tv));
        } else {
          int32_t* out = p.cand_idx + gq * (TC_GROUPS * LS) + lgrp * LS;
          for (int e = 0; e < LSO; ++e) out[e] = (e < cnt) ? (int32_t)p.cand_buf[boff + e].y : -1;
          p.tau[gq * TC_GROUPS + lgrp] = tv;
          if (QT == 2) p.tau[gq * TC_GROUPS + 1] = tv;
        }
      }
    }
    }  // rounds
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
  if (CL > 1) cluster_sync_all();               // no CTA exits while a peer may still signal its barriers
}

// ---------------------------------------------------------------- merge of a split last round
// One warp per row of the piece launch: the row's split_k piece lists (<= LS entries each after the piece's final
// compaction) are concatenated in shared memory; if the union exceeds LS entries the LS smallest are selected with the
// same quickselect as in the sweep.  Every point that is not in the result lies above its piece's threshold or above
// the LS-th smallest of the union, so tau = min(piece thresholds, LS-th smallest of the union).
constexpr int TC_SPLIT_MAX = 4, TC_MERGE_WARPS = 4;

template <int LS>
__global__ void __launch_bounds__(TC_MERGE_WARPS * 32) merge_pieces_kernel(TcParams p) {
  constexpr int CAP = TC_GROUPS * TC_CAP, MCAP = TC_SPLIT_MAX * LS;
  __shared__ uint2 stage_s[TC_MERGE_WARPS][MCAP];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t r = (int64_t)blockIdx.x * TC_MERGE_WARPS + warp;
  const int64_t gq = p.split_row0 + r;
  if (r >= p.split_rows || gq >= p.nq) return;               // whole warp
  uint2* stage = stage_s[warp];
  const float nx = p.qn2[gq];
  float tau = gtb_inf_f();
  int total = 0;
  for (int pc = 0; pc < (int)p.split_k; ++pc) {
    const uint2 meta = p.piece_meta[pc * p.split_rows + r];
    const int c = (int)meta.x < LS ? (int)meta.x : LS;
    tau = fminf(tau, __uint_as_float(meta.y));
    const uint2* src = p.piece_buf + (pc * p.split_rows + r) * CAP;
    for (int e = lane; e < c; e += 32) stage[total + e] = src[e];
    total += c;
  }
  __syncwarp();
  if (total > LS) {
    const float t = compact_row<LS, MCAP>(stage, total, lane);
    tau = fminf(tau, t + nx);
    total = LS;
    __syncwarp();
  }
  int32_t* out = p.cand_idx + gq * LS;
  for (int e = lane; e < LS; e += 32) out[e] = (e < total) ? (int32_t)stage[e].y : -1;
  if (lane == 0) { p.tau[gq * TC_GROUPS] = tau; p.tau[gq * TC_GROUPS + 1] = tau; }
}

// ---------------------------------------------------------------- operand preparation (row-major hi/lo)
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

__global__ void tc_norms_kernel(const float* __restrict__ X, int64_t n, int d, const float* __restrict__ mean,
                                int64_t n_pad, float* __restrict__ norm2, float* __restrict__ maxnorm) {
  const int lane = threadIdx.x & 31;
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_pad) return;
  float out = 0.f;
  if (r < n) {
    double s = 0.0;
    for (int k = lane; k < d; k += 32) {
      double v = (double)(X[r * d + k] - (mean ? mean[k] : 0.f));
      s += v * v;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    out = __double2float_ru(s);
  }
  if (lane == 0) {
    norm2[r] = (r < n) ? out : TC_PAD_NORM;
    if (maxnorm && r < n) atomicMax((int*)maxnorm, __float_as_int(out));
  }
}

__global__ void tc_split_kernel(const float* __restrict__ X, int64_t n, int d, const float* __restrict__ mean,
                                int role, const float* __restrict__ norm2, int64_t n_pad, int Kp,
                                float* __restrict__ hi, float* __restrict__ lo) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_pad * Kp) return;
  const int64_t r = e / Kp;
  const int k = (int)(e - r * Kp);
  float v = 0.f;
  if (r < n) {
    if (k < d) {
      v = X[r * d + k] - (mean ? mean[k] : 0.f);
      if (role == 1) v *= -2.f;
    } else if (k == d) {
      v = (role == 1) ? norm2[r] : 1.f;
    }
  } else if (role == 1 && k == d) {
    v = TC_PAD_NORM;
  }
  const float h = to_tf32(v);
  hi[e] = h;
  lo[e] = to_tf32(v - h);
}

__global__ void tc_split16_kernel(const float* __restrict__ X, int64_t n, int d, const float* __restrict__ mean,
                                  int role, const float* __restrict__ norm2, int64_t n_pad, int Kp,
                                  __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_pad * Kp) return;
  const int64_t r = e / Kp;
  const int k = (int)(e - r * Kp);
  float v = 0.f;
  if (r < n) {
    if (k < d) {
      v = X[r * d + k] - (mean ? mean[k] : 0.f);
      if (role == 1) v *= -2.f;
    } else if (k == d) {
      v = (role == 1) ? norm2[r] : 1.f;
    }
  } else if (role == 1 && k == d) {
    v = TC_PAD_NORM;
  }
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[e] = h;
  lo[e] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// fp16 pairs of the scaled data: hi = fp16(s v), lo = fp16(s v - hi); the norm column carries s^2 |y|^2
__global__ void tc_split16h_kernel(const float* __restrict__ X, int64_t n, int d, const float* __restrict__ mean,
                                   int role, const float* __restrict__ norm2, int64_t n_pad, int Kp, float scale,
                                   __half* __restrict__ hi, __half* __restrict__ lo) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_pad * Kp) return;
  const int64_t r = e / Kp;
  const int k = (int)(e - r * Kp);
  float v = 0.f;
  if (r < n) {
    if (k < d) {
      v = (X[r * d + k] - (mean ? mean[k] : 0.f)) * scale;
      if (role == 1) v *= -2.f;
    } else if (k == d) {
      v = (role == 1) ? norm2[r] * scale * scale : 1.f;
    } else if (k == d + 1) {
      // spare column: the low part of |y|^2 rides in the hi array (query side: 1), so the one-product flavour sees
      // |y|^2 to 22 bits as well; the lo array carries nothing for the norm
      if (role == 1) {
        const float nv = norm2[r] * scale * scale;
        v = nv - __half2float(__float2half_rn(nv));
      } else {
        v = 1.f;
      }
    }
  } else if (role == 1 && k == d) {
    v = TC_PAD_NORM_H;
  }
  const __half h = __float2half_rn(v);
  hi[e] = h;
  lo[e] = (k >= d) ? __float2half_rn(0.f) : __float2half_rn(v - __half2float(h));
}

// ---------------------------------------------------------------- host side
// 2-D map over a row-major [rows][Kp] float32 / bfloat16 array; box = {box_k elements, box_rows}
int make_map(CUtensorMap* m, const void* ptr, int64_t rows, int Kp, int box_k, int box_rows, bool sw128, int fmt) {
  const bool bf16 = fmt != 0;
  EncodeTiledFn enc = get_encode();
  if (!enc) { gtb_set_error("cuTensorMapEncodeTiled entry point not available"); return GTB_ERR_CUDA; }
  cuuint64_t dims[2] = {(cuuint64_t)Kp, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)Kp * (bf16 ? 2 : 4)};
  cuuint32_t box[2] = {(cuuint32_t)box_k, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, fmt == 1 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : (fmt >= 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32), 2, (void*)ptr, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { gtb_set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return GTB_ERR_CUDA; }
  return GTB_OK;
}

template <int MODE, int CL, int FMT, int LS, int QT = 1, bool WIDE = false>
int launch_tc_cl(const void* q_hi, const void* q_lo, const void* r_hi, const void* r_lo, int Kp, TcParams& p,
                 cudaStream_t st) {
  CUtensorMap mBh, mBht, mBl, mBlt;
  int rc;
  constexpr bool BF16 = FMT != 0;
  constexpr int EPK = BF16 ? 16 : 8;
  p.nks = Kp / EPK;
  if ((rc = make_map(&mBh, r_hi, p.nr_pad, Kp, 4 * EPK, TC_N / CL, true, FMT))) return rc;
  if ((rc = make_map(&mBht, r_hi, p.nr_pad, Kp, EPK, TC_N / CL, false, FMT))) return rc;
  if ((rc = make_map(&mBl, r_lo, p.nr_pad, Kp, 4 * EPK, TC_N / CL, true, FMT))) return rc;
  if ((rc = make_map(&mBlt, r_lo, p.nr_pad, Kp, EPK, TC_N / CL, false, FMT))) return rc;
  constexpr int NPART = (FMT == 3) ? 1 : 2;
  constexpr int NS = BF16 ? (NPART == 1 ? 4 : 3) : 2;
  size_t smem = 1024 + (size_t)NPART * NS * TC_N * (WIDE ? 8 : p.nks) * 32 + 256 + 1024;
  auto kern = search_tc_kernel<MODE, CL, FMT, LS, QT, false, WIDE>;
  GTB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, nsm = 0;
  GTB_CUDA(cudaGetDevice(&dev));
  GTB_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
  const int64_t n_cluster_tiles = gtb_cdiv(p.nq_pad / TC_M, CL * QT);
  int64_t n_clusters = n_cluster_tiles < (nsm / CL) ? n_cluster_tiles : (nsm / CL);
  p.nrounds = gtb_cdiv(n_cluster_tiles, n_clusters);
  if (p.tile_stride < 1 || MODE == 1) p.tile_stride = 1;
  const int64_t total_tiles = gtb_cdiv(p.nr_pad / TC_N, p.tile_stride);
  p.n_qclusters = n_clusters;
  p.tiles_per_split = total_tiles;
  int64_t splits = 1;
  if (MODE == 1 && n_cluster_tiles * 2 <= nsm / CL && total_tiles >= 16) {
    splits = (nsm / CL) / n_cluster_tiles;
    if (splits > total_tiles / 8) splits = total_tiles / 8;
    p.tiles_per_split = gtb_cdiv(total_tiles, splits);
    splits = gtb_cdiv(total_tiles, p.tiles_per_split);
    n_clusters = n_cluster_tiles * splits;
  }
  // one-product top-k: a last round with work for at most half of the clusters becomes a second launch in which
  // every remaining cluster-unit is swept by split_k clusters, each over a piece of the reference range
  int64_t rem_units = 0, piece_k = 0, piece_tpp = 0;
  uint2* piece_space = p.piece_buf;
  p.q_unit0 = 0; p.split_k = 0;
  const bool listed = p.unit_ptr != nullptr;
  p.n_units = n_cluster_tiles;
  if constexpr (MODE == 0 && FMT == 3 && !WIDE) {
    const int64_t full = n_cluster_tiles / n_clusters, rem = n_cluster_tiles % n_clusters;
    if (!listed && piece_space != nullptr && full >= 1 && rem > 0 && rem * 2 <= n_clusters && total_tiles >= 64) {
      int64_t k = n_clusters / rem;
      if (k > TC_SPLIT_MAX) k = TC_SPLIT_MAX;
      piece_tpp = gtb_cdiv(total_tiles, k);
      k = gtb_cdiv(total_tiles, piece_tpp);
      if (k >= 2 && rem * CL * QT * TC_M <= TC_SPLIT_ROWS_MAX) {
        rem_units = rem; piece_k = k;
        p.nrounds = full;                        // first launch: the full rounds only
      }
    }
  }
  const unsigned nblk = (unsigned)(n_clusters * CL);
  // pacing counter: one caller-owned device word, zeroed per launch (no state is kept in the library)
  if (p.sync_ctr != nullptr && nblk > (unsigned)CL && splits == 1 && !listed) {
    GTB_CUDA(cudaMemsetAsync(p.sync_ctr, 0, sizeof(unsigned int), st));
  } else {
    p.sync_ctr = nullptr;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(nblk);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if constexpr (MODE == 0 && FMT == 3 && !WIDE) {
    if (listed) {
      auto lkern = search_tc_kernel<MODE, CL, FMT, LS, QT, false, false, true>;
      GTB_CUDA(cudaFuncSetAttribute(lkern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      GTB_CUDA(cudaLaunchKernelEx(&cfg, lkern, mBh, mBht, mBl, mBlt, q_hi, q_lo, p));
      GTB_CHECK_LAUNCH();
      return GTB_OK;
    }
  }
  GTB_CUDA(cudaLaunchKernelEx(&cfg, kern, mBh, mBht, mBl, mBlt, q_hi, q_lo, p));
  GTB_CHECK_LAUNCH();
  if constexpr (MODE == 0 && FMT == 3 && !WIDE) {
    if (rem_units > 0) {
      // piece launch: cluster c = unit (c % rem_units) of the remaining ones, piece c / rem_units of the reference
      // range (the mapping of the RADIUS launches), one round, no pacing; then the merge
      TcParams q = p;
      q.q_unit0 = p.nrounds * n_clusters;
      q.nrounds = 1;
      q.n_qclusters = rem_units;
      q.tiles_per_split = piece_tpp;
      q.sync_ctr = nullptr;
      q.split_k = piece_k;
      q.split_rows = rem_units * CL * QT * TC_M;
      q.split_row0 = q.q_unit0 * CL * QT * TC_M;
      q.piece_buf = piece_space;
      q.piece_meta = piece_space + q.split_rows * piece_k * (TC_GROUPS * TC_CAP);
      cfg.gridDim = dim3((unsigned)(rem_units * piece_k * CL));
      auto pkern = search_tc_kernel<MODE, CL, FMT, LS, QT, true>;
      GTB_CUDA(cudaFuncSetAttribute(pkern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      GTB_CUDA(cudaLaunchKernelEx(&cfg, pkern, mBh, mBht, mBl, mBlt, q_hi, q_lo, q));
      GTB_CHECK_LAUNCH();
      merge_pieces_kernel<2 * LS><<<(unsigned)gtb_cdiv(q.split_rows, TC_MERGE_WARPS), TC_MERGE_WARPS * 32, 0, st>>>(q);
      GTB_CHECK_LAUNCH();
    }
  }
  return GTB_OK;
}

template <int MODE, int FMT>
int launch_tc_fmt(const void* q_hi, const void* q_lo, const void* r_hi, const void* r_lo, int Kp, int list, int cluster,
                  int qtiles, TcParams& p, cudaStream_t st) {
  constexpr int LS_SHORT = (MODE == 0) ? 16 : 32;
  const bool short_list = (MODE == 0) && list == 16;
  if constexpr (FMT == 3) {
    // one product: two query tiles per CTA; top-k keeps one list of 64 per row (list = 32), the seed sweep none
    if constexpr (MODE != 1) {
      if (qtiles != 2 || list != 32 || (cluster != 1 && cluster != 2)) {
        gtb_set_error("the one-product flavour needs qtiles = 2, list = 32, cluster = 1 or 2");
        return GTB_ERR_ARG;
      }
      return cluster == 1 ? launch_tc_cl<MODE, 1, 3, 32, 2>(q_hi, q_lo, r_hi, r_lo, Kp, p, st)
                          : launch_tc_cl<MODE, 2, 3, 32, 2>(q_hi, q_lo, r_hi, r_lo, Kp, p, st);
    } else {
      gtb_set_error("the one-product flavour has no radius mode (use dtype 2 on the same operands)");
      return GTB_ERR_ARG;
    }
  } else {
  if constexpr (MODE == 2) {
    gtb_set_error("seed sweeps use the one-product flavour (dtype 3)");
    return GTB_ERR_ARG;
  } else {
  if (Kp > 128) {
    // operand rows beyond 8 k-steps: chunked reference stream (fp16x2 only, one query tile per CTA)
    if constexpr (FMT == 2) {
      if (qtiles != 1 || (cluster != 1 && cluster != 2)) {
        gtb_set_error("wide operand rows (Kp > 128) need qtiles = 1 and cluster = 1 or 2");
        return GTB_ERR_ARG;
      }
      if (cluster == 1)
        return short_list ? launch_tc_cl<MODE, 1, 2, LS_SHORT, 1, true>(q_hi, q_lo, r_hi, r_lo, Kp, p, st)
                          : launch_tc_cl<MODE, 1, 2, 32, 1, true>(q_hi, q_lo, r_hi, r_lo, Kp, p, st);
      return short_list ? launch_tc_cl<MODE, 2, 2, LS_SHORT, 1, true>(q_hi, q_lo, r_hi, r_lo, Kp, p, st)
                        : launch_tc_cl<MODE, 2, 2, 32, 1, true>(q_hi, q_lo, r_hi, r_lo, Kp, p, st);
    } else {
      gtb_set_error("operand rows beyond 128 elements are supported by the fp16x2 flavour (dtype 2) only");
      return GTB_ERR_ARG;
    }
  }
  if (qtiles == 2) {
    if constexpr (FMT == 2 && MODE == 0) {
      if (!short_list) { gtb_set_error("two query tiles per CTA need list = 16 (one list of 32 per row)"); return GTB_ERR_ARG; }
      if (cluster == 1) return launch_tc_cl<0, 1, 2, 16, 2>(q_hi, q_lo, r_hi, r_lo, Kp, p, st);
      if (cluster == 2) return launch_tc_cl<0, 2, 2, 16, 2>(q_hi, q_lo, r_hi, r_lo, Kp, p, st);
      gtb_set_error("cluster size must be 1 or 2");
      return GTB_ERR_ARG;
    } else {
      gtb_set_error("two query tiles per CTA: fp16x2 top-k only");
      return GTB_ERR_ARG;
    }
  }
  switch (cluster) {
    case 1: return short_list ? launch_tc_cl<MODE, 1, FMT, LS_SHORT>(q_hi, q_lo, r_hi, r_lo, Kp, p, st)
                              : launch_tc_cl<MODE, 1, FMT, 32>(q_hi, q_lo, r_hi, r_lo, Kp, p, st);
    case 2: return short_list ? launch_tc_cl<MODE, 2, FMT, LS_SHORT>(q_hi, q_lo, r_hi, r_lo, Kp, p, st)
                              : launch_tc_cl<MODE, 2, FMT, 32>(q_hi, q_lo, r_hi, r_lo, Kp, p, st);
    case 4:
      if (FMT == 0)
        return short_list ? launch_tc_cl<MODE, 4, 0, LS_SHORT>(q_hi, q_lo, r_hi, r_lo, Kp, p, st)
                          : launch_tc_cl<MODE, 4, 0, 32>(q_hi, q_lo, r_hi, r_lo, Kp, p, st);
      // fall through: the 2-byte flavours support clusters of 1 or 2
    default: gtb_set_error("cluster size must be 1 or 2 (or 4 for the tf32 flavour)"); return GTB_ERR_ARG;
  }
  }
  }
}

template <int MODE>
int launch_tc(const void* q_hi, const void* q_lo, const void* r_hi, const void* r_lo, int Kp, int dtype, int list,
              int cluster, int qtiles, TcParams& p, cudaStream_t st) {
  if (dtype == 1) return launch_tc_fmt<MODE, 1>(q_hi, q_lo, r_hi, r_lo, Kp, list, cluster, qtiles, p, st);
  if (dtype == 2) return launch_tc_fmt<MODE, 2>(q_hi, q_lo, r_hi, r_lo, Kp, list, cluster, qtiles, p, st);
  if (dtype == 3) return launch_tc_fmt<MODE, 3>(q_hi, q_lo, r_hi, r_lo, Kp, list, cluster, qtiles, p, st);
  return launch_tc_fmt<MODE, 0>(q_hi, q_lo, r_hi, r_lo, Kp, list, cluster, qtiles, p, st);
}

}  // namespace

// largest operand row: 13 k-steps of 32 bytes = 104 tf32 or 208 bf16 elements (TMEM: 2 x 104 columns for A)
extern "C" int gtb_tc_max_kp(void) { return 104; }

// squared norms of the centred rows (rounded up) and their maximum: what the fp16 flavour needs BEFORE the split, to
// pick the power-of-two scale that brings the data into fp16 range
extern "C" int gtb_row_norms(const float* X, int64_t n, int d, const float* mean, int64_t n_pad, float* norm2,
                             float* maxnorm, void* stream) {
  GTB_CHECK_ARG(n > 0 && d > 0 && n_pad >= n, "bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  if (maxnorm) GTB_CUDA(cudaMemsetAsync(maxnorm, 0, sizeof(float), st));
  tc_norms_kernel<<<(unsigned)gtb_cdiv(n_pad * 32, 256), 256, 0, st>>>(X, n, d, mean, n_pad, norm2, maxnorm);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

// largest scaled squared norm the fp16 flavour accepts: scale^2 * max|row|^2 must stay <= this
extern "C" float gtb_tc_fp16_maxnorm(void) { return TC_H_MAXNORM; }

// Argument checks and the split into hi/lo pairs of `dtype`, shared by gtb_prepare_operand_tc and gtb_split_operand_tc;
// with `norms`, the squared norms (and their maximum) are computed first, into norm2
static int tc_operand(const float* X, int64_t n, int d, const float* mean, int role, void* hi, void* lo, int64_t n_pad,
                      int Kp, int dtype, float scale, float* norm2, float* maxnorm, bool norms, cudaStream_t st) {
  GTB_CHECK_ARG(n > 0 && d > 0 && n_pad >= n && n_pad % 128 == 0, "bad shape");
  GTB_CHECK_ARG(dtype >= 0 && dtype <= 2, "dtype must be 0 (tf32 pairs in float32), 1 (bfloat16 pairs) or 2 (float16 pairs)");
  const int epk = dtype ? 16 : 8;
  GTB_CHECK_ARG(Kp % epk == 0 && Kp >= d + 1 + (dtype == 2) && Kp / epk <= (dtype == 2 ? 32 : (dtype ? 8 : 13)),
                "Kp must be a multiple of 8 (tf32, <= 104) / 16 (bf16 <= 128, fp16 <= 512) and >= d+1 (fp16: d+2)");
  GTB_CHECK_ARG(role == 0 || role == 1, "role must be 0 (query) or 1 (reference)");
  GTB_CHECK_ARG(dtype != 2 || scale > 0.f, "the fp16 flavour needs a positive scale");
  if (norms) {
    if (maxnorm) GTB_CUDA(cudaMemsetAsync(maxnorm, 0, sizeof(float), st));
    tc_norms_kernel<<<(unsigned)gtb_cdiv(n_pad * 32, 256), 256, 0, st>>>(X, n, d, mean, n_pad, norm2, maxnorm);
    GTB_CHECK_LAUNCH();
  }
  if (dtype == 0)
    tc_split_kernel<<<(unsigned)gtb_cdiv(n_pad * Kp, 256), 256, 0, st>>>(X, n, d, mean, role, norm2, n_pad, Kp,
                                                                        (float*)hi, (float*)lo);
  else if (dtype == 1)
    tc_split16_kernel<<<(unsigned)gtb_cdiv(n_pad * Kp, 256), 256, 0, st>>>(X, n, d, mean, role, norm2, n_pad, Kp,
                                                                          (__nv_bfloat16*)hi, (__nv_bfloat16*)lo);
  else
    tc_split16h_kernel<<<(unsigned)gtb_cdiv(n_pad * Kp, 256), 256, 0, st>>>(X, n, d, mean, role, norm2, n_pad, Kp, scale,
                                                                           (__half*)hi, (__half*)lo);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_prepare_operand_tc(const float* X, int64_t n, int d, const float* mean, int role, void* hi,
                                      void* lo, int64_t n_pad, int Kp, int dtype, float scale, float* norm2,
                                      float* maxnorm, void* stream) {
  return tc_operand(X, n, d, mean, role, hi, lo, n_pad, Kp, dtype, scale, norm2, maxnorm, true, (cudaStream_t)stream);
}

// The split alone, from norms that are already on hand (gtb_row_norms): both roles of an in-sample build share one pass
// over the norms instead of recomputing them per role
extern "C" int gtb_split_operand_tc(const float* X, int64_t n, int d, const float* mean, int role, void* hi, void* lo,
                                    int64_t n_pad, int Kp, int dtype, float scale, const float* norm2, void* stream) {
  GTB_CHECK_ARG(norm2 != nullptr, "norm2 (from gtb_row_norms) is required");
  return tc_operand(X, n, d, mean, role, hi, lo, n_pad, Kp, dtype, scale, const_cast<float*>(norm2), nullptr, false,
                    (cudaStream_t)stream);
}

// candidate buffers of every row + the piece buffers and piece records of a split last round
extern "C" int64_t gtb_tc_scratch_bytes(int64_t nq_pad) {
  return (nq_pad * TC_GROUPS * TC_CAP + TC_SPLIT_ROWS_MAX * TC_SPLIT_MAX * (TC_GROUPS * TC_CAP + 1)) * (int64_t)sizeof(uint2);
}

static int tc_check(int64_t nq, int64_t nr, int64_t nq_pad, int64_t nr_pad, int Kp, int dtype) {
  GTB_CHECK_ARG(nq > 0 && nr > 0 && nq_pad % TC_M == 0 && nr_pad % TC_N == 0, "bad shape (pads must be x128)");
  GTB_CHECK_ARG(dtype >= 0 && dtype <= 3, "dtype must be 0 (tf32), 1 (bf16), 2 (fp16, two products) or 3 (fp16, one)");
  const int epk = dtype ? 16 : 8;
  GTB_CHECK_ARG(Kp % epk == 0 && Kp >= epk && Kp / epk <= (dtype == 2 ? 32 : (dtype ? 8 : 13)), "Kp out of range");
  GTB_CHECK_ARG(nr_pad < (1ll << 31) && nq_pad < (1ll << 31), "too many rows for 32-bit TMA coordinates");
  return GTB_OK;
}

extern "C" int gtb_knn_topk_tc_seeded(const void* q_hi, const void* q_lo, const float* qn2, int64_t nq, int64_t nq_pad,
                                      const void* r_hi, const void* r_lo, int64_t nr, int64_t nr_pad, int Kp, int dtype,
                                      int list, int cluster, int qtiles, const float* seed_tau, int tile_stride,
                                      int32_t* cand_idx, void* scratch, float* tau, unsigned int* pace,
                                      const int64_t* unit_ptr, const int32_t* unit_tiles, const int32_t* unit_order,
                                      void* stream) {
  int rc = tc_check(nq, nr, nq_pad, nr_pad, Kp, dtype);
  if (rc) return rc;
  GTB_CHECK_ARG(list == 16 || list == 32, "list size must be 16 or 32");
  GTB_CHECK_ARG(qtiles == 1 || qtiles == 2, "query tiles per CTA: 1 or 2");
  GTB_CHECK_ARG(tile_stride >= 1, "tile_stride must be >= 1");
  const bool listed = unit_ptr != nullptr || unit_tiles != nullptr || unit_order != nullptr;
  GTB_CHECK_ARG(!listed || (unit_ptr && unit_tiles && unit_order), "tile lists need unit_ptr, unit_tiles and unit_order");
  GTB_CHECK_ARG(!listed || (dtype == 3 && tile_stride == 1), "tile lists: the one-product flavour (dtype 3), tile_stride 1");
  TcParams p{};
  p.unit_ptr = unit_ptr; p.unit_tiles = unit_tiles; p.unit_order = unit_order;
  p.nq = nq; p.nq_pad = nq_pad; p.nr = nr; p.nr_pad = nr_pad; p.qn2 = qn2;
  p.cand_idx = cand_idx; p.cand_buf = reinterpret_cast<uint2*>(scratch); p.tau = tau; p.sync_ctr = pace;
  p.seed_tau = seed_tau; p.tile_stride = tile_stride;
  p.piece_buf = p.cand_buf + nq_pad * TC_GROUPS * TC_CAP;   // second part of the scratch (gtb_tc_scratch_bytes)
  return launch_tc<0>(q_hi, q_lo, r_hi, r_lo, Kp, dtype, list, cluster, qtiles, p, (cudaStream_t)stream);
}

// Threshold seeds for gtb_knn_topk_tc_seeded: tau[nq][2] (both slots) = the TC_SEED_K-th smallest TILE MINIMUM of the
// approximate squared distances over every tile_stride-th 128-row reference tile (+inf with fewer sampled tiles)
extern "C" int gtb_knn_seed_tc(const void* q_hi, const float* qn2, int64_t nq, int64_t nq_pad, const void* r_hi,
                               int64_t nr, int64_t nr_pad, int Kp, int cluster, int tile_stride, float* tau,
                               unsigned int* pace, void* stream) {
  int rc = tc_check(nq, nr, nq_pad, nr_pad, Kp, 3);
  if (rc) return rc;
  GTB_CHECK_ARG(tile_stride >= 1, "tile_stride must be >= 1");
  TcParams p{};
  p.nq = nq; p.nq_pad = nq_pad; p.nr = nr; p.nr_pad = nr_pad; p.qn2 = qn2;
  p.tau = tau; p.sync_ctr = pace; p.tile_stride = tile_stride;
  return launch_tc<2>(q_hi, q_hi, r_hi, r_hi, Kp, 3, 32, cluster, 2, p, (cudaStream_t)stream);
}

extern "C" int gtb_knn_seed_k(void) { return TC_SEED_K; }

extern "C" int gtb_knn_topk_tc(const void* q_hi, const void* q_lo, const float* qn2, int64_t nq, int64_t nq_pad,
                               const void* r_hi, const void* r_lo, int64_t nr, int64_t nr_pad, int Kp, int dtype,
                               int list, int cluster, int qtiles, int32_t* cand_idx, void* scratch, float* tau,
                               unsigned int* pace, void* stream) {
  return gtb_knn_topk_tc_seeded(q_hi, q_lo, qn2, nq, nq_pad, r_hi, r_lo, nr, nr_pad, Kp, dtype, list, cluster, qtiles,
                                nullptr, 1, cand_idx, scratch, tau, pace, nullptr, nullptr, nullptr, stream);
}

extern "C" int gtb_knn_radius_tc(const void* q_hi, const void* q_lo, const float* qn2, const float* lim2,
                                 int64_t nq, int64_t nq_pad, const void* r_hi, const void* r_lo, int64_t nr,
                                 int64_t nr_pad, int Kp, int dtype, int cluster, int32_t* pairs, int64_t capacity,
                                 unsigned long long* counter, int32_t* rowcnt, unsigned int* pace, void* stream) {
  int rc = tc_check(nq, nr, nq_pad, nr_pad, Kp, dtype);
  if (rc) return rc;
  TcParams p{};
  p.nq = nq; p.nq_pad = nq_pad; p.nr = nr; p.nr_pad = nr_pad; p.qn2 = qn2; p.lim2 = lim2;
  p.pairs = reinterpret_cast<int2*>(pairs); p.capacity = (unsigned long long)capacity; p.counter = counter;
  p.rowcnt = rowcnt; p.sync_ctr = pace; p.tile_stride = 1;
  return launch_tc<1>(q_hi, q_lo, r_hi, r_lo, Kp, dtype, 32, cluster, 1, p, (cudaStream_t)stream);
}
