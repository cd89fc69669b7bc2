/* gtb200 -- C ABI of the B200-native graph-construction engine (libgtb200.so).
 *
 * The reference (KrishnaswamyLab/graphtools v2.1.0) is pure Python and has no FFI: its seam is
 * the pair of abstract methods BaseGraph.build_kernel() (graphtools/base.py:805-818) and
 * DataGraph.build_kernel_to_data(Y) (base.py:1102-1127) plus the BaseGraph post-processing
 * (base.py:534-592, :629-698).  Every entry point below replaces the third-party call the
 * reference makes at the cited site.  INTEGRATION.md shows the ctypes stub a graphtools
 * maintainer would add to call them.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless stated otherwise; the caller owns every buffer
 *     (the Python host allocates them as torch tensors and passes tensor.data_ptr());
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on that stream and
 *     never synchronise;
 *   - return value: 0 on success, negative on error (GTB_ERR_*); gtb_last_error() returns a
 *     thread-local description;
 *   - matrices are row-major; CSR uses int64 row pointers on the device (cast with
 *     gtb_cast_indptr for the scipy int32 contract), int32 column indices, float64 values.
 */
#ifndef GTB200_H
#define GTB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* gtb_last_error(void);
int gtb_version(void);

/* ---- operand preparation (no reference counterpart: sklearn NearestNeighbors.fit keeps a
 * pointer for brute force, graphs.py:763-768) ------------------------------------------------ */
/* column means of X[n,d] (float32); ws holds gtb_col_mean_ws_doubles(d) doubles */
int64_t gtb_col_mean_ws_doubles(int d);
int gtb_col_mean(const float* X, int64_t n, int d, double* ws, float* mean, void* stream);
/* XT[d_pad][n_pad] = transpose(X - mean) zero padded (n_pad % 128 == 0, d_pad % 8 == 0);
 * norm2[n_pad] = |row|^2 of the centred rows, +inf on padding; *maxnorm = max norm2 (optional) */
int gtb_prepare_operand(const float* X, int64_t n, int d, const float* mean, float* XT, int64_t n_pad,
                        int d_pad, float* norm2, float* maxnorm, void* stream);
/* dstT[:, t] = srcT[:, rows[t]] for t < nt (query sub-set for the radius pass) */
int gtb_gather_operand(const float* srcT, int64_t src_pad, const float* src_n2, const int32_t* rows,
                       int64_t nt, float* dstT, int64_t dst_pad, int d_pad, float* dst_n2, void* stream);

/* ---- K1/K2 distance + selection: replaces knn_tree.kneighbors (graphs.py:883, :922, :957),
 * kneighbors_graph (:875-877) and radius_neighbors (:966-973) ------------------------------- */
/* top-S candidates per query by approximate squared distance; cand_idx[nq][S] (-1 = empty),
 * tau[nq] = S-th smallest approximate d^2 (+inf when fewer than S references). S in {16,32,48,64,128} */
int gtb_knn_topk_simt(const float* QT, const float* qn2, int64_t nq, int64_t nq_pad, const float* RT,
                      const float* rn2, int64_t nr, int64_t nr_pad, int d_pad, int S, int32_t* cand_idx,
                      float* tau, void* stream);
/* every (query slot, ref) pair with approximate d^2 <= lim2[slot] appended to pairs[capacity][2];
 * *counter (zeroed by the caller) receives the number of qualifying pairs even past capacity;
 * rowcnt[nq] (zeroed by the caller) receives the per-slot counts */
int gtb_knn_radius_simt(const float* QT, const float* qn2, const float* lim2, int64_t nq, int64_t nq_pad,
                        const float* RT, const float* rn2, int64_t nr, int64_t nr_pad, int d_pad,
                        int32_t* pairs, int64_t capacity, unsigned long long* counter, int32_t* rowcnt,
                        void* stream);
/* cityblock (L1) metric -- sklearn's brute-force manhattan search behind knn_tree for distance="cityblock"
 * (graphs.py:763-768; the reference's landmark tests run it, test/test_landmark.py:195-322): the tile accumulates
 * sum_k |x_k - y_k| in float32 on the CUDA cores (the L1 distance has no GEMM form), operands are the k-major rows
 * WITHOUT centring, tau / lim hold distances (not squared) */
int gtb_knn_topk_simt_l1(const float* QT, int64_t nq, int64_t nq_pad, const float* RT, int64_t nr, int64_t nr_pad,
                         int d_pad, int S, int32_t* cand_idx, float* tau, void* stream);
int gtb_knn_radius_simt_l1(const float* QT, const float* lim, int64_t nq, int64_t nq_pad, const float* RT, int64_t nr,
                           int64_t nr_pad, int d_pad, int32_t* pairs, int64_t capacity, unsigned long long* counter,
                           int32_t* rowcnt, void* stream);

/* Tensor-core variant (tcgen05.mma, TMA-fed, TMEM accumulators, persistent 2-CTA clusters).  Operands are
 * row-major [n_pad][Kp] hi/lo pairs built by gtb_prepare_operand_tc: role 0 (query) = [x~, 1, 0..],
 * role 1 (reference) = [-2y~, |y~|^2, 0..].
 *   dtype 0: 3xTF32 -- float32 storage, hi = tf32(v), lo = tf32(v - hi), kind::tf32, Kp = roundup(d+1, 8) <= 104
 *   dtype 1: bf16x3 -- bfloat16 storage, hi = bf16(v), lo = bf16(v - hi), kind::f16,  Kp multiple of 16, <= 128
 *            (3 smem stages, 3 TMEM accumulators); products A_hi.B_hi + A_hi.B_lo + A_lo.B_hi like dtype 0
 *   dtype 2: fp16x2 -- float16 storage of the data scaled by the power of two `scale` (scale^2 max|row|^2 <=
 *            gtb_tc_fp16_maxnorm(); gtb_row_norms gives the norms beforehand), TWO products A_hi.B_hi + A_hi.B_lo:
 *            2/3 of the tensor work, rounding bound 2^-11 (|x~|^2 + |y~|^2) on the (scaled) squared distance.  tau and
 *            the radius limits are in scaled units (scale^2 x squared distance); the caller converts.
 * topk: cand_idx[nq][2 * list] = two lists of `list` = 32 or 16 entries (disjoint halves of the reference tiles, -1 = empty; shorter
 * lists halve the selection work -- rows whose kernel support they do not cover fail certification in gtb_refine_topk and are
 * completed by the radius pass, so the result does not depend on `list`) with their
 * thresholds tau[nq][2]; scratch = gtb_tc_scratch_bytes(nq_pad) bytes.  radius: contract of gtb_knn_radius_simt.
 * qtiles: query tiles per CTA.  1: the layout above.  2 (dtype 2, list 16 only): every reference stage is multiplied
 * against two resident query tiles -- half the L2 -> SM bytes per unit of tensor work -- and each row keeps ONE list of
 * 2 * list entries (same cand_idx / tau layout; both tau slots carry the list's threshold).
 * cluster: 1, 2 (or 4, tf32 only) CTAs share each reference tile through TMA multicast.  pace: one caller-owned device
 * word for the grid-wide pacing of the TMA producers (so that one DRAM read of a reference tile serves all SMs), or
 * NULL for no pacing -- the library keeps no state between calls. */
int gtb_tc_max_kp(void);
float gtb_tc_fp16_maxnorm(void);
int gtb_row_norms(const float* X, int64_t n, int d, const float* mean, int64_t n_pad, float* norm2, float* maxnorm,
                  void* stream);
int gtb_prepare_operand_tc(const float* X, int64_t n, int d, const float* mean, int role, void* hi, void* lo,
                           int64_t n_pad, int Kp, int dtype, float scale, float* norm2, float* maxnorm, void* stream);
/* the split of gtb_prepare_operand_tc alone, from norms computed by gtb_row_norms (norm2 is an INPUT here) */
int gtb_split_operand_tc(const float* X, int64_t n, int d, const float* mean, int role, void* hi, void* lo,
                         int64_t n_pad, int Kp, int dtype, float scale, const float* norm2, void* stream);
int gtb_knn_topk_tc(const void* q_hi, const void* q_lo, const float* qn2, int64_t nq, int64_t nq_pad,
                    const void* r_hi, const void* r_lo, int64_t nr, int64_t nr_pad, int Kp, int dtype,
                    int list, int cluster, int qtiles, int32_t* cand_idx, void* scratch, float* tau,
                    unsigned int* pace, void* stream);
/* The same sweep with (a) dtype = 3: float16 operands of dtype 2 (hi arrays only), ONE product A_hi.B_hi -- rounding
 * bound 2^-10 (|x|^2 + |y|^2); qtiles = 2 and list = 32 only (one list of 64 per row, cand_idx [nq][64]); (b)
 * tile_stride > 1: only every tile_stride-th 128-row reference tile is visited; (c) seed_tau != NULL (layout of tau,
 * slot 0 read): the row's threshold starts at the seed instead of +inf, every reference point under it is kept
 * (compacting to the list length when the buffer fills) and a list that never filled reports the seed as its tau -- a
 * seed from gtb_knn_seed_tc removes most of the list * ln(N / list) threshold updates of a cold start.
 * seed_tau = NULL, tile_stride = 1 is gtb_knn_topk_tc.  (d) tile lists (dtype 3, tile_stride 1; all three or none):
 * unit u = the cluster * qtiles query tiles of rows [u * cluster * qtiles * 128, ...), u < cdiv(nq_pad / 128,
 * cluster * qtiles), sweeps only the reference tiles unit_tiles[unit_ptr[u] .. unit_ptr[u + 1]); unit_order lists every
 * unit once, in the order the clusters take them (longest list first balances the rounds); pace is not used.  A row's
 * list and tau then cover the listed tiles only. */
int gtb_knn_topk_tc_seeded(const void* q_hi, const void* q_lo, const float* qn2, int64_t nq, int64_t nq_pad,
                           const void* r_hi, const void* r_lo, int64_t nr, int64_t nr_pad, int Kp, int dtype,
                           int list, int cluster, int qtiles, const float* seed_tau, int tile_stride,
                           int32_t* cand_idx, void* scratch, float* tau, unsigned int* pace,
                           const int64_t* unit_ptr, const int32_t* unit_tiles, const int32_t* unit_order, void* stream);
/* Threshold seeds (one-product float16 sweep over every tile_stride-th reference tile, no candidate lists): tau[nq][2]
 * (both slots) = the gtb_knn_seed_k()-th smallest TILE MINIMUM of the approximate squared distances, an upper bound of
 * the k-th smallest sampled value kept in registers by a branch-free insertion network -- no hit servicing at all */
int gtb_knn_seed_k(void);
int gtb_knn_seed_tc(const void* q_hi, const float* qn2, int64_t nq, int64_t nq_pad, const void* r_hi, int64_t nr,
                    int64_t nr_pad, int Kp, int cluster, int tile_stride, float* tau, unsigned int* pace, void* stream);
int64_t gtb_tc_scratch_bytes(int64_t nq_pad);
/* Locality order and tile lists for the listed sweep (csrc/order.cu).  d <= 128 throughout.
 * gtb_order_assign: cell[r] = nearest of the P (<= 512, <= n) pivot rows p * floor(n / P) of X (float32).
 * gtb_order_sort: perm[i] = row at position i of the stable sort of the rows by cell; ws: gtb_order_ws_elems int32.
 * gtb_tile_geometry: per group g of the rows perm[g * rows .. min(n, (g + 1) * rows)) of X (float64 if x64, else
 * float32): centroid cent[k * ngroups + g] (float64) and radius rad[g] = max |x - c| rounded up (-1: no rows).
 * gtb_tile_lists_count: keep[u * nt + t] = 0 iff (|c_u - c_t| - r_u - r_t)^2 >= ub[u] (rounded against skipping), every
 * distance between the rows of unit u and tile t then reaching ub[u]; count[u] = kept tiles.
 * gtb_tile_lists_fill: tiles[ptr[u] ..] = the kept tiles of unit u, ascending (ptr = exclusive scan of count).
 * gtb_unpermute_candidates: cand[perm_q[i]][s] = perm_r[cand_p[i][s]] (-1 stays), tau[perm_q[i]] = tau_p[i]. */
int gtb_order_assign(const float* X, int64_t n, int d, int P, int32_t* cell, void* stream);
int64_t gtb_order_ws_elems(int64_t n, int P);
int gtb_order_sort(const int32_t* cell, int64_t n, int P, int32_t* ws, int32_t* perm, void* stream);
int gtb_tile_geometry(const void* X, int64_t n, int d, int x64, const int32_t* perm, int64_t rows, int64_t ngroups,
                      double* cent, double* rad, void* stream);
int gtb_tile_lists_count(const double* uc, const double* ur, const double* ub, int64_t nu, const double* rc,
                         const double* rr, int64_t nt, int d, uint8_t* keep, int32_t* count, void* stream);
int gtb_tile_lists_fill(const uint8_t* keep, int64_t nu, int64_t nt, const int64_t* ptr, int32_t* tiles, void* stream);
int gtb_unpermute_candidates(const int32_t* cand_p, const float* tau_p, int64_t nq, int S, int ntau,
                             const int32_t* perm_q, const int32_t* perm_r, int32_t* cand, float* tau, void* stream);
int gtb_knn_radius_tc(const void* q_hi, const void* q_lo, const float* qn2, const float* lim2, int64_t nq,
                      int64_t nq_pad, const void* r_hi, const void* r_lo, int64_t nr, int64_t nr_pad, int Kp,
                      int dtype, int cluster, int32_t* pairs, int64_t capacity, unsigned long long* counter,
                      int32_t* rowcnt, unsigned int* pace, void* stream);
/* Histogram count sweeps (kNN graphs whose knn is beyond the candidate lists): per query row, counts of the approximate
 * squared distances w (search units) by float32 bits, into hist[nq_pad][bins] (zeroed by the call, filled with
 * atomics).  top == NULL: coarse pass, 64 bins: bin b holds exponent field elo + b (bin 0 everything below, bin 63
 * everything above); counting stops `margin` octaves above the first bin whose cumulative count reaches k.  Otherwise
 * fine pass, 17 bins: w < top[i]/2, then the 16 sub-bins of [top[i]/2, top[i]) by the top four mantissa bits (rows
 * with top = +inf are not counted).  _tc: the fp16x2 operands of gtb_knn_radius_tc (dtype 2); _simt: the operands of
 * gtb_knn_radius_simt, or with qn2 = rn2 = NULL those of gtb_knn_radius_simt_l1 (cityblock distances). */
int gtb_knn_count_tc(const void* q_hi, const void* q_lo, const float* qn2, const float* top, int64_t nq, int64_t nq_pad,
                     const void* r_hi, const void* r_lo, int64_t nr, int64_t nr_pad, int Kp, int dtype, int cluster,
                     int k, int margin, int elo, uint32_t* hist, unsigned int* pace, void* stream);
int gtb_knn_count_simt(const float* QT, const float* qn2, const float* top, int64_t nq, int64_t nq_pad,
                       const float* RT, const float* rn2, int64_t nr, int64_t nr_pad, int d_pad, int k, int margin,
                       int elo, uint32_t* hist, void* stream);

/* ---- K3 float64 re-evaluation, bandwidth, affinities, CSR emission: replaces graphs.py:886-911
 * and _build_csr_from_neighbors (graphs.py:450-559) ------------------------------------------ */
/* Xq / Xr are the ORIGINAL rows used for the exact distances; x_kind bit 0: rows are float64 (e.g. PCA output)
 * instead of float32; bits 1-3: metric -- 1 = cosine: exact distances 1 - x.y/(|x||y|) (sklearn cosine_distances, the
 * metric behind knn_tree for distance="cosine", graphs.py:763-768) while the fast pass ran on the row-normalised
 * copies, where |x^ - y^|^2 = 2 d_cos; 2 = cityblock: exact sum |x - y|, fast pass = gtb_knn_topk_simt_l1 (tau is a
 * distance, the rounding bound is eps_rel * tau, qn2 / maxrn2 carry L1 norms for float64 inputs or NULL / 0); 3 =
 * sqeuclidean: exact sum (x - y)^2 on the Euclidean fast pass and operands (radii in squared units); 4 = correlation:
 * cosine of the rows centred by their own float64 means, fast pass on the row-centred, row-normalised copies as for
 * cosine.  decay < 0 means binary kNN (decay=None); kmax <= 0 means knn_max=None;
 * bw_mode 0: bandwidth = distance to the knn-th candidate (graphs.py:892), 1: scalar bw_fixed[0],
 * 2: per-row bw_fixed[nq].  cand_idx rows are cand_stride apart (first S entries used); tau holds ntau
 * thresholds per row (lists built over disjoint reference subsets), the row's bound is their minimum.  status: 1 done, 0 needs radius pass, 2 needs radius pass and its
 * bandwidth is not yet certified.  st_idx/st_val[nq][S]: kept entries sorted by column. */
int gtb_refine_topk(const void* Xq, int64_t nq, const void* Xr, int d, int x_kind, const int32_t* cand_idx, int S,
                    int cand_stride, const float* tau, int ntau, const float* qn2, float maxrn2, double eps_rel, int knn, int64_t kmax,
                    double decay, double thresh, const double* bw_fixed, int bw_mode, double bw_scale,
                    int32_t* st_idx, double* st_val, int32_t* n_keep, double* bw_out, float* lim2_out,
                    int32_t* status, int32_t* nzero, void* stream);
int gtb_compact_todo(const int32_t* status, int64_t nq, int32_t* todo_rows, int32_t* count, void* stream);
int gtb_scatter_pairs(const int32_t* pairs, int64_t npairs, const int64_t* seg_ptr, int32_t* cursor,
                      int64_t nt, int32_t* seg_idx, void* stream);
/* block per radius-pass row; *overflow receives the longest row length that exceeded `cap` */
int gtb_refine_ball(const void* Xq, const int32_t* todo_rows, const int32_t* status, int64_t nt,
                    const void* Xr, int d, int x_kind, const int64_t* seg_ptr, int32_t* seg_idx, double* seg_val, int knn,
                    int64_t kmax, double decay, double thresh, const double* bw_fixed, int bw_mode,
                    double bw_scale, int32_t* n_keep_t, int32_t* n_keep, double* bw_out, int32_t* nzero,
                    int32_t* overflow, int cap, void* stream);
int gtb_csr_gather(const int32_t* st_idx, const double* st_val, const int32_t* n_keep, const int32_t* status,
                   const int64_t* indptr, int64_t nq, int S, const int32_t* todo_rows, int64_t nt,
                   const int64_t* seg_ptr, const int32_t* seg_idx, const double* seg_val,
                   const int32_t* n_keep_t, int32_t* out_idx, double* out_val, void* stream);
/* Collect limits of the count path (rows whose knn is beyond the candidate lists), by the rule of the status-2 rows of
 * gtb_refine_topk with the knn-th distance bounded from the histograms: fine == NULL: top[nq] = upper edge of the
 * first coarse bin whose cumulative count reaches knn (+inf: none); otherwise lim2[nq] (data units, as lim2_out) and
 * bounds on the ball size: ball_lo <= |ball| <= ball_hi (-1: not known).  s2: search units per data unit (fp16 scale
 * squared, else 1); qn2 / maxrn2 / eps_rel / x_kind as for gtb_refine_topk.  coarse == NULL: fixed bandwidth
 * (bw_mode 1 or 2), lim2 = the kernel support alone. */
int gtb_knn_count_bound(const uint32_t* coarse, const uint32_t* fine, int64_t nq, int64_t nr, int elo, int margin,
                        float s2, const float* qn2, float maxrn2, double eps_rel, int x_kind, int knn, int64_t kmax,
                        double decay, double thresh, const double* bw_fixed, int bw_mode, double bw_scale, float* top,
                        float* lim2, int32_t* ball_lo, int32_t* ball_hi, void* stream);

/* ---- K4 sparse symmetrise / normalise: replaces base.py:557-577, :579-592, :645, :648-666 --- */
int64_t gtb_scan_ws_elems(int64_t n);
/* out[n+1] = exclusive prefix sums of in[n] (int32 -> int64), one launch (decoupled look-back);
 * ws: gtb_scan_ws_elems(n) int64 of scratch */
int gtb_exclusive_scan(const int32_t* in, int64_t n, int64_t* out, int64_t* ws, void* stream);
int gtb_cast_indptr(const int64_t* in, int64_t n1, int32_t* out, void* stream);
/* Sort-based transpose of a CSR (K^T of base.py:561-571 without scipy's csr_tocsc), as 16-byte edge records
 * {int32 i, int32 j, float64 w}: cnt[n_cols] = histogram of (idx - col0); gtb_exclusive_scan(cnt) -> ptr_t, whose
 * 32-bit copy (gtb_cast_indptr) is the per-row cursor; scatter then places every edge (row0 + r, j, w) in row j - col0
 * of t_rec with ONE atomic on the cursor and ONE 16-byte store.  Rows come out in arrival order. */
int gtb_transpose_count(const int32_t* idx, int64_t nnz, int32_t col0, int32_t* cnt, int64_t n_cols, void* stream);
int gtb_transpose_scatter(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n_rows, int32_t row0,
                          int32_t col0, int32_t* cursor, void* t_rec, void* stream);
/* The same transpose for a list of k packed edge records (what the multi-GPU all-to-all delivers): row j - col0 of
 * t_rec receives the record */
int gtb_records_count(const void* rec, int64_t k, int32_t col0, int32_t* cnt, int64_t n_cols, void* stream);
int gtb_records_scatter(const void* rec, int64_t k, int32_t col0, int32_t* cursor, void* t_rec, void* stream);
/* In-place segmented sort of CSR rows by column (columns unique within a row; has_long: one int of scratch):
 * separate index / value arrays, or record rows keyed by .i.  For records, rows r with
 * len(r) + (pa ? pa[r+1] - pa[r] : 0) <= min_total are skipped (the merge handles them unsorted). */
int gtb_csr_sort_rows(const int64_t* ptr, int32_t* idx, double* val, int64_t n, int32_t* has_long, void* stream);
int gtb_rec_sort_rows(const int64_t* ptr, void* rec, int64_t n, const int64_t* pa, int min_total, int32_t* has_long,
                      void* stream);
/* Merge of the raw kernel rows A = (pa, ia, va), column-sorted, with the record rows T = (pt, t_rec) of the transposed
 * matrix -- in ARRIVAL order -- under mode 0 '+' ((w + w')/2), 1 '*' (w w'), 2 'mnn' (theta min + (1 - theta) max):
 * count -> gtb_exclusive_scan -> fill.  Rows with |A| + |T| <= gtb_sym_merge_reg_rows() are merged unsorted, one entry
 * per lane; count queues the longer ones (worklist: n_rows + 1 ints of scratch) and orders their T entries by column in
 * place before it returns, which is what fill's two-pointer merge of those rows reads.  fill emits the column-sorted K row,
 * P = K / sum|K| (base.py:645), the degree vector (base.py:648-666) and sets flags bit 1 when a row lacks its diagonal
 * (base.py:553-554; global row id = row0 + r, columns are global).  Used on the whole matrix (one GPU) and on a row
 * shard (multi-GPU, after the all-to-all) alike, so the two builds agree bit for bit. */
int gtb_sym_merge_reg_rows(void);
int gtb_sym_merge_count(const int64_t* pa, const int32_t* ia, const double* va, const int64_t* pt, void* t_rec,
                        int64_t n_rows, int mode, double theta, int32_t* newlen, int32_t* worklist, void* stream);
int gtb_sym_merge_fill(const int64_t* pa, const int32_t* ia, const double* va, const int64_t* pt, const void* t_rec,
                       int64_t n_rows, int32_t row0, int mode, double theta, const int64_t* outptr, int32_t* out_idx,
                       double* out_val, double* p_val, double* degree, int32_t* flags, void* stream);
/* kernel_symm=None: flags bit 0 set when max(K - K^T) > 1e-5 (base.py:551-552) */
int gtb_asym_check(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n, int32_t* flags,
                   void* stream);
/* p_val = val / sum|val| and degree = sum|val| per row (each optional); flags bit 1: a row lacks its diagonal */
int gtb_row_finalize(const int64_t* ptr, const int32_t* idx, const double* val, int64_t n, double* p_val,
                     double* degree, int32_t* flags, int check_diag, void* stream);
int gtb_anisotropy(const int64_t* indptr, const int32_t* idx, double* val, const double* deg, double alpha,
                   int64_t n, void* stream);
/* Multi-GPU edge exchange (SURVEY 8e collective 2): bucket the raw edges of a row shard by the rank that owns their
 * column, owner(j) = min(j / per, world - 1).  count: cnt[o * m + r] = entries of local row r bound for rank o
 * (destination-major); after gtb_exclusive_scan(cnt) -> pos, fill packs the 16-byte records {row0 + r, j, w} into
 * the send buffer in (destination, row, column) order -- the layout ncclAllToAll consumes, no sort. */
int gtb_route_count(const int64_t* indptr, const int32_t* idx, int64_t m, int32_t per, int world, int32_t* cnt,
                    void* stream);
int gtb_route_fill(const int64_t* indptr, const int32_t* idx, const double* val, int64_t m, int32_t row0, int32_t per,
                   int world, const int32_t* cnt, const int64_t* pos, void* send, void* stream);
/* out[n_rows][n_cols] (float64) = dense form of the CSR matrix (zero fill + scatter): exact graphs with a
 * threshold are built sparse on the tensor-core path and densified once (reference container contract:
 * TraditionalGraph.K is an ndarray, graphs.py:1594-1609) */
int gtb_csr_to_dense(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n_rows, int64_t n_cols,
                     double* out, void* stream);

/* MNN block assembly: scatter a CSR block (local indices) into the global staging CSR.  Row i of the
 * block goes to global row row_map[i], column j to col_map[j], values scaled by
 * min(1, within[i] / between[i]) * beta when `within` is non-NULL (reference graphs.py:1904-1935,
 * matrix.py:49-51).  block_count adds the block's row lengths to rowlen[]; block_fill appends at
 * outptr[row] + cursor[row] and advances cursor (calls on one stream are ordered). */
int gtb_block_count(const int64_t* indptr, int64_t nb, const int32_t* row_map, int32_t* rowlen, void* stream);
int gtb_block_fill(const int64_t* indptr, const int32_t* idx, const double* val, int64_t nb,
                   const int32_t* row_map, const int32_t* col_map, const double* within, const double* between,
                   double beta, const int64_t* outptr, int32_t* cursor, int32_t* out_idx, double* out_val,
                   void* stream);

/* ---- K6 landmark operator: replaces LandmarkGraph._landmarks_to_data, build_landmark_op and
 * extend_to_data (graphs.py:1169-1182, :1232-1246, :1272-1288) ------------------------------- */
/* per row: aggregate entries by label[col]; cnt[row] = number of distinct labels.  ws: gtb_cluster_aggregate_ws_elems
 * 8-byte words of scratch (long-row flag + dense per-label tables for rows longer than 256 entries) */
int64_t gtb_cluster_aggregate_ws_elems(int n_label);
int gtb_cluster_aggregate_count(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n,
                                const int32_t* label, int n_label, int32_t* cnt, void* ws, void* stream);
/* out rows sorted by label: out_raw = sums (column order inside a label, as the reference's
 * kernel[clusters == l, :].sum(axis=0)), out_norm = sums / row L1 norm (optional), colsum[n_label] = column L1 sums
 * of out_raw (optional; accumulated in 96-bit fixed point in colsum_fx[2 * n_label] -- order independent, hence
 * bit-reproducible) */
int gtb_cluster_aggregate_fill(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n,
                               const int32_t* label, const int64_t* outptr, int32_t* out_idx, double* out_raw,
                               double* out_norm, double* colsum, void* colsum_fx, int n_label, void* ws,
                               void* stream);
/* op[L][L] = rownorm(pnm^T) . rownorm(pnm) from the aggregated rows; op_fx: 2 * L * L 8-byte words of scratch (the
 * fixed-point accumulator: integer atomics, so the operator is identical from run to run and for any row split) */
int gtb_landmark_op(const int64_t* ptr, const int32_t* lab, const double* raw, const double* nrm,
                    const double* colsum, int64_t n, int L, double* op, void* op_fx, void* stream);

/* ---- K5 dense exact graph: replaces TraditionalGraph.build_kernel / build_kernel_to_data
 * (graphs.py:1546-1609, :1651-1677) and the dense branches of base.py:557-592, :645 ---------- */
/* Xq / Xr: float32 rows, or float64 rows when x_is_f64 (distances are float64 differences of the rows as given,
 * what pdist / cdist compute).  what 0: out = distances; 1: out = thresholded affinities exp(-(d/bw_q[i])^decay);
 * 2: additionally symmetrised with the transposed entry (symm 0 '+', 1 '*', 2 'mnn', 3 none);
 * rowsum (optional) receives the row L1 sums (a separate deterministic pass).  metric 0: Euclidean distances;
 * 1: cosine distances 1 - x.y/(|x||y|) with |cos| clamped to 1; 2: cityblock; 3: sqeuclidean (scipy pdist / cdist,
 * graphs.py:1552, :1653).  Correlation distances are metric 1 on rows centred by their float64 means, as scipy computes
 * them. */
int gtb_dense_kernel(const void* Xq, int64_t nq, const void* Xr, int64_t nr, int d, int x_is_f64, int what, int metric,
                     const double* bw_q, const double* bw_r, double decay, double thresh, int symm, double theta,
                     double* out, double* rowsum, void* stream);
int gtb_dense_row_scale(const double* in, const double* rowsum, int64_t nq, int64_t nr, double* out, void* stream);
int gtb_dense_anisotropy(double* K, const double* deg, double alpha, int64_t n, double* newsum, void* stream);
int gtb_dense_rowsum(const double* K, int64_t nq, int64_t nr, double* sum, void* stream);

/* ---- sparse x dense product (section 8f "next" rows): replaces scipy csr_matvecs behind
 * `transitions.dot(transform)` (DataGraph.interpolate, base.py:1195-1229), the callers' repeated
 * `diff_op.dot(X)` diffusion, and the sparse products inside sklearn randomized_svd(diff_aff)
 * (graphs.py:1216-1218) ---------------------------------------------------------------------- */
/* out[n_rows][ldo] (first f columns) = A . B, A = CSR float64, B row-major [n_cols][ldb] float64; every element
 * accumulated in stored order with separate multiply and add (bit-identical to scipy's A.dot(B)) */
int gtb_spmm_csr(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n_rows, const double* B,
                 int64_t ldb, int f, double* out, int64_t ldo, void* stream);
/* Chebyshev filter step of the diffusion-map eigensolver (graphtools_b200/eigen.py): out[n][ldo] (first f columns)
 * = (alpha (A . Y) + beta Y) + gamma Z for a square CSR float64 A [n x n] and row-major float64 Y, Z.  A . Y is
 * accumulated as gtb_spmm_csr does and every product and sum of the epilogue is rounded separately, so the result
 * is bit-identical to scipy's S = A.dot(Y) followed by numpy's alpha*S + beta*Y + gamma*Z.  out may be Z itself
 * (same pointer, ldo == ldz: the three-term recurrence rotates two buffers); out overlapping Y, or overlapping Z
 * in any other way, is rejected (GTB_ERR_ARG). */
int gtb_spmm_cheb(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n, const double* Y,
                  int64_t ldy, int f, double alpha, double beta, double gamma, const double* Z, int64_t ldz,
                  double* out, int64_t ldo, void* stream);
/* Step of a Chebyshev filter bank (graphtools_b200/gsp.py, pygsp's cheby_op): gtb_spmm_cheb's out, then for every
 * a < F: R[a * ldrb + i * ldr + k] = R[...] + coef[a] * out[i][k] (product and sum rounded separately, numpy's
 * `r += c * out`).  coef: F doubles in device memory; R: F blocks of [n][ldr] (first f columns), ldrb apart.  The
 * aliasing rules of gtb_spmm_cheb hold; R overlapping Y, Z or out, blocks of R overlapping each other, and coef
 * overlapping R or out are rejected (GTB_ERR_ARG). */
int gtb_spmm_cheb_acc(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n, const double* Y,
                      int64_t ldy, int f, double alpha, double beta, double gamma, const double* Z, int64_t ldz,
                      double* out, int64_t ldo, const double* coef, int F, double* R, int64_t ldr, int64_t ldrb,
                      void* stream);
/* Graph Laplacian of a square column-sorted CSR kernel K, W = K without its diagonal (pygsp's compute_laplacian;
 * csrc/gsp.cu): count writes dw[n] (sequential column-order sums of W's rows) and len[n] (row lengths of L: W's
 * entries plus one diagonal); after gtb_exclusive_scan(len) -> lptr, fill writes L's column-sorted indices and
 * values, lap_type 0 combinatorial (L = D - W) or 1 normalized (I - D^-1/2 W D^-1/2; zero-degree rows get L_ii = 0) */
int gtb_laplacian_count(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n, double* dw,
                        int32_t* len, void* stream);
int gtb_laplacian_fill(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n, const double* dw,
                       const int64_t* lptr, int lap_type, int32_t* lidx, double* lval, void* stream);
/* out[i][:] = in[i][:] * s[i]   (power_neg_half = 0)   or   in[i][:] / sqrt(s[i])   (power_neg_half = 1) */
int gtb_row_scale(const double* in, const double* s, int64_t n, int f, int power_neg_half, double* out,
                  void* stream);

/* ---- float64-faithful dense product on the INT8 tensor cores (section 8f row 3: the landmark diffusion chain
 * landmark_op^t the callers run through np.linalg.matrix_power on the operator of graphs.py:1240-1243) ------- */
/* Digit planes of a float64 operand.  Logical operand rows r < R of length K: row r of X[R][ld] (transposed = 0)
 * or column r of X[K][ld] (transposed = 1).  scale[r] = power of two with |row r| / scale[r] < 1/4; digits is
 * int8 [slices][R_pad][K_pad], zero padded, v / scale = sum_s digits[s] 2^(-8 (s + 1)) (balanced base-256 digits,
 * exact up to the truncation at 2^(-8 slices)).  R_pad, K_pad multiples of 128; 2 <= slices <= 7 */
int gtb_slice_f64(const double* X, int64_t R, int64_t K, int64_t ld, int transposed, int slices, int64_t R_pad,
                  int64_t K_pad, int8_t* digits, double* scale, void* stream);
/* C[M][ldc] (first N columns) = A . B from the digit planes of A's rows and B's columns (gtb_slice_f64): every digit
 * pair product of order s + t < slices is accumulated EXACTLY in int32 by tcgen05.mma kind::i8 and combined in
 * float64, C_ij = sa_i sb_j sum_o 2^(-8 (o + 2)) ACC_o.  K_pad <= gtb_gemm_max_k(); row_bytes = 32, 64 or 128
 * selects the shared-memory row length (swizzle) of one k-block and with it the pipeline depth (4, 2, 1 stages) */
int gtb_gemm_max_k(void);
int gtb_gemm_i8(const int8_t* a_digits, const int8_t* b_digits, int slices, int64_t M, int64_t N, int64_t K_pad,
                int64_t M_pad, int64_t N_pad, const double* sa, const double* sb, double* C, int64_t ldc,
                int row_bytes, void* stream);

/* ---- K10 all-pairs shortest paths: replaces scipy.sparse.csgraph.shortest_path behind BaseGraph.shortest_path
 * (base.py:934-988) ---------------------------------------------------------------------------------------------- */
/* Present (non-zero) entries of a dense float64 matrix as a column-sorted CSR, what csr_matrix(K) stores:
 * count -> gtb_exclusive_scan -> fill */
int gtb_dense_to_csr_count(const double* K, int64_t n_rows, int64_t n_cols, int32_t* cnt, void* stream);
int gtb_dense_to_csr_fill(const double* K, int64_t n_rows, int64_t n_cols, const int64_t* indptr, int32_t* idx,
                          double* val, void* stream);
/* len[nnz] = edge length of every stored entry: mode 0 K_ij, 1 |x_i - x_j|_2 of the rows X[n][d] (float32, or float64
 * when x_is_f64; numpy's pairwise summation order in that dtype), 2 -log(K_ij) correctly rounded.  *flags |= 1 when a
 * length is negative or NaN (the caller zeroes flags) */
int gtb_sp_lengths(const int64_t* indptr, const int32_t* idx, const double* val, int64_t n, const void* X, int d,
                   int x_is_f64, int mode, double* len, int32_t* flags, void* stream);
/* label[n] = smallest vertex of the weakly connected component (union-find over the stored entries) */
int gtb_sp_components(const int64_t* indptr, const int32_t* idx, int64_t n, int32_t* label, void* stream);
/* dist[n][batch] = shortest-path lengths from the nb <= batch sources src[] (column b: source src[b], +inf where
 * unreachable); batch is a multiple of 32, at most 1024; ws: gtb_sp_ws_bytes(n, batch) bytes.  Lengths must be
 * non-negative.  One cooperative launch (grid-wide barriers between relaxation rounds). */
int64_t gtb_sp_ws_bytes(int64_t n, int batch);
int gtb_sp_traverse(const int64_t* indptr, const int32_t* idx, const double* len, int64_t n, const int32_t* src, int nb,
                    int batch, double* dist, void* ws, void* stream);
/* out[src[b]][v] = dist[v][b] for b < nb (row stride ldo) */
int gtb_sp_store_rows(const double* dist, int batch, int64_t n, const int32_t* src, int nb, double* out, int64_t ldo,
                      void* stream);
/* in place on D[n][n]: (D + D^T) / 2, then 0 -> +inf off the diagonal, 0 on the diagonal */
int gtb_sp_finish(double* D, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GTB200_H */
