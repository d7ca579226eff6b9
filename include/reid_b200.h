/*
 * reid_b200.h -- C ABI of libreid_b200.so: the B200 (sm_100a) implementation of the
 * pseudo-label hot path of cluster-contrast-reid (daemon-219/ReID-GAN).
 *
 * The reference is 100% Python and has no FFI of its own; each entry point below
 * replaces the Python statement(s) cited next to it (paths relative to
 * cluster-contrast-reid-main/).  INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - every call is asynchronous on `stream` unless stated; no call allocates
 *     device memory: the caller owns inputs, outputs and scratch;
 *   - indices are int32, CSR row pointers int64, sets are sorted ascending;
 *   - rows [row_begin, row_end) are the caller's shard of the N query rows;
 *     "local" arrays are indexed by (row - row_begin), "global" arrays by row;
 *   - return value: REID_OK or a negative code; reid_last_error() (thread local)
 *     describes the last failure.  No exception crosses this boundary and there
 *     is no CPU fallback behind any entry.
 */
#ifndef REID_B200_H_
#define REID_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define REID_OK 0
#define REID_ERR_INVALID_ARG (-1)
#define REID_ERR_CUDA (-2)
#define REID_ERR_NCCL (-3)          /* reserved: collectives live in the host layer (torch.distributed), no entry returns it */
#define REID_ERR_CERTIFICATE (-4)
#define REID_ERR_UNSUPPORTED (-5)

#define REID_MAX_K1 64 /* rank positions are kept in 64-bit masks */

int reid_abi_version(void);
const char* reid_last_error(void);
/* kernels launched by the library in this process (bench.py's gpu_launches) */
uint64_t reid_launch_count(void);

/* ---- utilities ---------------------------------------------------------- */

/* ptr_out[0..n] = exclusive prefix sum of cnt[0..n-1] (ptr_out[n] = total);
 * stats_out (optional, 3 x int64) = {total, max(cnt), sum(cnt^2)}.  One multi-CTA pass (decoupled look-back), 64-bit
 * sums throughout.  The tile state lives in a small library-owned buffer per (device, stream), created at the first
 * call on that stream -- so the first call must not happen inside a stream capture. */
int reid_scan_counts(const int32_t* cnt, int64_t n, int64_t* ptr_out, int64_t* stats_out, void* stream);

/* ---- a1: kNN search  (utils/faiss_rerank.py:58-62, faiss IndexFlatL2.search) ----
 * Exact top-k of  key(i,j) = fp32( sum_d x[i,d]*x[j,d] accumulated in fp64 ),
 * ordered by (key descending, j ascending) -- for unit-norm rows the L2-ascending
 * order faiss returns.  Query rows are rows_list[0..n_rows) (or row_begin + r when
 * rows_list is NULL); all N rows are searched, self included.
 * scratch: at least reid_knn_exact_scratch_bytes(N, 1) bytes; more lets more query
 * rows go per pass. */
size_t reid_knn_exact_scratch_bytes(int64_t N, int64_t n_rows);
int reid_knn_exact(const float* x, int64_t N, int64_t D, const int32_t* rows_list, int64_t row_begin,
                   int64_t n_rows, int k, int32_t* out_idx, float* out_key, void* scratch,
                   size_t scratch_bytes, void* stream);
/* The same search for rows that do NOT all have one norm (faiss IndexFlatL2 ranks by squared L2, which is the
 * inner-product order only then):  key(i,j) = fp32( x_i.x_j - ||x_j||^2 / 2 in fp64 ), descending, j ascending --
 * squared L2 ascending with the per-query constant ||x_i||^2 dropped.  out_key receives that key (not the dot).
 * scratch: 256-byte-rounded N doubles (the half norms) + at least N floats. */
/* sqnorm_range[0..1] = { max_i ||x_i||^2, min_i ||x_i||^2 } (fp32): decides between the two keys */
int reid_sqnorm_range(const float* x, int64_t N, int64_t D, float* sqnorm_range, void* stream);
int reid_knn_exact_l2(const float* x, int64_t N, int64_t D, const int32_t* rows_list, int64_t row_begin,
                      int64_t n_rows, int k, int32_t* out_idx, float* out_key, void* scratch,
                      size_t scratch_bytes, void* stream);

/* Tensor-core candidate search: fp16 tcgen05 GEMM (TMA-fed, TMEM accumulators) of query rows
 * [row_begin,row_end) against all N rows with a fused per-row running top-`keep` selection in the
 * epilogue.  xh = fp16(x * 2^scale_log2), row-major N x D, D % 64 == 0, 16-byte aligned.
 * The N columns are cut into n_splits ranges (reid_knn_tc_plan picks the count that fills the SMs) and
 * inside a range the 256-column tiles alternate between the two epilogue groups of the kernel, so every
 * row owns n_lists = 2 * n_splits candidate lists:
 *   cand[((row-row_begin)*n_lists + l)*REID_TC_CAP + p] = (fp32 score bits << 32) | column,
 *   p < cand_cnt[(row-row_begin)*n_lists + l] <= REID_TC_CAP.
 * A column appears at most once across a row's lists (reid_knn_rescore ranks by counting strictly greater keys).
 * row_tau[row-row_begin] (order-preserving integer image of a float, 0 = none) is the row's final
 * rejection threshold: every column that is in none of the row's lists scored <= that value, and at
 * least `keep` listed columns score >= it.  Scores are approximate (fp16 inputs); see reid_knn_rescore.
 * cta_group = 1: one CTA per 128-row tile; 2: a CTA pair per 256-row tile (tcgen05 cta_group::2,
 * the column tile is fetched once per pair). */
#define REID_TC_CAP 512
#define REID_TC_KEEP_MAX 64
#define REID_TC_MAX_SPLITS 4
int reid_knn_tc_plan(int64_t N, int64_t n_rows, int cta_group, int* n_splits_out);
int reid_knn_candidates_tc(const void* xh, int64_t N, int64_t D, int scale_log2, int64_t row_begin,
                           int64_t row_end, int keep, int n_splits, int cta_group, uint64_t* cand,
                           int32_t* cand_cnt, uint32_t* row_tau, void* stream);
/* Same kernel with distinct operands: query rows [row_begin,row_end) of xa (Na x D) against all N rows of xb
 * (column ids = row index in xb).  Used by the sampling prepass of the symmetric search below: a NEGATIVE keep
 * selects its mode (|keep| entries kept; every list seeds its threshold with the 5th largest of its first 32
 * scores instead of taking the first tiles unfiltered -- good for an order statistic, not for a top-k). */
int reid_knn_candidates_tc_ab(const void* xa, int64_t Na, const void* xb, int64_t N, int64_t D, int scale_log2,
                              int64_t row_begin, int64_t row_end, int keep, int n_splits, int cta_group,
                              uint64_t* cand, int32_t* cand_cnt, uint32_t* row_tau, void* stream);

/* Symmetric candidate search (single GPU, all N rows): S = Xh Xh^T is symmetric, so only the 256 x 256 tiles
 * (I, J), I <= J, go through the tensor cores and each off-diagonal tile feeds the lists of both its row
 * block and its column block -- half the tcgen05 work and half the operand traffic of reid_knn_candidates_tc.
 * Selection is against a FIXED per-row threshold tau[i] (reid_knn_sample_tau): every column j with
 * approximate score > tau[i] is appended to row i's single list
 *   cand[i * cap + p] = (fp32 score bits << 32) | j,  p < min(cand_cnt[i], cap);
 * cand_cnt[i] > cap means the list overflowed (reid_knn_rescore un-certifies such rows).
 * tiles: n_tiles (I, J) int32 pairs in processing order (the host orders them for L2 locality). */
#define REID_SYM_CAP 1024
int reid_knn_candidates_sym(const void* xh, int64_t N, int64_t D, int scale_log2, const float* tau,
                            const int32_t* tiles, int64_t n_tiles, int cap, uint64_t* cand, int32_t* cand_cnt,
                            int reset_counts, void* stream);
/* reset_counts = 0 keeps appending to the lists of earlier launches: the tiles may be issued in several launches
 * as the feature rows arrive from the host (tiles whose rows are all resident), see knn_tc.knn_search_upload. */
/* The same search over 256 x 512 strips: units = n_units int32 triples (I, J0, J1), the tiles (I, J0) and (I, J1) of
 * one row block (J1 = -1: a single tile), both accumulated from ONE A slice per K step -- 48 KB instead of 64 KB of
 * operands per pair of tiles through the L2 -> shared-memory feed that bounds the kernel.  Same lists (as sets; the
 * order inside a list is the order of the atomics in either flavour).  knn_tc.pair_units builds the triples from the
 * tile order.  (replaces the same lines as reid_knn_candidates_sym: utils/faiss_rerank.py:39-62) */
int reid_knn_candidates_sym_wide(const void* xh, int64_t N, int64_t D, int scale_log2, const float* tau,
                                 const int32_t* units, int64_t n_units, int cap, uint64_t* cand, int32_t* cand_cnt,
                                 int reset_counts, void* stream);
/* n_rows rows of row_bytes each, src_pitch_bytes apart in (pinned) HOST memory -> packed on the device
 * (cudaMemcpy2DAsync): the regularly strided threshold sample goes up before the bulk of the features. */
int reid_upload_rows_strided(void* dst, const void* src_host, size_t row_bytes, size_t src_pitch_bytes,
                             int64_t n_rows, void* stream);
/* xs[m] = xh[(m * stride) mod N], m < n_sample: a low-discrepancy sample of the rows (stride coprime with N). */
int reid_features_sample(const void* xh, int64_t N, int64_t D, int64_t n_sample, int64_t stride, void* xs,
                         void* stream);
/* tau[row] = r-th largest score over the row's prepass lists (reid_knn_candidates_tc_ab against the sample),
 * tau_ord = its order-preserving integer image (0 / -inf when fewer than r scores are listed). */
int reid_knn_sample_tau(const uint64_t* cand, const int32_t* cand_cnt, const uint32_t* row_tau, int n_lists,
                        int64_t n_rows, int r, float* tau, uint32_t* tau_ord, void* stream);

/* ---- sample-first layout of the symmetric search (knn_tc._candidates_sym_sf; replaces the same lines,
 * utils/faiss_rerank.py:39-62).  The fp16 operand is written with the threshold sample in its first m rows
 * (reid_features_to_half_gather), and the block column [0, m) of the matrix -- all rows against the sample --
 * gives both the thresholds and candidates the symmetric pass needs: it is scored once, its scores go to the main
 * lists in both directions, and the symmetric pass runs only the tiles (I, J) with m / 256 <= I <= J (12 % fewer
 * tcgen05 tiles at N = 32,621, m = 2,048).  The sample rows against the sample run through the prepass entries:
 *   reid_knn_candidates_tc_abt : reid_knn_candidates_tc_ab + the transposed direction -- tau_col[j] is the (already
 *       known) threshold of column row j; every score above it is appended to cand_col[j * cap_col + ..] with the
 *       query row as its column (tau_col = NULL: off); publish_final: row_tau additionally receives every list's final
 *       rejection threshold (the seeds of the prepass mode included), so that it bounds everything any list of the
 *       row ever rejected;
 *   reid_knn_sample_tau_emit   : reid_knn_sample_tau + the direct direction -- the listed scores above tau[row] go to
 *       the main list of row row0 + row (cand_main = NULL: plain reid_knn_sample_tau).  Here tau is raised to the
 *       published floor of the prepass lists (they are complete only above it; needs publish_final), which is also the
 *       threshold when fewer than r scores are listed above the floor;
 *   reid_knn_rescore_mapped    : reid_knn_rescore on lists that live in the permuted row space -- row r's lists and
 *       threshold are those of position row_pos[r], a listed column p is the original row col_orig[p] (both NULL:
 *       plain reid_knn_rescore).
 * The other rows against the sample run on the symmetric kernel with a provisional threshold: a row only needs a
 * threshold that every unlisted column scored at or below, and a lower one only lengthens its list:
 *   reid_knn_tau_floor         : tau' = the smallest of the sample rows' thresholds tau_ord[0, m), written to tau[m, N)
 *       and tau_ord[m, N) -- on the device, no host round trip;
 *   reid_knn_candidates_sym_tiles : reid_knn_candidates_sym, for the tiles (I, J) with I < m / 256 <= J: sample row i
 *       lists column j above tau[i], row j lists sample column i above tau[j] = tau'.  A separate entry so that the
 *       per-entry timings keep the block column apart from the symmetric pass over the other tiles;
 *   reid_knn_list_tau          : for rows [row0, row0 + n_rows) whose list holds exactly their scores above tau_ord[row]
 *       (here: the sample scores above tau'), raise tau[row] / tau_ord[row] to the r-th best listed score (its top 16
 *       bits, rounded down) when at least r are listed and it is higher; otherwise tau' stays.  Only the first
 *       min(cand_cnt[row], cap, 1024) entries are read (a subset can only lower the result). */
/* xh[i] = fp16(2^s x[src_row[i]]), i < n_rows; max_sqnorm_inout accumulates like reid_features_to_half_acc */
int reid_features_to_half_gather(const float* x, const int32_t* src_row, int64_t n_rows, int64_t D, int scale_log2,
                                 void* xh, float* max_sqnorm_inout, void* stream);
int reid_knn_candidates_tc_abt(const void* xa, int64_t Na, const void* xb, int64_t N, int64_t D, int scale_log2,
                               int64_t row_begin, int64_t row_end, int keep, int n_splits, int cta_group,
                               uint64_t* cand, int32_t* cand_cnt, uint32_t* row_tau, int publish_final,
                               const float* tau_col, uint64_t* cand_col, int32_t* cand_col_cnt, int cap_col,
                               void* stream);
int reid_knn_sample_tau_emit(const uint64_t* cand, const int32_t* cand_cnt, const uint32_t* row_tau, int n_lists,
                             int64_t n_rows, int r, float* tau, uint32_t* tau_ord, uint64_t* cand_main,
                             int32_t* cand_main_cnt, int cap_main, int64_t row0, void* stream);
int reid_knn_rescore_mapped(const float* x, int64_t N, int64_t D, int64_t row_begin, int64_t row_end,
                            const uint64_t* cand, const int32_t* cand_cnt, const uint32_t* row_tau, int n_lists,
                            int list_cap, int64_t list_pitch_rows, int k, float err_bound, const float* max_sqnorm,
                            int locality_order, const int32_t* row_pos, const int32_t* col_orig, int32_t* out_idx,
                            float* out_key, int32_t* uncertified_flag, float* max_err_out, void* workspace,
                            uint64_t* uncertified_count, void* stream);
int reid_knn_tau_floor(float* tau, uint32_t* tau_ord, int64_t m, int64_t N, void* stream);
int reid_knn_candidates_sym_tiles(const void* xh, int64_t N, int64_t D, int scale_log2, const float* tau,
                                  const int32_t* tiles, int64_t n_tiles, int cap, uint64_t* cand, int32_t* cand_cnt,
                                  int reset_counts, void* stream);
int reid_knn_list_tau(const uint64_t* cand, const int32_t* cand_cnt, int cap, int64_t row0, int64_t n_rows, int r,
                      float* tau, uint32_t* tau_ord, void* stream);

/* fp32 features -> scaled fp16 operand; max_sqnorm_out (optional, TWO floats) = { max_i ||x_i||^2, min_i ||x_i||^2 }:
 * the maximum scales the fp16 rounding bound  |approx - exact| <= 2^-10 ||x_i|| ||x_j||, the pair tells the caller
 * whether all rows have one norm (inner-product order == the reference's L2 order) or reid_knn_exact_l2 is needed.
 * Limit: a component with |x| * 2^scale_log2 >= 65520 rounds to +-inf in fp16 and no bound holds for its row's scores;
 * the maximum is then reported as +inf (no row can be certified), and the minimum stays the true one -- a caller that
 * needs the true maximum recomputes it with reid_sqnorm_range.  The same holds for _acc and _gather. */
int reid_features_to_half(const float* x, int64_t n_rows, int64_t D, int scale_log2, void* xh,
                          float* max_sqnorm_out, void* stream);
/* { 0, 3.4e38 }: the identities of the { max, min } pair, for reid_features_to_half_acc */
int reid_sqnorm_range_reset(float* sqnorm_range, void* stream);
/* same, but max_sqnorm_inout (two floats, initialised by the caller to { 0, a huge value }) is NOT reset: a matrix
 * converted in several row blocks accumulates one maximum and one minimum */
int reid_features_to_half_acc(const float* x, int64_t n_rows, int64_t D, int scale_log2, void* xh,
                              float* max_sqnorm_inout, void* stream);

/* Exact re-score of the candidates with the canonical key, certificate, final order.
 * Let a_(k) be the k-th best approximate score of a row.  Every member of the exact top-k has an
 * approximate score >= a_(k) - 2*err_bound (the "window").  The row is certified when its rejection
 * threshold row_tau lies below the window -- then the window, hence the exact top-k, is entirely among
 * the listed candidates.  Window members are re-scored with
 * fp32(fp64 dot) and ordered by (key desc, index asc): bit-identical to reid_knn_exact.
 * |approx - exact| is audited against err_bound; a violation un-certifies the row.
 * uncertified_flag[row-row_begin] = 1 marks rows the caller must redo with reid_knn_exact;
 * max_err_out (1 float) = largest |approx - exact| seen.
 * max_sqnorm (optional device scalar from reid_features_to_half): when given, err_bound is derived on the
 * device as 1.02 * 2^-10 * max_sqnorm + 2^-14 and the err_bound argument is ignored (no host round trip).
 * locality_order != 0: the exact stage gathers ~36 feature rows per query row and is HBM bound; rows of one
 * identity cluster share their candidates, so they are visited back to back (counting sort on the smallest
 * index among a row's strong candidates) and repeats become L2 hits.
 * The lists must be free of duplicates: no column twice across one row's lists.
 * list_cap: entries reserved per list (REID_TC_CAP for reid_knn_candidates_tc, the cap given to
 * reid_knn_candidates_sym); a count above it marks an overflowed list and un-certifies the row.
 * list_pitch_rows: 0 = lists are row-major, list l of local row r at index r * n_lists + l (what the candidate
 * kernels write); > 0 = list-major, index l * list_pitch_rows + r (what an all-to-all of per-rank partial lists
 * leaves behind in the tile-sharded multi-GPU search).
 * workspace: reid_knn_rescore_workspace_bytes(N, row_end - row_begin). */
int reid_knn_rescore(const float* x, int64_t N, int64_t D, int64_t row_begin, int64_t row_end,
                     const uint64_t* cand, const int32_t* cand_cnt, const uint32_t* row_tau, int n_lists,
                     int list_cap, int64_t list_pitch_rows, int k, float err_bound, const float* max_sqnorm, int locality_order, int32_t* out_idx, float* out_key,
                     int32_t* uncertified_flag, float* max_err_out, void* workspace, uint64_t* uncertified_count,
                     void* stream);
/* uncertified_count (optional device scalar): += number of rows whose flag is set -- lets a caller that does not
 * want a host round trip here read the count later together with its other sizes. */
size_t reid_knn_rescore_workspace_bytes(int64_t N, int64_t n_rows);
/* byte offset, inside that workspace, of the int32[n_rows] window sizes of the last call (for reporting the
 * bytes the exact stage really had to gather) */
size_t reid_knn_rescore_window_counts_offset(int64_t N, int64_t n_rows);
/* byte offset of the int32[n_rows] cluster-locality visiting order (a permutation of the local rows; valid when the
 * call had locality_order != 0): reid_v_weights can walk the rows in the same order */
size_t reid_knn_rescore_order_offset(int64_t N, int64_t n_rows);

/* ---- a2: reciprocal sets  (faiss_rerank.py:23-27, 65-69) -----------------------
 * mask_out[row - row_begin] bit r  <=>  row in rank[rank[row,r], :cols], cols = min(k+1, ncols).
 * R_k(row) = { rank[row, r] : bit r set }, in rank order. */
int reid_reciprocal_masks(const int32_t* rank, int64_t N, int ncols, int k, int64_t row_begin,
                          int64_t row_end, uint64_t* mask_out, void* stream);
/* Both sets of the loop at :65-69 in one pass: R_out[row - row_begin] = mask for k_full (rows [row_begin, row_end) only),
 * Rhalf_out[row] = mask for k_half (ALL N rows: a row-sharded pass needs R_half of every row, R only of its own). */
int reid_reciprocal_masks2(const int32_t* rank, int64_t N, int ncols, int k_full, int k_half, int64_t row_begin,
                           int64_t row_end, uint64_t* R_out, uint64_t* Rhalf_out, void* stream);

/* ---- a3: expansion  (faiss_rerank.py:72-80) ------------------------------------
 * E(row) = sort_unique( R(row) + all R_half(c), c in R(row), 3*|R_half(c) & R(row)| > 2*|R_half(c)| ).
 * One pass into padded rows: E_pad[(row-row_begin)*stride + t], t < E_cnt[row-row_begin].  A row that does
 * not fit reports E_cnt = stride + 1 (stride >= k1 + k1*(k1/2 + 1) always fits).  Rmask is local,
 * Rhalf_mask is global (all N rows); half_cols = the `cols` of the reid_reciprocal_masks call that made it
 * (no R_half mask has a bit at or above it) -- it sizes the per-warp pair buffer. */
int reid_expand(const int32_t* rank, int64_t N, int ncols, int half_cols, const uint64_t* Rmask,
                const uint64_t* Rhalf_mask, int64_t row_begin, int64_t row_end, int stride, int32_t* E_pad,
                int32_t* E_cnt, void* stream);

/* ---- a4: Gaussian weights  (faiss_rerank.py:81-85) ------------------------------
 * V_val[p] = softmax over the row of -(2 - 2 x_row.x_e), e in E(row); fp32.  Reads the padded sets of
 * reid_expand and writes the CSR (E_idx, V_val) at E_ptr (local, from a scan of E_cnt) in the same pass.
 * rank/rank_key (optional, the shard's rows of the search result) let the kernel reuse the search keys
 * for members that are among the row's k1 neighbours instead of gathering 4*D bytes.
 * visit_order (optional): a permutation of the local rows to walk them in (reid_knn_rescore's cluster-locality
 * order): cluster mates gather the same feature rows and find them in L2.  The output does not depend on it. */
int reid_v_weights(const float* x, int64_t N, int64_t D, const int32_t* E_pad, int stride, const int64_t* E_ptr,
                   int64_t row_begin, int64_t row_end, const int32_t* rank_local, const float* rank_key_local,
                   int ncols, const int32_t* visit_order, int32_t* E_idx, float* V_val, int half_precision, void* stream);
/* half_precision (here, in reid_query_expand, reid_jaccard_eps_graph and reid_jaccard_dense) = the reference's
 * use_float16=True (faiss_rerank.py:37): V, V_qe, the running Jaccard sums and the distances are float16 ARRAYS there,
 * and numpy evaluates every float16 operation in float32 and rounds the result to float16.  The kernels keep fp32
 * storage and apply exactly those roundings (V after the fp32 softmax; V_qe after sum / k2, entries that round to zero
 * leave the structure; the min-sum after every column; each of the three operations of 1 - t / (2 - t)). */

/* ---- a5: k2 query expansion  (faiss_rerank.py:89-94) ----------------------------
 * Vq[row] = (V[rank[row,0]] + ... + V[rank[row,k2-1]]) / k2, adds in that order, fp32.
 * V is the GLOBAL CSR (all N rows); max_row_nnz = max |E|.  One pass into padded rows of
 * reid_query_expand_stride(k2, max_row_nnz) slots; reid_csr_compact packs them into a CSR.
 * A caller that has not read max |E| back may pass a guess: a row whose distinct columns do not fit the table
 * sized from it reports Q_cnt = 0 and is counted in *overflow_rows (optional device scalar, accumulates); with the
 * true maximum no row can overflow. */
int reid_query_expand_stride(int k2, int max_row_nnz);
int reid_query_expand(const int32_t* rank, int64_t N, int ncols, int k2, const int64_t* V_ptr,
                      const int32_t* V_idx, const float* V_val, int max_row_nnz, int64_t row_begin,
                      int64_t row_end, int32_t* Q_cnt, int32_t* Q_pad_idx, float* Q_pad_val, uint64_t* overflow_rows,
                      int half_precision, void* stream);
int reid_csr_compact(const int32_t* pad_idx, const float* pad_val, int64_t stride, const int32_t* cnt,
                     const int64_t* ptr, int64_t n_rows, int32_t* out_idx, float* out_val, void* stream);

/* neighbour lists kept in upper-bound slots (reid_jaccard_neighbors) -> packed at ptr (before an all-gather) */
int reid_lists_compact(const int64_t* slot_ptr, const int32_t* idx, const int32_t* cnt, const int64_t* ptr,
                       int64_t n_rows, int32_t* out, void* stream);

/* ---- multi-GPU exchange format of the row-sharded plan -------------------------------------
 * One fixed-stride record per row: rec[row] = { count, idx[stride], (val bits[stride]) } in int32 words, so that a
 * single all-gather moves a ragged stage output (V rows, V_qe rows, eps-neighbour lists).
 *   pack   : local rows (cnt, starts `ptr` into idx / val; val may be NULL) -> n_rows_padded records (padding: count 0)
 *   unpack : gathered records of `world` ranks (max_rows records each; rank r owns rows [bounds[r], bounds[r+1]))
 *            -> global counts; after the caller's scan -> global CSR.  A count above `stride` means the row did
 *            not fit: the caller must fall back to a variable-length exchange. */
int reid_rows_pack(const int32_t* cnt, const int64_t* ptr, const int32_t* idx, const float* val, int64_t n_rows,
                   int64_t n_rows_padded, int stride, int32_t* rec, void* stream);
int reid_rows_unpack_counts(const int32_t* rec, int stride, int has_val, int world, int64_t max_rows,
                            const int64_t* bounds, int64_t N, int32_t* g_cnt, uint64_t* overflow_rows, void* stream);
/* overflow_rows (optional device scalar, accumulates): with it a row whose count exceeds `stride` is counted there and
 * its count clamped to what travelled -- for a pass that does not read sizes back and is redone if the scalar is set. */
int reid_rows_unpack_fill(const int32_t* rec, int stride, int world, int64_t max_rows, const int64_t* bounds,
                          int64_t N, const int64_t* g_ptr, int32_t* out_idx, float* out_val, void* stream);

/* ---- a6: inverted index  (faiss_rerank.py:98-100) -------------------------------
 * CSC of a CSR with n_rows x n_cols; column lists sorted by row.
 * Step 1 writes col_cnt; caller scans it into C_ptr; step 2 fills.  cursor: n_cols int32 scratch.
 * nnz_dev (optional device scalar): the real nnz when the host only knows the upper bound `nnz` (no read-back).
 * max_col_len: the longest column (sizes the shared-memory sort), or <= 0 when the caller has not read it back:
 * columns of up to 256 entries are then sorted by warps and a second launch gives every longer one a whole CTA. */
int reid_transpose_count(const int32_t* idx, int64_t nnz, const int64_t* nnz_dev, int64_t n_cols, int32_t* col_cnt,
                         void* stream);
int reid_transpose_fill(const int64_t* ptr, const int32_t* idx, const float* val, int64_t n_rows,
                        int64_t n_cols, const int64_t* C_ptr, int32_t* cursor, int32_t* C_idx, float* C_val,
                        int max_col_len, void* stream);

/* ---- a7: Jaccard min-sum  (faiss_rerank.py:102-119) -----------------------------
 * t_ij = sum over shared columns c (ascending) of min(Vq[i,c], Vq[j,c]) in sequential fp32;
 * J = max(0, 1 - t/(2-t)); pairs without a shared column have J == 1 exactly.
 * Q (CSR) and C (CSC) are global. */
/* T_cnt[row-row_begin] = sum_c |col(c)|: the work of the row and an upper bound of its number of distinct partners.
 * S_cnt (optional, needs Q_val): a much tighter bound of the number of eps-NEIGHBOURS, min(T, B / t_min + 2) with
 * B = sum_c Vq[row,c] |col(c)| >= sum_j t_ij and t_min the smallest t with J(t) <= eps (Markov); scanning S_cnt
 * instead of T_cnt gives slots of about twice the edge count instead of sum_c |col(c)|^2. */
int reid_jaccard_bounds(const int64_t* Q_ptr, const int32_t* Q_idx, const float* Q_val, const int64_t* C_ptr,
                        int64_t row_begin, int64_t row_end, float eps, int32_t* T_cnt, int32_t* S_cnt, int32_t* P_cnt,
                        void* stream);
/* P_cnt (optional): a GUESS of the row's number of distinct partners, min(T-based, 3 x longest column + nnz(row)); it
 * only picks the hash-table class of the row's first attempt in reid_jaccard_eps_graph (NULL there: the T-based guess). */
/* eps-neighbourhoods { j : J_ij <= eps } (what DBSCAN consumes), written at slot_ptr (local, from a
 * scan of T_cnt); nbr_cnt[row-row_begin] = size, or -1 when the row overflowed the shared-memory
 * table (redo those rows with a larger table_slots).  J values optional (nbr_val may be NULL).
 * rows_list (optional): local row ids to process instead of the whole shard. */
int reid_jaccard_neighbors(const int64_t* Q_ptr, const int32_t* Q_idx, const float* Q_val,
                           const int64_t* C_ptr, const int32_t* C_idx, const float* C_val, int64_t N,
                           int64_t row_begin, int64_t row_end, const int32_t* rows_list, int64_t n_list,
                           float eps, const int64_t* slot_ptr, int32_t* nbr_idx, float* nbr_val,
                           int32_t* nbr_cnt, int table_slots, void* stream);
/* same contract for the rows of rows_list that overflowed every table ("hub" rows): dense accumulator
 * rows in `scratch` (n_list x N floats), neighbours written in ascending j. */
int reid_jaccard_neighbors_heavy(const int64_t* Q_ptr, const int32_t* Q_idx, const float* Q_val,
                                 const int64_t* C_ptr, const int32_t* C_idx, const float* C_val, int64_t N,
                                 int64_t row_begin, const int32_t* rows_list, int64_t n_list, float eps,
                                 const int64_t* slot_ptr, int32_t* nbr_idx, float* nbr_val, int32_t* nbr_cnt,
                                 float* scratch, void* stream);
/* The whole eps-graph of the shard in one call, no host round trip: rows are dealt to shared-memory table
 * classes (512 .. 8192 slots) on the device from T_cnt (reid_jaccard_bounds), overflowing rows move up a
 * class, the last resort is the dense-accumulator kernel.  nbr_cnt is never -1 on return.
 * slot_ptr: n + 1 entries (a scan of T_cnt or S_cnt); row r owns [slot_ptr[r], slot_ptr[r+1]).  No kernel writes
 * outside a row's slots or at / beyond nbr_capacity (<= 0: unlimited): a row with more neighbours than slots stores
 * (and counts in nbr_cnt) only what fits and is counted in *slot_overflow (optional device scalar) -- with slots
 * from T_cnt that cannot happen.
 * workspace: reid_jaccard_eps_graph_workspace_bytes(N, row_end - row_begin). */
size_t reid_jaccard_eps_graph_workspace_bytes(int64_t N, int64_t n_rows);
int reid_jaccard_eps_graph(const int64_t* Q_ptr, const int32_t* Q_idx, const float* Q_val, const int64_t* C_ptr,
                           const int32_t* C_idx, const float* C_val, int64_t N, int64_t row_begin,
                           int64_t row_end, float eps, const int32_t* T_cnt, const int32_t* P_cnt, const int64_t* slot_ptr,
                           int32_t* nbr_idx, float* nbr_val, int32_t* nbr_cnt, int64_t nbr_capacity,
                           uint64_t* slot_overflow, int half_precision, int owned_pairs_only, uint64_t* escalated_rows,
                           void* workspace, void* stream);
/* escalated_rows (optional device scalar, accumulates): rows whose first table was too small and that were moved to a
 * bigger class -- tells the caller whether the P_cnt guess suits the data. */
/* owned_pairs_only: J is bit-symmetric, so each unordered pair {i, j} may be accumulated and listed by only ONE of its
 * rows -- i owns (i, j) iff i == j, or i < j with i + j even, or i > j with i + j odd (every row keeps about half of its
 * partners).  Half the table updates; reid_dbscan_labels(owned_pairs = 1) consumes such lists. */
/* dense rows: out[(row-row_begin)*ld + j] for all j < N  (the reference's return value). */
int reid_jaccard_dense(const int64_t* Q_ptr, const int32_t* Q_idx, const float* Q_val, const int64_t* C_ptr,
                       const int32_t* C_idx, const float* C_val, int64_t N, int64_t row_begin,
                       int64_t row_end, float* out, int64_t ld, int half_precision, void* stream);

/* ---- a8: DBSCAN on precomputed distances -----------------------------------------
 * (examples/cluster_contrast_train_usl.py:160,163; sklearn/cluster/_dbscan.py:397-475)
 * neighbourhood = { j : d_ij <= eps } in fp32, self included; core <=> |nbr| >= min_samples;
 * cluster ids 0.. by ascending smallest core index; border -> smallest adjacent core label; noise -1. */
/* dense input (drop-in class): two passes over rows [row_begin,row_end) of an n x n matrix */
int reid_dbscan_dense_count(const float* dist, int64_t N, int64_t ld, float eps, int64_t row_begin,
                            int64_t row_end, int32_t* nbr_cnt, void* stream);
int reid_dbscan_dense_fill(const float* dist, int64_t N, int64_t ld, float eps, int64_t row_begin,
                           int64_t row_end, const int64_t* nbr_ptr, int32_t* nbr_idx, void* stream);
/* labelling from neighbour lists of ALL N rows: list of row i = nbr_idx[nbr_ptr[i] .. +nbr_cnt[i]).
 * workspace: reid_dbscan_workspace_bytes(N).  labels: int64 (numpy intp); core_mask: uint8 (optional). */
size_t reid_dbscan_workspace_bytes(int64_t N);
int reid_dbscan_labels(int64_t N, const int64_t* nbr_ptr, const int32_t* nbr_idx, const int32_t* nbr_cnt,
                       int min_samples, int64_t* labels, uint8_t* core_mask, int64_t* num_clusters_out,
                       void* workspace, int owned_pairs, void* stream);
/* owned_pairs != 0: the lists name every edge {i, j} ONCE (reid_jaccard_eps_graph with owned_pairs_only; the self pair
 * (i, i) is in i's list when d_ii <= eps): degrees are counted from both ends, the union-find needs each edge once
 * anyway, border points take the smallest adjacent core label from whichever end lists the edge. */

/* ---- f1 (next row): edge filter of the Infomap variant  (utils/infomap_cluster.py:129-144) ----
 * nbrs / dists: (N, k) neighbour lists in ascending distance 1 - sim (reid_knn_* keys give sim).  Row i links to
 * every non-self entry up to the first one with dist > 1 - min_sim (compared in fp64 like the reference's
 * float64 arrays); weight = 1 - dist.  Count, scan (reid_scan_counts), fill; rows with count 0 are "single". */
int reid_links_count(const int32_t* nbrs, const float* dists, int64_t N, int k, double min_sim, int32_t* link_cnt,
                     void* stream);
int reid_links_fill(const int32_t* nbrs, const float* dists, int64_t N, int k, double min_sim,
                    const int64_t* link_ptr, int32_t* link_dst, double* link_weight, void* stream);

/* ---- f2 (next row): evaluation-time re-ranking  (utils/rerank.py re_ranking :31-97) ----------
 * dense front end: dist (M x M, M = Q + G) = transpose( block^2 / column max ) of [[q_q, q_g], [q_g^T, g_g]]
 * (:36-41); scratch_mm: M*M floats, colmax: M floats.  The neighbour lists are reid_select_rows(dist, ascending)
 * (:43 argsort, first k1+1 columns; ties by index), the sets / V_qe / inverted index / Jaccard rows are the entries
 * above, the weights are exp(-dist) normalised per row (:66-67), the result is (1-lambda) J + lambda dist (:95-96). */
int reid_rr_normalised_distance(const float* q_g, const float* q_q, const float* g_g, int64_t Q, int64_t G,
                                float* scratch_mm, float* colmax, float* dist, void* stream);
int reid_rr_weights(const float* dist, int64_t M, const int32_t* E_pad, int stride, const int64_t* E_ptr,
                    int64_t n_rows, int32_t* E_idx, float* V_val, void* stream);
int reid_rr_final(const float* J, int64_t ldJ, const float* dist, int64_t Q, int64_t G, float one_minus_lambda,
                  float lambda, float* out, void* stream);

/* ---- f2 from features (re_ranking_features): the same result from the (M x D) union x = [query; gallery] ----
 * Nothing of M^2 elements exists.  With orig(r, c) = sq(r, c)^2 and colmax[c] = max_r orig(r, c), dist[i, j] =
 * orig(j, i) / colmax[i]: the neighbour lists are the squared-L2 kNN of x (reid_knn_*), colmax comes from a
 * farthest-neighbour search, the weights and the blend read gathered feature rows and the Q x G distance block.
 * Distance arithmetic of these entries: sqnorm[i] = sum_d x[i,d]^2 and the dot x_i.x_j accumulated in fp64 (one fixed
 * order, so sq(i, j) and sq(j, i) have the same bits), sq(i, j) = fp32((sqnorm[i] + sqnorm[j]) - 2 x_i.x_j) formed in
 * fp64, orig = fp32(sq * sq).
 *   reid_rr_row_sqnorm64     : sqnorm[i] (fp64) for i < n_rows -- the norms the other entries take.
 *   reid_rr_farthest_certify : colmax of rows [row_begin, row_end) from the candidate lists of
 *       reid_knn_candidates_tc_ab run with the NEGATED fp16 operand as xb (scores ~ -x_i.x_j; lists row-major,
 *       n_lists per row, list_cap entries each).  sqnorm_range = { max, min } fp32 squared norms
 *       (reid_features_to_half) gives the fp16 error bound eps and the norm spread.  With a_max the best listed score,
 *       the row is certified when no list overflowed and its rejection threshold lies below
 *       lo = a_max - 2 eps - (max - min) / 2; then the farthest row is among the listed entries >= lo, which are
 *       re-scored exactly (at most 128; every |approx - exact| is audited against eps).  A certified row gets its
 *       exact colmax; an uncertified one gets colmax 0, uncertified_flag[row - row_begin] = 1 and
 *       *uncertified_count += 1 (optional) -- the caller redoes it with reid_rr_farthest_exact.
 *   reid_rr_farthest_exact   : colmax[row] = max over all M rows of orig(row, j), exact CUDA-core scan, for the rows
 *       rows[0 .. n_rows) (or row_begin + r when rows is NULL).  D * 4 <= 200 KB.
 *   reid_rr_weights_features : reid_rr_weights with orig(e, i) / colmax[i] gathered from the feature rows (:66-67).
 *   reid_rr_final_qg         : rows [row_begin, row_end) of out (Q x G):  J[i - row_begin][Q + g] * (1 - lambda) +
 *       (q_g[i][g]^2 / colmax[i]) * lambda, fp32 in the reference's order; J holds those rows (leading dimension ldJ),
 *       q_g is the Q x G block of reid_pairwise_distance. */
int reid_rr_row_sqnorm64(const float* x, int64_t n_rows, int64_t D, double* sqnorm, void* stream);
int reid_rr_farthest_certify(const float* x, int64_t M, int64_t D, const double* sqnorm, const uint64_t* cand,
                             const int32_t* cand_cnt, const uint32_t* row_tau, int n_lists, int list_cap, int64_t row_begin,
                             int64_t row_end, const float* sqnorm_range, float* colmax, int32_t* uncertified_flag,
                             uint64_t* uncertified_count, void* stream);
int reid_rr_farthest_exact(const float* x, int64_t M, int64_t D, const double* sqnorm, const int32_t* rows,
                           int64_t row_begin, int64_t n_rows, float* colmax, void* stream);
int reid_rr_weights_features(const float* x, int64_t M, int64_t D, const double* sqnorm, const float* colmax,
                             const int32_t* E_pad, int stride, const int64_t* E_ptr, int64_t n_rows, int32_t* E_idx,
                             float* V_val, void* stream);
int reid_rr_final_qg(const float* J, int64_t ldJ, const float* q_g, const float* colmax, int64_t Q, int64_t G,
                     int64_t row_begin, int64_t row_end, float one_minus_lambda, float lambda, float* out, void* stream);
/* exact top-k of every row of a dense (n_rows x N) key matrix: descending (ties by smaller index), or the k
 * smallest in ascending order when `ascending` != 0. */
int reid_select_rows(const float* keys, int64_t N, int64_t n_rows, int k, int ascending, int32_t* out_idx,
                     float* out_key, void* stream);

/* ---- f3 (next row): evaluation metrics  (evaluators.py pairwise_distance :71-88; ----------------
 *      evaluation_metrics/ranking.py mean_ap :82-115, cmc :18-79)
 * out[i][j] = (||x_i||^2 + ||y_j||^2) - 2 x_i.y_j in fp32; scratch_norms: m + n floats. */
int reid_pairwise_distance(const float* x, const float* y, int64_t m, int64_t n, int64_t D, float* scratch_norms,
                           float* out, void* stream);
/* Per query i: valid gallery items = different id or different camera (and, with separate_camera_set, different
 * camera); positives = valid items of the same id.  ap_out[i] = uninterpolated average precision (sklearn's
 * average_precision_score: ties share a threshold), has_pos[i] = 1 / 0 (no positive: the query is skipped by the
 * reference) / -1 (more positives than the kernel handles).  With cmc buffers: cmc_contrib (m x topk doubles) gets
 * the query's additions to the CMC histogram (first_match_break or 1/P per match) and cmc_ret (topk) their sum over
 * the queries in order; ties in distance are ranked by gallery index (the reference's argsort leaves them unordered). */
size_t reid_rank_metrics_smem_bytes(int64_t n);
int reid_rank_metrics(const float* dist, int64_t m, int64_t n, int64_t ld, const int64_t* q_ids, const int64_t* g_ids,
                      const int64_t* q_cams, const int64_t* g_cams, int separate_camera_set, int topk,
                      int first_match_break, double* ap_out, int32_t* has_pos, double* cmc_contrib, double* cmc_ret,
                      void* stream);
/* cmc_ret[k] = sum over i = 0..m-1, in order, of cmc_contrib[i * topk + k]: the reduction reid_rank_metrics runs, on
 * contributions gathered from several ranks (distributed evaluation), so the sum has the single-process order. */
int reid_cmc_reduce(const double* cmc_contrib, int64_t m, int topk, double* cmc_ret, void* stream);

/* ---- a9: centroid init  (train_usl.py:169-182, 191) -------------------------------
 * out[k] = mean of x[i] over labels[i] == k, k = 0..C-1 (labels < 0 skipped), members added in
 * ascending i; normalize != 0 fuses the F.normalize of :191.  workspace: reid_centroids_workspace_bytes(N, C). */
size_t reid_centroids_workspace_bytes(int64_t N, int64_t C);
int reid_centroids(const float* x, int64_t N, int64_t D, const int64_t* labels, int64_t C, int normalize,
                   float* out, void* workspace, void* stream);
/* The same with the cluster count still on the device (reid_dbscan_labels' num_clusters_out): the grid covers
 * `capacity` clusters (<= N: every cluster holds a core point), rows >= *num_clusters_dev of `out` are not written.
 * Lets the whole pseudo-label pass run without a host round trip (train_usl.py:163-191 back to back). */
int reid_centroids_dev(const float* x, int64_t N, int64_t D, const int64_t* labels, const int64_t* num_clusters_dev,
                       int64_t capacity, int normalize, float* out, void* workspace, void* stream);
/* workspace (both entries; reid_centroids_workspace_bytes(N, C or capacity); NULL = none): with it the labels are binned
 * ONCE into per-cluster member lists (count, scan, scatter; each CTA sorts its short list ascending and adds the rows
 * four at a time) instead of every cluster's CTA streaming the whole label vector. */

/* ---- multi-GPU exchange over NVLink peer memory (SURVEY.md 8e; the reference has no multi-GPU hot path) --------
 * reid_peer_push_lists: the all-to-all of the tile-sharded search as plain peer stores.  part / part_cnt: this rank's
 * partial candidate lists of ALL rows (world blocks of block_rows rows, cap entries each).  peer_base[w] (device array
 * of `world` addresses): base of rank w's receive buffer, mapped into this process -- world * block_rows * cap
 * entries (list q of local row r at (q * block_rows + r) * cap), followed at cnt_offset_bytes by the
 * world * block_rows int32 counts.  Block w of `part` is stored as list `me` of rank w; only the valid entries
 * travel, the true count travels with them.  The caller separates the push from the consumers with a barrier
 * across the ranks. */
int reid_peer_push_lists(const uint64_t* part, const int32_t* part_cnt, int world, int64_t block_rows, int cap, int me,
                         const uint64_t* peer_base, int64_t cnt_offset_bytes, void* stream);
/* reid_peer_push_records: the ragged all-gathers of the row-sharded sparse stages (V rows, V_qe rows, eps-neighbour
 * lists) without a staging copy and without NCCL: the record of local row r -- { count, idx[stride], (val[stride]) }, the
 * format of reid_rows_pack -- is written as record (me * max_rows + r) into EVERY rank's receive buffer
 * (peer_base[w] + rec_offset_bytes); only the valid entries travel.  reid_rows_unpack_* then read the local buffer.
 * reid_peer_allgather: a fixed-size block (block_bytes, multiple of 4) to slot `me` of every rank's buffer. */
int reid_peer_push_records(const int32_t* cnt, const int64_t* ptr, const int32_t* idx, const float* val, int64_t n_rows,
                           int64_t max_rows, int stride, int me, int world, const uint64_t* peer_base,
                           int64_t rec_offset_bytes, void* stream);
int reid_peer_allgather(const void* src, int64_t block_bytes, int me, int world, const uint64_t* peer_base,
                        int64_t dst_offset_bytes, void* stream);
/* reid_peer_scatter_rows: the feature exchange of distributed evaluation.  src: this rank's n_rows extracted feature
 * rows (D floats each, D % 4 == 0, 16-byte aligned).  Local row r is stored as rows dst_rows[2r] and dst_rows[2r + 1]
 * (-1: not in that list) of the (M, D) fp32 matrix [query; gallery] at peer_base[w] + dst_offset_bytes, for every
 * w < world -- a file name in both lists is written twice.  A destination >= M is never written; bad_count (optional
 * device uint64) counts them.  With world = 1 and a local base it is a plain scatter (the collective fallback). */
int reid_peer_scatter_rows(const float* src, int64_t n_rows, int64_t D, const int32_t* dst_rows, int64_t M, int world,
                           const uint64_t* peer_base, int64_t dst_offset_bytes, uint64_t* bad_count, void* stream);

/* ---- f4: feature hand-off  (clustercontrast/evaluators.py:16-68, train_usl.py:152-153) ----------------
 * dst[r] = src[idx[r]] for r < n (rows of D floats, D % 4 == 0): re-orders a device-resident feature store into the
 * sorted-file-name order the pseudo-label pass expects, replacing the per-row `.cpu()` (evaluators.py:19) and the
 * N-way torch.cat on the host (train_usl.py:153). */
int reid_gather_rows(const float* src, int64_t n_src, const int64_t* idx, int64_t n, int64_t D, float* dst, void* stream);

/* ---- a10-a12: ClusterMemory  (models/cm.py:9-76, 110-137) --------------------------
 * forward: xhat = normalize(inputs); z = xhat . F^T / temp; loss_b = logsumexp(z_b) - z_b[y_b].
 * Saves xhat (B x D), inv_norm (B) and z (B x C) for backward.  (cm.py:125,16/47,134-135)
 * scratch: reid_cm_forward_scratch_bytes(B, C, D) bytes (split-K partial sums). */
size_t reid_cm_forward_scratch_bytes(int64_t B, int64_t C, int64_t D);
int reid_cm_forward(const float* inputs, const int64_t* targets, const float* centroids, int64_t B,
                    int64_t C, int64_t D, float temp, float* loss, float* xhat, float* inv_norm, float* z,
                    void* scratch, void* stream);
/* backward: grad_inputs through CE, /temp, mm with the PRE-update centroids (cm.py:26,56) and normalize. */
int reid_cm_backward(const float* grad_loss, const float* z, const int64_t* targets, const float* centroids,
                     const float* xhat, const float* inv_norm, int64_t B, int64_t C, int64_t D, float temp,
                     float* gz_scratch, float* grad_inputs, void* stream);
/* plain logits = a . F^T and grad = g . F for the module-level cm()/cm_hard() (cm.py:16,26,47,56) */
int reid_cm_logits(const float* a, const float* centroids, int64_t B, int64_t C, int64_t D, float* out,
                   void* stream);
int reid_cm_grad_inputs(const float* g, const float* centroids, int64_t B, int64_t C, int64_t D, float* out,
                        void* stream);
/* momentum update, in place on centroids.  hard = 0: per-sample sequential chain in batch order
 * (cm.py:29-31); hard = 1: per distinct label the first-argmin member of x.f[label] (cm.py:58-70).
 * workspace: B int32. */
int reid_cm_update(const float* xhat, const int64_t* targets, float* centroids, int64_t B, int64_t C,
                   int64_t D, float momentum, int hard, void* workspace, void* stream);
/* One ClusterMemory over `world` ranks (DistributedClusterMemory; the reference's nn.DataParallel gathers every GPU's
 * batch onto one memory, train_usl.py:189): reid_cm_forward on this rank's B rows, and the same CTA that writes row b's
 * xhat also stores it, with the row's target, into slot me * cap + b of EVERY rank's receive buffer.  peer_base[w]
 * (device array of `world` addresses) is rank w's buffer: world * cap int64 targets, then world * cap x D fp32 xhat.
 * Slots B <= b < cap of this rank get target -1.  After a barrier across the ranks, reid_cm_update on the local
 * buffer (B = world * cap rows) applies the update of the concatenated batch in rank order; the padding rows are
 * skipped.  The split-K count is that of B_split rows (pass world * cap): z, loss and the gradients then equal the
 * single-process values of the concatenated batch.  B <= cap, B <= B_split, D <= 4096.
 * scratch: reid_cm_forward_scratch_bytes(B_split, C, D) bytes. */
int reid_cm_forward_push(const float* inputs, const int64_t* targets, const float* centroids, int64_t B, int64_t C,
                         int64_t D, float temp, int64_t B_split, float* loss, float* xhat, float* inv_norm, float* z,
                         void* scratch, int me, int world, int64_t cap, const uint64_t* peer_base, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* REID_B200_H_ */
