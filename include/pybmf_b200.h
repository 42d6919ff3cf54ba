/*
 * pybmf_b200.h -- C ABI of the B200-native Asso hot path (libbmf_b200.so).
 *
 * The reference (PreferredAI/PyBMF) is pure Python and has no FFI: its "operator
 * API" for this path is a handful of Python functions (SURVEY.md section 8b).  Each entry
 * point below names the reference function (file:line under /root/reference) whose
 * arithmetic it replaces.  INTEGRATION.md shows the ctypes stub a PyBMF maintainer
 * would add at each of those call sites.
 *
 * Conventions
 *  - plain C types only; every pointer is a DEVICE pointer owned by the caller
 *    unless the parameter name ends in `_host`;
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and the
 *    call returns without synchronising;
 *  - return value: 0 ok, <0 invalid argument (BMF_E_*), >0 a cudaError_t;
 *    bmf_last_error() gives a thread-local message for the last non-zero return;
 *  - bit matrices are row-major arrays of uint64 words, bit c of a row lives in
 *    word c>>6 at position c&63; rows are `words` uint64 apart, `words` is EVEN
 *    (rows are 16-byte aligned so kernels can use 128-bit loads) and pad bits are 0;
 *  - int8 operand planes are row-major with leading dimension `ld` (bytes), a
 *    multiple of 128, rows padded to the tile multiple given per function, pad = 0.
 */
#ifndef PYBMF_B200_H
#define PYBMF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BMF_ABI_VERSION 1

#define BMF_E_ARG (-1)      /* bad shape / null pointer / misaligned leading dimension   */
#define BMF_E_NOGPU (-2)    /* no sm_100 device visible                                   */
#define BMF_E_DRIVER (-3)   /* cuTensorMapEncodeTiled unavailable / failed                */

/* tile multiples the int8 tensor-core kernels expect (callers pad to these) */
#define BMF_I8_CAND_TILE 128  /* rows of the "candidate" operand (MMA M)                  */
#define BMF_I8_ROW_TILE 256   /* rows of the "data row" operand (MMA N)                   */
#define BMF_I8_K_TILE 128     /* bytes of K per pipeline stage (= one 128B swizzle row)   */
/* FP4 (tcgen05 kind::mxf4) kernels: candidate rows padded to 256, data rows to 240, K to 256 elements */
#define BMF_F4_CAND_TILE 256
#define BMF_F4_ROW_TILE 240
#define BMF_F4_SUPER_ROWS 496 /* data rows padded to 496 select the super-tile kernel (256 + 240 sub-tiles)  */
#define BMF_F4_K_TILE 256     /* elements of K per stage = 128 bytes of packed E2M1         */

typedef void* bmf_stream_t;

int bmf_abi_version(void);
const char* bmf_last_error(void);
/* sm count and compute capability of the current device */
int bmf_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- input packing ------------------------------------------------------------------
 * Replaces the csr containers of BaseModel.load_dataset (PyBMF/models/BaseModel.py:146).
 * Non-zero pattern of a CSR matrix -> bit rows.  transposed=1 writes X^T (n rows of
 * ceil(m/64) words).  `bits` must be zero-filled by the caller (bmf_fill_zero). */
int bmf_pack_csr(const int64_t* indptr, const int32_t* indices, int64_t m, int64_t n,
                 int transposed, uint64_t* bits, int64_t words, bmf_stream_t stream);
int bmf_fill_zero(void* ptr, int64_t bytes, bmf_stream_t stream);
/* bits[rows][words] -> int8 plane[rows_pad][ld]: value `masked` wherever mask_bits (nullable,
 * same layout; the covered mask) has a 1, else `one` where the bit is set and `zero` where it is
 * clear; 0 in all padding (columns >= ncols, rows >= rows). */
int bmf_expand_bits_i8(const uint64_t* bits, const uint64_t* mask_bits, int64_t rows, int64_t ncols,
                       int64_t words, int8_t one, int8_t zero, int8_t masked, int8_t* plane,
                       int64_t rows_pad, int64_t ld, bmf_stream_t stream);

/* ---- association matrix: build_assoc, PyBMF/models/Asso.py:191-213 -------------------
 * cnt[i][j] = |col_i AND col_j| = (X^T X)[i][j], int32, leading dimension ldc.
 * popc variant: XT bits [n][words_m].  i8 variant (tcgen05 kind::i8, TMA, TMEM):
 * XT plane int8 [n_pad(256)][ld] of 0/1 with K = rows of X along ld. */
int bmf_assoc_counts_popc(const uint64_t* xt_bits, int64_t n, int64_t words_m, int32_t* cnt,
                          int64_t ldc, bmf_stream_t stream);
/* the primitive under both int8 paths, exported for parity tests:
 * c[i][j] = sum_k a[i][k]*b[j][k], a rows multiple of 128, b rows multiple of 256, int32 out */
int bmf_gemm_i8_nt(const int8_t* a_plane, int64_t a_rows_pad, const int8_t* b_plane, int64_t b_rows_pad,
                   int64_t ld, int32_t* c, int64_t ldc, bmf_stream_t stream);
int bmf_assoc_counts_i8(const int8_t* xt_plane, int64_t n, int64_t n_pad, int64_t ld, int32_t* cnt,
                        int64_t ldc, bmf_stream_t stream);
/* build_basis, Asso.py:216-235 + binarize, PyBMF/utils/common.py:75: bit (i,j) =
 * ((double)cnt[i][j] / (double)cnt[i][i] > tau) (IEEE division, strict >); the association
 * row of an empty column (cnt[i][i] = 0) is 0 (Asso.py:211), so its bits are (0 > tau).
 * Evaluated as cnt[i][j] >= c_min(cnt[i][i], tau): correctly rounded division is monotone in
 * the count, and c_min is found per column with the literal division -- the same predicate,
 * without n^2 fp64 divisions.  alive[i] = row i has any bit set (the reference drops all-zero
 * rows but keeps order, so candidate rank = rank among alive rows).  cand_plane
 * (nullable) receives the same rows as int8 0/1, [n_pad(128)][ld]. */
int bmf_basis_threshold(const int32_t* cnt, int64_t ldc, int64_t n, double tau, uint64_t* basis_bits,
                        int64_t words, int8_t* cand_plane, int64_t ld, uint8_t* alive,
                        int32_t* row_pop /* nullable: |b_i| per row */, bmf_stream_t stream);

/* ---- greedy cover-gain scoring: the hot loop Asso.py:83-95 -> get_vector Asso.py:144-188,
 *      coverage_score PyBMF/utils/metrics.py:189-201 ------------------------------------
 * For every candidate row b_j and data row i:
 *   P = |x_i & ~c_i & b_j|, N = |~x_i & ~c_i & b_j|,
 *   use(i,j) = (s_new > s_old) with s = (-w_fp)*FP + w_fn*TP evaluated in fp64, no FMA.
 * Integer mode (wa, wb > 0 given, w_fp = wa/2^s, w_fn = wb/2^s): use <=> wb*P - wa*N > 0,
 *   gain_p[j] = sum_i relu(wb*P - wa*N), gain_n untouched.
 * General mode (wa = wb = 0): gain_p[j] = sum_{use} P, gain_n[j] = sum_{use} N, with
 *   tp_old/fp_old the per-row counts of the current cover.
 * Outputs are overwritten (not accumulated). */
int bmf_cover_score_popc(const uint64_t* x_bits, const uint64_t* c_bits, int64_t m, int64_t n,
                         int64_t words, const uint64_t* basis_bits, const uint8_t* alive,
                         const int32_t* tp_old, const int32_t* fp_old, int32_t wa, int32_t wb,
                         double w_fp, double w_fn, int64_t* gain_p, int64_t* gain_n,
                         bmf_stream_t stream);
/* tcgen05 kind::i8 variant, integer mode only.  cand_plane = 0/1 basis rows and
 *   gain[j] = sum_i relu(sign * sum_k cand[j][k]*rows[i][k] - bias_scale * cand_pop[j]).
 * Two equivalent operand encodings give D = wb*P - wa*N:
 *   signed   : rows[i][k] = sign*wb (uncovered one), -sign*wa (uncovered zero), 0 (covered); cand_pop = NULL
 *   zero-dominant: rows[i][k] = wa+wb (uncovered one), 0 (uncovered zero), wa (covered), sign = +1,
 *              cand_pop[j] = |b_j|, bias_scale = wa   (since N = |b_j| - |b_j & c_i| - P);
 *              the dominant operand value is 0, which lowers tensor-core switching power.
 * gain has cand_pad entries. */
int bmf_cover_score_i8(const int8_t* cand_plane, int64_t cand_pad, const int8_t* rows_plane,
                       int64_t rows_pad, int64_t ld, int32_t sign, const int32_t* cand_pop,
                       int32_t bias_scale, int64_t* gain, bmf_stream_t stream);

/* tcgen05 kind::i8 variant for GENERAL weights (any fp64 w_fp, w_fn; e.g. the reference notebooks' w_fp = 0.2).
 * pq_plane interleaves, per block of 128 data rows, 128 rows of P_i = x_i & ~c_i and 128 rows of Q_i = c_i
 * (0/1 bytes; plane row of data row i = (i/128)*256 + i%128 for P, +128 for Q; 2*ceil(m/128)*128 rows of ld bytes,
 * written by bmf_expand_bits_pq and kept current by bmf_cover_apply_general).  One contraction then yields
 * P = |b_j & x_i & ~c_i| and Q = |b_j & c_i| side by side in the accumulator, N = cand_pop[j] - Q - P, and the
 * fused epilogue evaluates use(i,j) with the literal fp64 expression above:
 *   gain_p[j] = sum_{use} P, gain_n[j] = sum_{use} N   (cand_pad entries each, overwritten). */
int bmf_expand_bits_pq(const uint64_t* x_bits, const uint64_t* c_bits, int64_t rows, int64_t ncols, int64_t words,
                       int8_t* pq_plane, int64_t ld, bmf_stream_t stream);
int bmf_cover_score_i8_general(const int8_t* cand_plane, int64_t cand_pad, const int8_t* pq_plane, int64_t m,
                               int64_t ld, const int32_t* cand_pop, const int32_t* tp_old, const int32_t* fp_old,
                               double w_fp, double w_fn, int64_t* gain_p, int64_t* gain_n, bmf_stream_t stream);

/* ---- FP4 tensor-core variants (tcgen05 kind::mxf4, packed E2M1 operands, unit block scales, FP32 accumulate) ----
 * Twice the kind::i8 rate at half the operand bytes, and still EXACT for this path: the operand values are
 * non-negative integers that E2M1 represents exactly (0, 1, 2, 3, 4, 6) and every partial sum is an integer
 * below 2^24.  An f4 plane is row-major with `ld_bytes` bytes per row (a multiple of 128 covering ceil(ncols/2)),
 * two 4-bit E2M1 codes per byte, element k in byte k/2, low nibble for even k; padding is code 0.
 * bmf_expand_bits_f4: value codes `one`/`zero`/`masked` are E2M1 bit patterns (0 -> 0.0, 2 -> 1.0, 4 -> 2.0,
 * 5 -> 3.0, 6 -> 4.0, 7 -> 6.0), otherwise as bmf_expand_bits_i8.  bmf_e2m1_code maps an integer value to its
 * code or returns -1 when E2M1 cannot represent it (the caller then stays on the int8 kernels).
 * bmf_gemm_f4_nt: c[i][j] = sum_k a[i][k]*b[j][k] as int32 (a rows multiple of 256, b rows multiple of 240, or
 * of 496 = BMF_F4_SUPER_ROWS, which selects the faster super-tile kernel; likewise rows_pad of bmf_cover_score_f4).
 * accumulate bit 0 (496-padded b rows only): c += ..., so K (the data rows of X^T X) can be split over several launches
 * and the association of one row chunk overlaps the host-to-device copy of the next.  accumulate bit 1 (a_plane ==
 * b_plane, i.e. X^T X): the product is symmetric, super tiles entirely below the diagonal are skipped (their part of c
 * is left untouched) -- see bmf_basis_threshold_rows(symmetric).
 * bmf_cover_score_f4: the zero-dominant encoding of bmf_cover_score_i8 (sign = +1) on f4 planes. */
int bmf_e2m1_code(int32_t value);
int bmf_expand_bits_f4(const uint64_t* bits, const uint64_t* mask_bits, int64_t rows, int64_t ncols, int64_t words,
                       int32_t one, int32_t zero, int32_t masked, uint8_t* plane, int64_t rows_pad, int64_t ld_bytes,
                       bmf_stream_t stream);
int bmf_gemm_f4_nt(const uint8_t* a_plane, int64_t a_rows_pad, const uint8_t* b_plane, int64_t b_rows_pad,
                   int64_t ld_bytes, int32_t* c, int64_t ldc, int32_t accumulate, bmf_stream_t stream);
int bmf_cover_score_f4(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* rows_plane, int64_t rows_pad,
                       int64_t ld_bytes, const int32_t* cand_pop, int32_t bias_scale, int64_t* gain,
                       bmf_stream_t stream);
/* general (non-dyadic) weights on the FP4 pipe: the interleaved P/Q operand of bmf_cover_score_i8_general as packed
 * E2M1 0/1, in blocks of 120 data rows (plane row of data row i = (i/120)*240 + i%120 for P, +120 for Q;
 * 2*ceil(m/120)*120 rows of ld_bytes), same outputs as bmf_cover_score_i8_general. */
int bmf_expand_bits_pq_f4(const uint64_t* x_bits, const uint64_t* c_bits, int64_t rows, int64_t ncols, int64_t words,
                          uint8_t* pq_plane, int64_t ld_bytes, bmf_stream_t stream);
int bmf_cover_score_f4_general(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* pq_plane, int64_t m,
                               int64_t ld_bytes, const int32_t* cand_pop, const int32_t* tp_old, const int32_t* fp_old,
                               double w_fp, double w_fn, int64_t* gain_p, int64_t* gain_n, bmf_stream_t stream);
int bmf_cover_apply_f4_general(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                               const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                               int32_t* fp_old, double w_fp, double w_fn, uint8_t* pq_plane, int64_t ld_bytes,
                               uint64_t* u_bits, int64_t* totals, bmf_stream_t stream);
/* bmf_cover_apply on an f4 rows plane: newly covered entries of the used rows get the E2M1 code `covered_code` */
int bmf_cover_apply_f4(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                       const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                       int32_t* fp_old, int32_t wa, int32_t wb, uint8_t* rows_plane, int64_t ld_bytes,
                       int32_t covered_code, uint64_t* u_bits, int64_t* totals, bmf_stream_t stream);

/* ---- block-sparse FP4 scoring (integer weights, zero-dominant encoding) ----
 * Both planes may hold their K columns in an order sigma and the candidate plane its rows in an order pi: column k of X
 * is element col_pos[k] (col_pos = sigma^-1, int32 [ncols]) and candidate plane row p holds basis row row_src[p] = pi[p]
 * (int32 [rows]).  A common K permutation leaves every dot product unchanged; the scorer's epilogue writes the gain of
 * plane row p to gain[cand_id[p]] and reads the bias from cand_pop[cand_id[p]] (cand_id int32 [cand_pad], padding rows
 * map to themselves), so gains stay indexed by the original candidate.  The plain entry points above are these with
 * null maps.  Mapped expansion needs zero == 0 and ld_bytes <= 204800.
 * kb_table (int32, nullable = dense walk): [mt_total + 1] exclusive prefix sums of the per-candidate-tile counts of K
 * blocks (256 candidates x 256 columns) that hold a nonzero, then [mt_total][kb_total] the ascending K-block lists
 * (mt_total = cand_pad / 256, kb_total = ld_bytes / 128).  Blocks left out must be all zero in the candidate plane: they
 * add exactly 0 to the integer D.  With a table the (data-row super tile, candidate tile) units are walked super tile
 * outer and split over the CTA pairs by equal K-block cost.
 * bmf_bits_first_set: row_first[j] = lowest set column of bit row j (ncols when empty), col_first[k] = min row_rank[j]
 * over the rows holding column k (caller-filled with INT_MAX); both outputs nullable. */
int bmf_expand_bits_f4_mapped(const uint64_t* bits, const uint64_t* mask_bits, int64_t rows, int64_t ncols, int64_t words,
                              int32_t one, int32_t zero, int32_t masked, const int32_t* row_src, const int32_t* col_pos,
                              uint8_t* plane, int64_t rows_pad, int64_t ld_bytes, bmf_stream_t stream);
int bmf_cover_apply_f4_mapped(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                              const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                              int32_t* fp_old, int32_t wa, int32_t wb, uint8_t* rows_plane, int64_t ld_bytes,
                              int32_t covered_code, const int32_t* col_pos, uint64_t* u_bits, int64_t* totals,
                              bmf_stream_t stream);
int bmf_cover_apply_compact_mapped(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                                   const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                                   int32_t* fp_old, int32_t wa, int32_t wb, int32_t kind, int32_t v_one, int32_t v_zero,
                                   int32_t v_covered, uint8_t* comp_old, uint8_t* comp_new, int64_t comp_ld,
                                   int64_t comp_cap, int32_t tile_rows, int32_t* nused, uint64_t* u_bits,
                                   uint64_t* u_words, int64_t kw, int32_t factor_bit, uint64_t* vt_row,
                                   const int32_t* col_pos, int64_t* totals, bmf_stream_t stream);
int bmf_cover_score_f4_blocks(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* rows_plane, int64_t rows_pad,
                              int64_t ld_bytes, const int32_t* cand_pop, int32_t bias_scale, const int32_t* kb_table,
                              const int32_t* cand_id, int64_t* gain, bmf_stream_t stream);
int bmf_cover_rescore_f4_blocks(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* compact_plane,
                                int64_t rows_cap, int64_t ld_bytes, const int32_t* cand_pop, int32_t bias_scale,
                                const int32_t* kb_table, const int32_t* cand_id, const int32_t* dyn_rows,
                                int32_t gain_sign, int64_t* gain, bmf_stream_t stream);
int bmf_bits_first_set(const uint64_t* bits, int64_t rows, int64_t ncols, int64_t words, const int32_t* row_rank,
                       int32_t* row_first, int32_t* col_first, bmf_stream_t stream);

/* argmax of Asso.py:94: first j (lowest index) among alive candidates whose score is
 * strictly greater than `best_score` and than every earlier score.
 * integer mode: score_j = (double)(base_int + gain_p[j]) * scale
 * general mode: score_j = (-w_fp)*(double)(fp_tot + gain_n[j]) + w_fn*(double)(tp_tot + gain_p[j])
 * record[0] = winner index or -1, record[1] = bit pattern of the winning score (double). */
int bmf_select_first_max(const int64_t* gain_p, const int64_t* gain_n, const uint8_t* alive, int64_t n,
                         int32_t wa, int32_t wb, int64_t base_int, double scale, double w_fp,
                         double w_fn, int64_t tp_tot, int64_t fp_tot, double best_score,
                         int64_t* record, bmf_stream_t stream);

/* set_factors + cover update for the chosen candidate (Asso.py:103-110): recompute
 * use(i) for basis row *winner (device int64; <0 = no-op), write u_bits (bit i of a
 * ceil(m/64)-word vector, caller-zeroed), OR the row into c_bits where used, add P/N to
 * tp_old/fp_old, set the used rows' newly covered entries of rows_plane (nullable) to
 * covered_value, clear alive[winner].  totals[0..2] += (#used rows, sum P, sum N). */
int bmf_cover_apply(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                    const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                    int32_t* fp_old, int32_t wa, int32_t wb, double w_fp, double w_fn,
                    int8_t* rows_plane, int64_t ld, int8_t covered_value, uint64_t* u_bits,
                    int64_t* totals, bmf_stream_t stream);

/* same in general mode with the interleaved P/Q operand plane: newly covered entries get P = 0, Q = 1 */
int bmf_cover_apply_general(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                            const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                            int32_t* fp_old, double w_fp, double w_fn, int8_t* pq_plane, int64_t ld,
                            uint64_t* u_bits, int64_t* totals, bmf_stream_t stream);

/* ---- device-resident greedy loop (Asso._fit, PyBMF/models/Asso.py:62-110, without a host round trip per step) ----
 * bmf_greedy_select is bmf_select_first_max with the loop state in device memory:
 *   state[0] = bits of the inherited best score (Asso.py:71), [1] = TP total, [2] = FP total of the cover,
 *   [3] = stopped (a step found no improving candidate: Asso.py:98-100), [4] = number of steps selected.
 *   table_row (8 x int64, one per greedy step): winner, score bits, #used rows, sum P, sum N, TP total after,
 *   FP total after, status (0 no winner, 1 winner chosen / counters pending, 2 complete).
 * `tail` = (#used, sum P, sum N) of the PREVIOUS step's apply summed over all ranks -- the three counters ride at the
 * end of the all-reduced gain vector, so a step needs one collective -- and is folded into state / prev_row first;
 * tail_zero (the rank-local copy, may alias tail) and *nused are cleared for the coming apply.  first != 0 resets
 * the threshold to 0 (step 0).  table_row == NULL only folds the counters (the flush after the last step).
 * The winner is removed from alive[] here (Asso.py:106-107) and written to record[0] for bmf_cover_apply*.
 *
 * bmf_cover_apply_compact = bmf_cover_apply (integer weights) plus, for INCREMENTAL rescoring, the operand-plane rows of
 * the used data rows before (comp_old) and after (comp_new) the update, compacted at slots drawn from *nused
 * (kind 1: packed E2M1 codes v_one / v_zero / v_covered, kind 2: int8 values; kind 0: no compaction), rows
 * [*nused, round_up(*nused, tile_rows)) zeroed.  Only rows the winner uses change state, hence
 *   gain_j(t+1) = gain_j(t) - sum_{i used} relu(D_ij(t)) + sum_{i used} relu(D_ij(t+1)),
 * which bmf_cover_rescore_f4 / _i8 add to the running gain vector (gain_sign = -1 on comp_old, +1 on comp_new; the
 * kernels are the scoring GEMMs with the row-tile count read from *dyn_rows; gain is NOT cleared).
 * Optional extras: u_words/kw/factor_bit (bit of the row-major usage words), vt_row (copy of the winner's basis row). */
int bmf_greedy_select(const int64_t* gain_p, const int64_t* gain_n, const int64_t* tail, int64_t* tail_zero,
                      uint8_t* alive, int64_t n, int32_t wa, int32_t wb, double scale, double w_fp, double w_fn,
                      int32_t first, int64_t* state, int64_t* table_row, int64_t* prev_row, int64_t* record,
                      int32_t* nused, bmf_stream_t stream);
int bmf_cover_apply_compact(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                            const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                            int32_t* fp_old, int32_t wa, int32_t wb, int32_t kind, int32_t v_one, int32_t v_zero,
                            int32_t v_covered, uint8_t* comp_old, uint8_t* comp_new, int64_t comp_ld, int64_t comp_cap,
                            int32_t tile_rows, int32_t* nused, uint64_t* u_bits, uint64_t* u_words, int64_t kw,
                            int32_t factor_bit, uint64_t* vt_row, int64_t* totals, bmf_stream_t stream);
int bmf_cover_rescore_f4(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* compact_plane, int64_t rows_cap,
                         int64_t ld_bytes, const int32_t* cand_pop, int32_t bias_scale, const int32_t* dyn_rows,
                         int32_t gain_sign, int64_t* gain, bmf_stream_t stream);
int bmf_cover_rescore_i8(const int8_t* cand_plane, int64_t cand_pad, const int8_t* compact_plane, int64_t rows_cap,
                         int64_t ld, int32_t sign, const int32_t* cand_pop, int32_t bias_scale, const int32_t* dyn_rows,
                         int32_t gain_sign, int64_t* gain, bmf_stream_t stream);
/* The same for GENERAL (non-dyadic) weights: sum_use P and sum_use N update by the same identity.  The compacted operand
 * is the interleaved P/Q plane (kind 3: packed E2M1 in blocks of 120 rows, kind 4: int8 in blocks of 128 rows) and the used
 * rows' per-row TP / FP before and after the update travel with it (comp_tp_* / comp_fp_*, indexed by slot), because the
 * fp64 row test needs them.  bmf_cover_rescore_*_general = bmf_cover_score_*_general on the compacted rows, row count from
 * *dyn_rows, gain_p / gain_n accumulated with gain_sign instead of overwritten. */
int bmf_cover_apply_compact_general(const uint64_t* x_bits, uint64_t* c_bits, int64_t m, int64_t n, int64_t words,
                                    const uint64_t* basis_bits, uint8_t* alive, const int64_t* winner, int32_t* tp_old,
                                    int32_t* fp_old, double w_fp, double w_fn, int32_t kind, uint8_t* comp_old,
                                    uint8_t* comp_new, int64_t comp_ld, int64_t comp_cap, int32_t* nused,
                                    int32_t* comp_tp_old, int32_t* comp_fp_old, int32_t* comp_tp_new,
                                    int32_t* comp_fp_new, uint64_t* u_bits, int64_t* totals, bmf_stream_t stream);
int bmf_cover_rescore_f4_general(const uint8_t* cand_plane, int64_t cand_pad, const uint8_t* compact_pq_plane,
                                 int64_t rows_cap, int64_t ld_bytes, const int32_t* cand_pop, const int32_t* comp_tp,
                                 const int32_t* comp_fp, double w_fp, double w_fn, const int32_t* dyn_rows,
                                 int32_t gain_sign, int64_t* gain_p, int64_t* gain_n, bmf_stream_t stream);
int bmf_cover_rescore_i8_general(const int8_t* cand_plane, int64_t cand_pad, const int8_t* compact_pq_plane,
                                 int64_t rows_cap, int64_t ld, const int32_t* cand_pop, const int32_t* comp_tp,
                                 const int32_t* comp_fp, double w_fp, double w_fn, const int32_t* dyn_rows,
                                 int32_t gain_sign, int64_t* gain_p, int64_t* gain_n, bmf_stream_t stream);
/* bmf_basis_threshold on a row window [row0, row0 + nrows) (all pointers at row row0): with the rows of X sharded, every
 * rank thresholds the block of X^T X it received from the reduce-scatter and the bit rows are all-gathered.
 * symmetric != 0 (row0 = 0): entries below the diagonal were skipped by bmf_gemm_f4_nt(accumulate bit 1) and are read
 * as cnt[min(i,j)][max(i,j)]; with nrows = n the stored triangle is walked in 64 x 64 tiles, each emitting both of the
 * mirrored bit words (pop_rows, when given, is also used as scratch for the per-column minimal counts). */
int bmf_basis_threshold_rows(const int32_t* cnt_rows, int64_t ldc, int64_t n, int64_t row0, int64_t nrows,
                             int32_t symmetric, double tau, uint64_t* basis_rows, int64_t words, uint8_t* alive_rows,
                             int32_t* pop_rows, bmf_stream_t stream);

/* ---- Boolean product and confusion counts ------------------------------------------------
 * get_prediction / matmul(boolean=True): PyBMF/utils/common.py:98-107, boolean_utils.py:61-84.
 * u_words[m][kw]: bit l of row i = U[i][l]; vt_bits[k][words] = rows of V^T.
 * pd_bits[i] = OR_{l in U_i} vt_bits[l]. */
int bmf_bool_product(const uint64_t* u_words, int64_t m, int64_t kw, const uint64_t* vt_bits,
                     int64_t k, int64_t words, uint64_t* pd_bits, bmf_stream_t stream);
/* get_residual, PyBMF/utils/common.py:154-160: out[i] = x[i] AND NOT (OR_{l in U_i} vt_bits[l]) in one pass.
 * Same u_words / vt_bits layout as bmf_bool_product; k = 0 copies x; out must not alias x. */
int bmf_residual_factors(const uint64_t* x_bits, int64_t m, int64_t words, const uint64_t* u_words, int64_t kw,
                         const uint64_t* vt_bits, int64_t k, uint64_t* out_bits, bmf_stream_t stream);
/* TP/FP/FN of PyBMF/utils/metrics.py:56-76 against the product computed on the fly
 * (never materialised).  counts[0..2] = (TP, FP, FN) (overwritten); row_tp/row_fp nullable int32[m].
 * gt_ones = number of ones in gt_bits when the caller knows it (the csr nnz), which saves the
 * kernel a third of its popcounts; pass -1 to have it counted. */
int bmf_confusion_factors(const uint64_t* gt_bits, int64_t m, int64_t words, const uint64_t* u_words,
                          int64_t kw, const uint64_t* vt_bits, int64_t k, int64_t gt_ones, int64_t* counts,
                          int32_t* row_tp, int32_t* row_fp, bmf_stream_t stream);
/* same against a materialised prediction */
int bmf_confusion_bits(const uint64_t* gt_bits, const uint64_t* pd_bits, int64_t m, int64_t words,
                       int64_t gt_ones, int64_t* counts, int32_t* row_tp, int32_t* row_fp,
                       bmf_stream_t stream);
/* Stored-entry counts of evaluate_utils.py:32-44 (task='prediction') in ONE pass: ones = the stored non-zeros, zeros
 * (nullable) = the explicitly stored zeros, both [m][words] like pd_bits; counts[0..3] = (|ones & pd|, |zeros & pd|,
 * |ones|, |zeros|) (overwritten), so TP = counts[0], FP = counts[1], FN = counts[2] - TP, size = counts[2] + counts[3].
 * _factors computes the product of the factors once for both streams (panel-list form for k <= 64, row stream above). */
int bmf_confusion_entries_bits(const uint64_t* ones, const uint64_t* zeros, const uint64_t* pd_bits, int64_t m,
                               int64_t words, int64_t* counts, bmf_stream_t stream);
int bmf_confusion_entries_factors(const uint64_t* ones, const uint64_t* zeros, int64_t m, int64_t words,
                                  const uint64_t* u_words, int64_t kw, const uint64_t* vt_bits, int64_t k,
                                  int64_t* counts, bmf_stream_t stream);
/* add(boolean=True) / multiply(boolean=True), PyBMF/utils/boolean_utils.py:87-107 / 6-33:
 * out = a OR b (op 0), a AND b (op 1), a AND NOT b (op 2) on [rows][words] bit matrices. */
int bmf_bits_combine(const uint64_t* a_bits, const uint64_t* b_bits, int64_t rows, int64_t words, int op,
                     uint64_t* out_bits, bmf_stream_t stream);
/* eval(task='prediction'), PyBMF/utils/evaluate_utils.py:32-44: counts over stored triplets
 * (i, j, gt != 0); counts[0..3] += (TP, FP, FN, TN). */
int bmf_confusion_triplets(const int32_t* rows, const int32_t* cols, const uint8_t* gt, int64_t nnz,
                           const uint64_t* u_words, int64_t kw, const uint64_t* v_words,
                           int64_t* counts, bmf_stream_t stream);

/* ---- GreConDPlus._expansion, PyBMF/models/GreConDPlus.py:267-308 (SURVEY section 8f rank 1) ------------------
 * delta[i] = coverage_score(x_i, old_i | pattern) - coverage_score(x_i, old_i) in the reference's fp64 order for every row
 * whose bit in exclude_bits (nullable; a bit vector over the rows) is clear, +0.0 for excluded rows; best[0] = bits of
 * max(delta), best[1] = FIRST argmax (nullable).  Row-wise expansion (axis = 1): rows of X / X_old, pattern = v,
 * exclude = u; column-wise (axis = 0): rows of X^T / X_old^T, pattern = u, exclude = v. */
int bmf_expand_scores(const uint64_t* x_bits, const uint64_t* old_bits, int64_t rows, int64_t words,
                      const uint64_t* pattern_bits, const uint64_t* exclude_bits, double w_fp, double w_fn,
                      double* delta, int64_t* best, bmf_stream_t stream);
/* ---- GreConDPlus.expansion, PyBMF/models/GreConDPlus.py:207-264: the incremental, device-resident loop ----------
 * Row layout only.  A rank holds rows [row0, row0 + rows) of x / old; u_bits (m bits) and v_bits (n bits) are the whole,
 * replicated pattern.
 * bmf_expand_init: one pass over the rows.  row_cnt[i][0..3] = (TP_old, FP_old, P, N) of local row i (int32, written)
 * with P = |x & ~old & v|, N = |~x & ~old & v|; col_cnt[k][j] (int64 [4][n], written) = this rank's share of column j's
 * TP_old, FP_old, and over the rows in u, P = |x & ~old| and N = |~x & ~old| (pad bits masked).  Column counts are
 * summed over the ranks by the caller.
 * One iteration = bmf_expand_step_rows, a SUM of xbuf over the ranks (nothing with one rank), bmf_expand_step_decide.
 * state[8] (int64, caller-initialised to {0, -1, -1, 0, 0, 0, 0, 0}) = (stopped, row chosen last or -1, column chosen
 * last or -1, iterations logged, two block counters).  partials: 4 * 1024 int64 scratch.  xbuf: 2 * world + 2 * words
 * int64 = world slots (bits of the rank's max row delta, its logical row or -1) then the words of the row chosen last
 * (x & ~old, then ~x & ~old masked to n), filled by its owner and 0 elsewhere.  step_rows applies a column chosen last to
 * P / N of the rows and fills xbuf; step_decide applies the row in xbuf to the column counts, merges the slots (max, then
 * the lowest row), takes the max and FIRST argmax of the column deltas and applies the reference's rule: it sets the bit in
 * u / v and appends (0 row | 1 column | 2 stop, index) to log[log_cap][2].  Once stopped, both are no-ops.
 * bmf_expand_col_scores: _expansion(axis = 0) from summed column counts: delta[j], best as bmf_expand_scores. */
int bmf_expand_init(const uint64_t* x_bits, const uint64_t* old_bits, int64_t rows, int64_t n, int64_t words, int64_t row0,
                    const uint64_t* u_bits, const uint64_t* v_bits, int32_t* row_cnt, int64_t* col_cnt,
                    bmf_stream_t stream);
int bmf_expand_step_rows(const uint64_t* x_bits, const uint64_t* old_bits, int64_t rows, int64_t n, int64_t words,
                         int64_t row0, const uint64_t* u_bits, int32_t* row_cnt, double w_fp, double w_fn, int64_t* state,
                         int64_t* partials, int64_t* xbuf, int64_t world, int64_t rank, bmf_stream_t stream);
int bmf_expand_step_decide(int64_t* col_cnt, int64_t n, int64_t words, uint64_t* u_bits, uint64_t* v_bits, double w_fp,
                           double w_fn, int64_t* state, int64_t* partials, const int64_t* xbuf, int64_t world,
                           int64_t* log, int64_t log_cap, bmf_stream_t stream);
int bmf_expand_col_scores(const int64_t* col_cnt, int64_t n, const uint64_t* v_bits, double w_fp, double w_fn,
                          double* delta, int64_t* best, bmf_stream_t stream);
/* ---- AssoOpt.set_optimal_row, PyBMF/models/AssoOpt.py:69-80 (SURVEY section 8f rank 4) -------------------------
 * best_trial[i] = FIRST argmax over j in [0, 2^k) of (-w_fp) FP + w_fn TP of the OR of the V^T rows selected by j
 * (factor l = bit k-1-l of j, the MSB-first order of int2bin, AssoOpt.py:83-86) against data row i; best_score
 * (nullable) receives the winning score.  k <= 20. */
int bmf_optimal_rows(const uint64_t* x_bits, int64_t m, int64_t words, const uint64_t* vt_bits, int64_t k, double w_fp,
                     double w_fn, int64_t* best_trial, double* best_score, bmf_stream_t stream);

/* ---- on-device synthetic inputs (SURVEY section 8f rank 3) -----------------------------------------------------
 * The generators' recipe (PyBMF/generators/BaseGenerator.py:202-221, PyBMF/utils/generator_utils.py:30-49) on bit rows,
 * with a counter-based generator: bit (i, j) of a stream depends only on (seed, stream_id, i, j), so every rank can
 * generate its own row range [row0, row0 + rows) of the same logical matrix.
 * bmf_random_bits: bits[r][.] = Bernoulli(p) for logical row row0 + r (pad bits 0).
 * bmf_noise_bits : add_noise -- ones dropped with probability p_pos, then entries set with probability p_neg.
 * bmf_transpose_bits: bits [rows][words] -> bits_t [ncols][words_t] (caller zero-fills bits_t's pad words), the X^T the
 * association needs when X never existed as a csr.  `words` and `words_t` are row strides, so a column window of bits
 * (pointer advanced by whole words) or a word offset into bits_t can be passed; rows <= 4.19M per call.  Writes only
 * bits_t[c][w] with c < ncols and 64 w < rows. */
int bmf_random_bits(uint64_t* bits, int64_t rows, int64_t ncols, int64_t words, int64_t row0, uint64_t seed,
                    uint64_t stream_id, double p, bmf_stream_t stream);
int bmf_noise_bits(uint64_t* bits, int64_t rows, int64_t ncols, int64_t words, int64_t row0, uint64_t seed, double p_pos,
                   double p_neg, bmf_stream_t stream);
int bmf_transpose_bits(const uint64_t* bits, int64_t rows, int64_t ncols, int64_t words, uint64_t* bits_t,
                       int64_t words_t, bmf_stream_t stream);
/* bmf_split_bits: generate.ratio_split in one pass over x (rows [row0, row0 + rows) of an ncols-column matrix).  A one at
 * global bit index b = (row * ceil(ncols / 64) + w) * 64 + bit draws u = 32-bit half (b & 1) of
 * splitmix64(key(seed, stream_ones) + b / 2), the draw of bmf_random_bits, and goes to val ones if u < t_v, to test ones
 * if u < t_v + t_t, else to train; a zero inside the ncols columns draws from stream_zeros and becomes a val zero if
 * u < q_v, a test zero if u < q_v + q_t, else nothing.  Thresholds are 32-bit (p * 2^32, as bmf_random_bits).  out_bits
 * = 5 consecutive [rows][words] matrices: train, val ones, val zeros, test ones, test zeros; every word is written and
 * pad bits are zero. */
int bmf_split_bits(const uint64_t* x_bits, int64_t rows, int64_t ncols, int64_t words, int64_t row0, uint64_t seed,
                   uint64_t stream_ones, uint64_t stream_zeros, uint64_t t_v, uint64_t t_t, uint64_t q_v, uint64_t q_t,
                   uint64_t* out_bits, bmf_stream_t stream);

/* ---- measurement aid (bench.py): tensor-pipe ceiling measured on the box -----------------------------------
 * One launch in which a CTA pair per TPC issues iters x 4 back-to-back tcgen05.mma instructions of the production shape
 * (kind 0: kind::i8 256 x 256 x 32; kind 1: kind::mxf4 256 x 256 x 64, unit scales) on sparse small-integer operands
 * resident in shared memory -- no TMA, no epilogue.  The caller times the launch with CUDA events; *ops_out_host (HOST
 * pointer, nullable) receives the operations performed.  This is the roofline denominator of the scoring kernels. */
int bmf_probe_mma_rate(int32_t kind, int32_t iters, double* ops_out_host, bmf_stream_t stream);

/* ---- AssoIter.get_refined_column, PyBMF/models/AssoIter.py:80-100 -------------------------
 * One streaming pass over the rows: cover without factor `col`, get_vector with basis
 * V[:, col], overwrite bit `col` of u_words (AssoIter.py:60), and accumulate
 * out[0..4] += (TP, FP of the new cover, #used rows, sum_{use} P, sum_{use} N). */
int bmf_refine_column(const uint64_t* x_bits, int64_t m, int64_t n, int64_t words, uint64_t* u_words,
                      int64_t kw, const uint64_t* vt_bits, int64_t k, int64_t col, int32_t wa,
                      int32_t wb, double w_fp, double w_fn, int64_t* out, bmf_stream_t stream);

/* Columns col0 .. col0+ncols-1 of AssoIter.get_refined_column in ONE pass over the rows; out[c][0..4] += what
 * bmf_refine_column(col0 + c) would accumulate after columns col0 .. col0+c-1 were refined (TP, FP, #used, sum P,
 * sum N), and u_words ends as after those ncols launches.  0 <= col0, ncols >= 1, col0 + ncols <= k; the shape rules
 * are those of bmf_refine_column.  Rows are independent: a caller holding a slice of the rows gets that slice's share
 * of every counter. */
int bmf_refine_sweep(const uint64_t* x_bits, int64_t m, int64_t n, int64_t words, uint64_t* u_words, int64_t kw,
                     const uint64_t* vt_bits, int64_t k, int64_t col0, int64_t ncols, int32_t wa, int32_t wb,
                     double w_fp, double w_fn, int64_t* out, bmf_stream_t stream);

/* ---- GreConD's concept search (bmf_concept.cu, pybmf_b200/concept.py) ------------------------------------------------
 * Bit rows x / res (the residual) are [rows][words] with n <= 64 words columns; a row mask (nullable: every row) selects
 * the extent C.  Columns are scored a column word (64 columns) at a time, for the column words cw0 .. cw0 + ncw - 1; the
 * live candidates are the columns j with lo <= j < n and j not in d_bits (nullable), where lo = state[0] + 1 when state
 * (nullable; int64 [pos, best, done, accepted]) is given, else col_lo.  With state[2] != 0 the kernels do nothing.
 * bmf_concept_intents: intents[(j - 64 cw0)][.] = AND of the rows of C with bit j (all ones when there are none) for
 *   every live j; counts (nullable, int64 [64 ncw]) = the number of those rows.  Other rows of intents are unspecified.
 * bmf_concept_covers : covers[(j - 64 cw0)] = sum over the rows r of C with bit j of popc(res[r] & I_j), where I_j is the
 *   AND over q < parts of intents[q * part_stride + (j - 64 cw0) * words + .]; 0 for the other columns.
 * bmf_concept_decide : one block: the first live j (state given) with covers[j] > state[1]; if there is one, pos = j,
 *   best = covers[j], accepted += 1, d_bits = intents[j], c_bits &= X[:, j] (c_bits: rows bits over the rows of xc);
 *   else done = 1.  covers / intents hold column j at index j.
 * bmf_concept_extent : the rows of x with bit col, compacted: xc / rc [cap][words] get their x / res rows and idx [cap]
 *   their logical rows row0 + r (-1 after the last); fill (int64) = the number of such rows; rows beyond cap are dropped.
 * bmf_concept_residual: res[idx[c] - row0] &= ~d_bits for every compact row c < rows in c_bits with row0 <= idx[c] < row1
 *   (res holds rows [row0, row1)). */
int bmf_concept_intents(const uint64_t* x, int64_t rows, int64_t words, int64_t n, const uint64_t* row_mask, int64_t cw0,
                        int64_t ncw, int64_t col_lo, const int64_t* state, const uint64_t* d_bits, uint64_t* intents,
                        int64_t* counts, bmf_stream_t stream);
int bmf_concept_covers(const uint64_t* x, const uint64_t* res, int64_t rows, int64_t words, int64_t n,
                       const uint64_t* row_mask, int64_t cw0, int64_t ncw, int64_t col_lo, const int64_t* state,
                       const uint64_t* d_bits, const uint64_t* intents, int64_t parts, int64_t part_stride, int64_t* covers,
                       bmf_stream_t stream);
int bmf_concept_decide(const uint64_t* xc, int64_t rows, int64_t words, int64_t n, const int64_t* covers,
                       const uint64_t* intents, int64_t* state, uint64_t* c_bits, uint64_t* d_bits, bmf_stream_t stream);
int bmf_concept_extent(const uint64_t* x, const uint64_t* res, int64_t rows, int64_t words, int64_t row0, int64_t col,
                       int64_t cap, uint64_t* xc, uint64_t* rc, int64_t* idx, int64_t* fill, bmf_stream_t stream);
int bmf_concept_residual(uint64_t* res, int64_t row0, int64_t row1, int64_t words, const int64_t* idx, int64_t rows,
                         const uint64_t* c_bits, const uint64_t* d_bits, bmf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PYBMF_B200_H */
