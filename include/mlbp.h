/*
 * mlbp.h -- C ABI of libmlbp.so: the B200 (sm_100a) loopy-belief-propagation hot path of
 * MacaronicUserModeling.  Plain pointers and sizes only; no torch / C++ types cross this boundary.
 *
 * The reference has no FFI of its own: its seam is two Python modules (SURVEY.md §8(b)):
 *     LBP.py                          (FactorGraph / VariableNode / FactorNode message loop)
 *     array_utils/c_array_utils.pyx   (Cython helpers, imported as `au` at LBP.py:6)
 * Every entry point below cites the reference lines it replaces (paths relative to /root/reference).
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 (MLBP_OK) or an MLBP_ERR_* code; mlbp_last_error() gives the text.
 *   - all data pointers are DEVICE pointers unless the parameter name starts with h_ (host).
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered, nothing synchronises.
 *   - the caller owns every buffer; the library owns only plan handles (host memory).
 *   - rows of "[rows, ld]" arrays are padded: ld is a multiple of 64 elements and >= V.
 *   - messages are scale-free: every consumer renormalises, so producers may emit any positive scale.
 */
#ifndef MLBP_H_
#define MLBP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MLBP_OK               0
#define MLBP_ERR_INVALID      1   /* bad argument (shape, alignment, null pointer)            */
#define MLBP_ERR_CUDA         2   /* a CUDA runtime / driver call failed                      */
#define MLBP_ERR_UNSUPPORTED  3   /* e.g. device is not sm_100, more than 2 variables/factor  */
#define MLBP_ERR_ALLOC        4

#define MLBP_N_PLANES        20   /* fp16 operand planes written by mlbp_build_pairwise_tables */
#define MLBP_N_TABLES        10   /* plane pairs (hi, lo): see MLBP_TABLE_*                    */
#define MLBP_TABLE_T          0   /* B[n=a][k=b] = T[a,b]      : message to the dim-0 variable, gap > 1 (LBP.py:509) */
#define MLBP_TABLE_TT         1   /* B[n=b][k=a] = T[a,b]      : message to the dim-1 variable, gap > 1 (LBP.py:518) */
#define MLBP_TABLE_T1         2   /* same two with the gap == 1 table pot_en_en_w1 (LBP.py:460-461)                 */
#define MLBP_TABLE_T1T        3
#define MLBP_TABLE_G          4   /* T  o PMI     : pairwise belief expectation of the pmi feature (LBP.py:566-569, :610) */
#define MLBP_TABLE_G1         5   /* T1 o PMI                                                                         */
#define MLBP_TABLE_G1W        6   /* T1 o PMI_w1  : expectation of the pmi_w1 feature, gap == 1 factors only          */
#define MLBP_TABLE_GT         7   /* transposes of G, G1, G1W: a COLUMN of a gradient table as a contiguous row, read by   */
#define MLBP_TABLE_G1T        8   /* mlbp_spike_correct when it restores the lo part of a spike in a gradient-stage row   */
#define MLBP_TABLE_G1WT       9

#define MLBP_N_SUMS           7   /* per-theta sum vectors written by mlbp_build_pairwise_tables                */
#define MLBP_D_CONST_ROWS     5   /* D rows 1..4 hold the constant messages of the 4 message tables (row 0 spare) */
#define MLBP_A_SCALE_LOG2    14   /* var->factor rows are stored as 2^14 * normalised message, split hi + lo fp16 */
#define MLBP_SPIKE_SLOTS      4   /* spikes recorded per A row (mlbp_spike_scan / mlbp_spike_correct)             */

const char *mlbp_last_error(void);
int mlbp_version(void);
/* 1 if the current device is compute capability 10.x, else 0 (also 0 when there is no device). */
int mlbp_device_ok(void);

/* ------------------------------------------------------------------------------------------------
 * (1) array_utils/c_array_utils.pyx dense helpers, float64 like the reference.
 * ------------------------------------------------------------------------------------------------ */
/* pyx:12-16  np.multiply(m1, m2)  (LBP.py:728) */
int mlbp_pointwise_multiply_f64(const double *m1, const double *m2, double *out, int64_t n, void *stream);
/* pyx:29-40  s = sum(m1); s > 0 ? m1 / s : zero-fill.  *d_sum (device, 1 double) receives s. (LBP.py:540,569,653) */
int mlbp_normalize_f64(const double *m1, double *out, int64_t n, double *d_sum, void *stream);
/* pyx:90-91  m1.dot(m2), row-major (m,k) x (k,n): the GEMV / outer product of LBP.py:509,518,566 */
int mlbp_dense_dot_f64(const double *m1, const double *m2, double *out, int m, int k, int n, void *stream);
/* pyx:93-94  np.multiply(m1, m2) on 2-D arrays (LBP.py:568) */
int mlbp_dense_pointwise_multiply_f64(const double *m1, const double *m2, double *out, int64_t n, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (2) potentials that depend on theta only -- replaces the per-sentence rebuild of train.py:218-253.
 * ------------------------------------------------------------------------------------------------ */
/* K2.  pmi, pmi_w1: [V, ldf] fp32 row-major feature planes (train.py:589-595).
 *   T  = exp(th[0]*pmi + th[2]),  T1 = exp(th[0]*pmi + th[1]*pmi_w1 + th[2])            (train.py:218-219, :252-253)
 *   planes: MLBP_N_PLANES fp16 arrays [V, ldv], plane p at planes + p*plane_stride, in the order
 *           T.hi T.lo Tt.hi Tt.lo T1.hi T1.lo T1t.hi T1t.lo G.hi G.lo G1.hi G1.lo G1w.hi G1w.lo Gt.hi Gt.lo G1t.hi G1t.lo G1wt.hi G1wt.lo,
 *           every value multiplied by 2^scale_exp before the hi/lo split (hi + lo carries 22 bits).
 *   colsums: [MLBP_N_SUMS, V] float64, UNscaled: sum_e T[e,y], sum_e T1[e,y], sum_e G[e,y], sum_e G1[e,y], sum_e G1w[e,y]
 *           (the normaliser and feature expectations of the unary en_en factors, LBP.py:540, :600-603), then the
 *           row sums sum_b T[a,b], sum_b T1[a,b]: together with the column sums they are the factor->variable
 *           messages of a pairwise factor whose incoming message is still the uniform initial one (LBP.py:211-216).
 *   with_grad_planes = 0 skips planes 8..19 (inference only).
 *   r_planes (or NULL): four more fp16 planes [V, ldv], same stride, R.hi Rt.hi R1.hi R1t.hi with R = T - tbar, R1 = T1 - tbar
 *           (scaled like the others, stochastic rounding of the magnitude), tbar = 2^scale_exp * exp(th[2]) = the table at
 *           phi = 0, returned in *h_tbar (a positive *h_tbar on entry overrides it): the operand of the ONE-pass message rows, whose GEMM adds tbar * sum(message) back as
 *           a constant (mlbp_factor_to_var_gemm_gated add_const) -- the fp16 rounding is then relative to |T - tbar|.        */
int mlbp_build_pairwise_tables(const float *pmi, const float *pmi_w1, int V, int ldf, const double *h_theta_ee,
                               int scale_exp, void *planes, int64_t plane_stride, int ldv, double *colsums,
                               int with_grad_planes, void *r_planes, float *h_tbar, void *stream);
/* edT, pedT: [Vd, ldf] fp32, de-major (row d = phi_en_de[:, d, k] of LBP.py:602 made contiguous).
 *   edstats[d] = { sum_e psi, sum_e psi*ed, sum_e psi*ped },  psi = exp(th[0]*ed + th[1]*ped + th[5])  (train.py:240,251) */
int mlbp_build_unary_tables(const float *edT, const float *pedT, int V, int Vd, int ldf, const double *h_theta_ed,
                            double *edstats, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (3) unary factors of a batch of sentences (LBP.py:492-498, :540, :600-603; train.py:176-215, :255-297)
 *     nv variables; variable v observes German word var_de[v], has supervised label var_label[v],
 *     sparse per-sentence en_de features sp_*[sp_off[v] .. sp_off[v+1]) already filtered to de == var_de[v],
 *     and unary en_en factors giv_*[giv_off[v] .. giv_off[v+1]) (label of the given token, gap == 1 flag).
 * ------------------------------------------------------------------------------------------------ */
/* per-variable normaliser and the closed-form unary gradient terms:
 *   inv_sigma[v]  = 1 / sum_e psi_v(e)                      (psi_v includes the sparse features)
 *   g_unary[v][9] = sum over v's unary factors of  phi[label, obs, :] - sum_e belief(e) phi[e, obs, :]
 *                   laid out [pmi, pmi_w1, bias | ed, ped, correct, full_history, hit_history, bias]   */
int mlbp_unary_stats(int nv, const int32_t *var_de, const int32_t *var_label, const int32_t *sp_off,
                     const int32_t *sp_en, const int32_t *sp_feat, const float *sp_val, const int32_t *giv_off,
                     const int32_t *giv_label, const int32_t *giv_gap1, const float *pmi, const float *pmi_w1,
                     const float *edT, const float *pedT, int V, int ldf, const double *h_theta_ed,
                     const double *edstats, const double *colsums, double *inv_sigma, double *g_unary, void *stream);
/* K1.  U[v, e] = V^(1+g) * prod over v's unary factors of their normalised message (mean-one scaling),
 *   the en_de factor recomputed from the de-major feature rows (coalesced gather-dot + exp), the en_en
 *   factors read as rows of the transposed table planes.  U: [nv, ldv] fp32.                            */
int mlbp_unary_products(int nv, const int32_t *var_de, const int32_t *sp_off, const int32_t *sp_en,
                        const int32_t *sp_feat, const float *sp_val, const int32_t *giv_off,
                        const int32_t *giv_label, const int32_t *giv_gap1, const float *edT, const float *pedT,
                        int V, int ldf, const double *h_theta_ed, const double *inv_sigma, const void *planes,
                        int64_t plane_stride, int ldv, int scale_exp, const double *colsums, float *U, void *stream);

/* ------------------------------------------------------------------------------------------------
 * (4) message kernels
 * ------------------------------------------------------------------------------------------------ */
/* uniform 1/V messages of FactorGraph.initialize (LBP.py:211-216) as fp16 hi/lo rows: rows[i] of A := 2^14 / V.
 * keep (optional, may be NULL): uint8 [V]; entries with keep[e] == 0 are written as 0 (top-K mask of a uniform message). */
int mlbp_fill_uniform_rows(void *A_hi, void *A_lo, int ldv, int V, const int32_t *rows, int n_rows,
                           const uint8_t *keep, void *stream);
/* K3.  VariableNode.update_message_to (LBP.py:377-389) for n_groups (variable, level) groups at once.
 *   group g multiplies U[grp_u[g]] with the factor->variable rows D[in_row[i]], i in [grp_off[g], grp_off[g+1]);
 *   for every i with destinations it emits the leave-one-out product (all inputs except i), renormalised
 *   (sum <= 0 or non-finite -> uniform, LBP.py:650-657; nan_to_num LBP.py:729), scaled by 2^14 and split into
 *   A_hi/A_lo rows dest[dest_off[i] .. dest_off[i+1]); first_dest[i] / second_dest[i] = dest[dest_off[i]] /
 *   dest[dest_off[i] + 1] (-1 if absent), stored per slot so that the kernels need no dependent index load for the two
 *   readers a message usually has (a message GEMM row and a gradient-stage row).  in_row < 0 means "uniform message": the kernels read the
 *   constant-one row D[0] in its place (messages are scale-free), so the caller keeps D row 0 filled with 1.0f.
 *   range_log2: caller's bound on |log2| of any product of one U element with max_in D elements; in [0, 100) the
 *   products are formed in fp32, otherwise (or negative = unknown) in fp64 (slow on B200: the fp64 pipe is narrow).
 */
int mlbp_var_to_factor(int n_groups, const int32_t *grp_u, const int32_t *grp_off, const int32_t *in_row,
                       const int32_t *dest_off, const int32_t *dest, const int32_t *first_dest,
                       const int32_t *second_dest, const float *U, const float *D, int ldv, int V, void *A_hi,
                       void *A_lo, int max_in, float range_log2, void *stream);
/* K4a. Spikes of the var->factor messages in A rows [a_row0, a_row0 + n_rows) (one GEMM block; run before the block's GEMM).
 *   A reduced-pass GEMM row (MLBP_GEMM_A_HI_ONLY) drops the lo half of every message element; for the bulk of a message that
 *   rounding averages away in the contraction, for an element that carries more than spike_prob of the mass (a history
 *   feature's word, say) it does not.  For every row the kernel files up to MLBP_SPIKE_SLOTS such elements as
 *   (column, float bits of the A_lo value) in spike_entries[row][slot] (int32 pairs, ascending columns), writes their number
 *   to spike_cnt[row] (MLBP_SPIKE_SLOTS + 1 = more than fit), and appends rows with spikes to block_rows[0 .. *block_n)
 *   (optional; *block_n zeroed by the caller).  spike_words (5 device int32, zeroed by the caller per theta / batch as noted):
 *     [0] PEAK   set when a row has more spikes than slots: mlbp_factor_to_var_gemm_gated then keeps the lo half        (per theta)
 *     [2] the largest spike seen so far, bits of the float 2^14 * probability (atomic max; diagnostics)                 (per theta)
 *     [3] SPIKE  set when any spike was seen (diagnostics)                                                               (per theta)
 *     [4] number of rows with spikes (diagnostics)                                                                      (per batch) */
int mlbp_spike_scan(const void *A_hi, const void *A_lo, int ldv, int V, int a_row0, int n_rows, float spike_prob,
                    int32_t *spike_words, int32_t *spike_cnt, int32_t *spike_entries, int32_t *block_rows, int32_t *block_n,
                    void *stream);
/* K4b. Spike compensation of a GEMM block that dropped the lo half of A (rows [a_row0, a_row0 + n_rows) of A -> D rows d_row0 ..):
 *   D[r, n] += alpha * sum over the recorded spikes s of row r of  lo_s * B[n, col_s],  with B[n, col] read as row `col` of
 *   the TRANSPOSED table's plane pair Bt_hi / Bt_lo (MLBP_TABLE_T <-> TT, T1 <-> T1T, G <-> GT, G1 <-> G1T, G1W <-> G1WT).
 *   block_rows / block_n: this block's list of spiky rows and its length (mlbp_spike_scan).  Returns at once (on the device) when spike_words[0] is set: the block then ran with the lo half.
 *   Spikes of a row are applied in ascending column order (deterministic).
 *   A_hi_one_pass (or NULL): the block ran ONE pass (A_hi . B_hi, MLBP_GEMM_A_HI_ONLY | MLBP_GEMM_B_HI_ONLY), so the spikes' share
 *   of the other dropped term is restored too:  D[r, n] += alpha * hi_s * B_lo[n, col_s]  with hi_s read from A_hi[r, col_s].
 *   Rt_hi (or NULL; needs A_hi_one_pass) + tbar: the one-pass block contracted with the RESIDUAL plane R = T - tbar; Rt_hi is the
 *   residual plane of the transposed table:  D[r, n] += alpha * ((hi_s + lo_s) * (B[n, col_s] - tbar) - hi_s * R_hi[n, col_s]).  */
int mlbp_spike_correct(const int32_t *spike_words, const int32_t *spike_cnt, const int32_t *spike_entries,
                       const int32_t *block_rows, const int32_t *block_n, int a_row0, int n_rows, const void *Bt_hi,
                       const void *Bt_lo, int V, int ldv, float *D, int64_t d_row0, int ldd, float alpha,
                       const void *A_hi_one_pass, const void *Rt_hi, float tbar, void *stream);
/* K5c. The K most probable words of each of n_rows belief rows X[r, 0..V) (fp32, row stride ldx), best first, on the device:
 *   VariableNode.get_max_vocab (LBP.py:402-411: np.argpartition + np.argsort on the host marginal; K = 50 for
 *   FactorGraph.to_string / get_precision_counts, LBP.py:87, :115).
 *   idx[r, 0..K) / val[r, 0..K): word indices and probabilities, descending value, ascending index among equal values.
 *   n_ties[r] (or NULL): > 0 when the order of row r is not decided by the values alone (equal neighbours inside the list, or
 *   more entries equal to the K-th value than were listed): NumPy's order among exactly equal values is an implementation
 *   detail, so a caller that has to reproduce it falls back to the host calls for that row.  1 <= K <= min(V, 1024).       */
int mlbp_topk_rows(const float *X, int ldx, int V, int n_rows, int K, int32_t *idx, float *val, int32_t *n_ties, void *stream);
/* K7.  The .dist text of n_rows belief rows (FactorGraph.to_dist, LBP.py:125-143), on the device: row r of X (fp32, row stride
 *   ldx, V entries) becomes the bytes of  ' '.join('%0.6f' % x for x in np.log(row.astype(np.float64)))  at
 *   out[offsets[r] .. offsets[r + 1]), offsets[0] = 0 (int64, n_rows + 1 entries); no separator after a row's last number.
 *   The log is the correctly rounded float64 log of each input and the decimals are CPython's (round half to even on the exact
 *   binary value): 0 -> "-inf", NaN or x < 0 -> "nan", +inf -> "inf", a negative value that rounds to zero -> "-0.000000".
 *   out_bytes (the capacity of out) must be at least MLBP_FMT_MAX_BYTES * V * n_rows: checked on the host, nothing is launched
 *   otherwise.  Deterministic.  n_rows = 0 only writes offsets[0].                                                      */
#define MLBP_FMT_MAX_BYTES   12   /* "-103.278930" (log of the smallest subnormal) plus its separator                 */
int mlbp_format_log_rows(const float *X, int ldx, int V, int n_rows, char *out, int64_t out_bytes, int64_t *offsets,
                         void *stream);
/* K8.  np.loadtxt(path, dtype=float64) of a feature matrix (train.py:589-603) on the device, one chunk of the file at a time:
 *   text[0 .. n_bytes) (16-byte aligned) starts at byte file_offset of the file and ends on a line boundary (after a '\n', or
 *   at the end of the file).  Grammar, for ASCII text: fields separated by runs of ' ' \t \v \f (and \r before \n); blank and
 *   whitespace-only lines are skipped; '#' starts a comment that runs to the end of the line; a field is
 *   [+-] (digits [. digits] | . digits) [(e|E) [+-] digits] or [+-] (inf | infinity | nan), case-insensitive.
 *   Field k of the file (state[MLBP_PARSE_FIELDS] counts the fields of the earlier chunks) is converted to the correctly rounded
 *   float64, rounded to nearest-even fp32 and stored at out[row * ld_out + col], (row, col) = divmod(k, n_cols); NaN keeps its sign.
 *   state: MLBP_PARSE_STATE_WORDS device words, zeroed by the caller before the first chunk of a file and read once after the
 *   last:  [MLBP_PARSE_FIELDS] fields so far; [MLBP_PARSE_ERROR] ~(offset << 3 | kind) of the first offending byte (0 = none);
 *   [MLBP_PARSE_MIN] ~key of the smallest value, [MLBP_PARSE_MAX] key of the largest (key(b) = b ^ (sign ? ~0 : 1 << 63) of the
 *   float64 bits b; NaN and hard fields are not included); [MLBP_PARSE_NAN] bit 0 / 1: a positive / negative NaN was read;
 *   [MLBP_PARSE_HARD] number of hard fields.
 *   Hard fields (more than 19 significant digits whose rounding the first 19 do not decide) are not written: their (file byte
 *   offset, field index) pairs go to hard[2 * i], hard[2 * i + 1] for i < hard_cap, in no particular order; the caller converts them.
 *   tile_ws: ceil(n_bytes / MLBP_PARSE_TILE_BYTES) device words of scratch.  n_bytes <= MLBP_PARSE_MAX_CHUNK.             */
#define MLBP_PARSE_TILE_BYTES   4096
#define MLBP_PARSE_MAX_CHUNK    (((int64_t)1 << 31) - 1)
#define MLBP_PARSE_STATE_WORDS  8
#define MLBP_PARSE_FIELDS       0
#define MLBP_PARSE_ERROR        1
#define MLBP_PARSE_MIN          2
#define MLBP_PARSE_MAX          3
#define MLBP_PARSE_NAN          4
#define MLBP_PARSE_HARD         5
#define MLBP_PARSE_ERR_FIELD    1   /* a field outside the grammar                                  */
#define MLBP_PARSE_ERR_COLS     2   /* a line whose field count is not n_cols                        */
#define MLBP_PARSE_ERR_ROWS     3   /* more than max_rows rows                                       */
#define MLBP_PARSE_ERR_BYTE     4   /* a byte >= 0x80, another control byte, or \r not before \n      */
int mlbp_parse_float_text(const char *text, int64_t n_bytes, int64_t file_offset, int n_cols, int64_t max_rows, float *out,
                          int64_t ld_out, uint64_t *state, int64_t *hard, int hard_cap, uint64_t *tile_ws, void *stream);
/* Approximate paths (use_approx_inference LBP.py:506-507, :515-516 -> au.sparse_vec_mat_dot pyx:193-205;
 *   use_approx_beliefs LBP.py:554-563 -> au.sparse_dot / sparse_pointwise_multiply / sparse_normalize pyx:108-129, :23-26):
 *   keep the K largest entries of each of the n_rows operand rows A[row0 ..], zero the others (K = 100 in the reference);
 *   the dense kernels then produce exactly the reference's restricted sums.  No-op when K >= V.                  */
int mlbp_topk_mask_rows(void *A_hi, void *A_lo, int ldv, int V, int64_t row0, int n_rows, int K, void *stream);
/* K4.  FactorNode.update_message_to for pairwise factors (LBP.py:499-526; au.dense_dot pyx:90-91), batched:
 *   D[d_row0 + r, n] = alpha * sum_k (A_hi + A_lo)[a_row0 + r, k] * (B_hi + B_lo)[n, k],  r < n_rows, n < V
 *   as three tcgen05 passes hi*hi + hi*lo + lo*hi with fp32 accumulation in tensor memory.
 *   A_*: [a_rows_total, ldv] fp16, B_*: one plane pair [V, ldv] fp16, D: [*, ldd] fp32.
 *   impl: 0 = tcgen05 (product path: the CTA-pair kernel for V > 2048, the one-CTA kernel below), 1 = SIMT cross-check
 *   kernel (tests only), 2 / 3 = the CTA-pair / one-CTA kernel of the product path at any V (tests); further tile and
 *   pipeline variants exist only in a -DMLBP_PROBES build (scripts/gemm_probe.py).  OR-ed with MLBP_GEMM_A_HI_ONLY the
 *   A_lo term is dropped (two passes hi*hi + hi*lo, A_lo is not even loaded).  The gradient stage uses it: the
 *   expectation N/Z of a pairwise belief is a RATIO of two rows computed from the same message r, so the 2^-12
 *   rounding of r largely cancels (measured <= 2e-7 relative on a sentence's gradient; the contract is 1e-4).      */
#define MLBP_GEMM_A_HI_ONLY 256
/* additionally drops the B_lo term: one pass, plain fp16 x fp16 with fp32 accumulation (gradient rows at large V only) */
#define MLBP_GEMM_B_HI_ONLY 512
int mlbp_factor_to_var_gemm(const void *A_hi, const void *A_lo, int64_t a_rows_total, int a_row0, int n_rows,
                            const void *B_hi, const void *B_lo, int V, int ldv, float *D, int64_t d_row0, int ldd,
                            float alpha, int impl, void *stream);
/* The same launch, DECIDED ON THE DEVICE: every CTA first reads *gate (device int32) and returns at once unless
 * (*gate != 0) == (run_if_set != 0).  The engine issues a level's message rows twice -- two passes (A_HI_ONLY) with
 * run_if_set = 0 and all three passes with run_if_set = 1 -- on the PEAK word that mlbp_spike_scan raises when a message has
 * more spikes than it can record (the one-pass gradient rows fall back to two passes on the same word); exactly one of the two launches
 * does the work and no host synchronisation is needed.
 * gate == NULL runs unconditionally.  tcgen05 kernels only (impl 1, the SIMT cross-check, ignores the gate on the host: error).
 * K range: [k0, k0 + k_len) in elements, multiples of 64 (k_len == 0: up to V).  A launch whose range does not start at 0
 * ADDS its product to D.  The engine splits a long K (V = 50 000) into several launches: the CTA pairs of one launch drift
 * apart in K and stop sharing operand slabs in L2, a kernel boundary re-aligns them.  CTA-pair kernel only.
 * add_const: added to every element of the product (by the launch whose K range starts at 0):  D = alpha * A . B^T + add_const.
 * With B_hi a residual plane R = T - tbar (mlbp_build_pairwise_tables r_planes) and message rows that sum to 2^14,
 * add_const = alpha * 2^14 * tbar makes a ONE-pass launch (A_HI_ONLY | B_HI_ONLY) the product with T itself.                 */
int mlbp_factor_to_var_gemm_gated(const void *A_hi, const void *A_lo, int64_t a_rows_total, int a_row0, int n_rows,
                                  const void *B_hi, const void *B_lo, int V, int ldv, float *D, int64_t d_row0, int ldd,
                                  float alpha, int impl, const int32_t *gate, int run_if_set, int k0, int k_len,
                                  float add_const, void *stream);
/* K5.  VariableNode.get_marginal / get_posterior_probs / get_precision_counts / argmax
 *   (LBP.py:392-411, :247-259, :80-106).  Same group layout as K3, all inputs multiplied.
 *   logp[g] = log b[label] (-99.99 if b[label] == 0), top1[g] = argmax b (first index on ties),
 *   rank[g] = #{e : b[e] > b[label]}, beliefs (optional, may be NULL): [n_groups, ldv] fp32 normalised.
 *   range_log2 as in mlbp_var_to_factor (bound for ALL incoming messages of a variable); max_in = the largest number of
 *   incoming pairwise messages of any variable (MLBP_ERR_UNSUPPORTED above 64).
 *   Near-tie detection (flags != NULL, else the five pointers may be NULL): flags[g] bit 0 = the runner-up product is within
 *   the relative band tau of the largest, bit 1 = some other candidate is within tau_label of the label's product while at
 *   most 50 candidates are certainly above the label (its rank can still decide P@25 / P@50, LBP.py:80-106);
 *   aux[g] = {largest product, label's product} (float64), cnts[g] = {#products > label's, #of those inside the band};
 *   flagged[0 .. *n_flagged) lists the variables with flags != 0 (atomic append: zero *n_flagged before the call).   */
int mlbp_marginals(int n_groups, const int32_t *grp_u, const int32_t *grp_off, const int32_t *in_row,
                   const int32_t *label, const float *U, const float *D, int ldv, int V, double *logp,
                   int32_t *top1, int32_t *rank, float *beliefs, float range_log2, int max_in, float tau,
                   float tau_label, double *aux, int32_t *cnts, int32_t *flags, int32_t *flagged, int32_t *n_flagged,
                   void *stream);
/* K5b. Exact re-score of the flagged variables' near-tied candidates (LBP.py:392-411: arg-max; :80-106: label rank).
 *   For every candidate e inside the bands of mlbp_marginals and every incoming message row the ONE element
 *   D_j[e] = sum_k (A_hi + A_lo)[row_j, k] * (B_hi + B_lo)[table_j][e, k] is recomputed from the full 22-bit operands
 *   (fp32 products, float64 reduction), the ratios are multiplied in float64, and top1[g] / rank[g] are overwritten with
 *   the decisions taken on those values.  This makes the last hop into a belief -- the only place where the rounding of a
 *   reduced-pass message row is not damped by a later contraction -- exact wherever it can change a decision.
 *   msg_blocks: the plan's flat list of message GEMM blocks, 4 int32 each {table, first A row, first D row, rows}, ascending
 *   (blob header H_MSG_BLK_*); a D row r of a message block has A row r - MLBP_D_CONST_ROWS.  planes / plane_stride as in
 *   mlbp_build_pairwise_tables.  counters[8] (device int32, accumulated): [0] variables re-scored, [1] skipped (more than 64
 *   candidates: a mass tie), [2] skipped (degenerate products), [3] arg-max decisions changed, [4] ranks changed.          */
int mlbp_rescore_candidates(int n_vars, const int32_t *flagged, const int32_t *n_flagged, const int32_t *flags,
                            const int32_t *grp_u, const int32_t *grp_off, const int32_t *in_row, const int32_t *label,
                            const float *U, const float *D, int ldv, int V, const void *A_hi, const void *A_lo,
                            const void *planes, int64_t plane_stride, const int32_t *msg_blocks, int n_blocks,
                            int n_msg_rows, const double *aux, const int32_t *cnts, float tau, float tau_label,
                            float range_log2, int32_t *top1, int32_t *rank, int32_t *counters, void *stream);
/* K6a. pairwise factor beliefs contracted with the features (LBP.py:544-569 + :610) in closed form:
 *   stats[f] = { z.u0, c.u1, c.u2 } with c = (A_hi + A_lo)[c_row[f]], z = (A_hi + A_lo)[z_row[f]],
 *   u* = D[u*_row[f]] (u2_row < 0 -> 0).  z_row == c_row with u0 = T r, or z_row = the r row with u0 = T'c
 *   (the plan reuses the D row of the factor's last message update when it read the final message).
 *   Spike cells (spike_words != NULL, else the seven arguments after stats are ignored): when the u rows come from ONE-pass
 *   gradient GEMMs (alpha * r_hi . B_hi) the lo half of the table planes is missing.  Its rounding averages away over the
 *   cells a belief spreads over, except where both messages have a spike; for those cells (spike lists of rows c_row[f]
 *   and r_row[f] from mlbp_spike_scan) the kernel adds  alpha * c[a] * r_hi[b] * B_lo[a, b]  to the three sums, B = T / G /
 *   G1w planes of the factor's gap class (pair_gap1).  Skipped on the device when spike_words[0] (PEAK) is set.        */
int mlbp_pair_expectations(int n_factors, const int32_t *c_row, const int32_t *z_row, const int32_t *u0_row,
                           const int32_t *u1_row, const int32_t *u2_row, const void *A_hi, const void *A_lo, const float *D,
                           int ldv, int V, double *stats, const int32_t *r_row, const int32_t *pair_gap1,
                           const int32_t *spike_words, const int32_t *spike_cnt, const int32_t *spike_entries,
                           const void *planes, int64_t plane_stride, float alpha, void *stream);
/* K6b. FactorGraph.get_unregularized_gradeint (LBP.py:301-320) as a segmented reduction:
 *   grad[s][9] = sum_{v in sentence s} g_unary[v] + sum_{pairwise f in s} (phi[l0,l1,:] - E_f[phi]),
 *   (l0, l1) = var_label[pair_v0[f]], var_label[pair_v1[f]] (the observed one-hot of LBP.py:584-589);
 *   sentence s owns variables [sent_var_off[s], sent_var_off[s+1]) and factors [sent_fac_off[s], ..);
 *   sent_fac_off == NULL: no pairwise factors (inference-only callers that want logp_sent).
 *   logp_sent[s] = sum of logp_var over the sentence (LBP.py:247-259).                                     */
int mlbp_gradient_reduce(int n_sent, const int32_t *sent_var_off, const int32_t *sent_fac_off, const double *g_unary,
                         const double *pair_stats, const int32_t *pair_v0, const int32_t *pair_v1,
                         const int32_t *var_label, const int32_t *pair_gap1, const float *pmi, const float *pmi_w1,
                         int ldf, const double *logp_var, double *grad, double *logp_sent, void *stream);
/* K6c. Batch level of the reduction: what train_mp.py's parent callback sums under its lock (train_mp.py:405-424), and the
 *   precision counts of FactorGraph.get_precision_counts (LBP.py:80-106).  ADDS this micro-batch to out16 (device, 16 float64,
 *   zeroed by the caller at the start of an SGD step; it is the buffer the NCCL all-reduce ships):
 *   [0..8] sum of grad[s][9], [9] sum of logp_sent, [10] #rank == 0, [11] #rank < 26, [12] #rank < 50, [13] n_vars, [14] n_sent;
 *   [15] = max([15], (spike_words[0] ? 1 : 0) + (spike_words[3] ? 2 : 0)) with peak_flag = the spike_words of
 *   mlbp_spike_scan (which reduced-pass GEMM variants this rank ran).  grad / logp_sent / rank / peak_flag may be NULL.
 *   One CTA, fixed summation order (deterministic).                                                              */
int mlbp_batch_reduce(int n_sent, const double *grad, const double *logp_sent, int n_vars, const int32_t *rank,
                      const int32_t *peak_flag, double *out16, void *stream);
/* K9.  Joint log-likelihood of each sentence's labels, the Bethe estimate at the final messages (not in the reference, whose
 *   one fit statistic is the sum of MARGINAL log-probabilities, LBP.py:247-259):
 *     logp_joint[s] = sum_{v in s} logp_var[v]
 *                   + sum_{pairwise f in s} [ log T_f(y0, y1) - log Z_f + sum_{k = 0, 1} ( log O_{f,k} - log mu_k[y_k] ) ]
 *   with y0, y1 = var_label[pair_v0[f]], var_label[pair_v1[f]]; nu_0 = (A_hi + A_lo)[c_row[f]], nu_1 = (A_hi + A_lo)[r_row[f]]
 *   the final variable->factor messages, mu_k = D[mk_row[f]] (mk_row < 0: the constant-one row D[0]) the final factor->variable
 *   messages of the factor's dim-0 / dim-1 variable, O_{f,k} = nu_k . mu_k (fp32 products, float64 sums in a fixed order),
 *   Z_f = pair_stats[f][0] * 2^-z_scale_log2 (mlbp_pair_expectations: 2^z_scale_log2 * nu_0' T nu_1 on the unscaled table),
 *   log T = th[0] * pmi + th[1] * pmi_w1 (gap == 1 only) + th[2] in float64 from the fp32 planes [V, ldf] (train.py:218-219).
 *   Row scales cancel (each row enters once with + and once with -).  Exact on trees; with one variable it is logp_var.
 *   A sentence with a variable whose logp_var is -99.99 (label of belief 0) gets -inf.  pair_term: n_pairs float64 of scratch.
 *   Sentence s owns variables [sent_var_off[s], ..) and factors [sent_fac_off[s], ..); n_pairs = sent_fac_off[n_sent].
 *   Two launches (one warp per factor, one warp per sentence), deterministic.  Bad arguments: MLBP_ERR_INVALID, nothing launched. */
int mlbp_joint_logp(int n_sent, int n_pairs, const int32_t *sent_var_off, const int32_t *sent_fac_off, const double *logp_var,
                    const int32_t *c_row, const int32_t *r_row, const int32_t *m0_row, const int32_t *m1_row,
                    const int32_t *pair_v0, const int32_t *pair_v1, const int32_t *var_label, const int32_t *pair_gap1,
                    const double *pair_stats, const void *A_hi, const void *A_lo, const float *D, int ldv, int V,
                    const float *pmi, const float *pmi_w1, int ldf, const double *h_theta_ee, int z_scale_log2,
                    double *pair_term, double *logp_joint, void *stream);
/* K10. Max-product factor->variable messages (not in the reference, which runs sum-product only): for r < n_rows, n < V
 *     D[d_row0 + r, n] = max_{k < V} ( a[r, k] / amax_r ) * T'[n, k]
 *   a[r, k] = (A_hi + A_lo)[a_row0 + r, k] in fp32 (exact), amax_r = max_k a[r, k] (a row with amax_r = 0 gives a zero D row),
 *   T' the message table `table` (MLBP_TABLE_T, TT, T1 or T1T) in the B[n][k] orientation documented above, formed from the fp32
 *   feature planes pmi / pmi_w1 [V, ldf]:  T'[a, b] = exp(th[0] pmi[a, b] + [T1, T1T] th[1] pmi_w1[a, b] + th[2] - centre_exp ln 2)
 *   with K2's compensated argument (~1 ulp; K2's fp16 planes are not read).  Every output lies within [min T', max T'] up to a few
 *   ulp.  Columns k >= V of A and of the planes are never used; only columns [0, V) of D are written.  fp32 products, exact max:
 *   bit-identical for any row slicing.  Needs ldv % 8 == 0, ldf % 4 == 0 and 16-byte aligned A_hi, A_lo, pmi, pmi_w1.
 *   MLBP_ERR_INVALID, nothing launched: a null pointer, an unknown table id, V < 1, ldv / ldf / ldd < V, a row range outside
 *   [0, a_rows_total), the alignment above.  n_rows == 0 is a no-op.                                                             */
int mlbp_factor_to_var_maxprod(const void *A_hi, const void *A_lo, int64_t a_rows_total, int a_row0, int n_rows, int table,
                               const float *pmi, const float *pmi_w1, int V, int ldv, int ldf, const double *h_theta_ee,
                               int centre_exp, float *D, int64_t d_row0, int ldd, void *stream);
/* K11. Log of the unnormalised joint potential of an assignment x (one int32 word per variable, sentence s owns variables
 *   [var_off[s], var_off[s + 1])), float64 per sentence (the model of SURVEY.md Appendix A; train.py:218-253, :255-297):
 *     score[s] = sum_{i in s} [ td[0] edT[d_i, x_i] + td[1] pedT[d_i, x_i] + td[5]
 *                               + sum over the sparse features (e, f, val) of i with e == x_i of td[f] val
 *                               + sum over the given tokens j of i of l_{gap1}(x_i, giv_label[j]) ]
 *              + sum over the pairwise factors (v0, v1) of s (pair indices local to the sentence) of l_{gap1}(x_v0, x_v1)
 *     l_g(a, b) = te[0] pmi[a, b] + te[2] + g te[1] pmi_w1[a, b]
 *   (no en_de term where var_de < 0).  Corpus arrays as in mlbp_unary_stats / mlbp_plan_compile; pmi, pmi_w1 [V, ldf] and edT,
 *   pedT [Vd, ldf] fp32.  One warp per sentence, fixed summation order (deterministic).  n_vars = var_off[n_sent] and n_given =
 *   giv_off[n_vars] are checked, and so is every x[i] and giv_label[j] against [0, V): on the host, after a copy that
 *   SYNCHRONISES the stream; MLBP_ERR_INVALID, nothing launched.                                                                */
int mlbp_assignment_score(int n_sent, int n_vars, int n_given, const int32_t *var_off, const int32_t *x, const int32_t *var_de,
                          const int32_t *sp_off, const int32_t *sp_en, const int32_t *sp_feat, const float *sp_val,
                          const int32_t *giv_off, const int32_t *giv_label, const int32_t *giv_gap1, const int32_t *pair_off,
                          const int32_t *pair_v0, const int32_t *pair_v1, const int32_t *pair_gap1, const float *pmi,
                          const float *pmi_w1, const float *edT, const float *pedT, int V, int ldf, const double *h_theta_ee,
                          const double *h_theta_ed, double *score, void *stream);
/* rows[0] = 1.0f (the constant-one row the kernels read for a message that is still uniform), rows[1 + t] = the message of a
 *   pairwise factor of message table t (MLBP_TABLE_T .. T1T) that is fed the uniform initial message (LBP.py:211-216 +
 *   :509 / :518): the row / column sums of the table, mean-one scaled.  rows: [MLBP_D_CONST_ROWS, ldv] fp32; the engine
 *   copies them to D rows 0..4 of every micro-batch.                                                            */
int mlbp_const_rows(const double *colsums, int V, int ldv, float *rows, void *stream);

/* 0, or the code of the mbarrier wait (1 = stage empty, 2 = stage full, 3 = accumulator full, 4 = accumulator drained) that
 * exceeded its ~4 s bound inside a tcgen05 GEMM kernel: the kernel records it in mapped host memory and traps (the launch
 * fails with a CUDA error) instead of hanging the GPU.                                                              */
int mlbp_gemm_barrier_timeout_code(void);

/* zero n device int32 words on the stream: the flag / counter words the kernels above communicate through */
int mlbp_zero_words(int32_t *words, int n, void *stream);

/* probe hook (scripts/k3_probe.py): per-CTA stage cycle counters of the resident K3 kernel are written to p[6 * CTA]
 * when the library is built with -DMLBP_K3_STAGE_TIMES; a no-op otherwise.  NULL switches it off.               */
void mlbp_debug_k3_times(long long *p);

/* ------------------------------------------------------------------------------------------------
 * (5) host-side schedule compiler: FactorGraph.initialize / has_loops / get_message_schedule /
 *     treelike_inference (LBP.py:155-245) for a batch of graphs, lowered to dependency levels.
 * ------------------------------------------------------------------------------------------------ */
typedef struct mlbp_plan mlbp_plan;
/* Graph g has variables [var_off[g], var_off[g+1]) and pairwise factors [pair_off[g], pair_off[g+1]) listed in the
 * order they were attached (defines facset order, LBP.py:367-369).  pair_v0/pair_v1 are variable indices LOCAL to
 * the graph (v0 = dim 0, v1 = dim 1 of the potential table), pair_gap1 selects pot_en_en_w1 (LBP.py:456-463).
 * roots: local variable index per graph and draw, [n_graphs, 1 + sweeps] (draw 0 = has_loops, LBP.py:176).
 * flags: bit 0 = plan the gradient stage, bit 1 = plan the marginal stage, bit 2 = do NOT constant-fold updates
 *        that read an initial uniform message (needed by the top-K approximate mode, which masks that message),
 *        bit 3 = give every pairwise belief normaliser Z its own GEMM row instead of reusing the D row of the factor's
 *        last message update (needed whenever message rows are masked: top-K approximate modes),
 *        bit 4 = with bits 0 and 1: also emit, per pairwise factor, the D rows of its final factor->variable messages (blob
 *        header words 29 / 30; what mlbp_joint_logp reads as m0_row / m1_row).  Without it the blob is unchanged.       */
int mlbp_plan_compile(int n_graphs, const int32_t *h_var_off, const int32_t *h_pair_off, const int32_t *h_pair_v0,
                      const int32_t *h_pair_v1, const int32_t *h_pair_gap1, const int32_t *h_roots, int sweeps,
                      int flags, mlbp_plan **out);
/* sizes[0..15]: see MLBP_PLAN_* below */
int mlbp_plan_sizes(const mlbp_plan *p, int64_t *h_sizes);
/* copies the flat int32 blob (sizes[MLBP_PLAN_BLOB_WORDS] words) that the kernels index into */
int mlbp_plan_export(const mlbp_plan *p, int32_t *h_blob);
void mlbp_plan_destroy(mlbp_plan *p);

#define MLBP_PLAN_BLOB_WORDS   0   /* length of the exported blob in int32 words                              */
#define MLBP_PLAN_A_ROWS       1   /* rows of the A_hi / A_lo buffers                                         */
#define MLBP_PLAN_D_ROWS       2   /* rows of the D buffer (row 0 is the constant-one row)                    */
#define MLBP_PLAN_N_LEVELS     3
#define MLBP_PLAN_N_PAIR       4   /* live pairwise factors in the gradient stage                             */
#define MLBP_PLAN_N_GEMM_ROWS  5   /* total GEMM rows (message + gradient), = algorithmic GEMV count          */
#define MLBP_PLAN_MAX_IN       6   /* largest number of incoming pairwise messages of any variable            */
#define MLBP_PLAN_HDR_WORDS    7   /* blob header length; layout documented in csrc/plan.cpp                  */
#define MLBP_PLAN_N_DEAD       8   /* updates removed because nothing reads their result                      */
#define MLBP_PLAN_TMPL_HITS    9   /* graphs whose schedule template was already compiled (csrc/plan.cpp)     */
#define MLBP_PLAN_TMPL_MISSES 10   /* graphs whose template this call compiled                                */

#ifdef __cplusplus
}
#endif
#endif /* MLBP_H_ */
