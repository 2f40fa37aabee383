/* snag_b200 — C ABI of the B200-native SNAG_MMEA hot path (libsnag_b200.so).
 *
 * Drop-in boundary for three parts of zjukg/SNAG's SNAG_MMEA trainer (citations relative to the
 * reference checkout, SNAG_MMEA/...):
 *   - Gauss modality noise masking        model/SNAG.py:66-98, model/SNAG_tools.py:127-128
 *   - ICL / IAL in-batch contrastive loss model/SNAG_loss.py:58-128, :148-202
 *   - alignment evaluation                src/utils.py:202-218 (pairwise_distances), :417-435 (csls_sim),
 *                                         main.py:359-455 (Runner._test ranking -> Hits@k / MR / MRR)
 *
 * Conventions
 *   - every function returns int: 0 = ok, < 0 = SNAG_ERR_* (bad argument / shape / alignment / driver /
 *     device), > 0 = a cudaError_t raised by the launch. Nothing is written on a negative return.
 *   - all pointers are DEVICE pointers owned by the caller; the library never allocates, frees or
 *     retains device memory, never synchronises, and enqueues on the cudaStream_t passed as `stream`
 *     (void* here so the header stays plain C).
 *   - bf16 operands are row-major [n, Dpad] with Dpad a multiple of 64, zero padded, 128-byte aligned
 *     (what snag_prep_bf16 writes). They feed TMA (128-byte swizzle) -> tcgen05.mma directly.
 *   - kernels are compiled for sm_100a only; on any other device the tcgen05 entry points return
 *     SNAG_ERR_DEVICE. There is no CPU or library fallback.
 */
#ifndef SNAG_B200_H
#define SNAG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNAG_OK 0
#define SNAG_ERR_ARG (-1)
#define SNAG_ERR_SHAPE (-2)
#define SNAG_ERR_ALIGN (-3)
#define SNAG_ERR_DRIVER (-4)
#define SNAG_ERR_DEVICE (-5)

#define SNAG_KT 16 /* candidate-list length of the CSLS top-k path; csls_k must be <= SNAG_KT */

/* ---- library ------------------------------------------------------------------------------ */
int snag_version(void);                      /* ABI version, currently 1 */
const char* snag_error_string(int code);     /* static string for SNAG_ERR_* codes; "cuda error" for > 0 */
int snag_device_check(void);                 /* 0 if the current device is sm_100, SNAG_ERR_DEVICE otherwise */
int snag_num_sms(void);

/* Work decomposition of an [n_rows x n_cols] similarity sweep. n_lists = number of partial per-row output
 * lists the sweep writes (column chunks x epilogue warpgroups): sizes the `part` / top3 / rowsum workspaces. */
int snag_sim_plan(int n_rows, int n_cols, int Dpad, int* tiles_per_chunk, int* n_lists);

/* ---- noise masking ------------------------------------------------------------------------ */
/* SNAG.add_noise_to_embeddings (model/SNAG.py:66-75):
 *   rows with mask: out = (1-rho)*x + rho*(mean + std*z), other rows: out = x   (out may alias x)
 * keep = (float)(1.0 - rho), rho = (float)mask_ratio are passed separately because the reference
 * computes 1.0 - mask_ratio in double before the fp32 multiply.
 * mask (uint8 [N]) / zsel (fp32 [n_sel, F], rows in selection order) / selpos (int32 [N]) inject the
 * reference's own draws for bit parity; pass all three NULL to draw in-kernel with Philox4x32-10:
 * row i selected iff u(seed, row0+i) < ratio; z is a function of (seed, (row0+i)*F + col) only. */
int snag_noise_mask(const float* x, float* out, const float* mean, const float* std_, const uint8_t* mask,
                    const float* zsel, const int32_t* selpos, int64_t N, int32_t F, int64_t ld_in, int64_t ld_out,
                    float ratio, float keep, float rho, uint64_t seed, int64_t row0, void* stream);
/* the Philox row selection itself (entity_noise_mask, model/SNAG.py:98) */
int snag_philox_rowmask(uint8_t* mask, int64_t N, float ratio, uint64_t seed, int64_t row0, void* stream);
/* out = mean + std * N(0,1) (entity_noise, model/SNAG.py:96) */
int snag_gauss_fill(float* out, const float* mean, const float* std_, int64_t N, int32_t F, int64_t ld, uint64_t seed,
                    int64_t row0, void* stream);
/* column mean / unbiased std over rows with valid[i] != 0 (valid may be NULL = all rows)
 * (SNAG.get_mean_std, model/SNAG.py:77-84; update_noise :94-95). workspace: (2*F+1)*8 bytes. */
int snag_col_mean_std(const float* x, const uint8_t* valid, int64_t N, int32_t F, int64_t ld, float* mean, float* std_,
                      void* workspace, void* stream);
/* entity-embedding blend of MultiModalEncoder.forward (model/SNAG_tools.py:127-128) and its gradient:
 *   fwd: out = mask ? a*e + c*noise : e      bwd: g_in = mask ? a*g_out : g_out
 * a = (float)(1.0 - mask_ratio*0.5), c = (float)(mask_ratio*0.5). */
int snag_rowblend_fwd(const float* e, const float* noise, const uint8_t* mask, float* out, int64_t N, int32_t D, float a,
                      float c, void* stream);
int snag_rowblend_bwd(const float* g_out, const uint8_t* mask, float* g_in, int64_t N, int32_t D, float a, void* stream);

/* ---- operand prologue ----------------------------------------------------------------------- */
/* out[r, :] = bf16( normalize ? emb[idx[r]] / max(||emb[idx[r]]||, 1e-12) : emb[idx[r]] ), zero padded
 * to Dpad; norm2[r] = ||out[r]||^2 (fp64 accumulate, one rounding). idx may be NULL (identity).
 * Replaces F.normalize + gather (main.py:379,386; model/SNAG_loss.py:60-64) + (x**2).sum(1)
 * (src/utils.py:210-212). out is uint16_t* = raw bf16. */
int snag_prep_bf16(const float* emb, int64_t ld, const int64_t* idx, int32_t n, int32_t D, int32_t normalize,
                   uint16_t* out, int32_t Dpad, float* norm2, void* stream);
/* Prologue of the fp32 evaluation (precision="fp32"). rows [n, Dpad] fp32 (16-byte aligned) = the values snag_prep_bf16
 * rounds, bit for bit (same normalisation arithmetic), zero padded; split [n, 3 Dpad] bf16 (128-byte aligned) = the
 * three-term split h = bf16(x), m = bf16(x - h) laid out as [m | h | h] for side 0 (sources) and [h | m | h] for side 1
 * (targets): a sweep over a side-0 and a side-1 operand (in either order) contracts m_x h_y + h_x m_y + h_x h_y, which
 * leaves out only m_x m_y and the split's residuals (|x y - that| <= 3 * 2^-16 |x y|). norm2[r] = ||rows[r]||^2 in fp64,
 * in index order, rounded once. Any sweep below accepts split operands (Dpad argument = 3 Dpad). */
int snag_prep_split(const float* emb, int64_t ld, const int64_t* idx, int32_t n, int32_t D, int32_t normalize, int32_t side,
                    float* rows, uint16_t* split, int32_t Dpad, float* norm2, void* stream);
/* ---- fusion-output (joint) embeddings, model/SNAG_tools.py:44-49 ------------------------------ */
/* joint[i, off_m + c] = w_ent[i, m] * e_m[i, c] / max(||e_m[i]||, 1e-12) and joint_fz[...] = w_glob[m] * (same), for the
 * M <= 6 present modalities concatenated along the row (off_m = widths[0] + .. + widths[m-1]). embs / widths are HOST
 * arrays of M device pointers (fp32 [N, widths[m]], contiguous) / M ints. joint or joint_fz may be NULL (with its
 * weights). Replaces 2M F.normalize + 2M scalings + 2 torch.cat. */
int snag_joint_fuse_fwd(const float* const* embs, const int32_t* widths, int32_t M, int64_t N, const float* w_ent, int64_t ldw,
                        const float* w_glob, float* joint, float* joint_fz, int64_t ld_out, void* stream);
/* Its backward: d_embs[m] [N, widths[m]] (written), d_w_ent [N, ldw] (columns 0..M-1 written; may be NULL),
 * d_w_glob [M] (ACCUMULATED: zero it first; may be NULL) from the upstream gradients d_joint / d_joint_fz (either may
 * be NULL). */
int snag_joint_fuse_bwd(const float* const* embs, float* const* d_embs, const int32_t* widths, int32_t M, int64_t N,
                        const float* w_ent, int64_t ldw, const float* w_glob, const float* d_joint, const float* d_joint_fz,
                        int64_t ld_out, float* d_w_ent, float* d_w_glob, void* stream);
/* Backward of snag_prep_bf16's (gather ->) L2-normalise as autograd sees it (F.normalize, model/SNAG_loss.py:60-64):
 * with e = emb[idx[r]] and g = dz[r] (fp32 [n, ld_dz]),  demb[idx[r]] += g/||e|| - e (e.g)/||e||^3  (atomic adds; demb
 * fp32 [N, ld_demb], zeroed by the caller). idx may be NULL (rows 0..n-1). normalize = 0: demb[idx[r]] += g. */
int snag_normalize_bwd_scatter(const float* emb, int64_t ld, const int64_t* idx, int32_t n, int32_t D, int32_t normalize,
                               const float* dz, int64_t ld_dz, int32_t n_parts, int64_t part_stride, float* demb,
                               int64_t ld_demb, void* stream);
/* dz may be given as n_parts partial sums, part_stride floats apart (the column splits of snag_icl_bwd_fused); they are
 * added in split order. n_parts = 1: a single gradient, part_stride ignored. */

/* Batched prologue / epilogue of the loss layer — the 2 + 2M icl_loss calls of a step (model/SNAG.py:106,147-159) share
 * the batch idx_l / idx_r [B]; all array arguments are HOST arrays with one entry per call (n_prob <= 16).
 * snag_icl_stack_prep: out[p] ([3 Bp, Dpad[p]] bf16) = [ z[idx_l] ; z[idx_r] ; z[idx_l] ] with z = F.normalize(emb[p])
 *   (model/SNAG_loss.py:59-64) rounded to bf16, every part zero padded to Bp rows and Dpad[p] columns.
 * snag_normalize_bwd_scatter_many: snag_normalize_bwd_scatter for both sides of every call in one launch (dz_a[p] /
 *   dz_b[p]: gradients w.r.t. the normalised rows of side a / b, n_parts[p] partial sums part_stride[p] floats apart). */
int snag_icl_stack_prep(int32_t n_prob, const float* const* emb, const int64_t* ld, const int32_t* D, uint16_t* const* out,
                        const int32_t* Dpad, const int64_t* idx_l, const int64_t* idx_r, int32_t B, int32_t Bp,
                        int32_t normalize, void* stream);
int snag_normalize_bwd_scatter_many(int32_t n_prob, const float* const* emb, const int64_t* ld, const int32_t* D,
                                    const float* const* dz_a, const float* const* dz_b, const int64_t* ld_dz,
                                    const int32_t* n_parts, const int64_t* part_stride, float* const* demb,
                                    const int64_t* ld_demb, const int64_t* idx_l, const int64_t* idx_r, int32_t n,
                                    int32_t normalize, void* stream);

/* Fused backward of icl_loss (model/SNAG_loss.py:98-126) w.r.t. the normalised rows for contraction widths
 * Dpad <= 320 (the per-modality calls, D = 300): for each of n_prob <= 16 calls that share the batch size,
 *   dz_x[split][i][:] = sum over the split's columns j of G_ij y_j,   G = dL/dlogits (see snag_icl_bwd_logits),
 * with the logits tile recomputed, turned into G in registers, kept in tensor memory as the A operand of a second
 * tcgen05.mma and contracted with the same shared-memory tile of the stacked embeddings — neither the [B, 2B] logits
 * nor G ever reach HBM. Per call: S3 = stacked operand [a ; b ; a] ([3 Bp, Dpad] bf16, each part zero padded to
 * Bp = multiple of 256 rows, from snag_prep_bf16), cr_a / cr_b [B] = g_x[i] * exp(1/tau - lse_x[i]),
 * dg [B] = g_a[i] + g_b[i]. The launch covers the anchors [128 rb0, 128 (rb0 + row_blocks)) of both sides (all of them:
 * rb0 = 0, row_blocks = Bp / 128; a rank's shard otherwise); outputs dz_a / dz_b = nsplit partial gradients
 * [128 row_blocks, Dpad] fp32 of those anchors, part_stride floats apart (sum them, e.g. through
 * snag_normalize_bwd_scatter). nsplit = snag_icl_bwd_fused_splits(n_prob, B, Bp, row_blocks) or any count that leaves
 * no split empty. Pointer arguments are HOST arrays of n_prob device pointers. */
int32_t snag_icl_bwd_fused_splits(int32_t n_prob, int32_t B, int32_t Bp, int32_t row_blocks);
int snag_icl_bwd_fused(int32_t n_prob, const uint16_t* const* S3, const float* const* cr_a, const float* const* cr_b,
                       const float* const* dg, float* const* dz_a, float* const* dz_b, int32_t B, int32_t Bp, int32_t rb0,
                       int32_t row_blocks, int32_t Dpad, float inv_tau, int32_t nsplit, int64_t part_stride, void* stream);

/* Forward of icl_loss (model/SNAG_loss.py:98-126) for n_prob <= 16 tables that share the batch, on HALF the Gram matrix
 * of the stacked rows Z = [a ; b] (S3[p]: [>= 2 Bp, Dpad] bf16, each part zero padded to Bp = multiple of 256 rows): the
 * four logit blocks of the reference are the quadrants of the symmetric Z.Z^T, and both directions' softmax denominators
 * are its row sums without the diagonal — only tiles meeting the strict upper triangle are computed, every element
 * E = exp(s/tau - 1/tau) is added to the row sum of its row and (as a column sum of the tile) of its column.
 *   snag_icl_fwd_sym_plan : sizes[0] = number of work units of the launch, sizes[1] / sizes[2] = floats of the per-table
 *                           workspaces rowpart / colpart
 *   snag_icl_fwd_sym      : processes the units [unit_begin, unit_end) (all of them: 0, sizes[0]; a rank's contiguous
 *                           share when the loss is sharded) and writes total[p][r] (fp32 [n_prob, 2 Bp]) = the sum over
 *                           those units' contributions to sum_{j != r} E[r, j], added in a fixed order, and
 *                           pos[p][i] = Z_i . Z_{Bp+i} ([n_prob, Bp]; only entries whose tile lies in the unit range are
 *                           written — zero the buffer first when sharding). Sharded: all-reduce(sum) total and pos.
 *   snag_icl_sym_finalize : out[p][0..3][i] ([n_prob, 4, B]) = lse_a, nll_a, lse_b, nll_b of anchor i:
 *                           lse = log(total) + 1/tau, nll = lse - pos/tau.
 * Pointer arguments S3 / rowpart / colpart are HOST arrays of n_prob device pointers. */
int snag_icl_fwd_sym_plan(int32_t n_prob, int32_t B, int32_t Bp, int64_t* sizes);
int snag_icl_fwd_sym(int32_t n_prob, const uint16_t* const* S3, float* const* rowpart, float* const* colpart, float* pos,
                     int32_t B, int32_t Bp, int32_t Dpad, float inv_tau, int32_t unit_begin, int32_t unit_end, float* total,
                     uint16_t* const* esave, void* stream);
/* esave (NULL, or a HOST array of n_prob device pointers, each NULL or a [2 Bp, 2 Bp] bf16 buffer, 32-byte aligned):
 * the forward also stores E of every computed element at esave[p][row][column] (row < column; other entries are left
 * untouched). snag_icl_g_from_e then forms dL/dlogits of one side (G [Bp, 2 Bp] bf16, the operand of the gradient GEMM
 * snag_sim_write_t_mn; same definition and arguments as snag_icl_bwd_logits) from it with a bandwidth kernel instead of
 * recomputing the logits — for tables too wide for snag_icl_bwd_fused. Requires a forward over ALL work units.
 * cr_this / cr_other [B] as cr / cc of snag_icl_bwd_logits; diag [B] = the value of the cross diagonal G[i, i] itself,
 * (g_a[i] expm1(-nll_a[i]) + g_b[i] expm1(-nll_b[i])) / tau from the forward's fp32 NLL: that element is a small
 * difference of large terms which the bf16 E cannot carry. */
int snag_icl_g_from_e(const uint16_t* E, int32_t side, int32_t B, int32_t Bp, const float* cr_this, const float* cr_other,
                      const float* diag, float inv_tau, uint16_t* G, void* stream);
int snag_icl_sym_finalize(const float* total, const float* pos, int32_t n_prob, int32_t B, int32_t Bp, float inv_tau,
                          float* out, void* stream);

/* ---- alignment evaluation ------------------------------------------------------------------- */
/* pairwise_distances (src/utils.py:202-218), materialising: mode 1: out[i,j] = clamp(xn_i + yn_j - 2 x_i.y_j, 0);
 * mode 0: out[i,j] = x_i.y_j. out is fp32 [n1, ld]. */
int snag_sim_write(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, int32_t n1, int32_t n2,
                   int32_t Dpad, int32_t mode, float* out, int64_t ld, void* stream);
/* Transposed, split-K form for products whose contraction is long and whose X side is narrow (the loss's gradient
 * GEMMs dA = G . [b ; a] with X = [b ; a]^T [D, 2B], Y = G [B, 2B]): out[s][j * ld + i] = sum over K slice s of
 * X[i,:] . Y[j,:], s = 0 .. ksplits-1 (slices split_stride floats apart; the caller adds them up). ksplits must be
 * the value snag_sim_write_t_splits(n1, n2, Dpad) returns (>= 1). */
int snag_sim_write_t_splits(int32_t n1, int32_t n2, int32_t Dpad);
int snag_sim_write_t(const uint16_t* X, const uint16_t* Y, int32_t n1, int32_t n2, int32_t Dpad, int32_t ksplits, float* out,
                     int64_t ld, int64_t split_stride, void* stream);
/* snag_sim_write_t with X given TRANSPOSED: XT is [Dpad rows (the contraction index), xt_ld columns] bf16 (xt_ld a
 * multiple of 64, first n1 columns valid) and its tiles are read MN-major by the tensor cores. For the loss's gradient
 * GEMMs dX = dL/dlogits . [other ; this] XT is the stacked, normalised embedding matrix as it lies in memory
 * ([2 Bp, Dpad_emb]): no transposed copy is made. Same outputs and split rules as snag_sim_write_t. */
int snag_sim_write_t_mn(const uint16_t* XT, int32_t xt_ld, const uint16_t* Y, int32_t n1, int32_t n2, int32_t Dpad,
                        int32_t ksplits, float* out, int64_t ld, int64_t split_stride, void* stream);
/* Measurement aid: the same TMA + tcgen05 sweep with the accumulators dropped (no epilogue, no output).
 * Times the mainloop alone so that bench.py can attribute a sweep's time to mainloop vs fused epilogue. */
int snag_sim_mainloop_only(const uint16_t* X, const uint16_t* Y, int32_t n1, int32_t n2, int32_t Dpad, void* stream);
/* Development aid: counters = zeroed device buffer of 4*snag_num_sms()*4 uint64 (or NULL to switch off). While set, the UMMA-
 * issuing thread of every CTA of every sweep records {total cycles, cycles waiting for a free accumulator stage
 * (epilogue-bound), cycles waiting for operands (TMA-bound), tiles}; the fused evaluation sweeps add their flag and
 * per-test counters (scripts/onepass_attrib.py reads them). Process-global, not thread-safe. */
int snag_debug_counters(uint64_t* counters);
/* CSLS sweep 1 (src/utils.py:431-432 without the matrix): for every row of X the SNAG_KT largest
 * c_ij = 1 - d_ij over the columns of each chunk. part: fp32 [n_lists][n1][SNAG_KT] (n_lists from
 * snag_sim_plan(n1, n2, Dpad)); part_idx (may be NULL): int32, same shape, the column j of every entry (-1 for the
 * -inf padding) — needed to re-score the neighbourhood canonically (snag_topk_rescore). Call with X and Y swapped
 * for the column neighbourhoods. */
int snag_eval_rowtopk(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, int32_t n1, int32_t n2,
                      int32_t Dpad, float* part, int32_t* part_idx, void* stream);
/* Two-sweep variant: CSLS neighbourhoods of BOTH directions from ONE pass over S (replaces the second
 * snag_eval_rowtopk call with swapped operands). Rows: as snag_eval_rowtopk (part). Columns: every element with
 * c_ij >= colthr[j] is appended, as a (j, c) pair, to the private stream of the CTA that computed it
 * (stream[cta][cta_cap] 8-byte entries, stream_cnt[cta] entries produced; both sized for snag_num_sms() CTAs,
 * stream_cnt zeroed by the caller). colthr / colb come from snag_col_threshold applied to the merged candidate lists
 * of a PRE-PASS snag_eval_rowtopk(Y, X_sample, ...) over a random sample of the rows of X: the k-th largest c of the
 * sample is a lower bound of the final k-th largest, so no neighbour is ever missed; a sample of m rows leaves
 * ~k*n1/m candidates per column. Then: snag_col_cand_hist (hist[j] = candidates of column j; sets *overflow if a
 * stream was full), offs = exclusive prefix sum of hist (caller), snag_col_cand_scatter (vals[offs[j] + ...]),
 * snag_col_cand_finalize (nv[j] = mean of the k largest and/or cand_val/cand_idx [n][SNAG_KT] = the column's SNAG_KT
 * best candidates with their rows; sets *overflow if a column has fewer than k). On overflow fall back to the swapped
 * snag_eval_rowtopk sweep. hist / cursor / overflow are zeroed by the caller. part_idx / stream_row carry the column
 * of every row candidate and the row of every stream entry (int32, same shapes as part / stream).
 * rowthr (may be NULL): per row a lower bound of its final SNAG_KT-th largest c (e.g. the SNAG_KT-th largest over a
 * sample of the columns, minus 2e-6); every partial list starts from it, slots it leaves unfilled read (rowthr, -1).
 * norm2_max: the largest squared row norm among xn / yn. Up to 1.05 (L2-normalised rows rounded to bf16) the per-element
 * pre-filter runs in fp16x2 with margins derived for such rows; above, the fp32 form is used (snag_eval_onepass: refused). */
int snag_eval_rowcoltopk(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, int32_t n1, int32_t n2,
                         int32_t Dpad, float* part, int32_t* part_idx, const float* rowthr, const float* colthr,
                         const float* colb, uint64_t* stream, int32_t* stream_row, int32_t* stream_cnt, int32_t cta_cap,
                         float norm2_max, void* stream_);
/* One-pass evaluation: snag_eval_rowcoltopk that ALSO streams out every element which may count towards a rank of
 * Runner._test (main.py:400-429), so that the second sweep over the similarity matrix (snag_eval_rank_band) is not needed.
 * rk_r / rk_rp [n1] and rk_c / rk_cp [n2] are relaxed (provably or speculatively lower) versions of the constants
 * R, R', C, C' of snag_eval_rank_band; every element with s > rk_r[i] + rk_c[j] or s > rk_rp[i] + rk_cp[j] is appended as
 * (column, s bits) + row to the CTA's rank stream (rk_stream[cta][rk_cap], rk_stream_row, rk_cnt[cta]; sized for
 * snag_num_sms() CTAs, rk_cnt zeroed by the caller). After the neighbourhood means are final, snag_rank_judge settles the
 * streamed elements against the final constants (entities whose relaxed constant was not below the final one are
 * skipped: row_ok / col_ok = 0 — recount them with snag_rank_exhaustive), elements inside the +-eps band go to the
 * `band` list for snag_band_rescore. *overflow is set when a rank stream was full (fall back to snag_eval_rank_band).
 * snag_spec_bounds: lo / hi [n] = lower bound / extrapolated upper guess of every entity's neighbourhood mean from the
 * merged sample lists cand [n][SNAG_KT] and the canonical c of its own pair (shift: extrapolation distance in units of
 * the list's tail scale, e.g. 1.5 ln(n / sample size); delta: tensor-core tolerance in c).
 * snag_rank_exhaustive: canonical recount of the listed rows of A against all n_b rows of B (cnt[row] += ...; the caller
 * zeroes those entries); swapped != 0 when A holds targets and B sources (the CSLS chain is not symmetric in fp32). */
int snag_eval_onepass(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, int32_t n1, int32_t n2,
                      int32_t Dpad, float* part, int32_t* part_idx, const float* rowthr, const float* colthr, const float* colb,
                      uint64_t* stream, int32_t* stream_row, int32_t* stream_cnt, int32_t cta_cap, const float* rk_r,
                      const float* rk_rp, const float* rk_c, const float* rk_cp, uint64_t* rk_stream, int32_t* rk_stream_row,
                      int32_t* rk_cnt, int32_t rk_cap, float norm2_max, void* stream_);
int snag_spec_bounds(const float* cand, int64_t n, int32_t k, const float* cdiag, float shift, float delta, float* lo,
                     float* hi, void* stream);
int snag_rank_judge(const uint64_t* rk_stream, const int32_t* rk_stream_row, const int32_t* rk_cnt, int32_t n_ctas,
                    int32_t rk_cap, const float* R, const float* Rp, const float* C, const float* Cp, const uint8_t* row_ok,
                    const uint8_t* col_ok, float eps, int32_t row_gid0, int32_t col_gid0, int32_t* cnt_row, int32_t* cnt_col,
                    uint64_t* band, uint32_t* band_cnt, uint32_t band_cap, int32_t* overflow, void* stream);
int snag_rank_exhaustive(const uint16_t* A, const uint16_t* B, int32_t Dpad, int64_t n_b, const float* an, const float* bn,
                         const float* nva, const float* nvb, const float* g, const int32_t* rows, int32_t n_rows,
                         int32_t a_gid0, int32_t b_gid0, int32_t use_csls, int32_t swapped, int32_t* cnt, void* stream);
int snag_col_threshold(const float* cand, int64_t n, int32_t k, const float* yn, float* colthr, float* colb, void* stream);
int snag_col_cand_hist(const uint64_t* stream, const int32_t* stream_cnt, int32_t n_ctas, int32_t cta_cap, int32_t* hist,
                       int32_t* overflow, void* stream_);
int snag_col_cand_scatter(const uint64_t* stream, const int32_t* stream_row, const int32_t* stream_cnt, int32_t n_ctas,
                          int32_t cta_cap, const int64_t* offs, int32_t* cursor, float* vals, int32_t* rows, void* stream_);
int snag_col_cand_finalize(const int64_t* offs, const int32_t* hist, const float* vals, const int32_t* rows, int64_t n,
                           int32_t k, float* nv, float* cand_val, int32_t* cand_idx, int32_t* overflow, void* stream);
/* merge n_lists candidate lists per row ([n_lists][n_rows][SNAG_KT]); nv[row] = mean of the k largest
 * (may be NULL); cand_out [n_rows][SNAG_KT] = merged list (may be NULL) for the cross-GPU exchange; with part_idx and
 * cand_idx_out the ids travel with the values. */
int snag_topk_merge_mean(const float* part, const int32_t* part_idx, int32_t n_lists, int64_t n_rows, int32_t k, float* nv,
                         float* cand_out, int32_t* cand_idx_out, void* stream);
/* Canonical neighbourhood means (the oracle's nv bit for bit): re-score the SNAG_KT candidates of every row of A
 * (cand_idx: rows of B, -1 = empty; cand_val: their tensor-core scores) with the fp64 index-order dot product and the
 * fp32 chain c = 1 - clamp((an + bn) - 2 s, 0); nv[row] = fp32 sum of the k largest taken largest-first, divided by
 * k. A row is verified when its k-th canonical score is >= (smallest tensor-core score of its full list) + delta, i.e.
 * no row of B outside the list can belong to the true neighbourhood; the others are appended to flagged[]
 * (*flagged_cnt counts them, zero it first) and must be completed by snag_topk_exhaustive, which scans all n_b rows
 * of B for each flagged row. outsider_bound (NULL or fp32 [n_rows]): for lists that were collected under an admission
 * threshold (the two-sweep path's column streams: only elements with c >= colthr[row] were ever candidates), that
 * threshold — a list that is not full is then verified against it instead of being trusted. */
int snag_topk_rescore(const uint16_t* A, const uint16_t* B, int32_t Dpad, int64_t n_rows, const float* an, const float* bn,
                      const int32_t* cand_idx, const float* cand_val, int32_t k, float delta, const float* outsider_bound,
                      float* nv, int32_t* flagged, int32_t* flagged_cnt, int32_t flagged_cap, float* best_d,
                      int32_t* best_idx, void* stream);
int snag_topk_exhaustive(const uint16_t* A, const uint16_t* B, int32_t Dpad, int64_t n_b, const float* an, const float* bn,
                         const int32_t* flagged, const int32_t* flagged_cnt, int32_t flagged_cap, int32_t k, float* nv,
                         float* best_d, int32_t* best_idx, void* stream);
/* best_d / best_idx (both NULL or fp32 / int32 [n_rows]): the nearest row of B for every row of A under the canonical
 * squared distance clamp((an + bn) - 2 s, 0), lowest index on ties (torch.argmin) — link mining, model/SNAG.py:199-200. */
/* ground-truth scores g[p] = distance of pair (x_p, y_p): CSLS distance 1 - ((2(1-d) - nv1_p) - nv2_p) if
 * use_csls else d; dot product accumulated in fp64 in index order. s_out (may be NULL) gets x_p.y_p. */
int snag_pair_score(const uint16_t* X, const uint16_t* Y, int32_t Dpad, int64_t n, const float* xn, const float* yn,
                    const float* nv1, const float* nv2, int32_t use_csls, float* g, float* s_out, void* stream);
/* CSLS sweep 2 = the two ranking loops of Runner._test (main.py:400-411, 422-429) without the matrix:
 *   cnt_row[i] += #{j != i : dist_ij < g_row[i] or (== and gid(j) < gid(i))}     l2r rank of pair gid(i)
 *   cnt_col[j] += #{i != j : dist_ij < g_col[j] or (== and gid(i) < gid(j))}     r2l rank of pair gid(j)
 * gid(i) = row_gid0 + i, gid(j) = col_gid0 + j (column shards of a multi-GPU evaluation pass their offset).
 * Counters are accumulated atomically: zero them first. top3_val/top3_idx (both NULL or both fp32/int32
 * [n_lists][n1][4]) receive each row's 3 nearest columns per list (merge with snag_top4_merge). */
int snag_eval_rank(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, const float* nv1,
                   const float* nv2, const float* g_row, const float* g_col, int32_t row_gid0, int32_t col_gid0,
                   int32_t n1, int32_t n2, int32_t Dpad, int32_t use_csls, int32_t* cnt_row, int32_t* cnt_col,
                   float* top3_val, int32_t* top3_idx, void* stream);
/* Default form of sweep 2: the same counters, decided in s-space with a deferral band (DESIGN.md 3.2). An element
 * whose margin to the ground-truth score exceeds `eps` (in units of the dot product) is counted in the sweep; the
 * others — exact ties included — are appended to band[] (x = view row | direction flags << 30, y = view column;
 * *band_cnt counts them and may exceed band_cap: re-run with a larger list) and must then be judged by
 * snag_band_rescore, which evaluates the reference's fp32 chain on the fp64 index-order dot product with the stable
 * tie-break. Together the two calls give ranks that do not depend on the tensor core's accumulation order.
 * top4_val/top4_idx (both NULL or fp32/int32 [n_lists][n1][4]): each row's 4 nearest candidate columns per list
 * (merge with snag_top4_merge, order and cut to ret1..ret3 with snag_top3_rescore). Zero *band_cnt first. */
int snag_eval_rank_band(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, const float* nv1,
                        const float* nv2, const float* g_row, const float* g_col, int32_t row_gid0, int32_t col_gid0,
                        int32_t n1, int32_t n2, int32_t Dpad, int32_t use_csls, float eps, int32_t* cnt_row, int32_t* cnt_col,
                        float* top4_val, int32_t* top4_idx, uint64_t* band, uint32_t* band_cnt, uint32_t band_cap,
                        void* stream);
int snag_band_rescore(const uint16_t* X, const uint16_t* Y, int32_t Dpad, const float* xn, const float* yn, const float* nv1,
                      const float* nv2, const float* g_row, const float* g_col, int32_t row_gid0, int32_t col_gid0,
                      int32_t use_csls, const uint64_t* band, const uint32_t* band_cnt, uint32_t band_cap, int32_t* cnt_row,
                      int32_t* cnt_col, void* stream);
/* Recount of SELECTED entities (one-pass evaluation: entities whose guessed bound failed): the same sweep and re-score
 * as snag_eval_rank_band / snag_band_rescore over a GATHERED subset of rows — X [n1][Dpad] holds the selected rows,
 * xn / nv1 / g_row their per-row values, row_gids [n1] their global pair ids (for the ground-truth exclusion and the
 * tie-break); only cnt_row [n1] is meaningful for the caller (cnt_col [n2] is scratch). To recount selected TARGETS call
 * it with the operands exchanged (X = gathered targets with yn / nv2 / g, Y = all sources with xn / nv1) and pass
 * swapped = 1 to the re-score, which then evaluates the fp32 CSLS chain in the reference's operand order. */
int snag_eval_rank_band_rows(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, const float* nv1,
                             const float* nv2, const float* g_row, const float* g_col, const int32_t* row_gids,
                             int32_t col_gid0, int32_t n1, int32_t n2, int32_t Dpad, int32_t use_csls, float eps,
                             int32_t* cnt_row, int32_t* cnt_col, uint64_t* band, uint32_t* band_cnt, uint32_t band_cap,
                             void* stream);
int snag_band_rescore_rows(const uint16_t* X, const uint16_t* Y, int32_t Dpad, const float* xn, const float* yn,
                           const float* nv1, const float* nv2, const float* g_row, const float* g_col, const int32_t* row_gids,
                           int32_t col_gid0, int32_t use_csls, int32_t swapped, const uint64_t* band, const uint32_t* band_cnt,
                           uint32_t band_cap, int32_t* cnt_row, int32_t* cnt_col, void* stream);
/* s_out[p] = X[rows[p]] . Y[cols[p]] with the canonical accumulation (fp64, index order, rounded once): the re-score of
 * explicitly listed similarity entries (unsupervised seed induction, src/data.py:367-375 + src/utils.py:437-443). */
int snag_pairs_dot(const uint16_t* X, const uint16_t* Y, int32_t Dpad, const int32_t* rows, const int32_t* cols,
                   int64_t n_pairs, float* s_out, void* stream);
int snag_top4_merge(const float* val, const int32_t* idx, int32_t n_lists, int64_t n_rows, float* oval, int32_t* oidx,
                    void* stream);
/* cand int32 [n_rows][4] column ids (0x7fffffff = empty) -> canonical distances, ascending (id ascending on ties) */
int snag_top3_rescore(const uint16_t* X, const uint16_t* Y, int32_t Dpad, int64_t n_rows, const float* xn, const float* yn,
                      const float* nv1, const float* nv2, int32_t use_csls, const int32_t* cand, float* oval, int32_t* oidx,
                      void* stream);
/* The canonical kernels above over fp32 rows [n, Dpad] (snag_prep_split's `rows`, 16-byte aligned) instead of bf16
 * operands: same arguments, same arithmetic (an fp32 x fp32 product is exact in fp64, so the fp64 index-order sum
 * rounded once is still the oracle's s_ij). The fp32 evaluation's sweeps run on the split operands and every verdict
 * inside their error bound is re-judged here. */
int snag_topk_rescore_f32(const float* A, const float* B, int32_t Dpad, int64_t n_rows, const float* an, const float* bn,
                          const int32_t* cand_idx, const float* cand_val, int32_t k, float delta, const float* outsider_bound,
                          float* nv, int32_t* flagged, int32_t* flagged_cnt, int32_t flagged_cap, float* best_d,
                          int32_t* best_idx, void* stream);
int snag_topk_exhaustive_f32(const float* A, const float* B, int32_t Dpad, int64_t n_b, const float* an, const float* bn,
                             const int32_t* flagged, const int32_t* flagged_cnt, int32_t flagged_cap, int32_t k, float* nv,
                             float* best_d, int32_t* best_idx, void* stream);
int snag_pair_score_f32(const float* X, const float* Y, int32_t Dpad, int64_t n, const float* xn, const float* yn,
                        const float* nv1, const float* nv2, int32_t use_csls, float* g, float* s_out, void* stream);
int snag_band_rescore_f32(const float* X, const float* Y, int32_t Dpad, const float* xn, const float* yn, const float* nv1,
                          const float* nv2, const float* g_row, const float* g_col, int32_t row_gid0, int32_t col_gid0,
                          int32_t use_csls, const uint64_t* band, const uint32_t* band_cnt, uint32_t band_cap, int32_t* cnt_row,
                          int32_t* cnt_col, void* stream);
int snag_band_rescore_rows_f32(const float* X, const float* Y, int32_t Dpad, const float* xn, const float* yn,
                               const float* nv1, const float* nv2, const float* g_row, const float* g_col,
                               const int32_t* row_gids, int32_t col_gid0, int32_t use_csls, int32_t swapped,
                               const uint64_t* band, const uint32_t* band_cnt, uint32_t band_cap, int32_t* cnt_row,
                               int32_t* cnt_col, void* stream);
int snag_rank_exhaustive_f32(const float* A, const float* B, int32_t Dpad, int64_t n_b, const float* an, const float* bn,
                             const float* nva, const float* nvb, const float* g, const int32_t* rows, int32_t n_rows,
                             int32_t a_gid0, int32_t b_gid0, int32_t use_csls, int32_t swapped, int32_t* cnt, void* stream);
int snag_pairs_dot_f32(const float* X, const float* Y, int32_t Dpad, const int32_t* rows, const int32_t* cols, int64_t n_pairs,
                       float* s_out, void* stream);
int snag_top3_rescore_f32(const float* X, const float* Y, int32_t Dpad, int64_t n_rows, const float* xn, const float* yn,
                          const float* nv1, const float* nv2, int32_t use_csls, const int32_t* cand, float* oval, int32_t* oidx,
                          void* stream);

/* csls_sim (src/utils.py:417-435) on a MATERIALISED fp32 similarity matrix [n1, ld]: nv1[i] / nv2[j] = mean of the k
 * largest entries of row i / column j; out[i,j] = (2*sim[i,j] - nv1[i]) - nv2[j] (out may be NULL to get only the
 * neighbourhood means, and may alias sim). workspace: snag_csls_workspace_bytes(n1, n2) bytes, 16-byte aligned.
 * k <= SNAG_KT runs the three bandwidth passes; SNAG_KT < k <= 1024 (the reference takes any k) selects per row /
 * column with a radix select + sorted largest-first sum (one block per vector; the column pass reads strided). */
int64_t snag_csls_workspace_bytes(int64_t n1, int64_t n2);
int snag_csls_sim(const float* sim, int64_t n1, int64_t n2, int64_t ld, int32_t k, float* out, int64_t ld_out, float* nv1,
                  float* nv2, void* workspace, void* stream);

/* --distance 1 (main.py:387-390, scipy cdist "cityblock" on the host in the reference): out[i,j] = fp32 of the fp64
 * index-order sum of |x_ik - y_jk| for fp32 x [n1, D], y [n2, D]. Materialising, like the reference. */
int snag_l1_distance(const float* x, const float* y, int64_t n1, int64_t n2, int32_t D, int64_t ldx, int64_t ldy, float* out,
                     int64_t ldo, void* stream);
/* The ranking loops of Runner._test (main.py:400-411, 422-429) on a materialised square distance matrix d [n, ld]:
 * cnt_row[i] / cnt_col[j] = 0-based position of the ground truth (the diagonal) in the stable ascending sort of row i /
 * column j. Used by the --distance 1 path, where no contraction exists to fuse the counting into. */
int snag_matrix_rank(const float* d, int64_t n, int64_t ld, int32_t* cnt_row, int32_t* cnt_col, void* stream);

/* ---- fused --distance 1 evaluation (no n x n matrix; the same generator as the L2 sweeps drives it) ------------------ */
/* Operands X [n1][Dp], Y [n2][Dp] are fp32 rows zero padded to Dp (a multiple of 8), 16-byte aligned; xn / yn are the
 * rows' L1 norms (sum of |x_k|, fp32). The CUDA-core sweep computes d~_ij = sum_k |x_ik - y_jk| in fp32 with packed adds
 * and |d~ - d| <= (ceil(Dp / 32) + 18) 2^-24 1.01 (xn_i + yn_j) against the canonical d = fp32 of the fp64 index-order
 * sum (scipy's cdist). snag_l1_plan: number of partial lists per row (n_lists) of an [n_rows x n_cols] sweep. */
int snag_l1_plan(int32_t n_rows, int32_t n_cols, int32_t Dp, int32_t* n_lists);
/* part / part_idx [n_lists][n1][SNAG_KT]: per list, the SNAG_KT largest c~ = 1 - d~ of every row (ascending, -inf / -1
 * padded) and their columns — the input of snag_topk_merge_mean, as from snag_eval_rowtopk. */
int snag_l1_rowtopk(const float* X, const float* Y, int32_t n1, int32_t n2, int32_t Dp, float* part, int32_t* part_idx,
                    void* stream);
/* Rank counts with a deferral band, as snag_eval_rank_band: dist~ = 1 - ((2 (1 - d~) - nv1_i) - nv2_j) (use_csls) or d~
 * is compared with g_row[i] and g_col[j]; clear "less" is counted into cnt_row / cnt_col, elements within the pair's
 * error bound are appended to band[] (x = row | direction flags << 30, y = column; *band_cnt may exceed band_cap: re-run
 * with a larger list) for snag_l1_band_rescore. top4_val / top4_idx (both NULL or [n_lists][n1][4]): each row's 4
 * nearest (x = -dist~, column gid) per list, for snag_top4_merge. Zero *band_cnt first. */
int snag_l1_rank_band(const float* X, const float* Y, const float* xn, const float* yn, const float* nv1, const float* nv2,
                      const float* g_row, const float* g_col, int32_t row_gid0, int32_t col_gid0, int32_t n1, int32_t n2,
                      int32_t Dp, int32_t use_csls, int32_t* cnt_row, int32_t* cnt_col, float* top4_val, int32_t* top4_idx,
                      uint64_t* band, uint32_t* band_cnt, uint32_t band_cap, void* stream);
/* Canonical CSLS neighbourhood means of the rows of A from their merged sweep candidates (as snag_topk_rescore, with
 * bn_max = the largest L1 norm of B); unverifiable rows are appended to flagged[] for snag_l1_topk_exhaustive. */
int snag_l1_topk_rescore(const float* A, const float* B, int32_t Dp, int64_t n_rows, const float* an, float bn_max,
                         const int32_t* cand_idx, const float* cand_val, int32_t k, float* nv, int32_t* flagged,
                         int32_t* flagged_cnt, int32_t flagged_cap, void* stream);
int snag_l1_topk_exhaustive(const float* A, const float* B, int32_t Dp, int64_t n_b, const int32_t* flagged,
                            const int32_t* flagged_cnt, int32_t flagged_cap, int32_t k, float* nv, void* stream);
/* g[p] = canonical (CSLS) distance of pair (x_p, y_p) */
int snag_l1_pair_score(const float* X, const float* Y, int32_t Dp, int64_t n, const float* nv1, const float* nv2,
                       int32_t use_csls, float* g, void* stream);
/* the deferred elements of snag_l1_rank_band judged canonically with the stable-sort tie-break */
int snag_l1_band_rescore(const float* X, const float* Y, int32_t Dp, const float* nv1, const float* nv2, const float* g_row,
                         const float* g_col, int32_t row_gid0, int32_t col_gid0, int32_t use_csls, const uint64_t* band,
                         const uint32_t* band_cnt, uint32_t band_cap, int32_t* cnt_row, int32_t* cnt_col, void* stream);
/* cand [n_rows][4] merged sweep candidates (ids into Y, 0x7fffffff = empty) -> canonical distances ascending (id
 * ascending on ties); rows whose 4th sweep candidate cannot rule out an outsider in the canonical top 3 (yn_max / nv2_absmax:
 * the largest L1 norm of Y and |nv2|) are appended to flagged[] (n_rows entries, *flagged_cnt zeroed by the caller) and
 * rescanned against all n_b rows of Y in the same call. */
int snag_l1_top3_rescore(const float* X, const float* Y, int32_t Dp, int64_t n_rows, int64_t n_b, const float* xn, float yn_max,
                         const float* nv1, const float* nv2, float nv2_absmax, int32_t use_csls, const int32_t* cand, float* oval,
                         int32_t* oidx, int32_t* flagged, int32_t* flagged_cnt, void* stream);

/* ---- mutual nearest neighbours (iterative-learning link mining) ------------------------------- */
/* The argmin pair of model/SNAG.py:192-208 (Iter_new_links: torch.argmin over the rows and over the columns of
 * pairwise_distances(final_emb[left], final_emb[right])) without forming the distance matrix.
 *   row_val / row_idx [n_lists][n1] (n_lists = snag_sim_plan(n1, n2)): per list, the smallest
 *       d_ij = clamp(xn_i + yn_j - 2 x_i.y_j, 0) of row i and its column (lowest column among equals); the caller
 *       reduces over lists lexicographically on (d, column).
 *   colkey [n2], initialised by the caller to all ones: receives min over rows of (d bits << 32 | row), i.e. the
 *       smallest d of column j and the lowest row attaining it — for every column whose minimum satisfies
 *       x_i.y_j > xn_i/2 + colb[j]. colb comes from an upper bound ub_j of the column minimum (the minimum over any
 *       subset of the rows): colb[j] = (yn_j - ub_j)/2 - 4e-6 admits every element with d_ij <= ub_j. */
int snag_mutual_nn(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, int32_t n1, int32_t n2,
                   int32_t Dpad, const float* colb, uint64_t* colkey, float* row_val, int32_t* row_idx, void* stream);

/* ---- ICL loss --------------------------------------------------------------------------------- */
/* One side of icl_loss.forward (model/SNAG_loss.py:98-126). Y = [other side ; this side] [2*Bp, Dpad], each part zero
 * padded from B to Bp rows (Bp multiple of 256). X = nx anchors of this side starting at batch index row0 (the whole
 * side: row0 = 0, nx = Bp; a rank of the anchor-sharded loss passes its own rows), [nx, Dpad], 128-byte aligned.
 *   rowsum_part[l][i] = partial sum l (of n_lists = snag_sim_plan(nx, 2*Bp)) of exp(logit_ij - 1/tau), self-similarity
 *                       excluded; i = local row, row stride nx
 *   pos[i] = x_i . other_(row0+i)                then snag_icl_finalize(.., B = valid local rows, Bp = nx, ..):
 *                                                lse, nll = lse - pos/tau */
int snag_icl_rowsum(const uint16_t* X, const uint16_t* Y, int32_t B, int32_t Bp, int32_t row0, int32_t nx, int32_t Dpad,
                    float inv_tau, float* rowsum_part, float* pos, void* stream);
int snag_icl_finalize(const float* rowsum_part, int32_t n_lists, int32_t B, int32_t Bp, const float* pos,
                      float inv_tau, float* lse, float* nll, void* stream);

/* ICL backward, stage 1: recompute one side's logits and write dL/dlogits as bf16 G [nx, 2*Bp] (same X / Y views
 * as snag_icl_rowsum; cr, cc, dg are [B], indexed by batch index). With g_x = dL/dnll_x (upstream) and lse_x from the
 * forward:
 *   cr[i] = g_this[i]*exp(1/tau - lse_this[i]), cc[j] = g_other[j]*exp(1/tau - lse_other[j]), dg[i] = g_this[i]+g_other[i]
 * Stage 2 is the contraction dX = G . [other ; this] (snag_sim_write_t on the transposed stacked operand and G).
 * Part 0 (cross columns): G[i,j] = (cr[i] + cc[j]) E_ij / tau - [i == j] dg[i] / tau; part 1 (self columns, diagonal
 * masked): G[i,j] = (cr[i] + (self_cols ? cr[j] : 0)) E_ij / tau. self_cols = 1 is the ICL / IAL gradient pattern;
 * self_cols = 0 with cc = dg = 0 and cr[i] = tau * exp(1/tau - lse[i]) writes the row softmax itself (IAL forward).
 * ebar is subtracted from E_ij (0 for ICL): IAL's gradient is the difference of two nearly uniform matrices at large tau;
 * centring E keeps their bf16 rounding relative to the deviations (the caller adds the common, rank-one part back). */
int snag_icl_bwd_logits(const uint16_t* X, const uint16_t* Y, int32_t B, int32_t Bp, int32_t row0, int32_t nx,
                        int32_t Dpad, float inv_tau, const float* cr, const float* cc, const float* dg, uint16_t* G,
                        int32_t self_cols, float ebar, void* stream);

/* ---- fp32 loss route (icl_loss with precision "fp32") ----------------------------------------- */
/* The contraction operands are a three-term bf16 split of the UNROUNDED normalised rows (as snag_prep_split): h = bf16(z),
 * m = bf16(z - h). One split stack per table, [3 Bp, 5 Dpad] bf16 (128-byte aligned): row r of [a ; b ; a] (each part
 * zero padded to Bp rows) laid out [m | h | h | m | h]; its side-0 window (columns [0, 3 Dpad)) is [m | h | h], its side-1
 * window (columns [2 Dpad, 5 Dpad)) is [h | m | h], so a side-0 row contracted with a side-1 row over 3 Dpad gives
 * m_i h_j + h_i m_j + h_i h_j (symmetric in i, j; |z_i z_j - that| <= 3 * 2^-16 |z_i| |z_j|). Dpad arguments below are
 * the table's Dpad (a multiple of 64), not the stack's width.
 * snag_icl_stack_prep_split : snag_icl_stack_prep with split stacks as out[p]; h is bit for bit snag_icl_stack_prep's
 *                             output, m bit for bit snag_prep_split's.
 * snag_icl_fwd_sym_split    : snag_icl_fwd_sym on split stacks S5[p] (no esave: a bf16 E would cap dL/dlogits at 2^-9);
 *                             same plan, workspaces, unit ranges and snag_icl_sym_finalize.
 * snag_icl_rowsum_split     : snag_icl_rowsum with X the side-0 window of the anchors' rows and Y the side-1 window of
 *                             [other ; this] (rows 5 Dpad apart); snag_icl_finalize as usual.
 * snag_icl_bwd_logits_split : snag_icl_bwd_logits (self_cols = 1, ebar = 0) on the same windows; G is formed in fp32 and
 *                             written as G3 [nx, 6 Bp] bf16 (32-byte aligned) = [G_h | G_h | G_m], G_h = bf16(G),
 *                             G_m = bf16(G - G_h). snag_sim_write_t_mn(XT = the K-stacked rows [Y_h ; Y_m ; Y_h]
 *                             ([6 Bp, Dpad]), Y = G3, contraction 6 Bp) then gives G_h Y_h + G_h Y_m + G_m Y_h. */
int snag_icl_stack_prep_split(int32_t n_prob, const float* const* emb, const int64_t* ld, const int32_t* D, uint16_t* const* out,
                              const int32_t* Dpad, const int64_t* idx_l, const int64_t* idx_r, int32_t B, int32_t Bp,
                              int32_t normalize, void* stream);
int snag_icl_fwd_sym_split(int32_t n_prob, const uint16_t* const* S5, float* const* rowpart, float* const* colpart, float* pos,
                           int32_t B, int32_t Bp, int32_t Dpad, float inv_tau, int32_t unit_begin, int32_t unit_end,
                           float* total, void* stream);
int snag_icl_rowsum_split(const uint16_t* X, const uint16_t* Y, int32_t B, int32_t Bp, int32_t row0, int32_t nx, int32_t Dpad,
                          float inv_tau, float* rowsum_part, float* pos, void* stream);
int snag_icl_bwd_logits_split(const uint16_t* X, const uint16_t* Y, int32_t B, int32_t Bp, int32_t row0, int32_t nx,
                              int32_t Dpad, float inv_tau, const float* cr, const float* cc, const float* dg, uint16_t* G3,
                              void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SNAG_B200_H */
