// extern "C" surface of libsnag_b200.so — see include/snag_b200.h for the contract.
#include "../../include/snag_b200.h"
#include "snag_internal.h"

using namespace snag;

static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline const __nv_bfloat16* BF(const uint16_t* p) { return reinterpret_cast<const __nv_bfloat16*>(p); }

extern "C" {

int snag_version(void) { return 1; }

const char* snag_error_string(int code) {
  switch (code) {
    case SNAG_OK: return "ok";
    case SNAG_ERR_ARG: return "bad argument (null pointer or non-positive size)";
    case SNAG_ERR_SHAPE: return "unsupported shape (Dpad not a multiple of 64, k > 16, ...)";
    case SNAG_ERR_ALIGN: return "pointer or leading dimension not aligned as required";
    case SNAG_ERR_DRIVER: return "cuTensorMapEncodeTiled unavailable or failed";
    case SNAG_ERR_DEVICE: return "current device is not sm_100 (B200); no fallback path exists";
    default: return code > 0 ? cudaGetErrorString(static_cast<cudaError_t>(code)) : "unknown error";
  }
}

int snag_device_check(void) { return device_is_sm100() ? SNAG_OK : SNAG_ERR_DEVICE; }
int snag_num_sms(void) { return num_sms(); }

int snag_sim_plan(int n_rows, int n_cols, int Dpad, int* tiles_per_chunk, int* n_lists) {
  SimPlan pl;
  const int rc = make_plan(n_rows, n_cols, Dpad, &pl);
  if (rc) return rc;
  if (tiles_per_chunk) *tiles_per_chunk = pl.tiles_per_chunk;
  if (n_lists) *n_lists = pl.n_lists;
  return SNAG_OK;
}

int snag_noise_mask(const float* x, float* out, const float* mean, const float* std_, const uint8_t* mask,
                    const float* zsel, const int32_t* selpos, int64_t N, int32_t F, int64_t ld_in, int64_t ld_out,
                    float ratio, float keep, float rho, uint64_t seed, int64_t row0, void* stream) {
  return launch_noise_mask(x, out, mean, std_, mask, zsel, selpos, N, F, ld_in, ld_out, ratio, keep, rho, seed, row0,
                           S(stream));
}
int snag_philox_rowmask(uint8_t* mask, int64_t N, float ratio, uint64_t seed, int64_t row0, void* stream) {
  return launch_philox_rowmask(mask, N, ratio, seed, row0, S(stream));
}
int snag_gauss_fill(float* out, const float* mean, const float* std_, int64_t N, int32_t F, int64_t ld, uint64_t seed,
                    int64_t row0, void* stream) {
  return launch_gauss_fill(out, mean, std_, N, F, ld, seed, row0, S(stream));
}
int snag_col_mean_std(const float* x, const uint8_t* valid, int64_t N, int32_t F, int64_t ld, float* mean, float* std_,
                      void* workspace, void* stream) {
  return launch_col_mean_std(x, valid, N, F, ld, mean, std_, workspace, S(stream));
}
int snag_rowblend_fwd(const float* e, const float* noise, const uint8_t* mask, float* out, int64_t N, int32_t D, float a,
                      float c, void* stream) {
  return launch_rowblend_fwd(e, noise, mask, out, N, D, a, c, S(stream));
}
int snag_rowblend_bwd(const float* g_out, const uint8_t* mask, float* g_in, int64_t N, int32_t D, float a, void* stream) {
  return launch_rowblend_bwd(g_out, mask, g_in, N, D, a, S(stream));
}

int snag_prep_bf16(const float* emb, int64_t ld, const int64_t* idx, int32_t n, int32_t D, int32_t normalize,
                   uint16_t* out, int32_t Dpad, float* norm2, void* stream) {
  return launch_prep_bf16(emb, ld, reinterpret_cast<const long long*>(idx), n, D, normalize,
                          reinterpret_cast<__nv_bfloat16*>(out), Dpad, norm2, S(stream));
}

int snag_joint_fuse_fwd(const float* const* embs, const int32_t* widths, int32_t M, int64_t N, const float* w_ent, int64_t ldw,
                        const float* w_glob, float* joint, float* joint_fz, int64_t ld_out, void* stream) {
  return launch_joint_fuse_fwd(embs, widths, M, N, w_ent, ldw, w_glob, joint, joint_fz, ld_out, S(stream));
}
int snag_joint_fuse_bwd(const float* const* embs, float* const* d_embs, const int32_t* widths, int32_t M, int64_t N,
                        const float* w_ent, int64_t ldw, const float* w_glob, const float* d_joint, const float* d_joint_fz,
                        int64_t ld_out, float* d_w_ent, float* d_w_glob, void* stream) {
  return launch_joint_fuse_bwd(embs, d_embs, widths, M, N, w_ent, ldw, w_glob, d_joint, d_joint_fz, ld_out, d_w_ent, d_w_glob,
                               S(stream));
}
int snag_normalize_bwd_scatter(const float* emb, int64_t ld, const int64_t* idx, int32_t n, int32_t D, int32_t normalize,
                               const float* dz, int64_t ld_dz, int32_t n_parts, int64_t part_stride, float* demb,
                               int64_t ld_demb, void* stream) {
  return launch_normalize_bwd_scatter(emb, ld, reinterpret_cast<const long long*>(idx), n, D, normalize, dz, ld_dz, n_parts,
                                      part_stride, demb, ld_demb, S(stream));
}
int snag_icl_stack_prep(int32_t n_prob, const float* const* emb, const int64_t* ld, const int32_t* D, uint16_t* const* out,
                        const int32_t* Dpad, const int64_t* idx_l, const int64_t* idx_r, int32_t B, int32_t Bp,
                        int32_t normalize, void* stream) {
  return launch_icl_stack_prep(n_prob, emb, reinterpret_cast<const long long*>(ld), D,
                               reinterpret_cast<__nv_bfloat16* const*>(out), Dpad, reinterpret_cast<const long long*>(idx_l),
                               reinterpret_cast<const long long*>(idx_r), B, Bp, normalize, S(stream));
}
int snag_normalize_bwd_scatter_many(int32_t n_prob, const float* const* emb, const int64_t* ld, const int32_t* D,
                                    const float* const* dz_a, const float* const* dz_b, const int64_t* ld_dz,
                                    const int32_t* n_parts, const int64_t* part_stride, float* const* demb,
                                    const int64_t* ld_demb, const int64_t* idx_l, const int64_t* idx_r, int32_t n,
                                    int32_t normalize, void* stream) {
  return launch_normalize_bwd_scatter_many(n_prob, emb, reinterpret_cast<const long long*>(ld), D, dz_a, dz_b,
                                           reinterpret_cast<const long long*>(ld_dz), n_parts,
                                           reinterpret_cast<const long long*>(part_stride), demb,
                                           reinterpret_cast<const long long*>(ld_demb),
                                           reinterpret_cast<const long long*>(idx_l),
                                           reinterpret_cast<const long long*>(idx_r), n, normalize, S(stream));
}
int snag_l1_distance(const float* x, const float* y, int64_t n1, int64_t n2, int32_t D, int64_t ldx, int64_t ldy, float* out,
                     int64_t ldo, void* stream) {
  return launch_l1_distance(x, y, n1, n2, D, ldx, ldy, out, ldo, S(stream));
}
int snag_matrix_rank(const float* d, int64_t n, int64_t ld, int32_t* cnt_row, int32_t* cnt_col, void* stream) {
  return launch_matrix_rank(d, n, ld, cnt_row, cnt_col, S(stream));
}

int snag_l1_plan(int32_t n_rows, int32_t n_cols, int32_t Dp, int32_t* n_lists) {
  SimPlan pl;
  const int rc = l1_plan(n_rows, n_cols, Dp, &pl);
  if (rc) return rc;
  if (n_lists) *n_lists = pl.n_lists;
  return SNAG_OK;
}
int snag_l1_rowtopk(const float* X, const float* Y, int32_t n1, int32_t n2, int32_t Dp, float* part, int32_t* part_idx,
                    void* stream) {
  return launch_l1_rowtopk(X, Y, n1, n2, Dp, part, part_idx, S(stream));
}
int snag_l1_rank_band(const float* X, const float* Y, const float* xn, const float* yn, const float* nv1, const float* nv2,
                      const float* g_row, const float* g_col, int32_t row_gid0, int32_t col_gid0, int32_t n1, int32_t n2,
                      int32_t Dp, int32_t use_csls, int32_t* cnt_row, int32_t* cnt_col, float* top4_val, int32_t* top4_idx,
                      uint64_t* band, uint32_t* band_cnt, uint32_t band_cap, void* stream) {
  return launch_l1_rank_band(X, Y, xn, yn, nv1, nv2, g_row, g_col, row_gid0, col_gid0, n1, n2, Dp, use_csls, cnt_row, cnt_col,
                             top4_val, top4_idx, reinterpret_cast<uint2*>(band), band_cnt, band_cap, S(stream));
}
int snag_l1_topk_rescore(const float* A, const float* B, int32_t Dp, int64_t n_rows, const float* an, float bn_max,
                         const int32_t* cand_idx, const float* cand_val, int32_t k, float* nv, int32_t* flagged,
                         int32_t* flagged_cnt, int32_t flagged_cap, void* stream) {
  return launch_l1_topk_rescore(A, B, Dp, n_rows, an, bn_max, cand_idx, cand_val, k, nv, flagged, flagged_cnt, flagged_cap,
                                S(stream));
}
int snag_l1_topk_exhaustive(const float* A, const float* B, int32_t Dp, int64_t n_b, const int32_t* flagged,
                            const int32_t* flagged_cnt, int32_t flagged_cap, int32_t k, float* nv, void* stream) {
  return launch_l1_topk_exhaustive(A, B, Dp, n_b, flagged, flagged_cnt, flagged_cap, k, nv, S(stream));
}
int snag_l1_pair_score(const float* X, const float* Y, int32_t Dp, int64_t n, const float* nv1, const float* nv2,
                       int32_t use_csls, float* g, void* stream) {
  return launch_l1_pair_score(X, Y, Dp, n, nv1, nv2, use_csls, g, S(stream));
}
int snag_l1_band_rescore(const float* X, const float* Y, int32_t Dp, const float* nv1, const float* nv2, const float* g_row,
                         const float* g_col, int32_t row_gid0, int32_t col_gid0, int32_t use_csls, const uint64_t* band,
                         const uint32_t* band_cnt, uint32_t band_cap, int32_t* cnt_row, int32_t* cnt_col, void* stream) {
  return launch_l1_band_rescore(X, Y, Dp, nv1, nv2, g_row, g_col, row_gid0, col_gid0, use_csls,
                                reinterpret_cast<const uint2*>(band), band_cnt, band_cap, cnt_row, cnt_col, S(stream));
}
int snag_l1_top3_rescore(const float* X, const float* Y, int32_t Dp, int64_t n_rows, int64_t n_b, const float* xn, float yn_max,
                         const float* nv1, const float* nv2, float nv2_absmax, int32_t use_csls, const int32_t* cand, float* oval,
                         int32_t* oidx, int32_t* flagged, int32_t* flagged_cnt, void* stream) {
  return launch_l1_top3_rescore(X, Y, Dp, n_rows, n_b, xn, yn_max, nv1, nv2, nv2_absmax, use_csls, cand, oval, oidx, flagged,
                                flagged_cnt, S(stream));
}
int32_t snag_icl_bwd_fused_splits(int32_t n_prob, int32_t B, int32_t Bp, int32_t row_blocks) {
  return icl_bwd_fused_splits(n_prob, B, Bp, row_blocks);
}
int snag_icl_bwd_fused(int32_t n_prob, const uint16_t* const* S3, const float* const* cr_a, const float* const* cr_b,
                       const float* const* dg, float* const* dz_a, float* const* dz_b, int32_t B, int32_t Bp, int32_t rb0,
                       int32_t row_blocks, int32_t Dpad, float inv_tau, int32_t nsplit, int64_t part_stride, void* stream) {
  return launch_icl_bwd_fused(n_prob, reinterpret_cast<const __nv_bfloat16* const*>(S3), cr_a, cr_b, dg, dz_a, dz_b, B, Bp,
                              rb0, row_blocks, Dpad, inv_tau, nsplit, part_stride, S(stream));
}

int snag_icl_fwd_sym_plan(int32_t n_prob, int32_t B, int32_t Bp, int64_t* sizes) {
  if (!sizes) return SNAG_ERR_ARG;
  long long out[3];
  const int rc = icl_fwd_sym_plan(n_prob, B, Bp, out);
  if (rc) return rc;
  sizes[0] = out[0]; sizes[1] = out[1]; sizes[2] = out[2];
  return SNAG_OK;
}
int snag_icl_fwd_sym(int32_t n_prob, const uint16_t* const* S3, float* const* rowpart, float* const* colpart, float* pos,
                     int32_t B, int32_t Bp, int32_t Dpad, float inv_tau, int32_t unit_begin, int32_t unit_end, float* total,
                     uint16_t* const* esave, void* stream) {
  return launch_icl_fwd_sym(n_prob, reinterpret_cast<const __nv_bfloat16* const*>(S3), rowpart, colpart, pos, B, Bp, Dpad,
                            inv_tau, unit_begin, unit_end, total, reinterpret_cast<__nv_bfloat16* const*>(esave), S(stream));
}
int snag_icl_g_from_e(const uint16_t* E, int32_t side, int32_t B, int32_t Bp, const float* cr_this, const float* cr_other,
                      const float* diag, float inv_tau, uint16_t* G, void* stream) {
  return launch_icl_g_from_e(BF(E), side, B, Bp, cr_this, cr_other, diag, inv_tau, reinterpret_cast<__nv_bfloat16*>(G), S(stream));
}
int snag_icl_sym_finalize(const float* total, const float* pos, int32_t n_prob, int32_t B, int32_t Bp, float inv_tau,
                          float* out, void* stream) {
  return launch_icl_sym_finalize(total, pos, n_prob, B, Bp, inv_tau, out, S(stream));
}

int snag_sim_mainloop_only(const uint16_t* X, const uint16_t* Y, int32_t n1, int32_t n2, int32_t Dpad, void* stream) {
  return launch_sim_null(BF(X), BF(Y), n1, n2, Dpad, S(stream));
}
int snag_debug_counters(uint64_t* counters) {
  set_debug_counters(reinterpret_cast<unsigned long long*>(counters));
  return SNAG_OK;
}
int snag_sim_write(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, int32_t n1, int32_t n2,
                   int32_t Dpad, int32_t mode, float* out, int64_t ld, void* stream) {
  return launch_sim_write(BF(X), BF(Y), xn, yn, n1, n2, Dpad, mode, out, ld, S(stream));
}
int snag_sim_write_t_splits(int32_t n1, int32_t n2, int32_t Dpad) { return sim_write_t_splits(n1, n2, Dpad); }
int snag_sim_write_t_mn(const uint16_t* XT, int32_t xt_ld, const uint16_t* Y, int32_t n1, int32_t n2, int32_t Dpad,
                        int32_t ksplits, float* out, int64_t ld, int64_t split_stride, void* stream) {
  return launch_sim_write_t_mn(BF(XT), xt_ld, BF(Y), n1, n2, Dpad, ksplits, out, ld, split_stride, S(stream));
}
int snag_sim_write_t(const uint16_t* X, const uint16_t* Y, int32_t n1, int32_t n2, int32_t Dpad, int32_t ksplits, float* out,
                     int64_t ld, int64_t split_stride, void* stream) {
  return launch_sim_write_t(BF(X), BF(Y), n1, n2, Dpad, ksplits, out, ld, split_stride, S(stream));
}
int snag_eval_rowtopk(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, int32_t n1, int32_t n2,
                      int32_t Dpad, float* part, int32_t* part_idx, void* stream) {
  return launch_eval_rowtopk(BF(X), BF(Y), xn, yn, n1, n2, Dpad, part, part_idx, S(stream));
}
int snag_topk_merge_mean(const float* part, const int32_t* part_idx, int32_t n_lists, int64_t n_rows, int32_t k, float* nv,
                         float* cand_out, int32_t* cand_idx_out, void* stream) {
  return launch_topk_merge_mean(part, part_idx, n_lists, n_rows, k, nv, cand_out, cand_idx_out, S(stream));
}
int snag_topk_rescore(const uint16_t* A, const uint16_t* B, int32_t Dpad, int64_t n_rows, const float* an, const float* bn,
                      const int32_t* cand_idx, const float* cand_val, int32_t k, float delta, const float* outsider_bound,
                      float* nv, int32_t* flagged, int32_t* flagged_cnt, int32_t flagged_cap, float* best_d,
                      int32_t* best_idx, void* stream) {
  return launch_topk_rescore(BF(A), BF(B), Dpad, n_rows, an, bn, cand_idx, cand_val, k, delta, outsider_bound, nv, flagged,
                             flagged_cnt, flagged_cap, best_d, best_idx, S(stream));
}
int snag_topk_exhaustive(const uint16_t* A, const uint16_t* B, int32_t Dpad, int64_t n_b, const float* an, const float* bn,
                         const int32_t* flagged, const int32_t* flagged_cnt, int32_t flagged_cap, int32_t k, float* nv,
                         float* best_d, int32_t* best_idx, void* stream) {
  return launch_topk_exhaustive(BF(A), BF(B), Dpad, n_b, an, bn, flagged, flagged_cnt, flagged_cap, k, nv, best_d, best_idx,
                                S(stream));
}
int snag_pair_score(const uint16_t* X, const uint16_t* Y, int32_t Dpad, int64_t n, const float* xn, const float* yn,
                    const float* nv1, const float* nv2, int32_t use_csls, float* g, float* s_out, void* stream) {
  return launch_pair_score(BF(X), BF(Y), Dpad, n, xn, yn, nv1, nv2, use_csls, g, s_out, S(stream));
}
int snag_eval_rank(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, const float* nv1,
                   const float* nv2, const float* g_row, const float* g_col, int32_t row_gid0, int32_t col_gid0,
                   int32_t n1, int32_t n2, int32_t Dpad, int32_t use_csls, int32_t* cnt_row, int32_t* cnt_col,
                   float* top3_val, int32_t* top3_idx, void* stream) {
  return launch_eval_rank(BF(X), BF(Y), xn, yn, nv1, nv2, g_row, g_col, row_gid0, col_gid0, n1, n2, Dpad, use_csls, cnt_row,
                          cnt_col, top3_val, top3_idx, S(stream));
}
int snag_eval_rank_band(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, const float* nv1,
                        const float* nv2, const float* g_row, const float* g_col, int32_t row_gid0, int32_t col_gid0,
                        int32_t n1, int32_t n2, int32_t Dpad, int32_t use_csls, float eps, int32_t* cnt_row, int32_t* cnt_col,
                        float* top4_val, int32_t* top4_idx, uint64_t* band, uint32_t* band_cnt, uint32_t band_cap,
                        void* stream) {
  return launch_eval_rank_band(BF(X), BF(Y), xn, yn, nv1, nv2, g_row, g_col, row_gid0, col_gid0, n1, n2, Dpad, use_csls, eps,
                               cnt_row, cnt_col, top4_val, top4_idx, reinterpret_cast<uint2*>(band), band_cnt, band_cap,
                               S(stream));
}
int snag_band_rescore(const uint16_t* X, const uint16_t* Y, int32_t Dpad, const float* xn, const float* yn, const float* nv1,
                      const float* nv2, const float* g_row, const float* g_col, int32_t row_gid0, int32_t col_gid0,
                      int32_t use_csls, const uint64_t* band, const uint32_t* band_cnt, uint32_t band_cap, int32_t* cnt_row,
                      int32_t* cnt_col, void* stream) {
  return launch_band_rescore(BF(X), BF(Y), Dpad, xn, yn, nv1, nv2, g_row, g_col, row_gid0, col_gid0, use_csls,
                             reinterpret_cast<const uint2*>(band), band_cnt, band_cap, cnt_row, cnt_col, S(stream));
}
int snag_eval_rank_band_rows(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, const float* nv1,
                             const float* nv2, const float* g_row, const float* g_col, const int32_t* row_gids,
                             int32_t col_gid0, int32_t n1, int32_t n2, int32_t Dpad, int32_t use_csls, float eps,
                             int32_t* cnt_row, int32_t* cnt_col, uint64_t* band, uint32_t* band_cnt, uint32_t band_cap,
                             void* stream) {
  if (!row_gids) return SNAG_ERR_ARG;
  return launch_eval_rank_band(BF(X), BF(Y), xn, yn, nv1, nv2, g_row, g_col, 0, col_gid0, n1, n2, Dpad, use_csls, eps,
                               cnt_row, cnt_col, nullptr, nullptr, reinterpret_cast<uint2*>(band), band_cnt, band_cap,
                               S(stream), row_gids);
}
int snag_band_rescore_rows(const uint16_t* X, const uint16_t* Y, int32_t Dpad, const float* xn, const float* yn,
                           const float* nv1, const float* nv2, const float* g_row, const float* g_col, const int32_t* row_gids,
                           int32_t col_gid0, int32_t use_csls, int32_t swapped, const uint64_t* band, const uint32_t* band_cnt,
                           uint32_t band_cap, int32_t* cnt_row, int32_t* cnt_col, void* stream) {
  if (!row_gids) return SNAG_ERR_ARG;
  return launch_band_rescore(BF(X), BF(Y), Dpad, xn, yn, nv1, nv2, g_row, g_col, 0, col_gid0, use_csls,
                             reinterpret_cast<const uint2*>(band), band_cnt, band_cap, cnt_row, cnt_col, S(stream), row_gids,
                             swapped);
}
int snag_pairs_dot(const uint16_t* X, const uint16_t* Y, int32_t Dpad, const int32_t* rows, const int32_t* cols,
                   int64_t n_pairs, float* s_out, void* stream) {
  return launch_pairs_dot(BF(X), BF(Y), Dpad, rows, cols, n_pairs, s_out, S(stream));
}
int snag_top4_merge(const float* val, const int32_t* idx, int32_t n_lists, int64_t n_rows, float* oval, int32_t* oidx,
                    void* stream) {
  return launch_top4_merge(val, idx, n_lists, n_rows, oval, oidx, S(stream));
}
int snag_top3_rescore(const uint16_t* X, const uint16_t* Y, int32_t Dpad, int64_t n_rows, const float* xn, const float* yn,
                      const float* nv1, const float* nv2, int32_t use_csls, const int32_t* cand, float* oval, int32_t* oidx,
                      void* stream) {
  return launch_top3_rescore(BF(X), BF(Y), Dpad, n_rows, xn, yn, nv1, nv2, use_csls, cand, oval, oidx, S(stream));
}

int64_t snag_csls_workspace_bytes(int64_t n1, int64_t n2) { return csls_workspace_floats(n1, n2) * 4; }
int snag_csls_sim(const float* sim, int64_t n1, int64_t n2, int64_t ld, int32_t k, float* out, int64_t ld_out, float* nv1,
                  float* nv2, void* workspace, void* stream) {
  return launch_csls_sim(sim, n1, n2, ld, k, out, ld_out, nv1, nv2, reinterpret_cast<float*>(workspace), S(stream));
}

int snag_icl_rowsum(const uint16_t* X, const uint16_t* Y, int32_t B, int32_t Bp, int32_t row0, int32_t nx, int32_t Dpad,
                    float inv_tau, float* rowsum_part, float* pos, void* stream) {
  return launch_icl_rowsum(BF(X), BF(Y), B, Bp, row0, nx, Dpad, inv_tau, rowsum_part, pos, S(stream));
}
int snag_icl_finalize(const float* rowsum_part, int32_t n_lists, int32_t B, int32_t Bp, const float* pos,
                      float inv_tau, float* lse, float* nll, void* stream) {
  if (!rowsum_part || !pos || !lse || !nll || B <= 0 || n_lists <= 0) return SNAG_ERR_ARG;
  return launch_icl_finalize(rowsum_part, n_lists, B, Bp, pos, inv_tau, lse, nll, S(stream));
}

int snag_eval_rowcoltopk(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, int32_t n1, int32_t n2,
                         int32_t Dpad, float* part, int32_t* part_idx, const float* rowthr, const float* colthr,
                         const float* colb, uint64_t* stream, int32_t* stream_row, int32_t* stream_cnt, int32_t cta_cap,
                         float norm2_max, void* stream_) {
  return launch_eval_rowcoltopk(BF(X), BF(Y), xn, yn, n1, n2, Dpad, part, part_idx, rowthr, colthr, colb,
                                reinterpret_cast<uint2*>(stream), stream_row, stream_cnt, cta_cap, norm2_max, S(stream_));
}
int snag_eval_onepass(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, int32_t n1, int32_t n2,
                      int32_t Dpad, float* part, int32_t* part_idx, const float* rowthr, const float* colthr, const float* colb,
                      uint64_t* stream, int32_t* stream_row, int32_t* stream_cnt, int32_t cta_cap, const float* rk_r,
                      const float* rk_rp, const float* rk_c, const float* rk_cp, uint64_t* rk_stream, int32_t* rk_stream_row,
                      int32_t* rk_cnt, int32_t rk_cap, float norm2_max, void* stream_) {
  return launch_eval_onepass(BF(X), BF(Y), xn, yn, n1, n2, Dpad, part, part_idx, rowthr, colthr, colb,
                             reinterpret_cast<uint2*>(stream), stream_row, stream_cnt, cta_cap, rk_r, rk_rp, rk_c, rk_cp,
                             reinterpret_cast<uint2*>(rk_stream), rk_stream_row, rk_cnt, rk_cap, norm2_max, S(stream_));
}
int snag_spec_bounds(const float* cand, int64_t n, int32_t k, const float* cdiag, float shift, float delta, float* lo,
                     float* hi, void* stream) {
  return launch_spec_bounds(cand, n, k, cdiag, shift, delta, lo, hi, S(stream));
}
int snag_rank_judge(const uint64_t* rk_stream, const int32_t* rk_stream_row, const int32_t* rk_cnt, int32_t n_ctas,
                    int32_t rk_cap, const float* R, const float* Rp, const float* C, const float* Cp, const uint8_t* row_ok,
                    const uint8_t* col_ok, float eps, int32_t row_gid0, int32_t col_gid0, int32_t* cnt_row, int32_t* cnt_col,
                    uint64_t* band, uint32_t* band_cnt, uint32_t band_cap, int32_t* overflow, void* stream) {
  return launch_rank_judge(reinterpret_cast<const uint2*>(rk_stream), rk_stream_row, rk_cnt, n_ctas, rk_cap, R, Rp, C, Cp,
                           row_ok, col_ok, eps, row_gid0, col_gid0, cnt_row, cnt_col, reinterpret_cast<uint2*>(band), band_cnt,
                           band_cap, overflow, S(stream));
}
int snag_rank_exhaustive(const uint16_t* A, const uint16_t* B, int32_t Dpad, int64_t n_b, const float* an, const float* bn,
                         const float* nva, const float* nvb, const float* g, const int32_t* rows, int32_t n_rows,
                         int32_t a_gid0, int32_t b_gid0, int32_t use_csls, int32_t swapped, int32_t* cnt, void* stream) {
  return launch_rank_exhaustive(BF(A), BF(B), Dpad, n_b, an, bn, nva, nvb, g, rows, n_rows, a_gid0, b_gid0, use_csls, swapped,
                                cnt, S(stream));
}
int snag_col_threshold(const float* cand, int64_t n, int32_t k, const float* yn, float* colthr, float* colb, void* stream) {
  return launch_col_threshold(cand, n, k, yn, colthr, colb, S(stream));
}
int snag_col_cand_hist(const uint64_t* stream, const int32_t* stream_cnt, int32_t n_ctas, int32_t cta_cap, int32_t* hist,
                       int32_t* overflow, void* stream_) {
  return launch_cand_hist(reinterpret_cast<const uint2*>(stream), stream_cnt, n_ctas, cta_cap, hist, overflow, S(stream_));
}
int snag_col_cand_scatter(const uint64_t* stream, const int32_t* stream_row, const int32_t* stream_cnt, int32_t n_ctas,
                          int32_t cta_cap, const int64_t* offs, int32_t* cursor, float* vals, int32_t* rows, void* stream_) {
  return launch_cand_scatter(reinterpret_cast<const uint2*>(stream), stream_row, stream_cnt, n_ctas, cta_cap,
                             reinterpret_cast<const long long*>(offs), cursor, vals, rows, S(stream_));
}
int snag_col_cand_finalize(const int64_t* offs, const int32_t* hist, const float* vals, const int32_t* rows, int64_t n,
                           int32_t k, float* nv, float* cand_val, int32_t* cand_idx, int32_t* overflow, void* stream) {
  return launch_col_cand_finalize(reinterpret_cast<const long long*>(offs), hist, vals, rows, n, k, nv, cand_val, cand_idx,
                                  overflow, S(stream));
}

int snag_mutual_nn(const uint16_t* X, const uint16_t* Y, const float* xn, const float* yn, int32_t n1, int32_t n2,
                   int32_t Dpad, const float* colb, uint64_t* colkey, float* row_val, int32_t* row_idx, void* stream) {
  return launch_mutual_nn(BF(X), BF(Y), xn, yn, n1, n2, Dpad, colb, reinterpret_cast<unsigned long long*>(colkey), row_val,
                          row_idx, S(stream));
}

int snag_icl_bwd_logits(const uint16_t* X, const uint16_t* Y, int32_t B, int32_t Bp, int32_t row0, int32_t nx,
                        int32_t Dpad, float inv_tau, const float* cr, const float* cc, const float* dg, uint16_t* G,
                        int32_t self_cols, float ebar, void* stream) {
  return launch_icl_bwd_logits(BF(X), BF(Y), B, Bp, row0, nx, Dpad, inv_tau, cr, cc, dg,
                               reinterpret_cast<__nv_bfloat16*>(G), self_cols, ebar, S(stream));
}

}  // extern "C"
