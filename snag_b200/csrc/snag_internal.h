// Internal C++ declarations shared by the translation units of libsnag_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace snag {

constexpr int SNAG_MAX_MODAL = 6;   // gph, rel, att, img, name, char (model/SNAG_tools.py:47)
constexpr int KT_LIST = 16;   // candidate-list length of the CSLS top-k path (must equal KT in simgemm.cuh)
#ifndef SNAG_EPI_WG
#define SNAG_EPI_WG 2
#endif
constexpr int LISTS_PER_CHUNK = SNAG_EPI_WG;   // partial per-row outputs per column chunk (= epilogue warpgroups)

int num_sms();                // SM count of the current device (cached per device)
int device_is_sm100();        // 1 if the current device is compute capability 10.x

struct SimPlan {
  int kblocks, row_blocks, col_tiles, tiles_per_chunk, n_chunks, n_units;
  int n_lists;   // partial per-row output lists a sweep produces: n_chunks * LISTS_PER_CHUNK
};
// Deterministic work decomposition for an [n_rows x n_cols] similarity sweep with padded width Dpad.
int make_plan(int n_rows, int n_cols, int Dpad, SimPlan* plan);

// ---- bandwidth kernels (bw_kernels.cu)
int launch_noise_mask(const float* x, float* out, const float* mean, const float* stdv, const uint8_t* mask,
                      const float* zsel, const int* selpos, long long N, int F, long long ld_in, long long ld_out,
                      float ratio, float keep, float rho, unsigned long long seed, long long row0, cudaStream_t st);
int launch_philox_rowmask(uint8_t* mask, long long N, float ratio, unsigned long long seed, long long row0, cudaStream_t st);
int launch_gauss_fill(float* out, const float* mean, const float* stdv, long long N, int F, long long ld,
                      unsigned long long seed, long long row0, cudaStream_t st);
int launch_col_mean_std(const float* x, const uint8_t* valid, long long N, int F, long long ld, float* mean, float* stdv,
                        void* workspace, cudaStream_t st);
int launch_rowblend_fwd(const float* e, const float* noise, const uint8_t* mask, float* out, long long N, int D, float a,
                        float c, cudaStream_t st);
int launch_rowblend_bwd(const float* g_out, const uint8_t* mask, float* g_in, long long N, int D, float a, cudaStream_t st);
int launch_prep_bf16(const float* emb, long long ld, const long long* idx, int n, int D, int normalize,
                     __nv_bfloat16* out, int Dpad, float* norm2, cudaStream_t st);
int launch_prep_split(const float* emb, long long ld, const long long* idx, int n, int D, int normalize, int side,
                      float* rows, __nv_bfloat16* split, int Dpad, float* norm2, cudaStream_t st);
int launch_joint_fuse_fwd(const float* const* embs, const int* widths, int M, long long N, const float* w_ent, long long ldw,
                          const float* w_glob, float* joint, float* joint_fz, long long ld_out, cudaStream_t st);
int launch_joint_fuse_bwd(const float* const* embs, float* const* d_embs, const int* widths, int M, long long N,
                          const float* w_ent, long long ldw, const float* w_glob, const float* d_joint, const float* d_joint_fz,
                          long long ld_out, float* d_w_ent, float* d_w_glob, cudaStream_t st);
int launch_normalize_bwd_scatter(const float* emb, long long ld, const long long* idx, int n, int D, int normalize,
                                 const float* dz, long long ld_dz, int n_parts, long long part_stride, float* demb,
                                 long long ld_demb, cudaStream_t st);
int launch_icl_stack_prep(int n_prob, const float* const* emb, const long long* ld, const int* D, __nv_bfloat16* const* out,
                          const int* Dpad, const long long* idx_l, const long long* idx_r, int B, int Bp, int normalize,
                          cudaStream_t st);
int launch_normalize_bwd_scatter_many(int n_prob, const float* const* emb, const long long* ld, const int* D,
                                      const float* const* dz_a, const float* const* dz_b, const long long* ld_dz,
                                      const int* n_parts, const long long* part_stride, float* const* demb,
                                      const long long* ld_demb, const long long* idx_l, const long long* idx_r, int n,
                                      int normalize, cudaStream_t st);
int launch_l1_distance(const float* x, const float* y, long long n1, long long n2, int D, long long ldx, long long ldy,
                       float* out, long long ldo, cudaStream_t st);
int launch_matrix_rank(const float* d, long long n, long long ld, int* cnt_row, int* cnt_col, cudaStream_t st);
// fused --distance 1 evaluation (l1_sweep.cu)
int l1_plan(int n_rows, int n_cols, int Dp, SimPlan* plan);
int launch_l1_rowtopk(const float* X, const float* Y, int n1, int n2, int Dp, float* part, int* part_idx, cudaStream_t st);
int launch_l1_rank_band(const float* X, const float* Y, const float* xn, const float* yn, const float* nv1, const float* nv2,
                        const float* g_row, const float* g_col, int row_gid0, int col_gid0, int n1, int n2, int Dp,
                        int use_csls, int* cnt_row, int* cnt_col, float* top4_val, int* top4_idx, uint2* band,
                        unsigned int* band_cnt, unsigned int band_cap, cudaStream_t st);
int launch_l1_topk_rescore(const float* A, const float* B, int Dp, long long n_rows, const float* an, float bn_max,
                           const int* cand_idx, const float* cand_val, int k, float* nv, int* flagged, int* flagged_cnt,
                           int flagged_cap, cudaStream_t st);
int launch_l1_topk_exhaustive(const float* A, const float* B, int Dp, long long n_b, const int* flagged, const int* flagged_cnt,
                              int flagged_cap, int k, float* nv, cudaStream_t st);
int launch_l1_pair_score(const float* X, const float* Y, int Dp, long long n, const float* nv1, const float* nv2, int use_csls,
                         float* g, cudaStream_t st);
int launch_l1_band_rescore(const float* X, const float* Y, int Dp, const float* nv1, const float* nv2, const float* g_row,
                           const float* g_col, int row_gid0, int col_gid0, int use_csls, const uint2* band,
                           const unsigned int* band_cnt, unsigned int band_cap, int* cnt_row, int* cnt_col, cudaStream_t st);
int launch_l1_top3_rescore(const float* X, const float* Y, int Dp, long long n_rows, long long n_b, const float* xn,
                           float yn_max, const float* nv1, const float* nv2, float nv2_absmax, int use_csls, const int* cand,
                           float* oval, int* oidx, int* flagged, int* flagged_cnt, cudaStream_t st);
// fused ICL backward for Dpad <= 320 (icl_fused.cu)
int icl_bwd_fused_splits(int n_prob, int B, int Bp, int row_blocks);
int launch_icl_bwd_fused(int n_prob, const __nv_bfloat16* const* S3, const float* const* cr_a, const float* const* cr_b,
                         const float* const* dg, float* const* dz_a, float* const* dz_b, int B, int Bp, int rb0,
                         int row_blocks, int Dpad, float inv_tau, int nsplit, long long part_stride, cudaStream_t st);
// ICL forward on half the Gram matrix, all tables of a step in one launch (icl_fwd_sym.cu)
int icl_fwd_sym_plan(int n_prob, int B, int Bp, long long* out);
int launch_icl_fwd_sym(int n_prob, const __nv_bfloat16* const* S3, float* const* rowpart, float* const* colpart, float* pos,
                       int B, int Bp, int Dpad, float inv_tau, int unit_begin, int unit_end, float* total,
                       __nv_bfloat16* const* esave, cudaStream_t st, int split = 0);
int launch_icl_g_from_e(const __nv_bfloat16* E, int side, int B, int Bp, const float* cr_this, const float* cr_other,
                        const float* diag, float inv_tau, __nv_bfloat16* G, cudaStream_t st);
int launch_icl_sym_finalize(const float* total, const float* pos, int n_prob, int B, int Bp, float inv_tau, float* out,
                            cudaStream_t st);
int launch_topk_merge_mean(const float* part, const int* part_idx, int n_lists, long long n_rows, int k, float* nv,
                           float* cand_out, int* cand_idx_out, cudaStream_t st);
template <typename T>
int launch_topk_rescore(const T* A, const T* B, int Dpad, long long n_rows, const float* an,
                        const float* bn, const int* cand_idx, const float* cand_val, int k, float delta,
                        const float* outsider_bound, float* nv, int* flagged, int* flagged_cnt, int flagged_cap,
                        float* best_d, int* best_idx, cudaStream_t st);
template <typename T>
int launch_topk_exhaustive(const T* A, const T* B, int Dpad, long long n_b, const float* an,
                           const float* bn, const int* flagged, const int* flagged_cnt, int flagged_cap, int k, float* nv,
                           float* best_d, int* best_idx, cudaStream_t st);
template <typename T>
int launch_pair_score(const T* X, const T* Y, int Dpad, long long n, const float* xn, const float* yn,
                      const float* nv1, const float* nv2, int use_csls, float* g, float* s_out, cudaStream_t st);
template <typename T>
int launch_band_rescore(const T* X, const T* Y, int Dpad, const float* xn, const float* yn,
                        const float* nv1, const float* nv2, const float* g_row, const float* g_col, int row_gid0, int col_gid0,
                        int use_csls, const uint2* band, const unsigned int* band_cnt, unsigned int band_cap, int* cnt_row,
                        int* cnt_col, cudaStream_t st, const int* row_gids = nullptr, int swapped = 0);
template <typename T>
int launch_pairs_dot(const T* X, const T* Y, int Dpad, const int* rows, const int* cols,
                     long long n_pairs, float* s_out, cudaStream_t st);
int launch_top4_merge(const float* val, const int* idx, int n_lists, long long n_rows, float* oval, int* oidx, cudaStream_t st);
template <typename T>
int launch_top3_rescore(const T* X, const T* Y, int Dpad, long long n_rows, const float* xn,
                        const float* yn, const float* nv1, const float* nv2, int use_csls, const int* cand, float* oval,
                        int* oidx, cudaStream_t st);
int launch_icl_finalize(const float* rowsum_part, int n_chunks, int B, int Bp, const float* pos, float inv_tau, float* lse,
                        float* nll, cudaStream_t st);

long long csls_workspace_floats(long long n1, long long n2);
int launch_csls_sim(const float* sim, long long n1, long long n2, long long ld, int k, float* out, long long ld_out,
                    float* nv1, float* nv2, float* workspace, cudaStream_t st);

// ---- tcgen05 similarity sweeps (sim_kernels.cu)
void set_debug_counters(unsigned long long* p);
int launch_sim_null(const __nv_bfloat16* X, const __nv_bfloat16* Y, int n1, int n2, int Dpad, cudaStream_t st);
int launch_sim_write(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, int n1, int n2,
                     int Dpad, int mode, float* out, long long ld, cudaStream_t st);
int sim_write_t_splits(int n1, int n2, int Dpad);
int launch_sim_write_t_mn(const __nv_bfloat16* XT, int xt_ld, const __nv_bfloat16* Y, int n1, int n2, int Dpad, int ksplits,
                          float* out, long long ld, long long split_stride, cudaStream_t st);
int launch_sim_write_t(const __nv_bfloat16* X, const __nv_bfloat16* Y, int n1, int n2, int Dpad, int ksplits, float* out,
                       long long ld, long long split_stride, cudaStream_t st);
int launch_eval_rowtopk(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, int n1, int n2,
                        int Dpad, float* part, int* part_idx, cudaStream_t st);
int launch_eval_rank(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, const float* nv1,
                     const float* nv2, const float* g_row, const float* g_col, int row_gid0, int col_gid0, int n1, int n2,
                     int Dpad, int use_csls, int* cnt_row, int* cnt_col, float* top3_val, int* top3_idx, cudaStream_t st);
int launch_eval_rank_band(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, const float* nv1,
                          const float* nv2, const float* g_row, const float* g_col, int row_gid0, int col_gid0, int n1, int n2,
                          int Dpad, int use_csls, float eps, int* cnt_row, int* cnt_col, float* top4_val, int* top4_idx,
                          uint2* band, unsigned int* band_cnt, unsigned int band_cap, cudaStream_t st,
                          const int* row_gids = nullptr);
int launch_icl_rowsum(const __nv_bfloat16* X, const __nv_bfloat16* Y, int B, int Bp, int row0, int nx, int Dpad, float inv_tau,
                      float* rowsum_part, float* pos, cudaStream_t st);

int launch_mutual_nn(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, int n1, int n2,
                     int Dpad, const float* colb, unsigned long long* colkey, float* row_val, int* row_idx,
                     cudaStream_t st);
int launch_eval_rowcoltopk(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, int n1, int n2,
                           int Dpad, float* part, int* part_idx, const float* rowthr, const float* colthr, const float* colb,
                           uint2* stream, int* stream_row, int* stream_cnt, int cta_cap, float norm2_max, cudaStream_t st);
int launch_eval_onepass(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, int n1, int n2,
                        int Dpad, float* part, int* part_idx, const float* rowthr, const float* colthr, const float* colb,
                        uint2* stream, int* stream_row, int* stream_cnt, int cta_cap, const float* rk_r, const float* rk_rp,
                        const float* rk_c, const float* rk_cp, uint2* rk_stream, int* rk_stream_row, int* rk_cnt, int rk_cap,
                        float norm2_max, cudaStream_t st);
// largest squared row norm for which the fp16x2 pre-filter of the fused CSLS sweep is used (F.normalize'd rows rounded to
// bf16 are 1 +- 4e-3); above it snag_eval_rowcoltopk runs its fp32 per-element tests and snag_eval_onepass refuses
#define SNAG_HALF_PREFILTER_NORM2_MAX 1.05f
int launch_spec_bounds(const float* cand, long long n, int k, const float* cdiag, float shift, float delta, float* lo,
                       float* hi, cudaStream_t st);
int launch_rank_judge(const uint2* rk_stream, const int* rk_stream_row, const int* rk_cnt, int n_ctas, int rk_cap,
                      const float* R, const float* Rp, const float* C, const float* Cp, const unsigned char* row_ok,
                      const unsigned char* col_ok, float eps, int row_gid0, int col_gid0, int* cnt_row, int* cnt_col,
                      uint2* band, unsigned int* band_cnt, unsigned int band_cap, int* overflow, cudaStream_t st);
template <typename T>
int launch_rank_exhaustive(const T* A, const T* B, int Dpad, long long n_b, const float* an,
                           const float* bn, const float* nva, const float* nvb, const float* g, const int* rows, int n_rows,
                           int a_gid0, int b_gid0, int use_csls, int swapped, int* cnt, cudaStream_t st);
int launch_col_threshold(const float* cand, long long n, int k, const float* yn, float* colthr, float* colb, cudaStream_t st);
int launch_cand_hist(const uint2* stream, const int* stream_cnt, int n_ctas, int cta_cap, int* hist, int* overflow,
                     cudaStream_t st);
int launch_cand_scatter(const uint2* stream, const int* stream_row, const int* stream_cnt, int n_ctas, int cta_cap,
                        const long long* offs, int* cursor, float* vals, int* rows, cudaStream_t st);
int launch_col_cand_finalize(const long long* offs, const int* hist, const float* vals, const int* rows, long long n, int k,
                             float* nv, float* cand_val, int* cand_idx, int* overflow, cudaStream_t st);
int launch_icl_bwd_logits(const __nv_bfloat16* X, const __nv_bfloat16* Y, int B, int Bp, int row0, int nx, int Dpad, float inv_tau,
                          const float* cr, const float* cc, const float* dg, __nv_bfloat16* G, int self_cols, float ebar, cudaStream_t st);
// the fp32 loss route: split stacks [3 Bp, 5 Dpad] rows [m | h | h | m | h] (bw_kernels.cu / sim_kernels.cu)
int launch_icl_stack_prep_split(int n_prob, const float* const* emb, const long long* ld, const int* D, __nv_bfloat16* const* out,
                                const int* Dpad, const long long* idx_l, const long long* idx_r, int B, int Bp, int normalize,
                                cudaStream_t st);
int launch_icl_rowsum_split(const __nv_bfloat16* X, const __nv_bfloat16* Y, int B, int Bp, int row0, int nx, int Dpad,
                            float inv_tau, float* rowsum_part, float* pos, cudaStream_t st);
int launch_icl_bwd_logits_split(const __nv_bfloat16* X, const __nv_bfloat16* Y, int B, int Bp, int row0, int nx, int Dpad,
                                float inv_tau, const float* cr, const float* cc, const float* dg, __nv_bfloat16* G3,
                                cudaStream_t st);

}  // namespace snag
