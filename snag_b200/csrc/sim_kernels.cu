// Host side of the tcgen05 similarity sweeps: TMA descriptors, work plan, launches.
#include <mutex>
#include "simgemm.cuh"
#include "snag_internal.h"

namespace snag {

static_assert(KT == KT_LIST, "candidate list length mismatch");
static_assert(NUM_EPI_WG == LISTS_PER_CHUNK, "partial list count mismatch");

// ------------------------------------------------------------------------------------------------
// device info
// ------------------------------------------------------------------------------------------------
static int g_sms[64];
static int g_cc[64];
static std::once_flag g_dev_once[64];

static void query_dev(int dev) {
  cudaDeviceProp p;
  if (cudaGetDeviceProperties(&p, dev) == cudaSuccess) {
    g_sms[dev] = p.multiProcessorCount;
    g_cc[dev] = p.major * 10 + p.minor;
  } else {
    g_sms[dev] = 1;
    g_cc[dev] = 0;
  }
}
int num_sms() {
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 63;
  std::call_once(g_dev_once[dev], query_dev, dev);
  return g_sms[dev];
}
int device_is_sm100() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  dev &= 63;
  std::call_once(g_dev_once[dev], query_dev, dev);
  return g_cc[dev] / 10 == 10;
}

// ------------------------------------------------------------------------------------------------
// work plan: chunk of Y kept <= ~40 MB (L2 resident while ~148 row blocks sweep it), and enough
// units (>= ~4 per SM) for the persistent grid to balance.
// ------------------------------------------------------------------------------------------------
// tiles the busiest CTA of the persistent grid processes when units (row block x chunk of `tpc` column tiles, the last
// chunk possibly shorter) are dealt round-robin in chunk-major order, plus a quarter tile of fixed cost per unit
static inline long long floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }
// ids congruent to b (mod m) in [lo, hi)
static inline long long count_congruent(long long lo, long long hi, long long b, long long m) {
  return floor_div(hi - 1 - b, m) - floor_div(lo - 1 - b, m);
}
static double busiest_cta_load(int row_blocks, int col_tiles, int tpc, int sms) {
  const int n_chunks = (col_tiles + tpc - 1) / tpc;
  const long long big_end = static_cast<long long>(n_chunks - 1) * row_blocks;       // ids [0, big_end): full chunks
  const long long end = big_end + row_blocks;                                        // ids [big_end, end): last chunk
  const int last_tiles = col_tiles - (n_chunks - 1) * tpc;
  double worst = 0.0;
  for (int b = 0; b < sms; ++b) {
    const double load = static_cast<double>(count_congruent(0, big_end, b, sms)) * (tpc + 0.25) +
                        static_cast<double>(count_congruent(big_end, end, b, sms)) * (last_tiles + 0.25);
    if (load > worst) worst = load;
  }
  return worst;
}

struct PlanMemo {
  int n_rows = 0, n_cols = 0, Dpad = 0, sms = 0;
  SimPlan plan{};
};
static thread_local PlanMemo g_plan_memo[4];
static thread_local int g_plan_memo_next = 0;

int make_plan(int n_rows, int n_cols, int Dpad, SimPlan* pl) {
  if (n_rows <= 0 || n_cols <= 0 || Dpad <= 0 || (Dpad % BK) != 0 || !pl) return SNAG_ERR_SHAPE;
  const int sms_now = num_sms();
  for (const PlanMemo& m : g_plan_memo)
    if (m.n_rows == n_rows && m.n_cols == n_cols && m.Dpad == Dpad && m.sms == sms_now) { *pl = m.plan; return SNAG_OK; }
  pl->kblocks = Dpad / BK;
  pl->row_blocks = (n_rows + BM - 1) / BM;
  pl->col_tiles = (n_cols + BN - 1) / BN;
  const long long tile_bytes = static_cast<long long>(BN) * Dpad * 2;
  long long max_tiles_l2 = (40ll << 20) / tile_bytes;
  if (max_tiles_l2 < 1) max_tiles_l2 = 1;
  const int sms = num_sms();
  long long want_chunks = (4ll * sms + pl->row_blocks - 1) / pl->row_blocks;
  if (want_chunks < 1) want_chunks = 1;
  long long tpc = (pl->col_tiles + want_chunks - 1) / want_chunks;
  if (tpc > max_tiles_l2) tpc = max_tiles_l2;
  if (tpc < 1) tpc = 1;
  // Units are dealt to the CTAs round-robin, so a launch lasts as long as its busiest CTA: among chunk sizes between
  // half of the above and the above, keep the one with the lightest busiest CTA (ties: the larger chunk = fewer partial
  // lists). E.g. 128 row blocks x 128 column tiles: 26-tile chunks give 640 units, 4 or 5 per CTA (85 % balanced);
  // 16-tile chunks give 1024 units, 6 or 7 per CTA (99 %).
  if (static_cast<long long>(pl->row_blocks) * ((pl->col_tiles + tpc - 1) / tpc) < 64ll * sms) {
    int best = static_cast<int>(tpc);
    double best_load = busiest_cta_load(pl->row_blocks, pl->col_tiles, best, sms);
    for (int t = static_cast<int>(tpc) - 1; t >= 1 && 2 * t >= tpc; --t) {
      const double load = busiest_cta_load(pl->row_blocks, pl->col_tiles, t, sms);
      if (load < best_load * 0.995) { best_load = load; best = t; }
    }
    tpc = best;
  }
  pl->tiles_per_chunk = static_cast<int>(tpc);
  pl->n_chunks = (pl->col_tiles + pl->tiles_per_chunk - 1) / pl->tiles_per_chunk;
  const long long units = static_cast<long long>(pl->row_blocks) * pl->n_chunks;
  if (units > 0x7fffffffll) return SNAG_ERR_SHAPE;
  pl->n_units = static_cast<int>(units);
  pl->n_lists = pl->n_chunks * LISTS_PER_CHUNK;
  PlanMemo& slot = g_plan_memo[g_plan_memo_next];
  g_plan_memo_next = (g_plan_memo_next + 1) & 3;
  slot.n_rows = n_rows; slot.n_cols = n_cols; slot.Dpad = Dpad; slot.sms = sms_now; slot.plan = *pl;
  return SNAG_OK;
}

// ------------------------------------------------------------------------------------------------
// TMA descriptors through the driver entry point (no link-time dependency on libcuda)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::once_flag g_encode_once;
static void load_encode() {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
      q == cudaDriverEntryPointSuccess)
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
}

// bf16 row-major [rows, Dpad] operand whose rows lie ld >= Dpad elements apart (a column window of a wider matrix),
// box = [box_rows x 64 elements], 128-byte swizzle, zero OOB fill
static int make_operand_map_ld(CUtensorMap* m, const __nv_bfloat16* ptr, long long rows, int Dpad, long long ld, int box_rows) {
  std::call_once(g_encode_once, load_encode);
  if (!g_encode) return SNAG_ERR_DRIVER;
  if (reinterpret_cast<uintptr_t>(ptr) & 127) return SNAG_ERR_ALIGN;
  if (ld != Dpad && (ld < Dpad || (ld % 8) != 0)) return SNAG_ERR_SHAPE;     // TMA: 16-byte row strides
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(Dpad), static_cast<cuuint64_t>(rows)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 2};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), static_cast<cuuint32_t>(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(ptr), dims, strides, box,
                              estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? SNAG_OK : SNAG_ERR_DRIVER;
}
int make_operand_map(CUtensorMap* m, const __nv_bfloat16* ptr, long long rows, int Dpad, int box_rows) {
  return make_operand_map_ld(m, ptr, rows, Dpad, Dpad, box_rows);
}

// development aid: when set (snag_debug_counters), every sweep's UMMA issuer records its wait cycles per CTA
static unsigned long long* g_dbg_counters = nullptr;
void set_debug_counters(unsigned long long* p) { g_dbg_counters = p; }

// xt_ld > 0: X is given transposed, as a [Dpad rows, xt_ld columns] matrix whose first n1 columns are the operand
// (SimShape::a_mn). row_ld > 0: the rows of X and Y lie row_ld elements apart (column windows of the loss's split stacks)
template <class Epi>
static int launch_sim(const __nv_bfloat16* X, const __nv_bfloat16* Y, int n1, int n2, int Dpad,
                      const typename Epi::Params& ep, cudaStream_t st, int ksplits = 1, int xt_ld = 0, int row_ld = 0) {
  if (!X || !Y) return SNAG_ERR_ARG;
  if (!device_is_sm100()) return SNAG_ERR_DEVICE;
  SimPlan pl;
  int rc = make_plan(n1, n2, Dpad, &pl);
  if (rc) return rc;
  CUtensorMap tmX, tmY;
  const int ld = row_ld > 0 ? row_ld : Dpad;
  if (xt_ld > 0) {
    if ((xt_ld % 64) != 0 || xt_ld < n1 || row_ld > 0) return SNAG_ERR_SHAPE;
    if ((rc = make_operand_map(&tmX, X, Dpad, xt_ld, 64))) return rc;
  } else if ((rc = make_operand_map_ld(&tmX, X, n1, Dpad, ld, BM))) return rc;
  if ((rc = make_operand_map_ld(&tmY, Y, n2, Dpad, ld, BN))) return rc;
  // the attribute is per device; setting it on every call is cheap and covers multi-device processes
  const cudaError_t attr_err =
      cudaFuncSetAttribute(sim_kernel<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, SIM_SMEM_BYTES);
  if (attr_err != cudaSuccess) return static_cast<int>(attr_err);
  SimShape shp;
  shp.n_rows = n1;
  shp.n_cols = n2;
  shp.kblocks = pl.kblocks;
  shp.row_blocks = pl.row_blocks;
  shp.col_tiles = pl.col_tiles;
  shp.tiles_per_chunk = pl.tiles_per_chunk;
  shp.n_chunks = pl.n_chunks;
  shp.n_units = pl.n_units;
  if (ksplits < 1 || ksplits > pl.kblocks) return SNAG_ERR_SHAPE;
  shp.kb_split = (pl.kblocks + ksplits - 1) / ksplits;
  shp.ksplits = (pl.kblocks + shp.kb_split - 1) / shp.kb_split;      // no empty slice
  if (shp.ksplits != ksplits) return SNAG_ERR_SHAPE;                 // the caller sized its partial buffers for ksplits
  if (static_cast<long long>(pl.n_units) * shp.ksplits > 0x7fffffffll) return SNAG_ERR_SHAPE;
  shp.dbg = g_dbg_counters;
  shp.a_mn = xt_ld > 0 ? 1 : 0;
  const long long all_units = static_cast<long long>(pl.n_units) * shp.ksplits;
  const int grid = all_units < num_sms() ? static_cast<int>(all_units) : num_sms();
  sim_kernel<Epi><<<grid, NUM_CTRL_THREADS + 128 * EpiWG<Epi>::value, SIM_SMEM_BYTES, st>>>(tmX, tmY, shp, ep);
  return static_cast<int>(cudaGetLastError());
}

int launch_sim_null(const __nv_bfloat16* X, const __nv_bfloat16* Y, int n1, int n2, int Dpad, cudaStream_t st) {
  EpiNull::Params p{0};
  return launch_sim<EpiNull>(X, Y, n1, n2, Dpad, p, st);
}

int launch_sim_write(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, int n1, int n2,
                     int Dpad, int mode, float* out, long long ld, cudaStream_t st) {
  if (!out || ld < n2) return SNAG_ERR_ARG;
  if (mode == 1 && (!xn || !yn)) return SNAG_ERR_ARG;
  EpiWrite::Params p{out, ld, xn, yn, mode, 0, 0};
  return launch_sim<EpiWrite>(X, Y, n1, n2, Dpad, p, st);
}

// number of K slices launch_sim_write_t will use for an [n1 x n2] product of contraction width Dpad: the smallest
// count whose units fill the persistent grid's waves to >= 90 % (else the best filling), with slices of at least 24
// k-blocks so that a unit's MMAs outweigh its pipeline fill and its 128 KB partial-tile write
int sim_write_t_splits(int n1, int n2, int Dpad) {
  SimPlan pl;
  if (make_plan(n1, n2, Dpad, &pl)) return 1;
  const int sms = num_sms();
  const int max_ks = pl.kblocks / 24 > 1 ? pl.kblocks / 24 : 1;
  int best = 1;
  double best_eff = 0.0;
  for (int ks = 1; ks <= max_ks && ks <= 64; ++ks) {
    const int kb_split = (pl.kblocks + ks - 1) / ks;
    if ((pl.kblocks + kb_split - 1) / kb_split != ks) continue;          // would leave an empty slice
    const long long units = static_cast<long long>(pl.n_units) * ks;
    const double eff = static_cast<double>(units) / (static_cast<double>((units + sms - 1) / sms) * sms);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = ks; }
    if (eff >= 0.9) break;
  }
  return best;
}

// out_t[s][j][i] = sum over K slice s of X[i,:] . Y[j,:]  — the product written TRANSPOSED ([n2, ld] with ld >= n1), one
// partial per K slice (split_stride floats apart). Used for the loss's gradient GEMMs, whose contraction runs over the
// whole batch while the output is only D wide: with the D rows as X a tile's 256 columns are anchors, dL/dlogits is
// read once (the row-block CTAs that share a column tile run side by side and meet in L2), and split-K fills the SMs.
int launch_sim_write_t(const __nv_bfloat16* X, const __nv_bfloat16* Y, int n1, int n2, int Dpad, int ksplits, float* out,
                       long long ld, long long split_stride, cudaStream_t st) {
  if (!out || ld < n1 || ksplits < 1 || (ksplits > 1 && split_stride < static_cast<long long>(n2) * ld)) return SNAG_ERR_ARG;
  EpiWrite::Params p{out, ld, nullptr, nullptr, 0, 1, split_stride};
  return launch_sim<EpiWrite>(X, Y, n1, n2, Dpad, p, st, ksplits);
}

// The same product with X given transposed: XT [Dpad rows (the contraction), xt_ld columns], first n1 columns valid — for
// the gradient GEMMs XT is the stacked embedding matrix itself ([2 Bp, Dpad_emb]), so no transposed copy is needed.
int launch_sim_write_t_mn(const __nv_bfloat16* XT, int xt_ld, const __nv_bfloat16* Y, int n1, int n2, int Dpad, int ksplits,
                          float* out, long long ld, long long split_stride, cudaStream_t st) {
  if (!out || ld < n1 || ksplits < 1 || (ksplits > 1 && split_stride < static_cast<long long>(n2) * ld)) return SNAG_ERR_ARG;
  EpiWrite::Params p{out, ld, nullptr, nullptr, 0, 1, split_stride};
  return launch_sim<EpiWrite>(XT, Y, n1, n2, Dpad, p, st, ksplits, xt_ld);
}

int launch_eval_rowtopk(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, int n1, int n2,
                        int Dpad, float* part, int* part_idx, cudaStream_t st) {
  if (!xn || !yn || !part) return SNAG_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(part) | reinterpret_cast<uintptr_t>(part_idx)) & 15) return SNAG_ERR_ALIGN;
  if (part_idx) {
    EpiRowTopK<true>::Params p{xn, yn, part, part_idx};
    return launch_sim<EpiRowTopK<true>>(X, Y, n1, n2, Dpad, p, st);
  }
  EpiRowTopK<false>::Params p{xn, yn, part, nullptr};
  return launch_sim<EpiRowTopK<false>>(X, Y, n1, n2, Dpad, p, st);
}

int launch_eval_rank(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, const float* nv1,
                     const float* nv2, const float* g_row, const float* g_col, int row_gid0, int col_gid0, int n1, int n2,
                     int Dpad, int use_csls, int* cnt_row, int* cnt_col, float* top3_val, int* top3_idx, cudaStream_t st) {
  if (!xn || !yn || !g_row || !g_col || !cnt_row || !cnt_col) return SNAG_ERR_ARG;
  if (use_csls && (!nv1 || !nv2)) return SNAG_ERR_ARG;
  if (!use_csls) { nv1 = xn; nv2 = yn; }   // never read for their values; keeps the staging loads valid
  if ((top3_val == nullptr) != (top3_idx == nullptr)) return SNAG_ERR_ARG;
  if (top3_val && ((reinterpret_cast<uintptr_t>(top3_val) | reinterpret_cast<uintptr_t>(top3_idx)) & 15)) return SNAG_ERR_ALIGN;
#define SNAG_RANK_CASE(T3, CS)                                                                                       \
  {                                                                                                                  \
    typename EpiRank<T3, CS>::Params p{xn, yn, nv1, nv2, g_row, g_col, row_gid0, col_gid0, cnt_row, cnt_col, top3_val, top3_idx}; \
    return launch_sim<EpiRank<T3, CS>>(X, Y, n1, n2, Dpad, p, st);                                                   \
  }
  if (top3_val) {
    if (use_csls) SNAG_RANK_CASE(true, true) else SNAG_RANK_CASE(true, false)
  } else {
    if (use_csls) SNAG_RANK_CASE(false, true) else SNAG_RANK_CASE(false, false)
  }
#undef SNAG_RANK_CASE
}

int launch_eval_rank_band(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, const float* nv1,
                          const float* nv2, const float* g_row, const float* g_col, int row_gid0, int col_gid0, int n1, int n2,
                          int Dpad, int use_csls, float eps, int* cnt_row, int* cnt_col, float* top4_val, int* top4_idx,
                          uint2* band, unsigned int* band_cnt, unsigned int band_cap, cudaStream_t st, const int* row_gids) {
  if (!xn || !yn || !g_row || !g_col || !cnt_row || !cnt_col || !band || !band_cnt) return SNAG_ERR_ARG;
  if (use_csls && (!nv1 || !nv2)) return SNAG_ERR_ARG;
  if (!(eps > 0.f) || n1 >= (1 << 30)) return SNAG_ERR_ARG;
  if (!use_csls) { nv1 = xn; nv2 = yn; }   // never read for their values
  if ((top4_val == nullptr) != (top4_idx == nullptr)) return SNAG_ERR_ARG;
  if (top4_val && ((reinterpret_cast<uintptr_t>(top4_val) | reinterpret_cast<uintptr_t>(top4_idx)) & 15)) return SNAG_ERR_ALIGN;
  if (reinterpret_cast<uintptr_t>(band) & 7) return SNAG_ERR_ALIGN;
#define SNAG_RANKB_CASE(T3, CS)                                                                                      \
  {                                                                                                                  \
    typename EpiRankBand<T3, CS>::Params p{xn, yn, nv1, nv2, g_row, g_col, row_gid0, col_gid0, cnt_row, cnt_col,     \
                                           top4_val, top4_idx, eps, band, band_cnt, band_cap, row_gids};             \
    return launch_sim<EpiRankBand<T3, CS>>(X, Y, n1, n2, Dpad, p, st);                                               \
  }
  if (top4_val) {
    if (use_csls) SNAG_RANKB_CASE(true, true) else SNAG_RANKB_CASE(true, false)
  } else {
    if (use_csls) SNAG_RANKB_CASE(false, true) else SNAG_RANKB_CASE(false, false)
  }
#undef SNAG_RANKB_CASE
}

int launch_icl_rowsum(const __nv_bfloat16* X, const __nv_bfloat16* Y, int B, int Bp, int row0, int nx, int Dpad,
                      float inv_tau, float* rowsum_part, float* pos, cudaStream_t st) {
  if (!rowsum_part || !pos || B <= 0 || Bp < B || (Bp % BN) != 0) return SNAG_ERR_ARG;
  if (row0 < 0 || nx <= 0 || row0 + nx > Bp) return SNAG_ERR_ARG;
  EpiIclFwd::Params p{inv_tau * 1.4426950408889634f, B, Bp, row0, nx, rowsum_part, pos};
  return launch_sim<EpiIclFwd>(X, Y, nx, 2 * Bp, Dpad, p, st);
}

// launch_icl_rowsum on split stacks (rows of 5 Dpad, see snag_icl_stack_prep_split): X at a side-0 window, Y at a
// side-1 window, contraction width 3 Dpad
int launch_icl_rowsum_split(const __nv_bfloat16* X, const __nv_bfloat16* Y, int B, int Bp, int row0, int nx, int Dpad,
                            float inv_tau, float* rowsum_part, float* pos, cudaStream_t st) {
  if (!rowsum_part || !pos || B <= 0 || Bp < B || (Bp % BN) != 0 || Dpad <= 0 || (Dpad % 64) != 0) return SNAG_ERR_ARG;
  if (row0 < 0 || nx <= 0 || row0 + nx > Bp) return SNAG_ERR_ARG;
  EpiIclFwd::Params p{inv_tau * 1.4426950408889634f, B, Bp, row0, nx, rowsum_part, pos};
  return launch_sim<EpiIclFwd>(X, Y, nx, 2 * Bp, 3 * Dpad, p, st, 1, 0, 5 * Dpad);
}

int launch_eval_rowcoltopk(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, int n1, int n2,
                           int Dpad, float* part, int* part_idx, const float* rowthr, const float* colthr, const float* colb,
                           uint2* stream, int* stream_row, int* stream_cnt, int cta_cap, float norm2_max, cudaStream_t st) {
  if (!xn || !yn || !part || !part_idx || !colthr || !colb || !stream || !stream_row || !stream_cnt || cta_cap < 1)
    return SNAG_ERR_ARG;
  if (((reinterpret_cast<uintptr_t>(part) | reinterpret_cast<uintptr_t>(part_idx)) & 15) ||
      (reinterpret_cast<uintptr_t>(stream) & 7))
    return SNAG_ERR_ALIGN;
  if (!(norm2_max <= SNAG_HALF_PREFILTER_NORM2_MAX)) {
    // rows that are not (nearly) unit norm: the fp16x2 pre-filter's margins do not hold — fp32 per-element tests
    EpiRowColTopKF32::Params p{xn, yn, part, part_idx, rowthr, colthr, colb, stream, stream_row, stream_cnt, cta_cap};
    return launch_sim<EpiRowColTopKF32>(X, Y, n1, n2, Dpad, p, st);
  }
  EpiRowColTopK::Params p{xn, yn, part, part_idx, rowthr, colthr, colb, stream, stream_row, stream_cnt, cta_cap,
                          nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0};
  return launch_sim<EpiRowColTopK>(X, Y, n1, n2, Dpad, p, st);
}

int launch_eval_onepass(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, int n1, int n2,
                        int Dpad, float* part, int* part_idx, const float* rowthr, const float* colthr, const float* colb,
                        uint2* stream, int* stream_row, int* stream_cnt, int cta_cap, const float* rk_r, const float* rk_rp,
                        const float* rk_c, const float* rk_cp, uint2* rk_stream, int* rk_stream_row, int* rk_cnt, int rk_cap,
                        float norm2_max, cudaStream_t st) {
  if (!(norm2_max <= SNAG_HALF_PREFILTER_NORM2_MAX)) return SNAG_ERR_ARG;    // unit-norm rows only (see EpiRowColTopKT)
  if (!xn || !yn || !part || !part_idx || !colthr || !colb || !stream || !stream_row || !stream_cnt || cta_cap < 1 ||
      !rk_r || !rk_rp || !rk_c || !rk_cp || !rk_stream || !rk_stream_row || !rk_cnt || rk_cap < 1)
    return SNAG_ERR_ARG;
  if (((reinterpret_cast<uintptr_t>(part) | reinterpret_cast<uintptr_t>(part_idx)) & 15) ||
      ((reinterpret_cast<uintptr_t>(stream) | reinterpret_cast<uintptr_t>(rk_stream)) & 7))
    return SNAG_ERR_ALIGN;
  EpiOnePass::Params p{xn, yn, part, part_idx, rowthr, colthr, colb, stream, stream_row, stream_cnt, cta_cap,
                       rk_r, rk_rp, rk_c, rk_cp, rk_stream, rk_stream_row, rk_cnt, rk_cap};
  return launch_sim<EpiOnePass>(X, Y, n1, n2, Dpad, p, st);
}

int launch_mutual_nn(const __nv_bfloat16* X, const __nv_bfloat16* Y, const float* xn, const float* yn, int n1, int n2,
                     int Dpad, const float* colb, unsigned long long* colkey, float* row_val, int* row_idx,
                     cudaStream_t st) {
  if (!xn || !yn || !colb || !colkey || !row_val || !row_idx) return SNAG_ERR_ARG;
  if (reinterpret_cast<uintptr_t>(colkey) & 7) return SNAG_ERR_ALIGN;
  EpiMutualNN::Params p{xn, yn, colb, colkey, row_val, row_idx};
  return launch_sim<EpiMutualNN>(X, Y, n1, n2, Dpad, p, st);
}

int launch_icl_bwd_logits(const __nv_bfloat16* X, const __nv_bfloat16* Y, int B, int Bp, int row0, int nx, int Dpad,
                          float inv_tau, const float* cr, const float* cc, const float* dg, __nv_bfloat16* G,
                          int self_cols, float ebar, cudaStream_t st) {
  if (!cr || !cc || !dg || !G || B <= 0 || Bp < B || (Bp % BN) != 0) return SNAG_ERR_ARG;
  if (row0 < 0 || nx <= 0 || row0 + nx > Bp) return SNAG_ERR_ARG;
  if (reinterpret_cast<uintptr_t>(G) & 15) return SNAG_ERR_ALIGN;
  EpiIclBwd::Params p{inv_tau * 1.4426950408889634f, inv_tau, B, Bp, row0, nx, cr, cc, dg, G, self_cols, ebar};
  return launch_sim<EpiIclBwd>(X, Y, nx, 2 * Bp, Dpad, p, st);
}

// dL/dlogits on split stacks (windows as launch_icl_rowsum_split), written as G3 = [G_h | G_h | G_m] [nx, 6 Bp]
int launch_icl_bwd_logits_split(const __nv_bfloat16* X, const __nv_bfloat16* Y, int B, int Bp, int row0, int nx, int Dpad,
                                float inv_tau, const float* cr, const float* cc, const float* dg, __nv_bfloat16* G3,
                                cudaStream_t st) {
  if (!cr || !cc || !dg || !G3 || B <= 0 || Bp < B || (Bp % BN) != 0 || Dpad <= 0 || (Dpad % 64) != 0) return SNAG_ERR_ARG;
  if (row0 < 0 || nx <= 0 || row0 + nx > Bp) return SNAG_ERR_ARG;
  if (reinterpret_cast<uintptr_t>(G3) & 31) return SNAG_ERR_ALIGN;
  EpiIclBwdSplit::Params p{inv_tau * 1.4426950408889634f, inv_tau, B, Bp, row0, nx, cr, cc, dg, G3, 1, 0.f};
  return launch_sim<EpiIclBwdSplit>(X, Y, nx, 2 * Bp, 3 * Dpad, p, st, 1, 0, 5 * Dpad);
}

}  // namespace snag
