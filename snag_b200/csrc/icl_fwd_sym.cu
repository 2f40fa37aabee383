// ICL forward on HALF the Gram matrix (model/SNAG_loss.py:98-126), all tables of a step in one launch.
//
// With Z = [a ; b] (the stacked, L2-normalised, bf16 rows of both sides; each part zero padded to Bp rows) the four
// logit blocks of the reference — a.b^T, a.a^T, b.a^T, b.b^T — are the four quadrants of ONE symmetric matrix
// S = Z.Z^T, and the softmax denominators of BOTH directions are its row sums without the diagonal:
//
//   lse_a[i] = log sum_{j != i}     exp(S[i, j] / tau)         (row i of S:       [ a.a^T | a.b^T ])
//   lse_b[i] = log sum_{j != Bp+i}  exp(S[Bp + i, j] / tau)    (row Bp + i of S:  [ b.a^T | b.b^T ])
//   nll_x[i] = lse_x[i] - S[i, Bp + i] / tau
//
// The per-side sweeps (sim_kernel<EpiIclFwd>, two launches per table) execute all of S: 8 B^2 D flop per call against
// 4 algorithmic. Here only the tiles that meet the strict upper triangle are computed; an element E = exp(S[i,j]/tau -
// 1/tau), i < j, is added to the row sum of i (registers, as before) AND to the row sum of j — a column sum of the
// tile, formed per 32 x 32 strip by a butterfly transposition across the warp (31 shuffles), combined over the tile's
// four row warps in shared memory and written once per (row block, column) to a partial buffer. A bandwidth kernel
// adds the partials in a fixed order (deterministic, unlike float atomics) and takes the logarithm.
//
//   unit = (table, chunk of T column tiles of 256, block of 128 rows) over the staircase  ct >= rb / 2 ;
//   units are enumerated in closed form, chunk-major (no table in memory), dealt round-robin to one persistent CTA per SM, and a
//   contiguous range [unit_begin, unit_end) of them is a rank's share when the loss is sharded (the partial sums of the
//   ranks are then all-reduced before the logarithm).
//
// Mainloop as sim_kernel (simgemm.cuh): TMA producer warp -> 4-stage ring of (128 x 64 | 256 x 64) bf16 k-blocks,
// single-thread tcgen05.mma 128x256x16 issuer, fp32 accumulator double-buffered in TMEM, FS_WG epilogue warpgroups
// owning 256 / FS_WG columns each.
#include <cstddef>
#include <mutex>
#include "common.cuh"
#include "snag_internal.h"

namespace snag {

constexpr int FS_BM = 128;
constexpr int FS_BN = 256;
constexpr int FS_BK = 64;
constexpr int FS_STAGES = 4;
constexpr int FS_ACC = 2;
constexpr int FS_A_BYTES = FS_BM * FS_BK * 2;          // 16 KB
constexpr int FS_B_BYTES = FS_BN * FS_BK * 2;          // 32 KB
constexpr int FS_STAGE_BYTES = FS_A_BYTES + FS_B_BYTES;
#ifndef SNAG_FS_WG
#define SNAG_FS_WG 4
#endif
constexpr int FS_WG = SNAG_FS_WG;                      // epilogue warpgroups, each owning FS_BN / FS_WG columns of every tile: the
                                                       // strip body is ~7 instructions per element (exp2 + row sum + the column
                                                       // butterfly), which two warps per scheduler cannot keep flowing at D = 300
constexpr int FS_WG_COLS = FS_BN / FS_WG;
constexpr int FS_WG_STRIPS = FS_WG_COLS / 32;
constexpr int FS_EPI_THREADS = 128 * FS_WG;
constexpr int FS_THREADS = FS_EPI_THREADS + 128;
constexpr int FS_BAR_BYTES = 256;
constexpr int FS_COLACC_FLOATS = 2 /*tile parity*/ * FS_WG * 4 /*row warps*/ * FS_WG_COLS;
constexpr int FS_SMEM_BYTES = 1024 + FS_STAGES * FS_STAGE_BYTES + FS_BAR_BYTES + FS_COLACC_FLOATS * 4;
constexpr int FS_MAX_PROB = 16;

struct alignas(64) FsProblem {
  CUtensorMap tm;          // stacked operand of the table: [>= 2 Bp, Dpad] bf16, box [128 rows x 64], SWIZZLE_128B
  float* rowpart;          // [nch_max][FS_WG][2 Bp]  row sums of the row's chunks, per epilogue warpgroup
  float* colpart;          // [R][2 Bp]        column sums per (row block, column)
  float* pos;              // [Bp]             S[i, Bp + i]
  __nv_bfloat16* esave;    // [2 Bp][2 Bp] or null: E = exp(S/tau - 1/tau) of every computed element (bf16), kept for a
                           // backward that forms dL/dlogits from it instead of recomputing S (wide tables)
  long long pad_[4];
};
static_assert(sizeof(FsProblem) == 192, "FsProblem layout");

struct FsGeom {
  int B, Bp;
  int R;                   // row blocks of 128 = 2 Bp / 128
  int C;                   // column tiles of 256 = 2 Bp / 256 (row blocks 2m and 2m+1 need tiles ct >= m)
  int T;                   // column tiles per chunk
  int nch_max;             // chunks of the longest rows = ceil(C / T)
  int units_per_prob;
};
struct FsParams {
  FsGeom g;
  int n_prob, kblocks;
  int unit_begin, unit_end;    // this launch's share of the n_prob * units_per_prob units
  float scale_log2;            // log2(e) / tau
  int koff_b;                  // split stacks: column of the side-1 window (2 Dpad); fits the padding before prob
  FsProblem prob[FS_MAX_PROB];
};
static_assert(offsetof(FsParams, prob) == 64, "FsParams header");

// ---- closed-form enumeration of the staircase --------------------------------------------------
// Column tiles are cut into G = ceil(C / T) chunks of T tiles, aligned globally: chunk gch = tiles [gch T, (gch + 1) T).
// Row block rb (needs tiles ct >= rb / 2) takes part in chunk gch iff rb < 2 (gch + 1) T, with the tiles
// [max(gch T, rb / 2), (gch + 1) T) — fewer than T only on the staircase itself. Units are numbered CHUNK-MAJOR,
//   uid = prefix(gch) + rb ,   prefix(gch) = sum_{g' < gch} 2 (g' + 1) T = T gch (gch + 1)       (the last chunk has R rows)
// so that the CTAs resident at any time sweep the same column chunk (T x 256 rows of Z: L2 resident even at D = 1800)
// while each reads its own 128-row block.
__host__ __device__ inline long long fs_prefix(const FsGeom& g, int gch) {
  return static_cast<long long>(g.T) * gch * (gch + 1);
}
__host__ __device__ inline int fs_unit_of(const FsGeom& g, int rb, int ct) {
  return static_cast<int>(fs_prefix(g, ct / g.T)) + rb;
}
struct FsUnit {
  int prob, rb, chunk, ct0, ct1;
};
__device__ __forceinline__ FsUnit fs_decode(const FsGeom& g, int uid) {
  FsUnit u;
  u.prob = uid / g.units_per_prob;
  const int v = uid - u.prob * g.units_per_prob;
  int lo = 0, hi = g.nch_max - 1;              // largest chunk with prefix(chunk) <= v
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (fs_prefix(g, mid) <= v) lo = mid; else hi = mid - 1;
  }
  u.chunk = lo;
  u.rb = v - static_cast<int>(fs_prefix(g, lo));
  u.ct0 = max(lo * g.T, u.rb >> 1);
  u.ct1 = min((lo + 1) * g.T, g.C);
  return u;
}

// column sums of a 32 (rows = lanes) x 32 (columns = v[]) strip: afterwards lane l holds in v[0] the sum over the warp's
// rows of column l
__device__ __forceinline__ float fs_transpose_sum(float (&v)[32], int lane) {
#pragma unroll
  for (int k = 16; k >= 1; k >>= 1) {
    const bool up = (lane & k) != 0;
#pragma unroll
    for (int j = 0; j < k; ++j) {
      const float send = up ? v[j] : v[j + k];
      const float keep = up ? v[j + k] : v[j];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, k);
    }
  }
  return v[0];
}

// kSplit: the tables are split stacks (snag_icl_stack_prep_split, [m | h | h | m | h] rows of 5 Dpad): the A rows of a
// tile are read from the side-0 window (columns [0, 3 Dpad)) and the B rows from the side-1 window (columns
// [2 Dpad, 5 Dpad), p.koff_b further), so every element is m_i h_j + h_i m_j + h_i h_j — symmetric in (i, j), like the
// bf16 Gram matrix, so the staircase, both sums and pos are unchanged. No E is saved (bf16 E would cap dL/dlogits at
// 2^-9 relative).
template <bool kSplit>
__device__ __forceinline__ void icl_fwd_sym_body(const FsParams& p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);
  const uint32_t bar0 = base + FS_STAGES * FS_STAGE_BYTES;
  auto full_bar = [&](uint32_t s) { return bar0 + 8u * s; };
  auto empty_bar = [&](uint32_t s) { return bar0 + 8u * (FS_STAGES + s); };
  auto tfull_bar = [&](uint32_t a) { return bar0 + 8u * (2 * FS_STAGES + a); };
  auto tempty_bar = [&](uint32_t a) { return bar0 + 8u * (2 * FS_STAGES + FS_ACC + a); };
  const uint32_t tmem_slot = bar0 + 8u * (2 * FS_STAGES + 2 * FS_ACC);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem + FS_STAGES * FS_STAGE_BYTES + 8 * (2 * FS_STAGES + 2 * FS_ACC));
  float* colacc = reinterpret_cast<float*>(smem + FS_STAGES * FS_STAGE_BYTES + FS_BAR_BYTES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cwarp = warp - FS_EPI_THREADS / 32;      // 0 = TMA producer, 1 = UMMA issuer, 2 = TMEM allocator; < 0: epilogue
  const FsGeom& g = p.g;

  if (cwarp == 1 && lane == 0) {
    for (int s = 0; s < FS_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < FS_ACC; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), FS_EPI_THREADS);
    }
    fence_mbar_init();
  }
  if (cwarp == 2) tmem_alloc(tmem_slot, FS_ACC * FS_BN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  const int u_first = p.unit_begin + blockIdx.x;

  if (cwarp == 0) {
    // ------------------------------------------------------------------ TMA producer
    const uint32_t leader = elect_one_sync();
    uint32_t stage = 0, phase = 0;
    for (int uid = u_first; uid < p.unit_end; uid += gridDim.x) {
      const FsUnit u = fs_decode(g, uid);
      const CUtensorMap* tm = &p.prob[u.prob].tm;
      for (int ct = u.ct0; ct < u.ct1; ++ct) {
        for (int kb = 0; kb < p.kblocks; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1);
          if (leader) {
            mbar_expect_tx(full_bar(stage), FS_STAGE_BYTES);
            const uint32_t sa = base + stage * FS_STAGE_BYTES;
            tma_load_2d(sa, tm, full_bar(stage), kb * FS_BK, u.rb * FS_BM);
            const int kb_b = kb * FS_BK + (kSplit ? p.koff_b : 0);
            tma_load_2d(sa + FS_A_BYTES, tm, full_bar(stage), kb_b, ct * FS_BN);
            tma_load_2d(sa + FS_A_BYTES + FS_A_BYTES, tm, full_bar(stage), kb_b, ct * FS_BN + FS_BM);
          }
          __syncwarp();
          if (++stage == FS_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (cwarp == 1) {
    // ------------------------------------------------------------------ UMMA issuer
    const uint32_t leader = elect_one_sync();
    const uint64_t adesc0 = make_sdesc_k128(base);
    const uint64_t bdesc0 = make_sdesc_k128(base + FS_A_BYTES);
    const uint32_t idesc = make_idesc_bf16(FS_BM, FS_BN);
    uint32_t stage = 0, phase = 0, as = 0, aphase = 0;
    for (int uid = u_first; uid < p.unit_end; uid += gridDim.x) {
      const FsUnit u = fs_decode(g, uid);
      for (int ct = u.ct0; ct < u.ct1; ++ct) {
        mbar_wait(tempty_bar(as), aphase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * FS_BN;
        uint32_t accumulate = 0;
        for (int kb = 0; kb < p.kblocks; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          if (leader) {
            const uint64_t adesc = adesc0 + static_cast<uint64_t>(stage * (FS_STAGE_BYTES >> 4));
            const uint64_t bdesc = bdesc0 + static_cast<uint64_t>(stage * (FS_STAGE_BYTES >> 4));
            umma_bf16_ss(tmem_d, adesc, bdesc, idesc, accumulate);
            umma_bf16_ss(tmem_d, adesc + 2u, bdesc + 2u, idesc, 1u);
            umma_bf16_ss(tmem_d, adesc + 4u, bdesc + 4u, idesc, 1u);
            umma_bf16_ss(tmem_d, adesc + 6u, bdesc + 6u, idesc, 1u);
            umma_commit(empty_bar(stage));
          }
          __syncwarp();
          accumulate = 1;
          if (++stage == FS_STAGES) { stage = 0; phase ^= 1; }
        }
        if (leader) umma_commit(tfull_bar(as));
        __syncwarp();
        if (++as == FS_ACC) { as = 0; aphase ^= 1; }
      }
    }
  } else if (cwarp < 0) {
    // ------------------------------------------------------------------ epilogue warpgroups
    const int tid = threadIdx.x;
    const int et = tid & 127;                          // row within the block == TMEM lane
    const int wg = tid >> 7;                           // which FS_WG_COLS of the tile's 256 columns
    const int wq = (tid >> 5) & 3;                     // row warp within the warpgroup
    const uint32_t lane_base = static_cast<uint32_t>((warp & 3) * 32) << 16;
    const float nb = -p.scale_log2;
    const int twoBp = 2 * g.Bp;
    uint32_t as = 0, aphase = 0, tile_seq = 0;
    for (int uid = u_first; uid < p.unit_end; uid += gridDim.x) {
      const FsUnit u = fs_decode(g, uid);
      const FsProblem& pr = p.prob[u.prob];
      const int i = u.rb * FS_BM + et;                 // row of S
      const int part_i = i >= g.Bp ? 1 : 0;
      const int idx_i = i - part_i * g.Bp;
      const bool row_ok = idx_i < g.B;
      const int w0 = u.rb * FS_BM + wq * 32 - part_i * g.Bp;       // batch index of the warp's first row
      const bool rows_all_ok = (u.rb * FS_BM - part_i * g.Bp) + FS_BM <= g.B;
      float sum = 0.f;
      for (int ct = u.ct0; ct < u.ct1; ++ct, ++tile_seq) {
        float* acc_s = colacc + ((tile_seq & 1) * FS_WG + wg) * 4 * FS_WG_COLS;
        mbar_wait(tfull_bar(as), aphase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + lane_base + as * FS_BN;
        const bool above = ct * FS_BN >= (u.rb + 1) * FS_BM;       // every column of the tile lies right of every row
#pragma unroll 1
        for (int s = 0; s < FS_WG_STRIPS; ++s) {
          const int c = wg * FS_WG_STRIPS + s;
          uint32_t r[32];
          SNAG_TMEM_LD32(taddr + c * 32, r);
          SNAG_TMEM_WAIT32(r);
          const int col0 = ct * FS_BN + c * 32;
          const int part_j = col0 >= g.Bp ? 1 : 0;
          const int idxj0 = col0 - part_j * g.Bp;
          float e[32];
          if (idxj0 >= g.B) {                           // strip entirely in the padding (warp-uniform)
            acc_s[wq * FS_WG_COLS + s * 32 + lane] = 0.f;
            continue;
          }
          // the strip may hold the positive logit S[i, Bp + i] of one of this warp's rows
          const bool has_pos = part_i == 0 && part_j == 1 && idxj0 < w0 + 32 && w0 < idxj0 + 32;
          const bool plain = above && rows_all_ok && (idxj0 + 32 <= g.B) && !has_pos;
          if (plain) {
            float a = 0.f;
#pragma unroll
            for (int q = 0; q < 32; ++q) {
              e[q] = ex2_approx(__fmaf_rn(__uint_as_float(r[q]), p.scale_log2, nb));
              a += e[q];
            }
            sum += a;
          } else {
#pragma unroll
            for (int q = 0; q < 32; ++q) {
              const int j = col0 + q;
              const float sv = __uint_as_float(r[q]);
              const bool ok = row_ok && (idxj0 + q < g.B) && (j > i);
              e[q] = ok ? ex2_approx(__fmaf_rn(sv, p.scale_log2, nb)) : 0.f;
              sum += e[q];
              if (has_pos && row_ok && j == i + g.Bp) pr.pos[idx_i] = sv;
            }
          }
          if (!kSplit && pr.esave != nullptr) {
            uint32_t pk[16];
#pragma unroll
            for (int q = 0; q < 32; q += 2) {
              const __nv_bfloat162 h2 = __floats2bfloat162_rn(e[q], e[q + 1]);
              pk[q >> 1] = *reinterpret_cast<const uint32_t*>(&h2);
            }
            uint8_t* dst = reinterpret_cast<uint8_t*>(pr.esave + static_cast<long long>(i) * twoBp + col0);
            st_global_256(dst, make_uint4(pk[0], pk[1], pk[2], pk[3]), make_uint4(pk[4], pk[5], pk[6], pk[7]));
            st_global_256(dst + 32, make_uint4(pk[8], pk[9], pk[10], pk[11]), make_uint4(pk[12], pk[13], pk[14], pk[15]));
          }
          acc_s[wq * FS_WG_COLS + s * 32 + lane] = fs_transpose_sum(e, lane);
        }
        tc_fence_before();
        mbar_arrive(tempty_bar(as));                    // accumulator stage drained
        if (++as == FS_ACC) { as = 0; aphase ^= 1; }
        // combine the four row warps' column sums (fixed order) and write them once per (row block, column)
        named_bar_sync(1 + wg, 128);
        if (et < FS_WG_COLS) {
          const float tot = (acc_s[et] + acc_s[FS_WG_COLS + et]) + (acc_s[2 * FS_WG_COLS + et] + acc_s[3 * FS_WG_COLS + et]);
          pr.colpart[static_cast<long long>(u.rb) * twoBp + ct * FS_BN + wg * FS_WG_COLS + et] = tot;
        }
      }
      // this warpgroup's share of the row sums of the chunk: the two warpgroups own different columns
      pr.rowpart[(static_cast<long long>(u.chunk) * FS_WG + wg) * twoBp + i] = sum;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (cwarp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, FS_ACC * FS_BN);
  }
}

__global__ void __launch_bounds__(FS_THREADS, 1) icl_fwd_sym_kernel(const __grid_constant__ FsParams p) {
  icl_fwd_sym_body<false>(p);
}
__global__ void __launch_bounds__(FS_THREADS, 1) icl_fwd_sym_split_kernel(const __grid_constant__ FsParams p) {
  icl_fwd_sym_body<true>(p);
}

// total[prob][r] = sum of the row partials of r's chunks + sum of the column partials of the row blocks whose tile
// (rb', ct(r)) was computed, in a fixed order; only partials produced by units in [unit_begin, unit_end) are read
struct FsTotalArgs {
  const float* rowpart[FS_MAX_PROB];
  const float* colpart[FS_MAX_PROB];
};
__global__ void __launch_bounds__(256) icl_sym_total_kernel(const FsTotalArgs a, const FsGeom g, int unit_begin, int unit_end,
                                                            float* __restrict__ total) {
  const int prob = blockIdx.y;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const int twoBp = 2 * g.Bp;
  if (r >= twoBp) return;
  const int ubase = prob * g.units_per_prob;
  const int rb = r / FS_BM;
  float tot = 0.f;
  for (int c = (rb >> 1) / g.T; c < g.nch_max; ++c) {          // the chunks row block rb takes part in
    const int uu = ubase + static_cast<int>(fs_prefix(g, c)) + rb;
    if (uu >= unit_begin && uu < unit_end)
      for (int w = 0; w < FS_WG; ++w) tot += a.rowpart[prob][(static_cast<long long>(c) * FS_WG + w) * twoBp + r];
  }
  const int ct = r / FS_BN;
  const int rb_hi = min(g.R - 1, 2 * ct + 1);
  for (int rbp = 0; rbp <= rb_hi; ++rbp) {
    const int uu = ubase + fs_unit_of(g, rbp, ct);
    if (uu >= unit_begin && uu < unit_end) tot += a.colpart[prob][static_cast<long long>(rbp) * twoBp + r];
  }
  total[static_cast<long long>(prob) * twoBp + r] = tot;
}
// out[prob][0..3][i] = lse_a, nll_a, lse_b, nll_b of anchor i (model/SNAG_loss.py:120-126 per row)
__global__ void __launch_bounds__(256) icl_sym_finalize_kernel(const float* __restrict__ total, const float* __restrict__ pos,
                                                               int B, int Bp, float inv_tau, float* __restrict__ out) {
  const int prob = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const float* t = total + static_cast<long long>(prob) * 2 * Bp;
  const float ps = pos[static_cast<long long>(prob) * Bp + i] * inv_tau;
  const float la = logf(t[i]) + inv_tau, lb = logf(t[Bp + i]) + inv_tau;
  float* o = out + static_cast<long long>(prob) * 4 * B;
  o[i] = la;
  o[B + i] = la - ps;
  o[2 * B + i] = lb;
  o[3 * B + i] = lb - ps;
}

// ------------------------------------------------------------------------------------------------ host side
int make_operand_map(CUtensorMap* m, const __nv_bfloat16* ptr, long long rows, int Dpad, int box_rows);   // sim_kernels.cu

static int fs_geometry(int n_prob, int B, int Bp, FsGeom* g) {
  if (n_prob < 1 || n_prob > FS_MAX_PROB || B <= 0 || Bp < B || (Bp % 256) != 0) return SNAG_ERR_ARG;
  g->B = B;
  g->Bp = Bp;
  g->R = 2 * Bp / FS_BM;
  g->C = 2 * Bp / FS_BN;
  // chunk length: long enough to amortise a unit's row-state flush and pipeline fill, short enough that every CTA gets
  // >= ~12 units (the units of a launch differ in length only in their last chunk)
  const long long tiles = static_cast<long long>(n_prob) * (static_cast<long long>(g->C) * g->C + g->C);
  long long T = tiles / (12ll * num_sms());
  if (T > 16) T = 16;
  if (T < 2) T = 2;
  if (T > g->C) T = g->C;
  g->T = static_cast<int>(T);
  g->nch_max = (g->C + g->T - 1) / g->T;
  const long long upp = fs_prefix(*g, g->nch_max - 1) + g->R;      // the last chunk is met by every row block
  if (upp * n_prob > 0x7fffffffll) return SNAG_ERR_SHAPE;
  g->units_per_prob = static_cast<int>(upp);
  return SNAG_OK;
}

// sizes a caller needs: out[0] = units in total, out[1] = floats of rowpart per table, out[2] = floats of colpart per table
int icl_fwd_sym_plan(int n_prob, int B, int Bp, long long* out) {
  FsGeom g;
  const int rc = fs_geometry(n_prob, B, Bp, &g);
  if (rc) return rc;
  out[0] = static_cast<long long>(g.units_per_prob) * n_prob;
  out[1] = static_cast<long long>(FS_WG) * g.nch_max * 2 * Bp;
  out[2] = static_cast<long long>(g.R) * 2 * Bp;
  return SNAG_OK;
}

int launch_icl_fwd_sym(int n_prob, const __nv_bfloat16* const* S3, float* const* rowpart, float* const* colpart, float* pos,
                       int B, int Bp, int Dpad, float inv_tau, int unit_begin, int unit_end, float* total,
                       __nv_bfloat16* const* esave, cudaStream_t st, int split) {
  if (!S3 || !rowpart || !colpart || !pos || !total) return SNAG_ERR_ARG;
  if (split && esave) return SNAG_ERR_ARG;
  if (Dpad <= 0 || (Dpad % FS_BK) != 0) return SNAG_ERR_SHAPE;
  if (!device_is_sm100()) return SNAG_ERR_DEVICE;
  FsParams p{};
  int rc = fs_geometry(n_prob, B, Bp, &p.g);
  if (rc) return rc;
  const int n_units = p.g.units_per_prob * n_prob;
  if (unit_begin < 0 || unit_end > n_units || unit_begin > unit_end) return SNAG_ERR_ARG;
  p.n_prob = n_prob;
  p.kblocks = (split ? 3 : 1) * Dpad / FS_BK;
  p.koff_b = split ? 2 * Dpad : 0;
  p.unit_begin = unit_begin;
  p.unit_end = unit_end;
  p.scale_log2 = inv_tau * 1.4426950408889634f;
  FsTotalArgs ta{};
  for (int i = 0; i < n_prob; ++i) {
    if (!S3[i] || !rowpart[i] || !colpart[i]) return SNAG_ERR_ARG;
    if ((rc = make_operand_map(&p.prob[i].tm, S3[i], 2ll * Bp, (split ? 5 : 1) * Dpad, FS_BM))) return rc;
    p.prob[i].rowpart = rowpart[i];
    p.prob[i].colpart = colpart[i];
    p.prob[i].pos = pos + static_cast<long long>(i) * Bp;
    p.prob[i].esave = esave ? esave[i] : nullptr;
    if (p.prob[i].esave && (reinterpret_cast<uintptr_t>(p.prob[i].esave) & 31)) return SNAG_ERR_ALIGN;
    ta.rowpart[i] = rowpart[i];
    ta.colpart[i] = colpart[i];
  }
  if (unit_end > unit_begin) {
    auto* kern = split ? icl_fwd_sym_split_kernel : icl_fwd_sym_kernel;
    const cudaError_t attr_err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, FS_SMEM_BYTES);
    if (attr_err != cudaSuccess) return static_cast<int>(attr_err);
    const int span = unit_end - unit_begin;
    const int grid = span < num_sms() ? span : num_sms();
    kern<<<grid, FS_THREADS, FS_SMEM_BYTES, st>>>(p);
  }
  icl_sym_total_kernel<<<dim3((2 * Bp + 255) / 256, n_prob), 256, 0, st>>>(ta, p.g, unit_begin, unit_end, total);
  return static_cast<int>(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------
// dL/dlogits of one side from the saved E (instead of recomputing the logits): the bandwidth-bound replacement of
// sim_kernel<EpiIclBwd> for tables too wide for the fused backward. With zi = side Bp + i the anchor's row of
// Z = [a ; b] and zj the column's row (part 0 = the other side, part 1 = this side), E[zi, zj] was stored at
// esave[min][max] by the half-Gram forward; a 64 x 64 tile is staged in shared memory and read straight, transposed
// or — on the diagonal — folded. Same formula as EpiIclBwd:
//   part 0: G[i,j] = ((cr_i + cc_j) E - [i == j] dg_i) / tau     part 1: G[i,j] = (cr_i + cr_j) E / tau, 0 on the diagonal
// The cross diagonal (the positive pair) is a small difference of large terms — g (P_ii - 1) / tau with P_ii close to 1 —
// that the bf16 rounding of E would swamp: the caller passes it ready-made, from the fp32 NLL of the forward,
//   diag_i = (g_a[i] expm1(-nll_a[i]) + g_b[i] expm1(-nll_b[i])) / tau .
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) icl_g_from_e_kernel(const __nv_bfloat16* __restrict__ E, int side, int B, int Bp,
                                                           const float* __restrict__ cr_this, const float* __restrict__ cr_other,
                                                           const float* __restrict__ diag, float inv_tau,
                                                           __nv_bfloat16* __restrict__ G) {
  __shared__ float tile[64][65];
  const int twoBp = 2 * Bp;
  const int i0 = blockIdx.y * 64;                    // anchors of the tile (batch index)
  const int c0 = blockIdx.x * 64;                    // output columns of G
  const int part = c0 >= Bp ? 1 : 0;
  const int j0 = c0 - part * Bp;                     // batch index of the first column
  const int zr0 = side * Bp + i0;                    // rows / columns of Z
  const int zc0 = (part == 0 ? (1 - side) : side) * Bp + j0;
  const bool any = i0 < B && j0 < B;
  const int cg = threadIdx.x & 7;                    // 8 groups of 8 consecutive columns: 16-byte loads and stores
  const int r0 = threadIdx.x >> 3;                   // 32 rows per pass
  if (any) {
    const int R0 = min(zr0, zc0), C0 = max(zr0, zc0);
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int r = r0 + 32 * pass;
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(E + static_cast<long long>(R0 + r) * twoBp + C0 + cg * 8));
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        tile[r][cg * 8 + 2 * k] = __uint_as_float(w[k] << 16);
        tile[r][cg * 8 + 2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
      }
    }
  }
  __syncthreads();
  const float* ccp = part ? cr_this : cr_other;
  float cc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int j = j0 + cg * 8 + k;
    cc[k] = (any && j < B) ? __ldg(ccp + j) * inv_tau : 0.f;
  }
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    const int r = r0 + 32 * pass;
    const int i = i0 + r;
    const bool row_ok = any && i < B;
    const float cri = row_ok ? __ldg(cr_this + i) * inv_tau : 0.f;
    uint32_t pk[4];
#pragma unroll
    for (int k = 0; k < 8; k += 2) {
      float gv[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c = cg * 8 + k + h;
        const int j = j0 + c;
        float v = 0.f;
        if (row_ok && j < B) {
          const float e = zc0 > zr0 ? tile[r][c] : (zc0 < zr0 ? tile[c][r] : tile[min(r, c)][max(r, c)]);
          v = (cri + cc[k + h]) * e;
          if (i == j) v = part ? 0.f : __ldg(diag + i);
        }
        gv[h] = v;
      }
      const __nv_bfloat162 h2 = __floats2bfloat162_rn(gv[0], gv[1]);
      pk[k >> 1] = *reinterpret_cast<const uint32_t*>(&h2);
    }
    *reinterpret_cast<uint4*>(G + static_cast<long long>(i) * twoBp + c0 + cg * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
}

int launch_icl_g_from_e(const __nv_bfloat16* E, int side, int B, int Bp, const float* cr_this, const float* cr_other,
                        const float* diag, float inv_tau, __nv_bfloat16* G, cudaStream_t st) {
  if (!E || !cr_this || !cr_other || !diag || !G || B <= 0 || Bp < B || (Bp % 256) != 0 || (side != 0 && side != 1))
    return SNAG_ERR_ARG;
  icl_g_from_e_kernel<<<dim3(2 * Bp / 64, Bp / 64), 256, 0, st>>>(E, side, B, Bp, cr_this, cr_other, diag, inv_tau, G);
  return static_cast<int>(cudaGetLastError());
}

int launch_icl_sym_finalize(const float* total, const float* pos, int n_prob, int B, int Bp, float inv_tau, float* out,
                            cudaStream_t st) {
  if (!total || !pos || !out || n_prob < 1 || B <= 0 || Bp < B) return SNAG_ERR_ARG;
  icl_sym_finalize_kernel<<<dim3((B + 255) / 256, n_prob), 256, 0, st>>>(total, pos, B, Bp, inv_tau, out);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace snag
