// Persistent, warp-specialised similarity contraction  S = X · Yᵀ  (bf16 in, fp32 accumulate in TMEM)
// with the consumer of S fused into the epilogue, so S never reaches HBM.
//
//   warps 0..7  epilogue       : two warpgroups (SNAG_EPI_WG), each owning half of the tile's columns; tcgen05.ld 32 lanes x
//                                32 columns at a time, thread <-> one row of the tile (TMEM lane = 32*(warp%4)+lane)
//   warp 8      TMA producer   : X tile [128 x 64] + Y tile [256 x 64] per k-block -> 4-stage smem ring
//   warp 9      UMMA issuer    : tcgen05.mma 128x256x16, 4 per k-block, accumulator double-buffered in TMEM
//   warp 10     TMEM allocator : 512 columns (2 accumulator stages x 256 fp32 columns)
//
// Work decomposition: a *unit* is (row block of 128 sources) x (chunk of `tiles_per_chunk` column tiles);
// per-row epilogue state (top-k list, rank counter, softmax row sum) lives in registers for the whole
// unit and is flushed once at the end. Units are ordered chunk-major so that the CTAs resident at any
// time sweep the same Y chunk (sized to stay L2 resident) while each re-reads its own X row block.
#pragma once
#include <type_traits>
#include <utility>
#include "common.cuh"

namespace snag {

constexpr int BM = 128;           // rows per tile  (UMMA M)
constexpr int BN = 256;           // columns per tile (UMMA N)
constexpr int BK = 64;            // bf16 per k-block = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int STAGES = 4;
constexpr int A_STAGE_BYTES = BM * BK * 2;   // 16 KB
constexpr int B_STAGE_BYTES = BN * BK * 2;   // 32 KB
constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
constexpr int ACC_STAGES = 2;
constexpr int TMEM_COLS = ACC_STAGES * BN;   // 512
constexpr int NUM_CTRL_THREADS = 128;
#ifndef SNAG_EPI_WG
#define SNAG_EPI_WG 2
#endif
constexpr int NUM_EPI_WG = SNAG_EPI_WG;       // epilogue warpgroups; WG w owns BN/NUM_EPI_WG consecutive columns of every tile
constexpr int NUM_EPI_THREADS = 128 * NUM_EPI_WG;
constexpr int NUM_THREADS = NUM_CTRL_THREADS + NUM_EPI_THREADS;
constexpr int STRIPS_PER_WG = BN / 32 / NUM_EPI_WG;
constexpr int EPI_VEC_FLOATS = 3584;      // per-tile column vectors (double-buffered): 14 KB
constexpr int EPI_STAGE_VALS = 4096 / NUM_EPI_THREADS;   // accumulators one thread can park at a time (16 KB in total)
constexpr int EPI_STAGE_FLOATS = NUM_EPI_THREADS * EPI_STAGE_VALS;
constexpr int EPI_SCRATCH_BYTES = (EPI_VEC_FLOATS + EPI_STAGE_FLOATS) * 4;
constexpr int BAR_BYTES = 256;
constexpr int SIM_SMEM_BYTES = 1024 /*align slack*/ + STAGES * STAGE_BYTES + BAR_BYTES + EPI_SCRATCH_BYTES;
constexpr int KT = 16;            // per-row candidate list length kept by the top-k epilogue (k <= KT)

struct SimShape {
  int n_rows;           // valid rows of the X view
  int n_cols;           // valid rows of the Y view (= columns of S)
  int kblocks;          // Dpad / 64
  int row_blocks;       // ceil(n_rows / 128)
  int col_tiles;        // ceil(n_cols / 256)
  int tiles_per_chunk;
  int n_chunks;         // ceil(col_tiles / tiles_per_chunk)
  int n_units;          // row_blocks * n_chunks
  int ksplits;          // split-K factor (1 for every epilogue that needs complete dot products); unit ids run over
  int kb_split;         // [0, n_units * ksplits): split = id / n_units owns k-blocks [split*kb_split, +kb_split)
  int a_mn;             // 1: the X operand is given TRANSPOSED — tmX maps a [K rows, n_rows columns] matrix (box 64 x 64) and
                        // the A tile is read MN-major (the gradient GEMMs contract over the rows of the stacked embeddings,
                        // which are stored with the output dimension contiguous; no transposed copy is made)
  unsigned long long* dbg;   // optional [4*gridDim.x][4] cycle counters (zeroed by the caller) or null. Row cta: UMMA issuer
                             // total, its wait for a free accumulator stage, sum over epilogue warps of strip time,
                             // tiles. Row gridDim.x + cta: sum over epilogue warps of commit + barrier time, then the
                             // fused evaluation epilogues' flag counters; rows 2*gridDim.x.. : EpiRowColTopKT's per-test
                             // counters.
};

struct EpiCtx {
  int et;        // row within the tile == TMEM lane (0..127)
  int wg;        // epilogue warpgroup (0..NUM_EPI_WG-1): which half of the tile's columns this thread consumes
  int tid;       // epilogue thread id 0..NUM_EPI_THREADS-1
  int list;      // index of this thread's partial output list: chunk * NUM_EPI_WG + wg
  int lane;      // lane in warp
  int row;       // row index inside the X view
  bool row_ok;   // row < n_rows
  int rb, chunk; // unit coordinates
  int split;     // split-K slice of the unit (0 when ksplits == 1)
  int useq;      // sequence number of the unit within this CTA (parity selects double-buffered per-unit scratch)
  float* scratch;  // EPI_SCRATCH_BYTES of shared memory private to the epilogue warpgroup
  uint32_t taddr;  // TMEM address of the strip handed to Epi::chunk (this warp's lanes, first of its 32 columns)
};

// Control warps (TMA producer, UMMA issuer): by default the whole warp walks the loop and one elected lane issues
// (convergent code, uniform datapath). SNAG_CTRL_CONVERGED=0 builds the single-lane form for A/B measurements.
// SNAG_PIPE_LD=1: software-pipelined TMEM read-out in the epilogue strip loop (A/B: scripts/build_variants.sh)
// SNAG_OPX: development bisect switches of the one-pass epilogue (bit 0: no rank terms in the fast path, bit 1: l2r term
// only, bit 2: no rank test / append in the slow path); 0 in the product build
#ifndef SNAG_OPX
#define SNAG_OPX 0
#endif
#ifndef SNAG_PIPE_LD
#define SNAG_PIPE_LD 0
#endif
#ifndef SNAG_CTRL_CONVERGED
#define SNAG_CTRL_CONVERGED 1
#endif
#if SNAG_CTRL_CONVERGED
#define SNAG_CTRL_ENTER true
#define SNAG_CTRL_LEADER elect_one_sync()
#define SNAG_CTRL_SYNC() __syncwarp()
#else
#define SNAG_CTRL_ENTER (lane == 0)
#define SNAG_CTRL_LEADER 1u
#define SNAG_CTRL_SYNC()
#endif

// number of 32-column strips of column tile ct that contain valid columns (BN/32 for every tile but a ragged last one)
__device__ __forceinline__ int tile_strips(const SimShape& shp, int ct) {
  return min(BN, shp.n_cols - ct * BN + 31) >> 5;
}

// registers carrying one column's prefetched per-tile values from tile_prefetch to tile_commit
struct EpiPre {
  float a, b, c, d, e;
};

// number of epilogue warpgroups of a kernel instantiation: Epi::kWG when the epilogue asks for its own count (a
// latency-bound epilogue with no per-row state wants more warps), else the build-wide NUM_EPI_WG
template <class E, class = void>
struct EpiWG { static constexpr int value = NUM_EPI_WG; };
template <class E>
struct EpiWG<E, std::void_t<decltype(E::kWG)>> { static constexpr int value = E::kWG; };

// optional per-CTA hook run by the epilogue threads after their last unit: Epi::kernel_end(params, shape, ctx)
template <class E, class = void>
struct HasKernelEnd : std::false_type {};
template <class E>
struct HasKernelEnd<E, decltype(E::kernel_end(std::declval<const typename E::Params&>(), std::declval<const SimShape&>(),
                                              std::declval<const EpiCtx&>()), void())>
    : std::true_type {};

template <class Epi>
__global__ void __launch_bounds__(NUM_CTRL_THREADS + 128 * EpiWG<Epi>::value, 1)
sim_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmY, const SimShape shp,
           const typename Epi::Params ep) {
  constexpr int kWG = EpiWG<Epi>::value;              // epilogue warpgroups of this instantiation
  constexpr int kEpiThreads = 128 * kWG;
  constexpr int kStripsPerWG = BN / 32 / kWG;
  static_assert(BN % (32 * kWG) == 0 && kEpiThreads >= BN, "epilogue warpgroup count");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw_addr);

  const uint32_t bar0 = base + STAGES * STAGE_BYTES;
  auto full_bar = [&](uint32_t s) { return bar0 + 8u * s; };
  auto empty_bar = [&](uint32_t s) { return bar0 + 8u * (STAGES + s); };
  auto tfull_bar = [&](uint32_t a) { return bar0 + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](uint32_t a) { return bar0 + 8u * (2 * STAGES + ACC_STAGES + a); };
  const uint32_t tmem_slot = bar0 + 8u * (2 * STAGES + 2 * ACC_STAGES);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + STAGES * STAGE_BYTES +
                                                                           8 * (2 * STAGES + 2 * ACC_STAGES));
  float* scratch = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES + BAR_BYTES);

  // Warp roles. The epilogue warps come FIRST and the control warps LAST on purpose: the SM's warp arbiter favours
  // the highest warp id among eligible warps, so the single-thread TMA producer and UMMA issuer must not sit below
  // 8-16 busy epilogue warps or their (few, latency-critical) instructions wait behind the epilogue's.
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cwarp = warp - kEpiThreads / 32;         // 0 = TMA producer, 1 = UMMA issuer, 2 = TMEM allocator; < 0: epilogue

  if (cwarp == 0 && lane == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmY);
  }
  if (cwarp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < ACC_STAGES; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), kEpiThreads);
    }
    fence_mbar_init();
  }
  if (cwarp == 2) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (cwarp == 0) {
    // ------------------------------------------------------------------ TMA producer
    // The whole warp walks the loop (so the code is convergent and stays on the uniform datapath); one elected
    // lane arms the barrier and issues the two bulk-tensor copies. Kept as short as possible: under a busy
    // epilogue every instruction of this warp waits for an issue slot.
    const uint32_t leader = SNAG_CTRL_LEADER;
    uint32_t stage = 0, phase = 0;
    for (int uid = blockIdx.x; SNAG_CTRL_ENTER && uid < shp.n_units * shp.ksplits; uid += gridDim.x) {
      const int u = uid % shp.n_units, split = uid / shp.n_units;
      const int rb = u % shp.row_blocks, ch = u / shp.row_blocks;
      const int ct0 = ch * shp.tiles_per_chunk;
      const int ct1 = min(ct0 + shp.tiles_per_chunk, shp.col_tiles);
      const int kb0 = split * shp.kb_split, kb1 = min(kb0 + shp.kb_split, shp.kblocks);
      for (int ct = ct0; ct < ct1; ++ct) {
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1);
          if (leader) {
            mbar_expect_tx(full_bar(stage), STAGE_BYTES);
            const uint32_t sa = base + stage * STAGE_BYTES;
            if (shp.a_mn) {          // two [64 k-rows x 64 output columns] boxes: MN-major atoms, 8 KB apart along M
              tma_load_2d(sa, &tmX, full_bar(stage), rb * BM, kb * BK);
              tma_load_2d(sa + A_STAGE_BYTES / 2, &tmX, full_bar(stage), rb * BM + 64, kb * BK);
            } else {
              tma_load_2d(sa, &tmX, full_bar(stage), kb * BK, rb * BM);
            }
            tma_load_2d(sa + A_STAGE_BYTES, &tmY, full_bar(stage), kb * BK, ct * BN);
          }
          SNAG_CTRL_SYNC();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (cwarp == 1) {
    // ------------------------------------------------------------------ UMMA issuer (same structure)
    const uint32_t leader = SNAG_CTRL_LEADER;
    // K-major A: +2 descriptor units (32 B) per 16-element K step; MN-major A: 16 k-rows = two 8-row groups = 2048 B
    const uint64_t adesc0 = shp.a_mn ? make_sdesc_mn128(base, A_STAGE_BYTES / 2) : make_sdesc_k128(base);
    const uint64_t a_kstep = shp.a_mn ? (2048u >> 4) : 2u;
    const uint32_t a_major = shp.a_mn ? (1u << 15) : 0u;
    const uint64_t bdesc0 = make_sdesc_k128(base + A_STAGE_BYTES);
    uint32_t stage = 0, phase = 0, as = 0, aphase = 0;
    const bool dbg = shp.dbg != nullptr;
    long long w_acc = 0, n_tiles = 0;
    const long long t_begin = dbg ? clock64() : 0;
    for (int uid = blockIdx.x; SNAG_CTRL_ENTER && uid < shp.n_units * shp.ksplits; uid += gridDim.x) {
      const int u = uid % shp.n_units, split = uid / shp.n_units;
      const int ch = u / shp.row_blocks;
      const int ct0 = ch * shp.tiles_per_chunk;
      const int ct1 = min(ct0 + shp.tiles_per_chunk, shp.col_tiles);
      const int n_kb = min(split * shp.kb_split + shp.kb_split, shp.kblocks) - split * shp.kb_split;
      for (int ct = ct0; ct < ct1; ++ct) {
        const long long tw = dbg ? clock64() : 0;
        mbar_wait(tempty_bar(as), aphase ^ 1);     // epilogue has drained this accumulator stage
        if (dbg) { w_acc += clock64() - tw; ++n_tiles; }
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * BN;
        // ragged last column tile: only the 32-column strips that hold valid columns are computed (UMMA N = 32..256);
        // the epilogue skips the others
        const uint32_t idesc = make_idesc_bf16(BM, tile_strips(shp, ct) * 32) | a_major;
        uint32_t accumulate = 0;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          if (leader) {
            // stage s starts (STAGE_BYTES >> 4) descriptor units after stage 0; +2 units (32 B) per 16-element K step
            const uint64_t adesc = adesc0 + static_cast<uint64_t>(stage * (STAGE_BYTES >> 4));
            const uint64_t bdesc = bdesc0 + static_cast<uint64_t>(stage * (STAGE_BYTES >> 4));
            umma_bf16_ss(tmem_d, adesc, bdesc, idesc, accumulate);
            umma_bf16_ss(tmem_d, adesc + a_kstep, bdesc + 2u, idesc, 1u);
            umma_bf16_ss(tmem_d, adesc + 2u * a_kstep, bdesc + 4u, idesc, 1u);
            umma_bf16_ss(tmem_d, adesc + 3u * a_kstep, bdesc + 6u, idesc, 1u);
            umma_commit(empty_bar(stage));           // smem slot free once these MMAs retire
          }
          SNAG_CTRL_SYNC();
          accumulate = 1;
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (leader) umma_commit(tfull_bar(as));      // accumulator complete -> epilogue
        SNAG_CTRL_SYNC();
        if (++as == ACC_STAGES) { as = 0; aphase ^= 1; }
      }
    }
    if (dbg && leader) {
      shp.dbg[blockIdx.x * 4 + 0] = clock64() - t_begin;
      shp.dbg[blockIdx.x * 4 + 1] = w_acc;
      shp.dbg[blockIdx.x * 4 + 3] = n_tiles;
    }
  } else if (cwarp < 0) {
    // ------------------------------------------------------------------ epilogue warpgroup
    EpiCtx cx;
    cx.tid = threadIdx.x;
    cx.et = cx.tid & 127;
    cx.wg = cx.tid >> 7;
    cx.lane = lane;
    cx.scratch = scratch;
    const uint32_t lane_base = static_cast<uint32_t>((warp & 3) * 32) << 16;
    uint32_t as = 0, aphase = 0;
    uint32_t tile_seq = 0;
    cx.useq = -1;
    const bool dbg = shp.dbg != nullptr;
    long long c_proc = 0, c_bar = 0;
    for (int uid = blockIdx.x; uid < shp.n_units * shp.ksplits; uid += gridDim.x) {
      const int u = uid % shp.n_units;
      cx.split = uid / shp.n_units;
      ++cx.useq;
      cx.rb = u % shp.row_blocks;
      cx.chunk = u / shp.row_blocks;
      cx.row = cx.rb * BM + cx.et;
      cx.list = cx.chunk * kWG + cx.wg;
      cx.row_ok = cx.row < shp.n_rows;
      const int ct0 = cx.chunk * shp.tiles_per_chunk;
      const int ct1 = min(ct0 + shp.tiles_per_chunk, shp.col_tiles);
      typename Epi::State st;
      Epi::unit_begin(ep, shp, cx, st);
      // per-column vectors of a tile (norms, CSLS means, thresholds ...) are fetched from global memory one tile
      // ahead (tile_prefetch: loads in flight while the current tile's strips are consumed) and parked in a
      // double-buffered shared-memory area (tile_commit) that all epilogue threads read after the barrier
      EpiPre pre = Epi::tile_prefetch(ep, shp, cx, ct0);
      for (int ct = ct0; ct < ct1; ++ct, ++tile_seq) {
        const int buf = tile_seq & 1;
        long long t0 = dbg ? clock64() : 0;
        Epi::tile_commit(ep, shp, cx, st, pre, ct, buf);
        named_bar_sync(1, kEpiThreads);
        if (dbg) c_bar += clock64() - t0;
        if (ct + 1 < ct1) pre = Epi::tile_prefetch(ep, shp, cx, ct + 1);
        mbar_wait(tfull_bar(as), aphase);
        tc_fence_after();
        t0 = dbg ? clock64() : 0;
        const uint32_t taddr = tmem_base + lane_base + as * BN;
        // Rolled on purpose: one copy of the strip body keeps the epilogue inside the instruction cache
        // (a fully unrolled tile body was ~150 KB of SASS and ran instruction-fetch bound).
        if constexpr (!Epi::kNoLoad) {
          const int c_beg = cx.wg * kStripsPerWG;
          const int c_end = min((cx.wg + 1) * kStripsPerWG, tile_strips(shp, ct));
#if SNAG_PIPE_LD
          // two strips in flight: the TMEM read of strip c+1 is issued before strip c is consumed, so its latency
          // hides behind the epilogue arithmetic (two copies of the strip body, still well inside the i-cache)
          uint32_t r0[32], r1[32];
          if (c_beg < c_end) SNAG_TMEM_LD32(taddr + c_beg * 32, r0);
#pragma unroll 1
          for (int c = c_beg; c < c_end; c += 2) {
            SNAG_TMEM_WAIT32(r0);
            if (c + 1 < c_end) SNAG_TMEM_LD32(taddr + (c + 1) * 32, r1);
            cx.taddr = taddr + c * 32;
            Epi::chunk(ep, shp, cx, st, ct, c, r0, buf);
            if (c + 1 < c_end) {
              SNAG_TMEM_WAIT32(r1);
              if (c + 2 < c_end) SNAG_TMEM_LD32(taddr + (c + 2) * 32, r0);
              cx.taddr = taddr + (c + 1) * 32;
              Epi::chunk(ep, shp, cx, st, ct, c + 1, r1, buf);
            }
          }
#else
#pragma unroll 1
          for (int c = c_beg; c < c_end; ++c) {
            uint32_t r[32];
            SNAG_TMEM_LD32(taddr + c * 32, r);
            SNAG_TMEM_WAIT32(r);
            cx.taddr = taddr + c * 32;
            Epi::chunk(ep, shp, cx, st, ct, c, r, buf);
          }
#endif
        }
        tc_fence_before();
        mbar_arrive(tempty_bar(as));
        if (dbg) c_proc += clock64() - t0;
        if (++as == ACC_STAGES) { as = 0; aphase ^= 1; }
        Epi::tile_end(ep, shp, cx, st, ct, buf);
      }
      Epi::unit_end(ep, shp, cx, st);
    }
    if constexpr (HasKernelEnd<Epi>::value) Epi::kernel_end(ep, shp, cx);
    if (dbg && lane == 0) {      // summed over the epilogue warps: cycles consuming strips / cycles in commit + barrier
      atomicAdd(shp.dbg + blockIdx.x * 4 + 2, static_cast<unsigned long long>(c_proc));
      atomicAdd(shp.dbg + (gridDim.x + blockIdx.x) * 4 + 0, static_cast<unsigned long long>(c_bar));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (cwarp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ================================================================================================
// Arithmetic shared by the evaluation epilogues: the reference's op order, one rounding per op.
//   d    = clamp((xn_i + yn_j) - 2 s_ij, 0)          src/utils.py:210-218
//   c    = 1 - d                                      main.py:393 (argument of csls_sim)
//   csls = (2 c - nv1_i) - nv2_j                      src/utils.py:433-434
//   dist = 1 - csls                                   main.py:393
// 2*s and 2*c are exact, so the FMAs below round exactly like the reference's separate mul and sub.
// ================================================================================================
__device__ __forceinline__ float sqdist_from_dot(float s, float xn, float yn) {
  const float t = __fadd_rn(xn, yn);
  return fmaxf(__fmaf_rn(-2.0f, s, t), 0.0f);
}
__device__ __forceinline__ float csls_dist_from_c(float c, float nv1, float nv2) {
  const float u = __fmaf_rn(2.0f, c, -nv1);
  const float v = __fsub_rn(u, nv2);
  return __fsub_rn(1.0f, v);
}

// ------------------------------------------------------------------------------------------------
// Epilogue: none (accumulators are dropped) — measures the TMA + UMMA mainloop alone (bench/diagnostics)
// ------------------------------------------------------------------------------------------------
struct EpiNull {
  static constexpr bool kNoLoad = true;
  struct Params { int unused; };
  struct State {};
  static __device__ __forceinline__ void unit_begin(const Params&, const SimShape&, const EpiCtx&, State&) {}
  static __device__ __forceinline__ EpiPre tile_prefetch(const Params&, const SimShape&, const EpiCtx&, int) { return EpiPre{}; }
  static __device__ __forceinline__ void tile_commit(const Params&, const SimShape&, const EpiCtx&, State&, const EpiPre&, int, int) {}
  static __device__ __forceinline__ void chunk(const Params&, const SimShape&, const EpiCtx&, State&, int, int,
                                               const uint32_t (&)[32], int) {}
  static __device__ __forceinline__ void tile_end(const Params&, const SimShape&, const EpiCtx&, State&, int, int) {}
  static __device__ __forceinline__ void unit_end(const Params&, const SimShape&, const EpiCtx&, State&) {}
};

// ------------------------------------------------------------------------------------------------
// Epilogue: write S (mode 0) or the squared-L2 distance (mode 1) — drop-in pairwise_distances
// ------------------------------------------------------------------------------------------------
struct EpiWrite {
  static constexpr bool kNoLoad = false;
  struct Params {
    float* out;        // [n_rows, ld]
    long long ld;
    const float* xn;   // [n_rows]  (mode 1)
    const float* yn;   // [n_cols]  (mode 1)
    int mode;
    int transposed;          // 1: out[col * ld + row] (mode 0 only) — a warp's 32 rows are 128 contiguous bytes per column
    long long split_stride;  // split-K: slice s writes its partial products to out + s * split_stride
  };
  struct State {
    float xn;
  };
  static __device__ __forceinline__ void unit_begin(const Params& p, const SimShape&, const EpiCtx& cx, State& st) {
    st.xn = (p.mode == 1 && cx.row_ok) ? p.xn[cx.row] : 0.f;
  }
  static __device__ __forceinline__ EpiPre tile_prefetch(const Params& p, const SimShape& shp, const EpiCtx& cx, int ct) {
    static_assert(NUM_EPI_THREADS >= BN, "one epilogue thread stages one column");
    EpiPre pre{};
    const int col = ct * BN + cx.tid;
    if (cx.tid < BN) pre.a = (p.mode == 1 && col < shp.n_cols) ? p.yn[col] : 0.f;
    return pre;
  }
  static __device__ __forceinline__ void tile_commit(const Params&, const SimShape&, const EpiCtx& cx, State&,
                                                     const EpiPre& pre, int, int buf) {
    if (cx.tid < BN) cx.scratch[buf * BN + cx.tid] = pre.a;
  }
  static __device__ __forceinline__ void chunk(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st,
                                               int ct, int c, const uint32_t (&r)[32], int buf) {
    if (p.transposed) {
      if (!cx.row_ok) return;
      const int col0 = ct * BN + c * 32;
      float* o = p.out + cx.split * p.split_stride + static_cast<long long>(col0) * p.ld + cx.row;
#pragma unroll
      for (int q = 0; q < 32; ++q)
        if (col0 + q < shp.n_cols) o[static_cast<long long>(q) * p.ld] = __uint_as_float(r[q]);
      return;
    }
    if (strip_coalesced(p, shp, cx, st, ct, c, r, buf)) return;       // warp-uniform
    const float* yn_s = cx.scratch + buf * BN + c * 32;
    const int col0 = ct * BN + c * 32;
    if (!cx.row_ok) return;
    float* orow = p.out + cx.split * p.split_stride + static_cast<long long>(cx.row) * p.ld + col0;
    float v[32];
#pragma unroll
    for (int q = 0; q < 32; ++q) {
      const float s = __uint_as_float(r[q]);
      v[q] = (p.mode == 1) ? sqdist_from_dot(s, st.xn, yn_s[q]) : s;
    }
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(orow) & 15) == 0) && (col0 + 32 <= shp.n_cols);
    if (vec_ok) {
#pragma unroll
      for (int q = 0; q < 32; q += 4)
        *reinterpret_cast<float4*>(orow + q) = make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]);
    } else {
#pragma unroll
      for (int q = 0; q < 32; ++q)
        if (col0 + q < shp.n_cols) orow[q] = v[q];
    }
  }
  // full strips of 32-byte aligned outputs: the thread's 128 bytes of the row leave as four 256-bit stores (full sectors)
  static __device__ __forceinline__ bool strip_coalesced(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st,
                                                         int ct, int c, const uint32_t (&r)[32], int buf) {
    const int col0 = ct * BN + c * 32;
    if (col0 + 32 > shp.n_cols ||
        ((reinterpret_cast<uintptr_t>(p.out) | static_cast<uintptr_t>(p.ld * 4) | static_cast<uintptr_t>(p.split_stride * 4)) & 31))
      return false;
    if (!cx.row_ok) return true;
    const float* yn_s = cx.scratch + buf * BN + c * 32;
    uint8_t* dst = reinterpret_cast<uint8_t*>(p.out + cx.split * p.split_stride + static_cast<long long>(cx.row) * p.ld + col0);
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      uint32_t w[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int q = 8 * h + e;
        const float sv = __uint_as_float(r[q]);
        w[e] = __float_as_uint((p.mode == 1) ? sqdist_from_dot(sv, st.xn, yn_s[q]) : sv);
      }
      st_global_256(dst + 32 * h, make_uint4(w[0], w[1], w[2], w[3]), make_uint4(w[4], w[5], w[6], w[7]));
    }
    return true;
  }
  static __device__ __forceinline__ void tile_end(const Params&, const SimShape&, const EpiCtx&, State&, int, int) {}
  static __device__ __forceinline__ void unit_end(const Params&, const SimShape&, const EpiCtx&, State&) {}
};

// ascending KT-list insertion (top[0] = current KT-th largest = admission threshold); with kIdx the column ids travel
// with the values (needed to re-score the neighbourhood canonically afterwards)
template <bool kIdx>
__device__ __forceinline__ void topk_list_insert(float (&top)[KT], int (&topi)[kIdx ? KT : 1], float x, int id) {
  top[0] = x;
  if (kIdx) topi[0] = id;
#pragma unroll
  for (int t = 0; t < KT - 1; ++t) {
    if (kIdx) {
      const bool sw = top[t] > top[t + 1];
      const float a = top[t], b = top[t + 1];
      const int ia = topi[t], ib = topi[t + 1];
      top[t] = sw ? b : a;
      top[t + 1] = sw ? a : b;
      topi[t] = sw ? ib : ia;
      topi[t + 1] = sw ? ia : ib;
    } else {
      const float lo = fminf(top[t], top[t + 1]);
      const float hi = fmaxf(top[t], top[t + 1]);
      top[t] = lo;
      top[t + 1] = hi;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Epilogue: per-row top-KT of c_ij = 1 - d_ij over the unit's columns (CSLS neighbourhood, sweep 1).
// Output: part[chunk][row][KT], ascending, -inf padded. A merge kernel reduces over chunks.
// ------------------------------------------------------------------------------------------------
template <bool kIdx>
struct EpiRowTopK {
  static constexpr bool kNoLoad = false;
  struct Params {
    const float* xn;   // [n_rows]
    const float* yn;   // [n_cols]
    float* part;       // [n_lists][n_rows][KT]
    int* part_idx;     // [n_lists][n_rows][KT] (kIdx) view column of every candidate, -1 for the -inf padding
  };
  struct State {
    float xn;
    float top[KT];     // ascending: top[0] is the current KT-th largest (the admission threshold)
    int topi[kIdx ? KT : 1];
  };
  static __device__ __forceinline__ void unit_begin(const Params& p, const SimShape&, const EpiCtx& cx, State& st) {
    st.xn = cx.row_ok ? p.xn[cx.row] : 0.f;
#pragma unroll
    for (int t = 0; t < KT; ++t) st.top[t] = -INFINITY;
    if (kIdx) {
#pragma unroll
      for (int t = 0; t < KT; ++t) st.topi[t] = -1;
    }
  }
  // scratch layout per buffer: yn[BN] then the minimum of yn over each 32-column strip [BN/32]
  static constexpr int kVecStride = BN + BN / 32;
  static __device__ __forceinline__ EpiPre tile_prefetch(const Params& p, const SimShape& shp, const EpiCtx& cx, int ct) {
    EpiPre pre{};
    const int col = ct * BN + cx.tid;
    // out-of-range columns get yn = +inf  ->  d = +inf, c = -inf: never admitted
    if (cx.tid < BN) pre.a = (col < shp.n_cols) ? p.yn[col] : INFINITY;
    return pre;
  }
  static __device__ __forceinline__ void tile_commit(const Params&, const SimShape&, const EpiCtx& cx, State&,
                                                     const EpiPre& pre, int, int buf) {
    static_assert(NUM_EPI_THREADS >= BN, "one epilogue thread stages one column");
    static_assert(2 * kVecStride <= EPI_VEC_FLOATS, "scratch too small");
    if (cx.tid >= BN) return;                      // whole warps leave: the shuffles below stay warp-complete
    float* yn_s = cx.scratch + buf * kVecStride;
    const float v = pre.a;
    yn_s[cx.tid] = v;
    float m = v;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (cx.lane == 0) yn_s[BN + (cx.tid >> 5)] = m;
  }
  static __device__ __forceinline__ void chunk(const Params&, const SimShape&, const EpiCtx& cx, State& st, int ct,
                                               int c, const uint32_t (&r)[32], int buf) {
    const float* yn_s = cx.scratch + buf * kVecStride + c * 32;
    // Conservative pre-filter in s-space. c_ij = fl(1 - max(fl(fl(xn_i + yn_j) - 2 s), 0)) can exceed the current
    // KT-th largest top0 only if s > ((xn_i + min_j yn_j) - 1 + top0)/2; every quantity is below 4 in magnitude, so
    // the roundings involved total < 2e-6 and a margin of 4e-6 makes the skip safe (false positives are re-checked
    // exactly below). Fast path: one compare + one predicated bit-set per element.
    const float tmin = __fadd_rn(st.xn, cx.scratch[buf * kVecStride + BN + c]);
    const float thr = __fmaf_rn(0.5f, __fadd_rn(__fadd_rn(tmin, -1.0f), st.top[0]), -4e-6f);
    uint32_t pm = 0;
#pragma unroll
    for (int q = 0; q < 32; ++q)
      if (__uint_as_float(r[q]) > thr) pm |= (1u << q);
    if (pm != 0) {
      // rare path, kept small on purpose (instruction cache): park the strip's accumulators in shared memory
      // ([q][thread] layout, conflict-free) and visit only the flagged elements
      float* stage = cx.scratch + EPI_VEC_FLOATS + cx.tid;
#pragma unroll
      for (int h = 0; h < 32 / EPI_STAGE_VALS; ++h) {      // the staging area holds EPI_STAGE_VALS values per thread
        uint32_t ph = (pm >> (EPI_STAGE_VALS * h)) & ((1u << EPI_STAGE_VALS) - 1u);
        if (ph == 0) continue;
#pragma unroll
        for (int q = 0; q < EPI_STAGE_VALS; ++q) stage[q * NUM_EPI_THREADS] = __uint_as_float(r[EPI_STAGE_VALS * h + q]);
        while (ph != 0) {
          const int q = __ffs(ph) - 1;
          ph &= ph - 1;
          const float x = __fsub_rn(1.0f, sqdist_from_dot(stage[q * NUM_EPI_THREADS], st.xn, yn_s[EPI_STAGE_VALS * h + q]));
          if (x > st.top[0]) topk_list_insert<kIdx>(st.top, st.topi, x, ct * BN + c * 32 + EPI_STAGE_VALS * h + q);
        }
      }
    }
  }
  static __device__ __forceinline__ void tile_end(const Params&, const SimShape&, const EpiCtx&, State&, int, int) {}
  static __device__ __forceinline__ void unit_end(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st) {
    if (!cx.row_ok) return;
    const long long o0 = (static_cast<long long>(cx.list) * shp.n_rows + cx.row) * KT;
    float4* o = reinterpret_cast<float4*>(p.part + o0);
#pragma unroll
    for (int t = 0; t < KT; t += 4) o[t / 4] = make_float4(st.top[t], st.top[t + 1], st.top[t + 2], st.top[t + 3]);
    if (kIdx) {
      int4* oi = reinterpret_cast<int4*>(p.part_idx + o0);
#pragma unroll
      for (int t = 0; t < KT; t += 4) oi[t / 4] = make_int4(st.topi[t], st.topi[t + 1], st.topi[t + 2], st.topi[t + 3]);
    }
  }
};

// ------------------------------------------------------------------------------------------------
// Epilogue: CSLS neighbourhoods of BOTH directions in one sweep. Rows as in EpiRowTopK (registers). Columns:
// column j's neighbourhood is the k largest c_ij over ALL rows, but a tile only sees 128 of them, so column
// state cannot live in the CTA. Instead every element that could still belong to column j's top-k is appended
// to a per-column candidate buffer in HBM and a tiny kernel selects the k largest afterwards:
//   * a pre-pass over a random sample of the rows gives colthr[j] <= (final k-th largest c of column j);
//     any row with c_ij >= colthr[j] is a candidate (a superset of the true top-k; ~k*n/m per column for a
//     sample of m rows, whatever the data distribution);
//   * fast path per element: s_ij > a_i + b_j with a_i = xn_i/2, b_j = (yn_j - 1 + colthr_j)/2 - margin — a
//     conservative s-space form of that test (same rounding argument as the row pre-filter);
//   * the 32x32 predicate bit-matrix of a warp's strip is transposed with 5 shuffles so that lane l owns column l;
//     it re-computes c exactly for the flagged rows (accumulators parked in shared memory) and appends the
//     survivors, as (column, c) pairs, to a stream private to the CTA (slot from a shared-memory counter);
//     bandwidth kernels bucket the streams by column afterwards. (Letting the row owner re-check its own flagged
//     columns through 32 predicated blocks needs no staging but measured 10-20 % slower.)
// ------------------------------------------------------------------------------------------------
// r[q] for a run-time q: a switch the compiler turns into a branch tree, so the register strip is never spilled to local
// memory; lanes that ask for different q take different leaves, one after the other
__device__ __forceinline__ uint32_t strip_value(const uint32_t (&r)[32], int q) {
  uint32_t v = 0;
  switch (q) {
#define SNAG_SV_CASE(i) case i: v = r[i]; break;
    SNAG_SV_CASE(0) SNAG_SV_CASE(1) SNAG_SV_CASE(2) SNAG_SV_CASE(3) SNAG_SV_CASE(4) SNAG_SV_CASE(5) SNAG_SV_CASE(6) SNAG_SV_CASE(7)
    SNAG_SV_CASE(8) SNAG_SV_CASE(9) SNAG_SV_CASE(10) SNAG_SV_CASE(11) SNAG_SV_CASE(12) SNAG_SV_CASE(13) SNAG_SV_CASE(14)
    SNAG_SV_CASE(15) SNAG_SV_CASE(16) SNAG_SV_CASE(17) SNAG_SV_CASE(18) SNAG_SV_CASE(19) SNAG_SV_CASE(20) SNAG_SV_CASE(21)
    SNAG_SV_CASE(22) SNAG_SV_CASE(23) SNAG_SV_CASE(24) SNAG_SV_CASE(25) SNAG_SV_CASE(26) SNAG_SV_CASE(27) SNAG_SV_CASE(28)
    SNAG_SV_CASE(29) SNAG_SV_CASE(30) SNAG_SV_CASE(31)
#undef SNAG_SV_CASE
    default: break;
  }
  return v;
}
__device__ __forceinline__ uint32_t transpose32(uint32_t x, int lane) {
#pragma unroll
  for (int sft = 16; sft >= 1; sft >>= 1) {
    const uint32_t m = sft == 16 ? 0x0000FFFFu : sft == 8 ? 0x00FF00FFu : sft == 4 ? 0x0F0F0F0Fu
                                               : sft == 2 ? 0x33333333u : 0x55555555u;
    const uint32_t y = __shfl_xor_sync(0xffffffffu, x, sft);
    x = (lane & sft) ? ((x & ~m) | ((y >> sft) & m)) : ((x & m) | ((y << sft) & ~m));
  }
  return x;
}

// kRank (the one-pass evaluation, EpiOnePass): the same sweep also streams out every element that may count towards a
// RANK, so that the second sweep over S is not needed. The rank verdicts are  s_ij > R_i + C_j  (l2r) and
// s_ij > R'_i + C'_j  (r2l) with per-row / per-column constants that depend on the CSLS means this very sweep
// produces (see EpiRankBand). The caller passes constants that are provably or speculatively BELOW the final ones —
// rk_row = min-side R, R' built from a lower bound of nv1 and a guessed upper bound of the pair's own nv2, rk_col
// likewise — and every element above either relaxed threshold is appended as (column, s bits, row) to a second
// per-CTA stream. rank_judge_kernel then settles the streamed elements against the final constants (counting,
// deferring the band to band_rescore); rows / columns whose guessed bound turned out too low are recounted
// exhaustively. A few 1e-4 of the elements are streamed.
template <bool kRank>
struct EpiRowColTopKT {
  static constexpr bool kNoLoad = false;
  struct Params {
    const float* xn;       // [n_rows]
    const float* yn;       // [n_cols]
    float* part;           // [n_lists][n_rows][KT]   row candidates, as EpiRowTopK
    int* part_idx;         // [n_lists][n_rows][KT]   their view columns
    const float* rowthr;   // [n_rows] or null: a lower bound of row i's final KT-th largest c (from a sample of the
                           // columns). Every list starts from it instead of -inf, which removes the ~KT*ln(cols/KT)
                           // warm-up insertions each unit would otherwise pay; unfilled slots keep (rowthr, -1).
    const float* colthr;   // [n_cols] admission threshold of column j in c-space (from the sample pre-pass)
    const float* colb;     // [n_cols] b_j of the s-space pre-filter
    uint2* stream;         // [gridDim.x][cta_cap] (column, c bits) candidates appended by each CTA
    int* stream_row;       // [gridDim.x][cta_cap] view row of every stream entry
    int* stream_cnt;       // [gridDim.x] entries each CTA produced (may exceed cta_cap: overflow, entries dropped)
    int cta_cap;
    // kRank only
    const float* rk_r;     // [n_rows] relaxed R_i   (l2r: s > rk_r[i] + rk_c[j])
    const float* rk_rp;    // [n_rows] relaxed R'_i  (r2l: s > rk_rp[i] + rk_cp[j])
    const float* rk_c;     // [n_cols] relaxed C_j
    const float* rk_cp;    // [n_cols] relaxed C'_j
    uint2* rk_stream;      // [gridDim.x][rk_cap] (column, s bits)
    int* rk_stream_row;    // [gridDim.x][rk_cap]
    int* rk_cnt;           // [gridDim.x]
    int rk_cap;
  };
  struct State {
    float xn, a;
    float rk_r, rk_rp;
    uint32_t a2, rk_r2, rk_rp2;      // half2 broadcasts of the row constants, rounded down and lowered by kHalfMargin
    float top[KT];
    int topi[KT];
  };
  // Pre-filter arithmetic in fp16x2 (two elements per instruction): for |values| < 2 every rounding involved (s to nearest:
  // 2.5e-4, the per-column terms and row constants DOWN, the half2 sum to nearest: 4.9e-4) is covered by lowering the row
  // constants by 1e-3 — the half2 test can only flag MORE than the exact fp32 test, which then decides. The caller must
  // not use this epilogue for rows that are not (nearly) unit norm (launch_eval_rowcoltopk checks norm_max).
  static constexpr float kHalfMargin = 1e-3f;
  static __device__ __forceinline__ uint32_t half2_bcast_rd(float v) {
    const __half h = __float2half_rd(v);
    const __half2 h2 = __halves2half2(h, h);
    return *reinterpret_cast<const uint32_t*>(&h2);
  }
  // scratch per tile buffer (floats): yn[BN], strip minima of yn [BN/32], colb[BN], colthr[BN] (+ rk_c[BN], rk_cp[BN]), then
  // the fp16x2 copies (rounded down) of colb (+ rk_c, rk_cp): BN/2 words each; after the two buffers the two stream counters
  static constexpr int kVecs = kRank ? 5 : 3;
  static constexpr int kHalfOff = kVecs * BN + BN / 32;             // 16-byte aligned: (kVecs*256 + 8) * 4 bytes
  static constexpr int kVecStride = kHalfOff + (kRank ? 3 : 1) * (BN / 2);
  static constexpr int kCntOff = 2 * kVecStride;         // int: candidates appended by this CTA so far (+1: rank stream)
  // diagnostics (shp.dbg set): what the exact tests made of the flagged elements, unsigned counters per CTA: accepted by
  // the row top-k test, appended as column candidates, above the l2r / r2l rank threshold, accepted by none of them
  enum { kDbgRow, kDbgCol, kDbgL2r, kDbgR2l, kDbgNone, kDbgN };
  static constexpr int kDbgOff = kCntOff + 2;
  static __device__ __forceinline__ void kernel_end(const Params& p, const SimShape& shp, const EpiCtx& cx) {
    named_bar_sync(1, NUM_EPI_THREADS);
    if (cx.tid == 0) {
      p.stream_cnt[blockIdx.x] = *reinterpret_cast<const int*>(cx.scratch + kCntOff);
      if (kRank) p.rk_cnt[blockIdx.x] = *reinterpret_cast<const int*>(cx.scratch + kCntOff + 1);
      if (shp.dbg != nullptr) {            // rows 2*gridDim.x + cta: row, col, l2r, r2l; 3*gridDim.x + cta: none
        const unsigned* d = reinterpret_cast<const unsigned*>(cx.scratch + kDbgOff);
        for (int t = 0; t < kDbgN; ++t) shp.dbg[((2 + t / 4) * gridDim.x + blockIdx.x) * 4 + t % 4] = d[t];
      }
    }
  }
  static __device__ __forceinline__ void unit_begin(const Params& p, const SimShape&, const EpiCtx& cx, State& st) {
    static_assert(kDbgOff + kDbgN <= EPI_VEC_FLOATS, "scratch too small");
    static_assert((kHalfOff % 4) == 0 && (kVecStride % 4) == 0, "fp16x2 vectors must be 16-byte aligned");
    if (cx.useq == 0 && cx.tid == 0) {                     // ordered by the tile barrier
      for (int t = 0; t < 2 + kDbgN; ++t) reinterpret_cast<int*>(cx.scratch + kCntOff)[t] = 0;
    }
    st.xn = cx.row_ok ? p.xn[cx.row] : 0.f;
    st.a = cx.row_ok ? 0.5f * st.xn : INFINITY;          // padding rows never produce column candidates
    st.a2 = half2_bcast_rd(st.a - kHalfMargin);
    if (kRank) {
      st.rk_r = cx.row_ok ? p.rk_r[cx.row] : INFINITY;
      st.rk_rp = cx.row_ok ? p.rk_rp[cx.row] : INFINITY;
      st.rk_r2 = half2_bcast_rd(st.rk_r - kHalfMargin);
      st.rk_rp2 = half2_bcast_rd(st.rk_rp - kHalfMargin);
    }
    const float t0 = (p.rowthr != nullptr && cx.row_ok) ? p.rowthr[cx.row] : -INFINITY;
#pragma unroll
    for (int t = 0; t < KT; ++t) { st.top[t] = t0; st.topi[t] = -1; }
  }
  static __device__ __forceinline__ EpiPre tile_prefetch(const Params& p, const SimShape& shp, const EpiCtx& cx, int ct) {
    EpiPre pre{};
    const int col = ct * BN + cx.tid;
    if (cx.tid < BN) {
      const bool ok = col < shp.n_cols;
      pre.a = ok ? p.yn[col] : INFINITY;
      pre.b = ok ? p.colb[col] : INFINITY;
      pre.c = ok ? p.colthr[col] : INFINITY;
      if (kRank) {
        pre.d = ok ? p.rk_c[col] : INFINITY;
        pre.e = ok ? p.rk_cp[col] : INFINITY;
      }
    }
    return pre;
  }
  static __device__ __forceinline__ void tile_commit(const Params&, const SimShape&, const EpiCtx& cx, State&,
                                                     const EpiPre& pre, int, int buf) {
    static_assert(NUM_EPI_THREADS >= BN, "one epilogue thread stages one column");
    if (cx.tid >= BN) return;                      // whole warps leave: the shuffles below stay warp-complete
    float* v_s = cx.scratch + buf * kVecStride;
    const float v = pre.a;
    v_s[cx.tid] = v;
    v_s[BN + BN / 32 + cx.tid] = pre.b;
    v_s[2 * BN + BN / 32 + cx.tid] = pre.c;
    if (kRank) {
      v_s[3 * BN + BN / 32 + cx.tid] = pre.d;
      v_s[4 * BN + BN / 32 + cx.tid] = pre.e;
    }
    float m = v;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (cx.lane == 0) v_s[BN + (cx.tid >> 5)] = m;
    // fp16x2 copies, rounded DOWN (a lower per-column term only flags more): even lanes pack (column, column + 1)
    uint32_t* h_s = reinterpret_cast<uint32_t*>(v_s + kHalfOff);
    const float b1 = __shfl_down_sync(0xffffffffu, pre.b, 1);
    const float d1 = __shfl_down_sync(0xffffffffu, pre.d, 1);
    const float e1 = __shfl_down_sync(0xffffffffu, pre.e, 1);
    if ((cx.tid & 1) == 0) {
      const __half2 hb = __halves2half2(__float2half_rd(pre.b), __float2half_rd(b1));
      h_s[cx.tid >> 1] = *reinterpret_cast<const uint32_t*>(&hb);
      if (kRank) {
        const __half2 hd = __halves2half2(__float2half_rd(pre.d), __float2half_rd(d1));
        const __half2 he = __halves2half2(__float2half_rd(pre.e), __float2half_rd(e1));
        h_s[BN / 2 + (cx.tid >> 1)] = *reinterpret_cast<const uint32_t*>(&hd);
        h_s[BN + (cx.tid >> 1)] = *reinterpret_cast<const uint32_t*>(&he);
      }
    }
  }
  // Fast path in fp16x2: two elements per instruction. flagged <=> s > min(row top-k pre-filter, a_i + b_j (column
  // candidate), R_i + C_j, R'_i + C'_j (rank candidates, kRank)) with every term rounded conservatively (see kHalfMargin):
  // per PAIR of elements one pack, 3 adds, 3 mins, one compare-to-mask and one LOP3 = 4.5 instructions per element
  // (2.5 without kRank) against 11 (6) for the fp32 per-element tests, which cost 27 % of the SM clock at the 1 kW power
  // cap. Strip-level (row x 32 columns) thresholds are useless here: column hubness — what CSLS corrects — moves the
  // per-column terms by as much as the element noise, and the minimum over 32 columns flagged 0.8 % of all elements.
  // Bit b of the mask: element 2b (b < 16) or 2(b - 16) + 1.
  static __device__ __forceinline__ void chunk(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st, int ct,
                                               int c, const uint32_t (&r)[32], int buf) {
    const float* v_s = cx.scratch + buf * kVecStride;
    const float* yn_s = v_s + c * 32;
    const float* cb_s = v_s + BN + BN / 32 + c * 32;
    const float* ct_s = v_s + 2 * BN + BN / 32 + c * 32;
    const float* kc_s = v_s + 3 * BN + BN / 32 + c * 32;
    const float* kp_s = v_s + 4 * BN + BN / 32 + c * 32;
    const uint32_t* h_s = reinterpret_cast<const uint32_t*>(v_s + kHalfOff) + c * 16;
    const float tmin = __fadd_rn(st.xn, v_s[BN + c]);
    const float thr = __fmaf_rn(0.5f, __fadd_rn(__fadd_rn(tmin, -1.0f), st.top[0]), -4e-6f);
    const uint32_t thr2w = half2_bcast_rd(thr - 3e-4f);
    const __half2 thr2 = *reinterpret_cast<const __half2*>(&thr2w);
    const __half2 a2 = *reinterpret_cast<const __half2*>(&st.a2);
    const __half2 r2 = *reinterpret_cast<const __half2*>(&st.rk_r2);
    const __half2 rp2 = *reinterpret_cast<const __half2*>(&st.rk_rp2);
    uint32_t fm = 0;
#pragma unroll
    for (int pq = 0; pq < 16; ++pq) {
      const __half2 h = __floats2half2_rn(__uint_as_float(r[2 * pq]), __uint_as_float(r[2 * pq + 1]));
      const __half2 cb2 = *reinterpret_cast<const __half2*>(h_s + pq);
      __half2 m = __hmin2(thr2, __hadd2(a2, cb2));
      if (kRank) {
#if !(SNAG_OPX & 1)
        const __half2 kc2 = *reinterpret_cast<const __half2*>(h_s + BN / 2 + pq);
#if (SNAG_OPX & 2)
        m = __hmin2(m, __hadd2(r2, kc2));
#else
        const __half2 kp2 = *reinterpret_cast<const __half2*>(h_s + BN + pq);
        m = __hmin2(m, __hmin2(__hadd2(r2, kc2), __hadd2(rp2, kp2)));
#endif
#endif
      }
      fm |= __hgt2_mask(h, m) & ((1u << pq) | (0x10000u << pq));
    }
    if (!__any_sync(0xffffffffu, fm != 0)) return;
    // Slow path. Each lane walks the columns IT flagged, so the warp iterates max over lanes of popc(fm) times (the union
    // of the flagged columns, walked by the whole warp, is several times longer when the flags sit in different rows and
    // columns, as they mostly do). The accumulator comes out of the register strip through an indexed branch that
    // diverges only over the distinct columns of one step; no shared-memory staging, no transposition. The row owner
    // runs all the exact tests: top-k insertion touches only its own registers, and the appends are warp-aggregated
    // (stream_slot). (Measured alternatives: staging the strip in shared memory + handing column candidates to a
    // column-owning lane: -20 % SM clock at the 1 kW power cap; re-reading the column from TMEM with tcgen05.ld.x1:
    // ~1 200 cycles per flagged column, epilogue-bound.)
    const bool dbg = shp.dbg != nullptr;
    if (dbg) {                              // diagnostics: flagged strips / flagged columns / flagged elements of this CTA
      const int nf = __reduce_add_sync(0xffffffffu, __popc(fm));
      const uint32_t um = __reduce_or_sync(0xffffffffu, fm);
      if (cx.lane == 0) {
        atomicAdd(shp.dbg + (gridDim.x + blockIdx.x) * 4 + 1, 1ull);
        atomicAdd(shp.dbg + (gridDim.x + blockIdx.x) * 4 + 2, static_cast<unsigned long long>(__popc(um)));
        atomicAdd(shp.dbg + (gridDim.x + blockIdx.x) * 4 + 3, static_cast<unsigned long long>(nf));
      }
    }
    const uint32_t col0 = static_cast<uint32_t>(ct * BN + c * 32);
    int* cnt = reinterpret_cast<int*>(cx.scratch + kCntOff);
    do {
      bool app_col = false, app_rk = false;
      uint32_t col = 0, dflags = 0;
      float sv = 0.f, x = 0.f;
      if (fm != 0) {
        const int b = __ffs(fm) - 1;
        fm &= fm - 1;
        const int q = b < 16 ? 2 * b : 2 * (b - 16) + 1;
        col = col0 + q;
        sv = __uint_as_float(strip_value(r, q));
        const bool want_row = sv > thr, want_col = sv > __fadd_rn(st.a, cb_s[q]);
        if (want_row || want_col) x = __fsub_rn(1.0f, sqdist_from_dot(sv, st.xn, yn_s[q]));
        const bool acc_row = want_row && x > st.top[0];
        if (acc_row) topk_list_insert<true>(st.top, st.topi, x, static_cast<int>(col));
        app_col = want_col && x >= ct_s[q];
        if (kRank && !(SNAG_OPX & 4)) {
          const float t_l2r = __fadd_rn(st.rk_r, kc_s[q]), t_r2l = __fadd_rn(st.rk_rp, kp_s[q]);
          app_rk = sv > fminf(t_l2r, t_r2l);
          if (dbg) dflags = (sv > t_l2r ? 1u << kDbgL2r : 0u) | (sv > t_r2l ? 1u << kDbgR2l : 0u);
        }
        if (dbg) {
          dflags |= (acc_row ? 1u << kDbgRow : 0u) | (app_col ? 1u << kDbgCol : 0u);
          if (dflags == 0) dflags = 1u << kDbgNone;
        }
      }
      // column candidate (column, c, row); rank candidate (column, tensor-core s, row)
      int slot = stream_slot(app_col, cnt, p.cta_cap, cx.lane);
      if (slot >= 0) {
        const long long o = static_cast<long long>(blockIdx.x) * p.cta_cap + slot;
        p.stream[o] = make_uint2(col, __float_as_uint(x));
        p.stream_row[o] = cx.row;
      }
      if (kRank) {
        slot = stream_slot(app_rk, cnt + 1, p.rk_cap, cx.lane);
        if (slot >= 0) {
          const long long o = static_cast<long long>(blockIdx.x) * p.rk_cap + slot;
          p.rk_stream[o] = make_uint2(col, __float_as_uint(sv));
          p.rk_stream_row[o] = cx.row;
        }
      }
      if (dbg) {
#pragma unroll
        for (int t = 0; t < kDbgN; ++t) {
          const int v = __popc(__ballot_sync(0xffffffffu, (dflags >> t) & 1u));
          if (cx.lane == 0 && v != 0) atomicAdd(reinterpret_cast<unsigned*>(cx.scratch + kDbgOff) + t, static_cast<unsigned>(v));
        }
      }
    } while (__any_sync(0xffffffffu, fm != 0));
  }
  // Slot of this lane's entry in a CTA-private stream (-1: nothing to append, or the stream is full). One shared-memory
  // atomicAdd per warp hands out consecutive slots to the lanes with pred set, in lane order. The counter stops growing
  // once it exceeds cap (overflow is detected by count > cap; letting it run on could wrap 32 bits when nearly everything
  // is streamed). Warp-collective: every lane of the warp calls it.
  static __device__ __forceinline__ int stream_slot(bool pred, int* cnt, int cap, int lane) {
    const uint32_t bal = __ballot_sync(0xffffffffu, pred);
    if (bal == 0) return -1;
    const int leader = __ffs(bal) - 1;
    int base = 0;
    if (lane == leader) base = *reinterpret_cast<volatile int*>(cnt) <= cap ? atomicAdd(cnt, __popc(bal)) : cap;
    base = __shfl_sync(0xffffffffu, base, leader) + __popc(bal & ((1u << lane) - 1u));
    return pred && base < cap ? base : -1;
  }
  static __device__ __forceinline__ void tile_end(const Params&, const SimShape&, const EpiCtx&, State&, int, int) {}
  static __device__ __forceinline__ void unit_end(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st) {
    if (!cx.row_ok) return;
    const long long o0 = (static_cast<long long>(cx.list) * shp.n_rows + cx.row) * KT;
    float4* o = reinterpret_cast<float4*>(p.part + o0);
    int4* oi = reinterpret_cast<int4*>(p.part_idx + o0);
#pragma unroll
    for (int t = 0; t < KT; t += 4) {
      o[t / 4] = make_float4(st.top[t], st.top[t + 1], st.top[t + 2], st.top[t + 3]);
      oi[t / 4] = make_int4(st.topi[t], st.topi[t + 1], st.topi[t + 2], st.topi[t + 3]);
    }
  }
};
struct EpiRowColTopKF32 {
  static constexpr bool kNoLoad = false;
  struct Params {
    const float* xn;       // [n_rows]
    const float* yn;       // [n_cols]
    float* part;           // [n_lists][n_rows][KT]   row candidates, as EpiRowTopK
    int* part_idx;         // [n_lists][n_rows][KT]   their view columns
    const float* rowthr;   // [n_rows] or null: a lower bound of row i's final KT-th largest c (from a sample of the
                           // columns). Every list starts from it instead of -inf, which removes the ~KT*ln(cols/KT)
                           // warm-up insertions each unit would otherwise pay; unfilled slots keep (rowthr, -1).
    const float* colthr;   // [n_cols] admission threshold of column j in c-space (from the sample pre-pass)
    const float* colb;     // [n_cols] b_j of the s-space pre-filter
    uint2* stream;         // [gridDim.x][cta_cap] (column, c bits) candidates appended by each CTA
    int* stream_row;       // [gridDim.x][cta_cap] view row of every stream entry
    int* stream_cnt;       // [gridDim.x] entries each CTA produced (may exceed cta_cap: overflow, entries dropped)
    int cta_cap;
  };
  struct State {
    float xn, a;
    float top[KT];
    int topi[KT];
  };
  // scratch per tile buffer: yn[BN], strip minima of yn [BN/32], colb[BN], colthr[BN]; then xn of the row block x2
  static constexpr int kVecStride = 3 * BN + BN / 32;
  static constexpr int kXnOff = 2 * kVecStride;
  static constexpr int kCntOff = kXnOff + 2 * BM;        // int: candidates appended by this CTA so far
  static __device__ __forceinline__ void kernel_end(const Params& p, const SimShape&, const EpiCtx& cx) {
    named_bar_sync(1, NUM_EPI_THREADS);
    if (cx.tid == 0) p.stream_cnt[blockIdx.x] = *reinterpret_cast<const int*>(cx.scratch + kCntOff);
  }
  static __device__ __forceinline__ void unit_begin(const Params& p, const SimShape&, const EpiCtx& cx, State& st) {
    static_assert(kCntOff + 1 <= EPI_VEC_FLOATS, "scratch too small");
    if (cx.useq == 0 && cx.tid == 0) *reinterpret_cast<int*>(cx.scratch + kCntOff) = 0;   // ordered by the tile barrier
    st.xn = cx.row_ok ? p.xn[cx.row] : 0.f;
    st.a = cx.row_ok ? 0.5f * st.xn : INFINITY;          // padding rows never produce column candidates
    const float t0 = (p.rowthr != nullptr && cx.row_ok) ? p.rowthr[cx.row] : -INFINITY;
#pragma unroll
    for (int t = 0; t < KT; ++t) { st.top[t] = t0; st.topi[t] = -1; }
    if (cx.wg == 0) cx.scratch[kXnOff + (cx.useq & 1) * BM + cx.et] = st.xn;   // visible after the tile barrier
  }
  static __device__ __forceinline__ EpiPre tile_prefetch(const Params& p, const SimShape& shp, const EpiCtx& cx, int ct) {
    EpiPre pre{};
    const int col = ct * BN + cx.tid;
    if (cx.tid < BN) {
      const bool ok = col < shp.n_cols;
      pre.a = ok ? p.yn[col] : INFINITY;
      pre.b = ok ? p.colb[col] : INFINITY;
      pre.c = ok ? p.colthr[col] : INFINITY;
    }
    return pre;
  }
  static __device__ __forceinline__ void tile_commit(const Params&, const SimShape&, const EpiCtx& cx, State&,
                                                     const EpiPre& pre, int, int buf) {
    static_assert(NUM_EPI_THREADS >= BN, "one epilogue thread stages one column");
    if (cx.tid >= BN) return;                      // whole warps leave: the shuffles below stay warp-complete
    float* v_s = cx.scratch + buf * kVecStride;
    const float v = pre.a;
    v_s[cx.tid] = v;
    v_s[BN + BN / 32 + cx.tid] = pre.b;
    v_s[2 * BN + BN / 32 + cx.tid] = pre.c;
    float m = v;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (cx.lane == 0) v_s[BN + (cx.tid >> 5)] = m;
  }
  static __device__ __forceinline__ void chunk(const Params& p, const SimShape&, const EpiCtx& cx, State& st, int ct,
                                               int c, const uint32_t (&r)[32], int buf) {
    const float* v_s = cx.scratch + buf * kVecStride;
    const float* yn_s = v_s + c * 32;
    const float* cb_s = v_s + BN + BN / 32 + c * 32;
    const float* ct_s = v_s + 2 * BN + BN / 32 + c * 32;
    const float tmin = __fadd_rn(st.xn, v_s[BN + c]);
    const float thr = __fmaf_rn(0.5f, __fadd_rn(__fadd_rn(tmin, -1.0f), st.top[0]), -4e-6f);
    uint32_t pm = 0, cm = 0;
#pragma unroll
    for (int q = 0; q < 32; ++q) {
      const float s = __uint_as_float(r[q]);
      if (s > thr) pm |= (1u << q);
      if (s > __fadd_rn(st.a, cb_s[q])) cm |= (1u << q);
    }
    const uint32_t cmT = transpose32(cm, cx.lane);       // lane l: bit t set <=> row t of this warp flagged column l
    if (__any_sync(0xffffffffu, (pm | cmT) != 0)) {
      float* stage_w = cx.scratch + EPI_VEC_FLOATS + (cx.tid & ~31);      // this warp's 32 columns of the staging area
      const float* xn_w = cx.scratch + kXnOff + (cx.useq & 1) * BM + (cx.et & ~31);
#pragma unroll
      for (int h = 0; h < 32 / EPI_STAGE_VALS; ++h) {      // the staging area holds EPI_STAGE_VALS values per thread
        uint32_t ph = (pm >> (EPI_STAGE_VALS * h)) & ((1u << EPI_STAGE_VALS) - 1u);
        const uint32_t ch = ((cx.lane / EPI_STAGE_VALS) == h) ? cmT : 0u;
        if (!__any_sync(0xffffffffu, (ph | ch) != 0)) continue;
#pragma unroll
        for (int q = 0; q < EPI_STAGE_VALS; ++q) stage_w[q * NUM_EPI_THREADS + cx.lane] = __uint_as_float(r[EPI_STAGE_VALS * h + q]);
        __syncwarp();
        while (ph != 0) {                                  // row direction: own staged values
          const int q = __ffs(ph) - 1;
          ph &= ph - 1;
          const float x = __fsub_rn(1.0f, sqdist_from_dot(stage_w[q * NUM_EPI_THREADS + cx.lane], st.xn, yn_s[EPI_STAGE_VALS * h + q]));
          if (x > st.top[0]) topk_list_insert<true>(st.top, st.topi, x, ct * BN + c * 32 + EPI_STAGE_VALS * h + q);
        }
        uint32_t cmask = ch;                               // column direction: lane l owns column l of the strip
        const int col = ct * BN + c * 32 + cx.lane;
        while (cmask != 0) {
          const int t = __ffs(cmask) - 1;
          cmask &= cmask - 1;
          const float s = stage_w[(cx.lane % EPI_STAGE_VALS) * NUM_EPI_THREADS + t];
          const float x = __fsub_rn(1.0f, sqdist_from_dot(s, xn_w[t], yn_s[cx.lane]));
          if (x >= ct_s[cx.lane]) {
            // append to this CTA's private stream: a shared-memory counter hands out the slot (no global-atomic
            // round trip on the epilogue's critical path); a later pass buckets the stream by column
            const int slot = atomicAdd(reinterpret_cast<int*>(cx.scratch + kCntOff), 1);
            if (slot < p.cta_cap) {
              const long long o = static_cast<long long>(blockIdx.x) * p.cta_cap + slot;
              p.stream[o] = make_uint2(static_cast<uint32_t>(col), __float_as_uint(x));
              p.stream_row[o] = cx.rb * BM + (cx.et & ~31) + t;
            }
          }
        }
        __syncwarp();
      }
    }
  }
  static __device__ __forceinline__ void tile_end(const Params&, const SimShape&, const EpiCtx&, State&, int, int) {}
  static __device__ __forceinline__ void unit_end(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st) {
    if (!cx.row_ok) return;
    const long long o0 = (static_cast<long long>(cx.list) * shp.n_rows + cx.row) * KT;
    float4* o = reinterpret_cast<float4*>(p.part + o0);
    int4* oi = reinterpret_cast<int4*>(p.part_idx + o0);
#pragma unroll
    for (int t = 0; t < KT; t += 4) {
      o[t / 4] = make_float4(st.top[t], st.top[t + 1], st.top[t + 2], st.top[t + 3]);
      oi[t / 4] = make_int4(st.topi[t], st.topi[t + 1], st.topi[t + 2], st.topi[t + 3]);
    }
  }
};

using EpiRowColTopK = EpiRowColTopKT<false>;
using EpiOnePass = EpiRowColTopKT<true>;

// ------------------------------------------------------------------------------------------------
// Epilogue: mutual nearest neighbours (model/SNAG.py:192-208, Iter_new_links): for every row the column with the
// smallest squared distance d_ij = clamp(xn_i + yn_j - 2 s_ij, 0) and for every column the row with the smallest
// d_ij, first index on ties (torch.argmin). The distance matrix the reference concatenates is never formed.
//   rows   : running (best d, its column) in registers, one partial result per list, merged afterwards;
//   columns: a pre-pass over a sample of the rows bounds every column's minimum from above; only elements at or
//            below that bound (a handful per column) reach a 64-bit atomicMin on  (d bits << 32 | row)  — d >= 0,
//            so unsigned order of the packed key is the lexicographic order (d, row).
// Both directions use the conservative s-space pre-filter of EpiRowTopK; survivors are re-checked exactly.
// ------------------------------------------------------------------------------------------------
struct EpiMutualNN {
  static constexpr bool kNoLoad = false;
  struct Params {
    const float* xn;              // [n_rows]
    const float* yn;              // [n_cols]
    const float* colb;            // [n_cols] b_j of the column pre-filter: flag when s_ij > xn_i/2 + b_j
    unsigned long long* colkey;   // [n_cols] packed (d bits << 32 | row), caller initialises to ~0
    float* row_val;               // [n_lists][n_rows] smallest d of the list's columns
    int* row_idx;                 // [n_lists][n_rows] its column (lowest index among equals)
  };
  struct State {
    float xn, a, best;
    int best_j;
  };
  static constexpr int kVecStride = 2 * BN + BN / 32;       // yn[BN], strip minima of yn, colb[BN]
  static __device__ __forceinline__ void unit_begin(const Params& p, const SimShape&, const EpiCtx& cx, State& st) {
    static_assert(2 * kVecStride <= EPI_VEC_FLOATS, "scratch too small");
    st.xn = cx.row_ok ? p.xn[cx.row] : 0.f;
    st.a = cx.row_ok ? 0.5f * st.xn : INFINITY;            // padding rows never reach a column
    st.best = INFINITY;
    st.best_j = 0x7fffffff;
  }
  static __device__ __forceinline__ EpiPre tile_prefetch(const Params& p, const SimShape& shp, const EpiCtx& cx, int ct) {
    EpiPre pre{};
    const int col = ct * BN + cx.tid;
    if (cx.tid < BN) {
      const bool ok = col < shp.n_cols;
      pre.a = ok ? p.yn[col] : INFINITY;                   // d = +inf: never the minimum of a row
      pre.b = ok ? p.colb[col] : INFINITY;                 // never flagged for the column side
    }
    return pre;
  }
  static __device__ __forceinline__ void tile_commit(const Params&, const SimShape&, const EpiCtx& cx, State&,
                                                     const EpiPre& pre, int, int buf) {
    static_assert(NUM_EPI_THREADS >= BN, "one epilogue thread stages one column");
    if (cx.tid >= BN) return;
    float* v_s = cx.scratch + buf * kVecStride;
    v_s[cx.tid] = pre.a;
    v_s[BN + BN / 32 + cx.tid] = pre.b;
    float m = pre.a;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (cx.lane == 0) v_s[BN + (cx.tid >> 5)] = m;
  }
  static __device__ __forceinline__ void chunk(const Params& p, const SimShape&, const EpiCtx& cx, State& st, int ct,
                                               int c, const uint32_t (&r)[32], int buf) {
    const float* v_s = cx.scratch + buf * kVecStride;
    const float* yn_s = v_s + c * 32;
    const float* cb_s = v_s + BN + BN / 32 + c * 32;
    // d_ij < best  =>  s_ij > (xn_i + yn_j - best)/2 >= (xn_i + min_strip yn - best)/2 ; 4e-6 covers the roundings
    const float thr = __fmaf_rn(0.5f, __fsub_rn(__fadd_rn(st.xn, v_s[BN + c]), st.best), -4e-6f);
    uint32_t pm = 0, cm = 0;
#pragma unroll
    for (int q = 0; q < 32; ++q) {
      const float s = __uint_as_float(r[q]);
      if (s > thr) pm |= (1u << q);
      if (s > __fadd_rn(st.a, cb_s[q])) cm |= (1u << q);
    }
    if ((pm | cm) != 0) {
      // rare after the first tiles of a unit / for a handful of elements per column: exact re-check by the row owner
      const int col0 = ct * BN + c * 32;
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        if ((pm | cm) & (1u << q)) {
          const float d = sqdist_from_dot(__uint_as_float(r[q]), st.xn, yn_s[q]);
          if (d < st.best) {                               // columns arrive in increasing order: strict keeps the first
            st.best = d;
            st.best_j = col0 + q;
          }
          if (cm & (1u << q))
            atomicMin(p.colkey + col0 + q, (static_cast<unsigned long long>(__float_as_uint(d)) << 32) |
                                               static_cast<unsigned int>(cx.row));
        }
      }
    }
  }
  static __device__ __forceinline__ void tile_end(const Params&, const SimShape&, const EpiCtx&, State&, int, int) {}
  static __device__ __forceinline__ void unit_end(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st) {
    if (!cx.row_ok) return;
    const long long o = static_cast<long long>(cx.list) * shp.n_rows + cx.row;
    p.row_val[o] = st.best;
    p.row_idx[o] = st.best_j;
  }
};

// ------------------------------------------------------------------------------------------------
// Epilogue: rank counting (sweep 2). For every pair (i, j) of the unit, with dist = CSLS distance:
//   cnt_row[i] += [dist < g_i] + [dist == g_i and gid(j) < gid(i)]      (j != i)     -> l2r rank of pair i
//   cnt_col[j] += [dist < g_j] + [dist == g_j and gid(i) < gid(j)]      (i != j)     -> r2l rank of pair j
// i.e. the position of the ground truth in a stable ascending sort (main.py:400-411, 422-429).
// Optionally tracks the 3 nearest columns per row (the ret1..ret3 of the prediction CSV, main.py:411).
// ------------------------------------------------------------------------------------------------
template <bool kTop3, bool kCsls>
struct EpiRank {
  static constexpr bool kNoLoad = false;
  struct Params {
    const float* xn;     // [n_rows]
    const float* yn;     // [n_cols]
    const float* nv1;    // [n_rows]
    const float* nv2;    // [n_cols]
    const float* g_row;  // [n_rows]  dist of pair(row gid)
    const float* g_col;  // [n_cols]  dist of pair(col gid)
    int row_gid0;        // global pair id of view row 0
    int col_gid0;        // global pair id of view column 0
    int* cnt_row;        // [n_rows]  (atomically accumulated, caller zeroes)
    int* cnt_col;        // [n_cols]
    float* top3_val;     // [n_lists][n_rows][4] (kTop3) ascending distance
    int* top3_idx;       // [n_lists][n_rows][4] (kTop3) column gid
  };                     // kCsls == false: rank on the plain squared distance d (args.csls False, main.py:392)
  struct State {
    float xn, nv1, g;
    int gid;
    int cnt;
    float t3v[3];
    int t3i[3];
  };
  static __device__ __forceinline__ void unit_begin(const Params& p, const SimShape&, const EpiCtx& cx, State& st) {
    st.xn = cx.row_ok ? p.xn[cx.row] : 0.f;
    st.nv1 = cx.row_ok ? p.nv1[cx.row] : 0.f;
    // invalid rows: g = -inf never counts anything on the row side; the column side masks by row_ok
    st.g = cx.row_ok ? p.g_row[cx.row] : -INFINITY;
    st.gid = p.row_gid0 + cx.row;
    st.cnt = 0;
    if (kTop3) {
#pragma unroll
      for (int t = 0; t < 3; ++t) { st.t3v[t] = INFINITY; st.t3i[t] = 0x7fffffff; }
    }
  }
  static __device__ __forceinline__ EpiPre tile_prefetch(const Params& p, const SimShape& shp, const EpiCtx& cx, int ct) {
    static_assert(NUM_EPI_THREADS >= BN, "one epilogue thread stages one column");
    EpiPre pre{};
    const int col = ct * BN + cx.tid;
    if (cx.tid < BN) {
      const bool ok = col < shp.n_cols;
      pre.a = ok ? p.yn[col] : INFINITY;        // d = inf -> dist = +inf: never smaller than anything
      pre.b = ok ? p.nv2[col] : 0.f;
      pre.c = ok ? p.g_col[col] : -INFINITY;
    }
    return pre;
  }
  static __device__ __forceinline__ void tile_commit(const Params&, const SimShape&, const EpiCtx& cx, State&,
                                                     const EpiPre& pre, int, int buf) {
    if (cx.tid >= BN) return;
    float* s = cx.scratch + buf * (3 * BN);
    s[cx.tid] = pre.a;
    s[BN + cx.tid] = pre.b;
    s[2 * BN + cx.tid] = pre.c;
  }
  static __device__ __forceinline__ void chunk(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st, int ct,
                                               int c, const uint32_t (&r)[32], int buf) {
    const float* s = cx.scratch + buf * (3 * BN) + c * 32;
    const int col0 = ct * BN + c * 32;
    const int cgid0 = p.col_gid0 + col0;
    // does this 32-column strip contain the ground-truth column of one of this warp's 32 rows? (warp-uniform)
    const int wgid0 = p.row_gid0 + cx.rb * BM + (cx.et & ~31);
    const bool diag_strip = (cgid0 <= wgid0 + 31) && (cgid0 + 31 >= wgid0);
    float dist[32];
    uint32_t rmask = 0, cmask = 0;
    bool tie = diag_strip;
    // fast path: strict comparisons only; any exact equality (or the diagonal) defers to the exact path below
#pragma unroll
    for (int q = 0; q < 32; ++q) {
      const float d = sqdist_from_dot(__uint_as_float(r[q]), st.xn, s[q]);
      dist[q] = kCsls ? csls_dist_from_c(__fsub_rn(1.0f, d), st.nv1, s[BN + q]) : d;
      const float gj = s[2 * BN + q];
      if (dist[q] < st.g) rmask |= (1u << q);
      if (dist[q] < gj) cmask |= (1u << q);
      tie |= (dist[q] == st.g);
      tie |= (dist[q] == gj);
    }
    if (tie) {
      // exact path: stable-sort tie-break on the pair id, ground-truth column excluded
      rmask = 0;
      cmask = 0;
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        const int jg = cgid0 + q;
        const float gj = s[2 * BN + q];
        bool prow = (dist[q] < st.g) || (dist[q] == st.g && jg < st.gid);
        bool pcol = (dist[q] < gj) || (dist[q] == gj && st.gid < jg);
        if (jg == st.gid) { prow = false; pcol = false; }
        if (prow) rmask |= (1u << q);
        if (pcol) cmask |= (1u << q);
      }
    }
    const int cnt = __popc(rmask);
    st.cnt += cnt;
    if (!cx.row_ok) cmask = 0;
    // column counts: transpose the warp's 32x32 predicate bit-matrix, then popc -> lane l owns column l
    uint32_t x = cmask;
#pragma unroll
    for (int sft = 16; sft >= 1; sft >>= 1) {
      const uint32_t m = sft == 16 ? 0x0000FFFFu : sft == 8 ? 0x00FF00FFu : sft == 4 ? 0x0F0F0F0Fu
                                                 : sft == 2 ? 0x33333333u : 0x55555555u;
      const uint32_t y = __shfl_xor_sync(0xffffffffu, x, sft);
      x = (cx.lane & sft) ? ((x & ~m) | ((y >> sft) & m)) : ((x & m) | ((y << sft) & ~m));
    }
    const int votes = __popc(x);
    if (votes != 0 && col0 + cx.lane < shp.n_cols) atomicAdd(p.cnt_col + col0 + cx.lane, votes);
    if (kTop3) {
      float mn = INFINITY;
#pragma unroll
      for (int q = 0; q < 32; ++q) mn = fminf(mn, dist[q]);
      if (mn <= st.t3v[2]) {
#pragma unroll
        for (int q = 0; q < 32; ++q) {
          const int jg = cgid0 + q;
          if (dist[q] < st.t3v[2] || (dist[q] == st.t3v[2] && jg < st.t3i[2])) {
            st.t3v[2] = dist[q]; st.t3i[2] = jg;
#pragma unroll
            for (int t = 2; t > 0; --t) {
              const bool sw = (st.t3v[t] < st.t3v[t - 1]) || (st.t3v[t] == st.t3v[t - 1] && st.t3i[t] < st.t3i[t - 1]);
              if (sw) {
                const float tv = st.t3v[t]; st.t3v[t] = st.t3v[t - 1]; st.t3v[t - 1] = tv;
                const int ti = st.t3i[t]; st.t3i[t] = st.t3i[t - 1]; st.t3i[t - 1] = ti;
              }
            }
          }
        }
      }
    }
  }
  static __device__ __forceinline__ void tile_end(const Params&, const SimShape&, const EpiCtx&, State&, int, int) {}
  static __device__ __forceinline__ void unit_end(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st) {
    if (!cx.row_ok) return;
    if (st.cnt != 0) atomicAdd(p.cnt_row + cx.row, st.cnt);
    if (kTop3) {
      const long long o = (static_cast<long long>(cx.list) * shp.n_rows + cx.row) * 4;
      *reinterpret_cast<float4*>(p.top3_val + o) = make_float4(st.t3v[0], st.t3v[1], st.t3v[2], 0.f);
      *reinterpret_cast<int4*>(p.top3_idx + o) = make_int4(st.t3i[0], st.t3i[1], st.t3i[2], 0);
    }
  }
};

// ------------------------------------------------------------------------------------------------
// Epilogue: rank counting in s-space with a deferral band (the default sweep 2).
// The CSLS chain is affine in s (apart from the clamp, which only acts within rounding distance of d = 0):
//   dist_ij = 2 (xn_i + yn_j - 2 s_ij) - 1 + nv1_i + nv2_j
// so   dist_ij < g_i   <=>   s_ij > R_i + C_j ,    R_i  = (2 xn_i + nv1_i - 1 - g_i)/4 ,  C_j  = (2 yn_j + nv2_j)/4
// and  dist_ij < g_j   <=>   s_ij > R'_i + C'_j ,  R'_i = (2 xn_i + nv1_i - 1)/4 ,        C'_j = (2 yn_j + nv2_j - g_j)/4
// (without CSLS: R = (xn - g)/2, C = yn/2, R' = xn/2, C' = (yn - g)/2).
// An element whose margin exceeds eps in magnitude has the same verdict under the reference's fp32 chain evaluated
// on the canonically accumulated dot product (eps covers the tensor-core accumulation error, the chain's roundings and
// the roundings of R, C): it is counted here with two subtractions and four compares. Elements inside the band —
// exact ties and the ground-truth column included — are NOT counted; they are appended to a list and judged afterwards
// by band_rescore_kernel with the canonical arithmetic (fp64 index-order dot, the reference's op order, stable-sort
// tie-break). The ranks therefore do not depend on the tensor core's accumulation order.
// kTop3: the four columns with the largest x = s - C_j per row (nearest first; re-scored and cut to three afterwards).
// ------------------------------------------------------------------------------------------------
template <bool kTop3, bool kCsls>
struct EpiRankBand {
  static constexpr bool kNoLoad = false;
  struct Params {
    const float* xn;     // [n_rows]
    const float* yn;     // [n_cols]
    const float* nv1;    // [n_rows]
    const float* nv2;    // [n_cols]
    const float* g_row;  // [n_rows]  dist of pair(row gid)
    const float* g_col;  // [n_cols]  dist of pair(col gid)
    int row_gid0;        // global pair id of view row 0
    int col_gid0;        // global pair id of view column 0
    int* cnt_row;        // [n_rows]  (atomically accumulated, caller zeroes)
    int* cnt_col;        // [n_cols]
    float* top4_val;     // [n_lists][n_rows][4] (kTop3) x = s - C_j, descending
    int* top4_idx;       // [n_lists][n_rows][4] (kTop3) column gid
    float eps;           // half-width of the deferral band in s-space
    uint2* band;         // [band_cap] deferred elements: x = view row | direction flags << 30, y = view column
    unsigned int* band_cnt;   // number of deferred elements (may exceed band_cap: overflow, caller re-runs)
    unsigned int band_cap;
    const int* row_gids;      // [n_rows] or null: global pair id of every view row when the rows are a gathered subset
                              // (recount of selected entities); null: row_gid0 + row
  };
  struct State {
    float r_lo, r_hi, rp;
    int gid;
    int cnt;
    float t4v[4];
    int t4i[4];
  };
  static __device__ __forceinline__ void unit_begin(const Params& p, const SimShape&, const EpiCtx& cx, State& st) {
    st.gid = (p.row_gids != nullptr && cx.row_ok) ? p.row_gids[cx.row] : p.row_gid0 + cx.row;
    st.cnt = 0;
    if (cx.row_ok) {
      const float xn = p.xn[cx.row], g = p.g_row[cx.row];
      float R, Rp;
      if (kCsls) {
        const float base = __fmaf_rn(2.0f, xn, p.nv1[cx.row]) - 1.0f;
        R = 0.25f * (base - g);
        Rp = 0.25f * base;
      } else {
        R = 0.5f * (xn - g);
        Rp = 0.5f * xn;
      }
      st.r_lo = R - p.eps;
      st.r_hi = R + p.eps;
      st.rp = Rp;
    } else {                       // padding rows: nothing is ever above +inf, and s - inf = -inf on the column side
      st.r_lo = st.r_hi = st.rp = INFINITY;
    }
    if (kTop3) {
#pragma unroll
      for (int t = 0; t < 4; ++t) { st.t4v[t] = -INFINITY; st.t4i[t] = 0x7fffffff; }
    }
  }
  static __device__ __forceinline__ EpiPre tile_prefetch(const Params& p, const SimShape& shp, const EpiCtx& cx, int ct) {
    static_assert(NUM_EPI_THREADS >= BN, "one epilogue thread stages one column");
    EpiPre pre{INFINITY, INFINITY, INFINITY};   // out-of-range columns: x = -inf, thresholds +inf
    const int col = ct * BN + cx.tid;
    if (cx.tid < BN && col < shp.n_cols) {
      const float yn = p.yn[col], g = p.g_col[col];
      float C, Cp;
      if (kCsls) {
        const float base = __fmaf_rn(2.0f, yn, p.nv2[col]);
        C = 0.25f * base;
        Cp = 0.25f * (base - g);
      } else {
        C = 0.5f * yn;
        Cp = 0.5f * (yn - g);
      }
      pre.a = C;
      pre.b = Cp - p.eps;
      pre.c = Cp + p.eps;
    }
    return pre;
  }
  static __device__ __forceinline__ void tile_commit(const Params&, const SimShape&, const EpiCtx& cx, State&,
                                                     const EpiPre& pre, int, int buf) {
    if (cx.tid >= BN) return;
    float* s = cx.scratch + buf * (3 * BN);
    s[cx.tid] = pre.a;
    s[BN + cx.tid] = pre.b;
    s[2 * BN + cx.tid] = pre.c;
  }
  static __device__ __forceinline__ void chunk(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st, int ct,
                                               int c, const uint32_t (&r)[32], int buf) {
    const float* s = cx.scratch + buf * (3 * BN) + c * 32;
    const int col0 = ct * BN + c * 32;
    const int cgid0 = p.col_gid0 + col0;
    uint32_t ra = 0, rb = 0, ca = 0, cb = 0, tm = 0;
#pragma unroll
    for (int q = 0; q < 32; ++q) {
      const float sv = __uint_as_float(r[q]);
      const float x = __fsub_rn(sv, s[q]);
      const float y = __fsub_rn(sv, st.rp);
      if (x > st.r_hi) ra |= (1u << q);
      if (x > st.r_lo) rb |= (1u << q);
      if (y > s[2 * BN + q]) ca |= (1u << q);
      if (y > s[BN + q]) cb |= (1u << q);
      if (kTop3) { if (x > st.t4v[3]) tm |= (1u << q); }
    }
    uint32_t rband = rb & ~ra, cband = cb & ~ca;
    // the ground-truth column of this row is never a competitor (main.py:400-411 ranks it, it does not count itself)
    const int qd = st.gid - cgid0;
    if (qd >= 0 && qd < 32) {
      const uint32_t keep = ~(1u << qd);
      ra &= keep; ca &= keep; rband &= keep; cband &= keep;
    }
    uint32_t deferred = rband | cband;
    while (deferred != 0) {                                   // rare: a handful of elements per row
      const int q = __ffs(deferred) - 1;
      deferred &= deferred - 1;
      const unsigned int slot = atomicAdd(p.band_cnt, 1u);
      if (slot < p.band_cap) {
        const uint32_t flags = ((rband >> q) & 1u) | (((cband >> q) & 1u) << 1);
        p.band[slot] = make_uint2(static_cast<uint32_t>(cx.row) | (flags << 30), static_cast<uint32_t>(col0 + q));
      }
    }
    st.cnt += __popc(ra);
    // column counts: transpose the warp's 32x32 predicate bit-matrix, then popc -> lane l owns column l
    const int votes = __popc(transpose32(ca, cx.lane));
    if (votes != 0 && col0 + cx.lane < shp.n_cols) atomicAdd(p.cnt_col + col0 + cx.lane, votes);
    if (kTop3) {
      while (tm != 0) {
        const int q = __ffs(tm) - 1;
        tm &= tm - 1;
        // r[] is indexed with a run-time q here: re-read the value through a select chain the compiler keeps in registers
        float sv = 0.f;
#pragma unroll
        for (int e = 0; e < 32; ++e) sv = (e == q) ? __uint_as_float(r[e]) : sv;
        const float x = __fsub_rn(sv, s[q]);
        if (x > st.t4v[3]) {                                  // columns arrive in increasing order: strict keeps the first
          st.t4v[3] = x; st.t4i[3] = cgid0 + q;
#pragma unroll
          for (int t = 3; t > 0; --t) {
            if (st.t4v[t] > st.t4v[t - 1]) {
              const float tv = st.t4v[t]; st.t4v[t] = st.t4v[t - 1]; st.t4v[t - 1] = tv;
              const int ti = st.t4i[t]; st.t4i[t] = st.t4i[t - 1]; st.t4i[t - 1] = ti;
            }
          }
        }
      }
    }
  }
  static __device__ __forceinline__ void tile_end(const Params&, const SimShape&, const EpiCtx&, State&, int, int) {}
  static __device__ __forceinline__ void unit_end(const Params& p, const SimShape& shp, const EpiCtx& cx, State& st) {
    if (!cx.row_ok) return;
    if (st.cnt != 0) atomicAdd(p.cnt_row + cx.row, st.cnt);
    if (kTop3) {
      const long long o = (static_cast<long long>(cx.list) * shp.n_rows + cx.row) * 4;
      *reinterpret_cast<float4*>(p.top4_val + o) = make_float4(st.t4v[0], st.t4v[1], st.t4v[2], st.t4v[3]);
      *reinterpret_cast<int4*>(p.top4_idx + o) = make_int4(st.t4i[0], st.t4i[1], st.t4i[2], st.t4i[3]);
    }
  }
};

// ------------------------------------------------------------------------------------------------
// Epilogue: in-batch contrastive row sums (ICL forward, model/SNAG_loss.py:98-126).
// X view = rows [row0, row0 + nx) of one side of the batch (the anchors this rank owns; the whole side when the
// loss is not sharded); Y view = [other side | same side], 2*Bp rows, B valid per part.
// Column c -> part p = c / Bp, idx = c - p*Bp; valid iff idx < B. With gr = row0 + row the anchor's index in the
// batch: p == 1 and idx == gr is the self-similarity the reference kills with -1e9; p == 0 and idx == gr is the
// positive logit.
// With unit-norm rows logits are bounded by 1/tau, so exp(logit - 1/tau) needs no running max.
//   rowsum_part[list][row] = sum_j exp2(s_ij * (log2e/tau) - log2e/tau)       (row = local row, stride nx)
//   pos[row]               = s_{row,gr} of part 0
// ------------------------------------------------------------------------------------------------
struct EpiIclFwd {
  static constexpr bool kNoLoad = false;
  struct Params {
    float scale_log2;   // log2(e) / tau
    int B;              // valid rows per part
    int Bp;             // padded rows per part (multiple of 256)
    int row0;           // batch index of X-view row 0
    int nx;             // rows of the X view
    float* rowsum_part; // [n_lists][nx]
    float* pos;         // [nx]
  };
  struct State {
    float sum;
  };
  static __device__ __forceinline__ void unit_begin(const Params&, const SimShape&, const EpiCtx&, State& st) {
    st.sum = 0.f;
  }
  static __device__ __forceinline__ EpiPre tile_prefetch(const Params&, const SimShape&, const EpiCtx&, int) { return EpiPre{}; }
  static __device__ __forceinline__ void tile_commit(const Params&, const SimShape&, const EpiCtx&, State&, const EpiPre&, int, int) {}
  static __device__ __forceinline__ void chunk(const Params& p, const SimShape&, const EpiCtx& cx, State& st, int ct,
                                               int c, const uint32_t (&r)[32], int) {
    const int col0 = ct * BN + c * 32;
    const int part = col0 >= p.Bp ? 1 : 0;
    const int idx0 = col0 - part * p.Bp;
    if (idx0 >= p.B) return;                              // strip entirely in the padding (warp-uniform)
    const int gr0 = p.row0 + cx.rb * BM;                 // batch index of the row block's first anchor
    const bool plain = (idx0 + 32 <= p.B) && (idx0 + 31 < gr0 || idx0 > gr0 + BM - 1);
    const float nb = -p.scale_log2;
    if (plain) {
      float acc = 0.f;
#pragma unroll
      for (int q = 0; q < 32; ++q) acc += ex2_approx(__fmaf_rn(__uint_as_float(r[q]), p.scale_log2, nb));
      st.sum += acc;
    } else {
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        const int idx = idx0 + q;
        const float s = __uint_as_float(r[q]);
        float e = ex2_approx(__fmaf_rn(s, p.scale_log2, nb));
        if (idx >= p.B) e = 0.f;
        if (idx == p.row0 + cx.row) {
          if (part == 1) e = 0.f;
          else if (cx.row_ok) p.pos[cx.row] = s;
        }
        st.sum += e;
      }
    }
  }
  static __device__ __forceinline__ void tile_end(const Params&, const SimShape&, const EpiCtx&, State&, int, int) {}
  static __device__ __forceinline__ void unit_end(const Params& p, const SimShape&, const EpiCtx& cx, State& st) {
    if (cx.row_ok) p.rowsum_part[static_cast<long long>(cx.list) * p.nx + cx.row] = st.sum;
  }
};

// ------------------------------------------------------------------------------------------------
// Epilogue: ICL backward, stage 1 — recompute the logits tile and write dL/dlogits as a bf16 matrix
// G [Bp, 2*Bp] (the left operand of the gradient GEMM  dX = G · [other side ; this side]).
// With nll_x[i] = lse_x[i] - s_ii/tau and upstream gradients gx = dL/dnll_x (Appendix A of SURVEY.md):
//   part 0 (cross):  G[i,j] = (cr_i + cc_j) * E_ij / tau  - [i == j] * dg_i / tau
//   part 1 (self) :  G[i,j] = (cr_i + cr_j) * E_ij / tau            (0 on the diagonal)
// where E_ij = exp(s_ij/tau - 1/tau), cr_i = g_this[i] * exp(1/tau - lse_this[i]) (row softmax term),
// cc_j = g_other[j] * exp(1/tau - lse_other[j]) (the same s_ij seen from the other side's softmax),
// dg_i = g_this[i] + g_other[i]. Anchors >= B and columns in the padding are written as zeros. As in the forward the
// X view is rows [row0, row0 + nx) of this side; cr / cc / dg are indexed by batch index, G by local row.
// ------------------------------------------------------------------------------------------------
#ifndef SNAG_ICLBWD_WG
#define SNAG_ICLBWD_WG 4
#endif
struct EpiIclBwd {
  static constexpr bool kNoLoad = false;
  // ncu (profiles/r01c): with 2 warpgroups this epilogue keeps the tensor pipe 40 % busy at D = 300 and issues on 32 %
  // of the cycles — 2 warps per scheduler cannot hide the TMEM-read -> exp -> pack -> shared -> global chain. It keeps
  // no per-row state across tiles, so it simply runs with 4 warpgroups (2 column strips each).
  static constexpr int kWG = SNAG_ICLBWD_WG;
  struct Params {
    float scale_log2;     // log2(e) / tau
    float inv_tau;
    int B, Bp;
    int row0, nx;
    const float* cr;      // [B] row-side coefficients (this side)
    const float* cc;      // [B] column-side coefficients of part 0 (other side)
    const float* dg;      // [B] diagonal term of part 0
    __nv_bfloat16* G;     // [nx, 2*Bp]
    int self_cols;        // 1: part 1 carries the transposed-role term cr_j (ICL / IAL gradients); 0: row term only
                          //    (G = cr_i E / tau in both parts: a plain row-softmax writer)
    float ebar;           // subtracted from E_ij before it is scaled (0 for ICL). IAL's gradient is a DIFFERENCE of two
                          // such matrices that are both nearly uniform at large tau; centring E on its value at s = 0
                          // keeps the bf16 rounding relative to the deviations, not to the common part (the common
                          // part's contribution to G.Y is rank one and is added back by the caller in fp32)
  };
  struct State {
    float cr, dg;
    int gr;               // batch index of this thread's anchor
    bool ok;
  };
  static __device__ __forceinline__ void unit_begin(const Params& p, const SimShape&, const EpiCtx& cx, State& st) {
    st.gr = p.row0 + cx.row;
    st.ok = cx.row_ok && st.gr < p.B;
    // coefficients carry the 1/tau factor from here on (one multiply per row / per staged column instead of per element)
    st.cr = st.ok ? p.cr[st.gr] * p.inv_tau : 0.f;
    st.dg = st.ok ? p.dg[st.gr] * p.inv_tau : 0.f;
  }
  static __device__ __forceinline__ EpiPre tile_prefetch(const Params& p, const SimShape&, const EpiCtx& cx, int ct) {
    static_assert(NUM_EPI_THREADS >= BN, "one epilogue thread stages one column");
    EpiPre pre{};
    if (cx.tid < BN) {
      const int col = ct * BN + cx.tid;
      const int part = col >= p.Bp ? 1 : 0;
      const int idx = col - part * p.Bp;
      if (idx < p.B) pre.a = (part ? (p.self_cols ? p.cr[idx] : 0.f) : p.cc[idx]) * p.inv_tau;
    }
    return pre;
  }
  static __device__ __forceinline__ void tile_commit(const Params&, const SimShape&, const EpiCtx& cx, State&,
                                                     const EpiPre& pre, int, int buf) {
    if (cx.tid < BN) cx.scratch[buf * BN + cx.tid] = pre.a;
  }
  // 16 consecutive elements of the strip (q0 = 0 or 16) -> 8 packed bf16 pairs
  static __device__ __forceinline__ void half_strip(const Params& p, const State& st, const float* cc_s, const uint32_t (&r)[32],
                                                    int q0, int idx0, int part, bool plain, uint32_t (&packed)[8]) {
    const float nb = -p.scale_log2;
    float cc[16];                                        // four 16-byte broadcast loads (not sixteen scalar ones)
#pragma unroll
    for (int q = 0; q < 16; q += 4) {
      const float4 t = *reinterpret_cast<const float4*>(cc_s + q0 + q);
      cc[q] = t.x; cc[q + 1] = t.y; cc[q + 2] = t.z; cc[q + 3] = t.w;
    }
    if (plain) {
#pragma unroll
      for (int q = 0; q < 16; q += 2) {
        const float e0 = ex2_approx(__fmaf_rn(__uint_as_float(r[q0 + q]), p.scale_log2, nb)) - p.ebar;
        const float e1 = ex2_approx(__fmaf_rn(__uint_as_float(r[q0 + q + 1]), p.scale_log2, nb)) - p.ebar;
        const __nv_bfloat162 h = __floats2bfloat162_rn((st.cr + cc[q]) * e0, (st.cr + cc[q + 1]) * e1);
        packed[q / 2] = *reinterpret_cast<const uint32_t*>(&h);
      }
    } else {
#pragma unroll
      for (int q = 0; q < 16; q += 2) {
        float v[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int idx = idx0 + q0 + q + e;
          const float E = ex2_approx(__fmaf_rn(__uint_as_float(r[q0 + q + e]), p.scale_log2, nb)) - p.ebar;
          float gval = (st.cr + cc[q + e]) * E;
          if (idx == st.gr) gval = part ? 0.f : gval - st.dg;
          if (!st.ok || idx >= p.B) gval = 0.f;
          v[e] = gval;
        }
        const __nv_bfloat162 h = __floats2bfloat162_rn(v[0], v[1]);
        packed[q / 2] = *reinterpret_cast<const uint32_t*>(&h);
      }
    }
  }
  static __device__ __forceinline__ void chunk(const Params& p, const SimShape&, const EpiCtx& cx, State& st, int ct,
                                               int c, const uint32_t (&r)[32], int buf) {
    const float* cc_s = cx.scratch + buf * BN + c * 32;
    const int col0 = ct * BN + c * 32;
    const int part = col0 >= p.Bp ? 1 : 0;
    const int idx0 = col0 - part * p.Bp;
    const int gr0 = p.row0 + cx.rb * BM;                 // batch index of the row block's first anchor
    // plain strip (CTA-uniform): every anchor of the row block and every column of the strip is valid and the strip
    // does not meet the block's diagonal -> 4 arithmetic instructions per element (FFMA, MUFU.EX2, FADD, FMUL)
    const bool plain = (gr0 + BM <= p.B) && ((cx.rb + 1) * BM <= p.nx) && (idx0 + 32 <= p.B) &&
                       (idx0 + 31 < gr0 || idx0 > gr0 + BM - 1);
    // Each thread owns one row of G: its 64 bytes of the strip leave as two 256-bit stores, i.e. two full 32-byte
    // sectors (16-byte stores left every sector half written by two instructions and ran at 1.4 TB/s; a shared-memory
    // transposition to 64-byte row segments fixed that but cost as many shared-memory wavefronts as the UMMA operand
    // reads leave free — ncu, profiles/r01c_summary.md).
    uint8_t* dst = reinterpret_cast<uint8_t*>(p.G + static_cast<long long>(cx.row) * (2 * p.Bp) + col0);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint32_t pk[8];
      half_strip(p, st, cc_s, r, 16 * h, idx0, part, plain, pk);
      if (cx.row_ok)
        st_global_256(dst + 32 * h, make_uint4(pk[0], pk[1], pk[2], pk[3]), make_uint4(pk[4], pk[5], pk[6], pk[7]));
    }
  }
  static __device__ __forceinline__ void tile_end(const Params&, const SimShape&, const EpiCtx&, State&, int, int) {}
  static __device__ __forceinline__ void unit_end(const Params&, const SimShape&, const EpiCtx&, State&) {}
};

// ------------------------------------------------------------------------------------------------
// Epilogue: ICL backward of the fp32 loss route. The logits tile comes from split operands (X rows [m | h | h], Y rows
// [h | m | h]), G is formed in fp32 registers exactly as EpiIclBwd forms it (the cross diagonal -dg/tau included), and
// stored as two bf16 terms, G3 = [G_h | G_h | G_m] ([nx, 6 Bp], G_h = bf16(G), G_m = bf16(G - G_h), the difference exact
// in fp32): the gradient GEMM over K = 6 Bp against the K-stacked rows [Y_h ; Y_m ; Y_h] then forms
// G_h Y_h + G_h Y_m + G_m Y_h, which leaves out G_m Y_m (<= 2^-16 |G| |Y|) and the residual of the two-term split of G
// (<= 2^-16 |G|). Every 32-byte piece is written with one 256-bit store, as in EpiIclBwd.
// ------------------------------------------------------------------------------------------------
struct EpiIclBwdSplit : EpiIclBwd {
  // EpiIclBwd::half_strip without the rounding: the 16 fp32 values of G
  static __device__ __forceinline__ void half_strip_f32(const Params& p, const State& st, const float* cc_s,
                                                        const uint32_t (&r)[32], int q0, int idx0, int part, bool plain,
                                                        float (&v)[16]) {
    const float nb = -p.scale_log2;
    float cc[16];
#pragma unroll
    for (int q = 0; q < 16; q += 4) {
      const float4 t = *reinterpret_cast<const float4*>(cc_s + q0 + q);
      cc[q] = t.x; cc[q + 1] = t.y; cc[q + 2] = t.z; cc[q + 3] = t.w;
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const float E = ex2_approx(__fmaf_rn(__uint_as_float(r[q0 + q]), p.scale_log2, nb)) - p.ebar;
      float gval = (st.cr + cc[q]) * E;
      if (!plain) {
        const int idx = idx0 + q0 + q;
        if (idx == st.gr) gval = part ? 0.f : gval - st.dg;
        if (!st.ok || idx >= p.B) gval = 0.f;
      }
      v[q] = gval;
    }
  }
  static __device__ __forceinline__ void chunk(const Params& p, const SimShape&, const EpiCtx& cx, State& st, int ct,
                                               int c, const uint32_t (&r)[32], int buf) {
    const float* cc_s = cx.scratch + buf * BN + c * 32;
    const int col0 = ct * BN + c * 32;
    const int part = col0 >= p.Bp ? 1 : 0;
    const int idx0 = col0 - part * p.Bp;
    const int gr0 = p.row0 + cx.rb * BM;
    const bool plain = (gr0 + BM <= p.B) && ((cx.rb + 1) * BM <= p.nx) && (idx0 + 32 <= p.B) &&
                       (idx0 + 31 < gr0 || idx0 > gr0 + BM - 1);
    const long long twoBp_bytes = 4ll * p.Bp;                  // bytes between the three column blocks of G3
    uint8_t* dst = reinterpret_cast<uint8_t*>(p.G + static_cast<long long>(cx.row) * (6 * p.Bp) + col0);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float v[16];
      half_strip_f32(p, st, cc_s, r, 16 * h, idx0, part, plain, v);
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int q = 0; q < 16; q += 2) {
        const __nv_bfloat162 g2 = __floats2bfloat162_rn(v[q], v[q + 1]);
        const __nv_bfloat162 m2 = __floats2bfloat162_rn(__fsub_rn(v[q], __low2float(g2)), __fsub_rn(v[q + 1], __high2float(g2)));
        hi[q / 2] = *reinterpret_cast<const uint32_t*>(&g2);
        lo[q / 2] = *reinterpret_cast<const uint32_t*>(&m2);
      }
      if (cx.row_ok) {
        const uint4 h0 = make_uint4(hi[0], hi[1], hi[2], hi[3]), h1 = make_uint4(hi[4], hi[5], hi[6], hi[7]);
        st_global_256(dst + 32 * h, h0, h1);
        st_global_256(dst + twoBp_bytes + 32 * h, h0, h1);
        st_global_256(dst + 2 * twoBp_bytes + 32 * h, make_uint4(lo[0], lo[1], lo[2], lo[3]), make_uint4(lo[4], lo[5], lo[6], lo[7]));
      }
    }
  }
};

}  // namespace snag
