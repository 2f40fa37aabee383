// Fused --distance 1 evaluation (main.py:387-429 with scipy's cdist "cityblock"): a CUDA-core sweep that never forms the
// n x n matrix, and the canonical re-scores that make its verdicts exact.
//
// The sweep. L1 is not a contraction, so the tensor cores cannot help; the lever sm_100a gives is the packed fp32 add:
// acc += |x - y| on two elements is two FADD2 (the second with the |.| operand modifier), one instruction per element.
//   operands  X [n1, Dp], Y [n2, Dp] fp32, rows zero padded to Dp (a multiple of 8; zeros add exactly 0)
//   units     (row block of 128 rows) x (chunk of column tiles of 64), dealt to a persistent grid round-robin in
//             chunk-major order as in sim_kernel: the CTAs running side by side share one Y chunk, which stays in L2
//   mainloop  k-slices of 32 columns of both operands staged in shared memory by cp.async (zero-filled past the row ends
//             and past n1 / n2), three stages in flight; the producer and the consumers are the same threads and only
//             __syncthreads orders them, so there is no wait that could hang
//   layout    256 threads as 16 x 16; thread (tx, ty) owns rows ty + 16 m (m < 8) and columns tx + 16 q (q < 4) of the
//             128 x 64 tile: 32 packed accumulators (even / odd k in the two halves), a k-slice read as float4 (two
//             pairs) per row and per column; smem rows are 36 floats apart so neither read pattern has bank conflicts
//
// Accumulation order and the error bound (l1_err_per_norm). Per element and lane half (even / odd k) the 16 terms of a
// k-slice are summed from 0 in fp32 (chunk), then total += (chunk_even + chunk_odd). With nc = ceil(Dp / 32) slices
// the computed d~ is the exact sum of the terms |x_k - y_k| with each term perturbed by at most
//   1 (the subtraction) + 15 (inside the chunk) + 1 (even + odd) + (nc - 1) (the running total) = nc + 16
// relative roundings of u = 2^-24 (first order; the higher-order terms and the final fp32 rounding of the canonical
// fp64 sum add less than 2u), and every term is <= |x_k| + |y_k|, so
//   |d~ - d_canonical| <= (nc + 18) u (||x||_1 + ||y||_1)          (x 1.01 for the higher-order terms)
// l1_approx below is the same sequence of operations on one pair, so a re-scorer can reproduce the sweep's d~ bit for bit.
// CSLS chain: |c~ - c| <= |d~ - d| + u (|c~| + |c|); the rank distance 1 - ((2 c - nv1) - nv2) adds 2 |c~ - c| and four
// more roundings on values bounded by 1 + S + |nv1| + |nv2| (S = ||x||_1 + ||y||_1): l1_rank_eps.
//
// Epilogue state. A row of the tile is spread over 16 threads (two warps), so per-row candidate lists live in shared
// memory: the list (ascending; [0] is the admission threshold) and a 64-entry inbox per row. After a tile every thread
// posts its elements that beat their row's threshold into the inbox (shared atomics), then one thread per row merges its
// inbox into the list; once the lists are full almost nothing passes the threshold and the merge costs nothing. The
// row-topk epilogue keeps KT candidates (c~ = 1 - d~, column ids); the rank epilogue keeps the 4 nearest (x = -dist~,
// column gids) when the prediction file is wanted. Rank counts: per-row counters in registers for the whole unit
// (reduced over the 16 threads of a row at its end), per-column counters reduced over the 8 rows of a thread and the 4
// row groups of a warp, then added with one global atomic per column and warp.
#include "common.cuh"
#include "snag_internal.h"

namespace snag {

constexpr int L1_BM = 128, L1_BN = 64, L1_BK = 32, L1_LD = L1_BK + 4, L1_STAGES = 3, L1_THREADS = 256;
constexpr int L1_INBOX = L1_BN;
constexpr int L1_STAGE_FLOATS = (L1_BM + L1_BN) * L1_LD;
constexpr int L1_SMEM_BYTES = L1_STAGES * L1_STAGE_FLOATS * 4 + L1_BM * KT_LIST * 8 + L1_BM * L1_INBOX * 8 + L1_BM * 4;
constexpr float L1_U = 5.9604645e-8f;   // 2^-24

__host__ __device__ __forceinline__ float l1_err_per_norm(int Dp) {
  return static_cast<float>((Dp + L1_BK - 1) / L1_BK + 18) * 1.01f * L1_U;
}
// half-width of the band around a ground-truth score (distance units) for a pair with S = ||x||_1 + ||y||_1
__host__ __device__ __forceinline__ float l1_rank_eps(float S, float nv1, float nv2, int use_csls, int Dp) {
  const float a = l1_err_per_norm(Dp) * S;
  if (!use_csls) return a;
  return 2.0f * a + 24.0f * L1_U * (2.0f + S + fabsf(nv1) + fabsf(nv2));
}
// tolerance on c = 1 - d between the sweep and the canonical arithmetic
__host__ __device__ __forceinline__ float l1_c_eps(float S, int Dp) {
  return l1_err_per_norm(Dp) * S + 3.0f * L1_U * (1.0f + S);
}

// the reference's fp32 chain from the distance to the (CSLS) rank distance, one rounding per op
__device__ __forceinline__ float l1_chain(float d, float nv1, float nv2, int use_csls) {
  if (!use_csls) return d;
  const float c = __fsub_rn(1.0f, d);
  return __fsub_rn(1.0f, __fsub_rn(__fmaf_rn(2.0f, c, -nv1), nv2));
}

// canonical cityblock distance: fp64 index-order sum of |x_k - y_k|, rounded once (scipy's cdist stored as fp32)
__device__ __forceinline__ float canonical_l1(const float* __restrict__ x, const float* __restrict__ y, int Dp) {
  const float4* xr = reinterpret_cast<const float4*>(x);
  const float4* yr = reinterpret_cast<const float4*>(y);
  double acc = 0.0;
  for (int c = 0; c < Dp / 4; ++c) {
    const float4 a = __ldg(xr + c), b = __ldg(yr + c);
    acc += fabs(static_cast<double>(a.x) - static_cast<double>(b.x));
    acc += fabs(static_cast<double>(a.y) - static_cast<double>(b.y));
    acc += fabs(static_cast<double>(a.z) - static_cast<double>(b.z));
    acc += fabs(static_cast<double>(a.w) - static_cast<double>(b.w));
  }
  return static_cast<float>(acc);
}

// the sweep's d~ of one pair, operation for operation (see the header)
__device__ __forceinline__ float l1_approx(const float* __restrict__ x, const float* __restrict__ y, int Dp) {
  float tot = 0.f;
  for (int k0 = 0; k0 < Dp; k0 += L1_BK) {
    float ae = 0.f, ao = 0.f;
    for (int k = k0; k < k0 + L1_BK; k += 2) {
      const float x0 = k < Dp ? x[k] : 0.f, x1 = k < Dp ? x[k + 1] : 0.f;
      const float y0 = k < Dp ? y[k] : 0.f, y1 = k < Dp ? y[k + 1] : 0.f;
      ae = __fadd_rn(ae, fabsf(__fsub_rn(x0, y0)));
      ao = __fadd_rn(ao, fabsf(__fsub_rn(x1, y1)));
    }
    tot = __fadd_rn(tot, __fadd_rn(ae, ao));
  }
  return tot;
}

__device__ __forceinline__ float2 absdiff2(float4 a, float4 b, bool hi) {
  const float2 x = hi ? make_float2(a.z, a.w) : make_float2(a.x, a.y);
  const float2 y = hi ? make_float2(b.z, b.w) : make_float2(b.x, b.y);
  const float2 d = __fadd2_rn(x, make_float2(-y.x, -y.y));
  return make_float2(fabsf(d.x), fabsf(d.y));
}

__device__ __forceinline__ void cp_async16(float* smem, const float* gmem, bool valid) {
  const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(valid ? 16 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// ascending list, [0] = admission threshold; the entry met first stays on ties
template <int L>
__device__ __forceinline__ void list_insert(float* val, int* idx, float v, int id) {
  if (!(v > val[0])) return;
  int t = 0;
  while (t + 1 < L && val[t + 1] < v) {
    val[t] = val[t + 1];
    idx[t] = idx[t + 1];
    ++t;
  }
  val[t] = v;
  idx[t] = id;
}

// the same on a register-resident list of values (fully unrolled, no dynamic indexing)
__device__ __forceinline__ void reg_insert(float (&top)[KT_LIST], float v) {
  if (!(v > top[0])) return;
  top[0] = v;
#pragma unroll
  for (int t = 0; t < KT_LIST - 1; ++t) {
    const float a = top[t], b = top[t + 1];
    top[t] = fminf(a, b);
    top[t + 1] = fmaxf(a, b);
  }
}

struct L1Params {
  const float* X;
  const float* Y;
  int n1, n2, Dp;
  int row_blocks, col_tiles, tiles_per_chunk, n_units;
  // row top-KT
  float* part;
  int* part_idx;
  // rank counts
  const float* xn;
  const float* yn;
  const float* nv1;
  const float* nv2;
  const float* g_row;
  const float* g_col;
  int row_gid0, col_gid0, use_csls;
  int* cnt_row;
  int* cnt_col;
  float* top4_val;
  int* top4_idx;
  uint2* band;
  unsigned int* band_cnt;
  unsigned int band_cap;
};

template <bool kRank>
__global__ void __launch_bounds__(L1_THREADS, 1) l1_sweep_kernel(const __grid_constant__ L1Params p) {
  extern __shared__ __align__(16) float l1_smem[];
  float* stage_base = l1_smem;
  float* list_val = l1_smem + L1_STAGES * L1_STAGE_FLOATS;                  // [BM][KT_LIST]
  int* list_idx = reinterpret_cast<int*>(list_val + L1_BM * KT_LIST);       // [BM][KT_LIST]
  float* inbox_val = reinterpret_cast<float*>(list_idx + L1_BM * KT_LIST);  // [BM][INBOX]
  int* inbox_idx = reinterpret_cast<int*>(inbox_val + L1_BM * L1_INBOX);    // [BM][INBOX]
  int* inbox_cnt = inbox_idx + L1_BM * L1_INBOX;                            // [BM]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tx = (lane & 7) | ((warp & 1) << 3);
  const int ty = (lane >> 3) | ((warp >> 1) << 2);
  const int Dp = p.Dp, nk = (Dp + L1_BK - 1) / L1_BK;
  constexpr int LIST = kRank ? 4 : KT_LIST;
  const bool want_list = !kRank || p.top4_val != nullptr;

  for (int unit = blockIdx.x; unit < p.n_units; unit += gridDim.x) {
    const int ch = unit / p.row_blocks, rb = unit - ch * p.row_blocks;
    const int r0 = rb * L1_BM;
    const int ct0 = ch * p.tiles_per_chunk, ct1 = min(ct0 + p.tiles_per_chunk, p.col_tiles);
    const int n_stages = (ct1 - ct0) * nk;
    if (want_list) {
      for (int t = tid; t < L1_BM * LIST; t += L1_THREADS) {
        list_val[t] = -INFINITY;
        list_idx[t] = kRank ? 0x7fffffff : -1;
      }
      if (tid < L1_BM) inbox_cnt[tid] = 0;
    }
    auto issue = [&](int s) {
      const int tile = ct0 + s / nk, k0 = (s % nk) * L1_BK;
      float* sx = stage_base + (s % L1_STAGES) * L1_STAGE_FLOATS;
      float* sy = sx + L1_BM * L1_LD;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int f = tid + q * L1_THREADS, row = f >> 3, kq = (f & 7) * 4;
        const bool ok = r0 + row < p.n1 && k0 + kq < Dp;
        cp_async16(sx + row * L1_LD + kq, ok ? p.X + static_cast<long long>(r0 + row) * Dp + k0 + kq : p.X, ok);
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int f = tid + q * L1_THREADS, row = f >> 3, kq = (f & 7) * 4;
        const long long j = static_cast<long long>(tile) * L1_BN + row;
        const bool ok = j < p.n2 && k0 + kq < Dp;
        cp_async16(sy + row * L1_LD + kq, ok ? p.Y + j * Dp + k0 + kq : p.Y, ok);
      }
    };
#pragma unroll
    for (int s = 0; s < L1_STAGES - 1; ++s) {
      if (s < n_stages) issue(s);
      cp_async_commit();
    }
    float2 acc[8][4];
    float tot[8][4];
    int rcnt[8];
#pragma unroll
    for (int m = 0; m < 8; ++m) {
      rcnt[m] = 0;
#pragma unroll
      for (int q = 0; q < 4; ++q) { acc[m][q] = make_float2(0.f, 0.f); tot[m][q] = 0.f; }
    }
    for (int s = 0; s < n_stages; ++s) {
      cp_async_wait<L1_STAGES - 2>();
      __syncthreads();
      if (s + L1_STAGES - 1 < n_stages) issue(s + L1_STAGES - 1);
      cp_async_commit();
      const float* sx = stage_base + (s % L1_STAGES) * L1_STAGE_FLOATS;
      const float* sy = sx + L1_BM * L1_LD;
#pragma unroll 2
      for (int kq = 0; kq < L1_BK; kq += 4) {
        float4 yv[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) yv[q] = *reinterpret_cast<const float4*>(sy + (tx + 16 * q) * L1_LD + kq);
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          const float4 xv = *reinterpret_cast<const float4*>(sx + (ty + 16 * m) * L1_LD + kq);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            acc[m][q] = __fadd2_rn(acc[m][q], absdiff2(xv, yv[q], false));
            acc[m][q] = __fadd2_rn(acc[m][q], absdiff2(xv, yv[q], true));
          }
        }
      }
#pragma unroll
      for (int m = 0; m < 8; ++m)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          tot[m][q] = __fadd_rn(tot[m][q], __fadd_rn(acc[m][q].x, acc[m][q].y));
          acc[m][q] = make_float2(0.f, 0.f);
        }
      if (s % nk != nk - 1) continue;

      // ---------------------------------------------------------------- tile epilogue
      const int tile = ct0 + s / nk;
      int ccnt[4] = {0, 0, 0, 0};
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        const int rl = ty + 16 * m, i = r0 + rl;
        const bool row_ok = i < p.n1;
        float a_n = 0.f, a_nv = 0.f, a_g = 0.f;
        if (kRank && row_ok) {
          a_n = __ldg(p.xn + i);
          a_nv = p.use_csls ? __ldg(p.nv1 + i) : 0.f;
          a_g = __ldg(p.g_row + i);
        }
        const float thr = want_list ? list_val[rl * LIST] : 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int j = tile * L1_BN + tx + 16 * q;
          if (!row_ok || j >= p.n2) continue;
          const float d = tot[m][q];
          if (!kRank) {
            const float c = __fsub_rn(1.0f, d);
            if (c > thr) {
              const int slot = atomicAdd(inbox_cnt + rl, 1);
              inbox_val[rl * L1_INBOX + slot] = c;
              inbox_idx[rl * L1_INBOX + slot] = j;
            }
            continue;
          }
          const float b_nv = p.use_csls ? __ldg(p.nv2 + j) : 0.f;
          const float dist = l1_chain(d, a_nv, b_nv, p.use_csls);
          const int ig = p.row_gid0 + i, jg = p.col_gid0 + j;
          if (want_list && -dist > thr) {
            const int slot = atomicAdd(inbox_cnt + rl, 1);
            inbox_val[rl * L1_INBOX + slot] = -dist;
            inbox_idx[rl * L1_INBOX + slot] = jg;
          }
          if (ig == jg) continue;                       // the ground-truth pair never competes with itself
          const float eps = l1_rank_eps(a_n + __ldg(p.yn + j), a_nv, b_nv, p.use_csls, Dp);
          uint32_t flags = 0;
          const float dr = __fsub_rn(dist, a_g);
          if (dr < -eps) ++rcnt[m];
          else if (dr <= eps) flags |= 1u;
          const float dc = __fsub_rn(dist, __ldg(p.g_col + j));
          if (dc < -eps) ++ccnt[q];
          else if (dc <= eps) flags |= 2u;
          if (flags) {
            const unsigned int slot = atomicAdd(p.band_cnt, 1u);
            if (slot < p.band_cap) p.band[slot] = make_uint2(static_cast<uint32_t>(i) | (flags << 30), static_cast<uint32_t>(j));
          }
        }
      }
      if (kRank) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          int v = ccnt[q];
          v += __shfl_xor_sync(0xffffffffu, v, 8);
          v += __shfl_xor_sync(0xffffffffu, v, 16);
          const int j = tile * L1_BN + tx + 16 * q;
          if (lane < 8 && v != 0 && j < p.n2) atomicAdd(p.cnt_col + j, v);
        }
      }
      if (want_list) {
        __syncthreads();
        if (tid < L1_BM) {
          const int cnt = inbox_cnt[tid];
          float* lv = list_val + tid * LIST;
          int* li = list_idx + tid * LIST;
          for (int e = 0; e < cnt; ++e) list_insert<LIST>(lv, li, inbox_val[tid * L1_INBOX + e], inbox_idx[tid * L1_INBOX + e]);
          inbox_cnt[tid] = 0;
        }
      }
#pragma unroll
      for (int m = 0; m < 8; ++m)
#pragma unroll
        for (int q = 0; q < 4; ++q) tot[m][q] = 0.f;
    }
    cp_async_wait<0>();
    __syncthreads();

    // ---------------------------------------------------------------- unit epilogue
    if (kRank) {
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        int v = rcnt[m];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        const int i = r0 + ty + 16 * m;
        if ((lane & 7) == 0 && v != 0 && i < p.n1) atomicAdd(p.cnt_row + i, v);
      }
    }
    if (want_list) {
      float* out_v = kRank ? p.top4_val : p.part;
      int* out_i = kRank ? p.top4_idx : p.part_idx;
      for (int t = tid; t < L1_BM * LIST; t += L1_THREADS) {
        const int rl = t / LIST, i = r0 + rl;
        if (i >= p.n1) continue;
        const long long o = (static_cast<long long>(ch) * p.n1 + i) * LIST + (t - rl * LIST);
        out_v[o] = list_val[t];
        if (out_i) out_i[o] = list_idx[t];
      }
      __syncthreads();                                   // the lists are re-initialised for the next unit
    }
  }
}

// ------------------------------------------------------------------------------------------------ plan
// Y chunk kept <= ~32 MB (L2 resident while the row blocks sweep it) and >= ~4 units per SM for the persistent grid.
int l1_plan(int n_rows, int n_cols, int Dp, SimPlan* pl) {
  if (n_rows <= 0 || n_cols <= 0 || Dp <= 0 || (Dp % 8) != 0 || !pl) return SNAG_ERR_SHAPE;
  pl->kblocks = (Dp + L1_BK - 1) / L1_BK;
  pl->row_blocks = (n_rows + L1_BM - 1) / L1_BM;
  pl->col_tiles = (n_cols + L1_BN - 1) / L1_BN;
  long long max_tiles_l2 = (32ll << 20) / (static_cast<long long>(L1_BN) * Dp * 4);
  if (max_tiles_l2 < 1) max_tiles_l2 = 1;
  long long want_chunks = (4ll * num_sms() + pl->row_blocks - 1) / pl->row_blocks;
  if (want_chunks < 1) want_chunks = 1;
  long long tpc = (pl->col_tiles + want_chunks - 1) / want_chunks;
  if (tpc > max_tiles_l2) tpc = max_tiles_l2;
  if (tpc < 1) tpc = 1;
  pl->tiles_per_chunk = static_cast<int>(tpc);
  pl->n_chunks = (pl->col_tiles + pl->tiles_per_chunk - 1) / pl->tiles_per_chunk;
  const long long units = static_cast<long long>(pl->row_blocks) * pl->n_chunks;
  if (units > 0x7fffffffll) return SNAG_ERR_SHAPE;
  pl->n_units = static_cast<int>(units);
  pl->n_lists = pl->n_chunks;
  return SNAG_OK;
}

template <bool kRank>
static int launch_l1_sweep(L1Params& p, cudaStream_t st) {
  if (!p.X || !p.Y) return SNAG_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(p.X) | reinterpret_cast<uintptr_t>(p.Y)) & 15) return SNAG_ERR_ALIGN;
  if (!device_is_sm100()) return SNAG_ERR_DEVICE;
  SimPlan pl;
  const int rc = l1_plan(p.n1, p.n2, p.Dp, &pl);
  if (rc) return rc;
  p.row_blocks = pl.row_blocks;
  p.col_tiles = pl.col_tiles;
  p.tiles_per_chunk = pl.tiles_per_chunk;
  p.n_units = pl.n_units;
  const cudaError_t e = cudaFuncSetAttribute(l1_sweep_kernel<kRank>, cudaFuncAttributeMaxDynamicSharedMemorySize, L1_SMEM_BYTES);
  if (e != cudaSuccess) return static_cast<int>(e);
  const int grid = pl.n_units < num_sms() ? pl.n_units : num_sms();
  l1_sweep_kernel<kRank><<<grid, L1_THREADS, L1_SMEM_BYTES, st>>>(p);
  return static_cast<int>(cudaGetLastError());
}

int launch_l1_rowtopk(const float* X, const float* Y, int n1, int n2, int Dp, float* part, int* part_idx, cudaStream_t st) {
  if (!part) return SNAG_ERR_ARG;
  L1Params p{};
  p.X = X; p.Y = Y; p.n1 = n1; p.n2 = n2; p.Dp = Dp;
  p.part = part; p.part_idx = part_idx;
  return launch_l1_sweep<false>(p, st);
}

int launch_l1_rank_band(const float* X, const float* Y, const float* xn, const float* yn, const float* nv1, const float* nv2,
                        const float* g_row, const float* g_col, int row_gid0, int col_gid0, int n1, int n2, int Dp,
                        int use_csls, int* cnt_row, int* cnt_col, float* top4_val, int* top4_idx, uint2* band,
                        unsigned int* band_cnt, unsigned int band_cap, cudaStream_t st) {
  if (!xn || !yn || !g_row || !g_col || !cnt_row || !cnt_col || !band || !band_cnt) return SNAG_ERR_ARG;
  if (use_csls && (!nv1 || !nv2)) return SNAG_ERR_ARG;
  if ((top4_val == nullptr) != (top4_idx == nullptr)) return SNAG_ERR_ARG;
  if (n1 >= (1 << 30)) return SNAG_ERR_SHAPE;                // band entries keep the row in 30 bits
  L1Params p{};
  p.X = X; p.Y = Y; p.n1 = n1; p.n2 = n2; p.Dp = Dp;
  p.xn = xn; p.yn = yn; p.nv1 = nv1; p.nv2 = nv2; p.g_row = g_row; p.g_col = g_col;
  p.row_gid0 = row_gid0; p.col_gid0 = col_gid0; p.use_csls = use_csls;
  p.cnt_row = cnt_row; p.cnt_col = cnt_col; p.top4_val = top4_val; p.top4_idx = top4_idx;
  p.band = band; p.band_cnt = band_cnt; p.band_cap = band_cap;
  return launch_l1_sweep<true>(p, st);
}

// ------------------------------------------------------------------------------------------------ canonical re-scores
// CSLS neighbourhood means from the KT sweep candidates (as topk_rescore_kernel): every candidate re-scored canonically,
// nv = mean of the k largest c summed largest-first in fp32; a row is verified when its k-th canonical score clears
// every outsider's bound (the list's smallest c~ plus l1_c_eps for the largest possible ||a||_1 + ||b||_1), else it goes
// to the exhaustive pass. 16 lanes per row, one candidate per lane.
__global__ void __launch_bounds__(128) l1_topk_rescore_kernel(const float* __restrict__ A, const float* __restrict__ B, int Dp,
                                                              long long n_rows, const float* __restrict__ an, float bn_max,
                                                              const int* __restrict__ cand_idx, const float* __restrict__ cand_val,
                                                              int k, float* __restrict__ nv, int* __restrict__ flagged,
                                                              int* __restrict__ flagged_cnt, int flagged_cap) {
  const long long gt = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const long long row = gt >> 4;
  const int sub = threadIdx.x & 15;
  const bool live = row < n_rows;
  const long long r = live ? row : n_rows - 1;
  const int id = cand_idx[r * KT_LIST + sub];
  const float tc = cand_val[r * KT_LIST + sub];
  float c = -INFINITY, d = INFINITY;
  if (id >= 0) {
    d = canonical_l1(A + r * Dp, B + static_cast<long long>(id) * Dp, Dp);
    c = __fsub_rn(1.0f, d);
  }
  const unsigned gmask = 0xffffu << (threadIdx.x & 16);
  const unsigned uid = id >= 0 ? static_cast<unsigned>(id) : (0x80000000u | static_cast<unsigned>(sub));
  int rank = 0;
  float tc_min = tc;
#pragma unroll
  for (int o = 0; o < 16; ++o) {
    const int src = (threadIdx.x & 16) | o;
    const float od = __shfl_sync(gmask, d, src);
    const unsigned oid = __shfl_sync(gmask, uid, src);
    const float otc = __shfl_sync(gmask, tc, src);
    rank += (od < d) || (od == d && oid < uid);
    tc_min = fminf(tc_min, otc);
  }
  float sum = 0.f, ck = 0.f;
#pragma unroll
  for (int t = 0; t < KT_LIST; ++t) {
    const unsigned who = __ballot_sync(gmask, rank == t) & gmask;
    const float v = __shfl_sync(gmask, c, __ffs(who) - 1);
    if (t < k) { sum = __fadd_rn(sum, v); ck = v; }
  }
  if (live && sub == 0) {
    nv[row] = __fdiv_rn(sum, static_cast<float>(k));
    // a list that is not full saw every row of B: nothing outside it
    if (tc_min > -INFINITY && !(ck >= tc_min + l1_c_eps(an[row] + bn_max, Dp))) {
      const int slot = atomicAdd(flagged_cnt, 1);
      if (slot < flagged_cap) flagged[slot] = static_cast<int>(row);
    }
  }
}

// exhaustive canonical neighbourhood of the flagged rows: one block per row, threads stride over all rows of B
__global__ void __launch_bounds__(256, 1) l1_topk_exhaustive_kernel(const float* __restrict__ A, const float* __restrict__ B, int Dp,
                                                                 long long n_b, const int* __restrict__ flagged,
                                                                 const int* __restrict__ flagged_cnt, int flagged_cap, int k,
                                                                 float* __restrict__ nv) {
  __shared__ float lists[256 * KT_LIST];
  const int total = min(*flagged_cnt, flagged_cap);
#pragma unroll 1
  for (int f = blockIdx.x; f < total; f += gridDim.x) {
    const long long row = flagged[f];
    float top[KT_LIST];
#pragma unroll
    for (int t = 0; t < KT_LIST; ++t) top[t] = -INFINITY;
    for (long long j = threadIdx.x; j < n_b; j += blockDim.x)
      reg_insert(top, __fsub_rn(1.0f, canonical_l1(A + row * Dp, B + j * Dp, Dp)));
#pragma unroll
    for (int t = 0; t < KT_LIST; ++t) lists[threadIdx.x * KT_LIST + t] = top[t];
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll 1
      for (int o = 1; o < static_cast<int>(blockDim.x); ++o)
#pragma unroll
        for (int t = 0; t < KT_LIST; ++t) reg_insert(top, lists[o * KT_LIST + t]);
      float s = 0.f;
#pragma unroll
      for (int t = 0; t < KT_LIST; ++t)
        if (t < k) s = __fadd_rn(s, top[KT_LIST - 1 - t]);
      nv[row] = __fdiv_rn(s, static_cast<float>(k));
    }
    __syncthreads();
  }
}

// ground-truth distances g[p] of the n pairs (x_p, y_p)
__global__ void __launch_bounds__(128) l1_pair_score_kernel(const float* __restrict__ X, const float* __restrict__ Y, int Dp,
                                                            long long n, const float* __restrict__ nv1,
                                                            const float* __restrict__ nv2, int use_csls, float* __restrict__ g) {
  const long long p = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (p >= n) return;
  const float d = canonical_l1(X + p * Dp, Y + p * Dp, Dp);
  g[p] = l1_chain(d, use_csls ? nv1[p] : 0.f, use_csls ? nv2[p] : 0.f, use_csls);
}

// deferred elements of the rank sweep, judged canonically with the stable-sort tie-break (as band_rescore_kernel)
__global__ void __launch_bounds__(128) l1_band_rescore_kernel(const float* __restrict__ X, const float* __restrict__ Y, int Dp,
                                                              const float* __restrict__ nv1, const float* __restrict__ nv2,
                                                              const float* __restrict__ g_row, const float* __restrict__ g_col,
                                                              int row_gid0, int col_gid0, int use_csls,
                                                              const uint2* __restrict__ band, const unsigned int* __restrict__ band_cnt,
                                                              unsigned int band_cap, int* __restrict__ cnt_row,
                                                              int* __restrict__ cnt_col) {
  const unsigned int total = min(*band_cnt, band_cap);
  for (unsigned int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const uint2 it = band[e];
    const int i = static_cast<int>(it.x & 0x3fffffffu), j = static_cast<int>(it.y);
    const uint32_t flags = it.x >> 30;
    const float d = canonical_l1(X + static_cast<long long>(i) * Dp, Y + static_cast<long long>(j) * Dp, Dp);
    const float dist = l1_chain(d, use_csls ? nv1[i] : 0.f, use_csls ? nv2[j] : 0.f, use_csls);
    const int ig = row_gid0 + i, jg = col_gid0 + j;
    if (flags & 1u) {
      const float g = g_row[i];
      if (dist < g || (dist == g && jg < ig)) atomicAdd(cnt_row + i, 1);
    }
    if (flags & 2u) {
      const float g = g_col[j];
      if (dist < g || (dist == g && ig < jg)) atomicAdd(cnt_col + j, 1);
    }
  }
}

// Prediction file: canonical distances of each row's 4 nearest sweep candidates, ascending with the lower id first on
// ties. The ids are exact when no column outside the list can reach the canonical 3rd: every outsider has
// dist~ >= dist~ of the list's 4th (re-computed here with the sweep's own arithmetic), so its canonical distance is at
// least that minus the band half-width; rows where that does not clear the canonical 3rd are flagged for the
// exhaustive scan.
__global__ void __launch_bounds__(128) l1_top3_rescore_kernel(const float* __restrict__ X, const float* __restrict__ Y, int Dp,
                                                              long long n_rows, const float* __restrict__ xn, float yn_max,
                                                              const float* __restrict__ nv1, const float* __restrict__ nv2,
                                                              float nv2_absmax, int use_csls, const int* __restrict__ cand,
                                                              float* __restrict__ oval, int* __restrict__ oidx,
                                                              int* __restrict__ flagged, int* __restrict__ flagged_cnt) {
  const long long row = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (row >= n_rows) return;
  const int4 ci = __ldg(reinterpret_cast<const int4*>(cand + row * 4));
  int id[4] = {ci.x, ci.y, ci.z, ci.w};
  const float a_nv = use_csls ? nv1[row] : 0.f;
  float v[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    if (id[e] == 0x7fffffff) { v[e] = INFINITY; continue; }
    const float d = canonical_l1(X + row * Dp, Y + static_cast<long long>(id[e]) * Dp, Dp);
    v[e] = l1_chain(d, a_nv, use_csls ? nv2[id[e]] : 0.f, use_csls);
  }
  float bound = INFINITY;                               // least canonical distance any outsider can have
  if (id[3] != 0x7fffffff) {
    const float d4 = l1_approx(X + row * Dp, Y + static_cast<long long>(id[3]) * Dp, Dp);
    const float t4 = l1_chain(d4, a_nv, use_csls ? nv2[id[3]] : 0.f, use_csls);
    bound = __fsub_rn(t4, l1_rank_eps(xn[row] + yn_max, a_nv, nv2_absmax, use_csls, Dp));
  }
#pragma unroll
  for (int a = 1; a < 4; ++a) {
#pragma unroll
    for (int t = a; t > 0; --t) {
      if (v[t] < v[t - 1] || (v[t] == v[t - 1] && id[t] < id[t - 1])) {
        const float tv = v[t]; v[t] = v[t - 1]; v[t - 1] = tv;
        const int ti = id[t]; id[t] = id[t - 1]; id[t - 1] = ti;
      }
    }
  }
  *reinterpret_cast<float4*>(oval + row * 4) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<int4*>(oidx + row * 4) = make_int4(id[0], id[1], id[2], id[3]);
  if (!(bound > v[2])) flagged[atomicAdd(flagged_cnt, 1)] = static_cast<int>(row);
}

// exhaustive canonical 4 nearest (dist, id) of the flagged rows against all n_b rows of Y: one block per row
__global__ void __launch_bounds__(256) l1_top3_exhaustive_kernel(const float* __restrict__ X, const float* __restrict__ Y, int Dp,
                                                                 long long n_b, const float* __restrict__ nv1,
                                                                 const float* __restrict__ nv2, int use_csls,
                                                                 const int* __restrict__ flagged, const int* __restrict__ flagged_cnt,
                                                                 float* __restrict__ oval, int* __restrict__ oidx) {
  __shared__ float sv[256 * 4];
  __shared__ int si[256 * 4];
  const int total = *flagged_cnt;
  for (int f = blockIdx.x; f < total; f += gridDim.x) {
    const long long row = flagged[f];
    const float a_nv = use_csls ? nv1[row] : 0.f;
    float v[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
    int id[4] = {0x7fffffff, 0x7fffffff, 0x7fffffff, 0x7fffffff};
    auto put = [&](float x, int j) {
      if (!(x < v[3] || (x == v[3] && j < id[3]))) return;
      v[3] = x; id[3] = j;
#pragma unroll
      for (int t = 3; t > 0; --t) {
        if (v[t] < v[t - 1] || (v[t] == v[t - 1] && id[t] < id[t - 1])) {
          const float tv = v[t]; v[t] = v[t - 1]; v[t - 1] = tv;
          const int ti = id[t]; id[t] = id[t - 1]; id[t - 1] = ti;
        }
      }
    };
    for (long long j = threadIdx.x; j < n_b; j += blockDim.x) {
      const float d = canonical_l1(X + row * Dp, Y + j * Dp, Dp);
      put(l1_chain(d, a_nv, use_csls ? nv2[j] : 0.f, use_csls), static_cast<int>(j));
    }
#pragma unroll
    for (int t = 0; t < 4; ++t) { sv[threadIdx.x * 4 + t] = v[t]; si[threadIdx.x * 4 + t] = id[t]; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int o = 1; o < static_cast<int>(blockDim.x); ++o)
        for (int t = 0; t < 4; ++t) put(sv[o * 4 + t], si[o * 4 + t]);
      *reinterpret_cast<float4*>(oval + row * 4) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<int4*>(oidx + row * 4) = make_int4(id[0], id[1], id[2], id[3]);
    }
    __syncthreads();
  }
}

static inline int blocks_for(long long items, int block) {
  long long g = (items + block - 1) / block;
  const long long cap = static_cast<long long>(num_sms()) * 16;
  if (g > cap) g = cap;
  return static_cast<int>(g < 1 ? 1 : g);
}

int launch_l1_topk_rescore(const float* A, const float* B, int Dp, long long n_rows, const float* an, float bn_max,
                           const int* cand_idx, const float* cand_val, int k, float* nv, int* flagged, int* flagged_cnt,
                           int flagged_cap, cudaStream_t st) {
  if (!A || !B || !an || !cand_idx || !cand_val || !nv || !flagged || !flagged_cnt || n_rows <= 0 || Dp % 8) return SNAG_ERR_ARG;
  if (k < 1 || k > KT_LIST) return SNAG_ERR_SHAPE;
  const long long threads = n_rows * 16;
  l1_topk_rescore_kernel<<<static_cast<unsigned>((threads + 127) / 128), 128, 0, st>>>(A, B, Dp, n_rows, an, bn_max, cand_idx,
                                                                                       cand_val, k, nv, flagged, flagged_cnt,
                                                                                       flagged_cap);
  return static_cast<int>(cudaGetLastError());
}

int launch_l1_topk_exhaustive(const float* A, const float* B, int Dp, long long n_b, const int* flagged, const int* flagged_cnt,
                              int flagged_cap, int k, float* nv, cudaStream_t st) {
  if (!A || !B || !flagged || !flagged_cnt || !nv || n_b <= 0 || flagged_cap <= 0 || Dp % 8) return SNAG_ERR_ARG;
  if (k < 1 || k > KT_LIST) return SNAG_ERR_SHAPE;
  l1_topk_exhaustive_kernel<<<blocks_for(static_cast<long long>(flagged_cap) * 256, 256), 256, 0, st>>>(
      A, B, Dp, n_b, flagged, flagged_cnt, flagged_cap, k, nv);
  return static_cast<int>(cudaGetLastError());
}

int launch_l1_pair_score(const float* X, const float* Y, int Dp, long long n, const float* nv1, const float* nv2, int use_csls,
                         float* g, cudaStream_t st) {
  if (!X || !Y || !g || n <= 0 || Dp % 8) return SNAG_ERR_ARG;
  if (use_csls && (!nv1 || !nv2)) return SNAG_ERR_ARG;
  l1_pair_score_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, st>>>(X, Y, Dp, n, nv1, nv2, use_csls, g);
  return static_cast<int>(cudaGetLastError());
}

int launch_l1_band_rescore(const float* X, const float* Y, int Dp, const float* nv1, const float* nv2, const float* g_row,
                           const float* g_col, int row_gid0, int col_gid0, int use_csls, const uint2* band,
                           const unsigned int* band_cnt, unsigned int band_cap, int* cnt_row, int* cnt_col, cudaStream_t st) {
  if (!X || !Y || !g_row || !g_col || !band || !band_cnt || !cnt_row || !cnt_col || Dp % 8) return SNAG_ERR_ARG;
  if (use_csls && (!nv1 || !nv2)) return SNAG_ERR_ARG;
  l1_band_rescore_kernel<<<num_sms() * 8, 128, 0, st>>>(X, Y, Dp, nv1, nv2, g_row, g_col, row_gid0, col_gid0, use_csls, band,
                                                        band_cnt, band_cap, cnt_row, cnt_col);
  return static_cast<int>(cudaGetLastError());
}

int launch_l1_top3_rescore(const float* X, const float* Y, int Dp, long long n_rows, long long n_b, const float* xn,
                           float yn_max, const float* nv1, const float* nv2, float nv2_absmax, int use_csls, const int* cand,
                           float* oval, int* oidx, int* flagged, int* flagged_cnt, cudaStream_t st) {
  if (!X || !Y || !xn || !cand || !oval || !oidx || !flagged || !flagged_cnt || n_rows <= 0 || n_b <= 0 || Dp % 8)
    return SNAG_ERR_ARG;
  if (use_csls && (!nv1 || !nv2)) return SNAG_ERR_ARG;
  l1_top3_rescore_kernel<<<static_cast<unsigned>((n_rows + 127) / 128), 128, 0, st>>>(
      X, Y, Dp, n_rows, xn, yn_max, nv1, nv2, nv2_absmax, use_csls, cand, oval, oidx, flagged, flagged_cnt);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return static_cast<int>(e);
  // the scan reads the flagged count on the device: a pass over nothing when every row was verified
  l1_top3_exhaustive_kernel<<<blocks_for(n_rows * 256, 256), 256, 0, st>>>(X, Y, Dp, n_b, nv1, nv2, use_csls, flagged,
                                                                           flagged_cnt, oval, oidx);
  return static_cast<int>(cudaGetLastError());
}

}  // namespace snag
