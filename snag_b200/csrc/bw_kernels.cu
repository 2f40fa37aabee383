// HBM-bound kernels of the SNAG hot path: normalise+gather+cast prologue, Gauss modality noise mask,
// column mean/std, entity-row blend (fwd/bwd), CSLS candidate merge, ground-truth ("diagonal") scores,
// and the materialised CSLS drop-in. All vectorised, coalesced, grid sized from the SM count.
#include <mutex>
#include <type_traits>
#include "common.cuh"
#include "snag_internal.h"

namespace snag {

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011) — counter-based, so the noise is a pure function of
// (seed, stream, global element index) and identical for any row sharding across GPUs.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}
__device__ __forceinline__ float u32_to_unit(uint32_t x) { return static_cast<float>(x >> 8) * (1.0f / 16777216.0f); }
// Box-Muller on two 32-bit draws; u1 in (0,1]
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
  const float u1 = (static_cast<float>(a >> 8) + 1.0f) * (1.0f / 16777216.0f);
  const float u2 = static_cast<float>(b >> 8) * (1.0f / 16777216.0f);
  const float rad = sqrtf(-2.0f * logf(u1));
  float s, c;
  sincospif(2.0f * u2, &s, &c);
  return make_float2(rad * c, rad * s);
}
__device__ __forceinline__ bool philox_row_selected(unsigned long long seed, long long row, float ratio) {
  const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(row), static_cast<uint32_t>(row >> 32), 0u, 1u),
                                make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
  return u32_to_unit(r.x) < ratio;
}

// ------------------------------------------------------------------------------------------------
// a1  SNAG.add_noise_to_embeddings  (model/SNAG.py:66-75)
//   selected rows:  out = (1-rho)*x + rho*(mean + std*z)     every op rounded separately, like torch
//   other rows:     out = x
// mask/z may be injected (bit parity with the reference's own draws) or generated in-kernel (Philox).
//   mask   : uint8 [N] or null          zsel : fp32 [n_sel, F] or null, row order = selected rows
//   selpos : int32 [N] (position of row in zsel; only read for selected rows) or null
// One float4 per thread-iteration; rows are contiguous so every access is a full 16-byte coalesced lane.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) noise_mask_kernel(const float* __restrict__ x, float* __restrict__ out,
                                                         const float* __restrict__ mean, const float* __restrict__ stdv,
                                                         const uint8_t* __restrict__ mask, const float* __restrict__ zsel,
                                                         const int* __restrict__ selpos, long long N, int F, long long ld_in,
                                                         long long ld_out, float ratio, float keep, float rho,
                                                         unsigned long long seed, long long row0) {
  const int f4 = F >> 2;
  const long long total = N * f4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / f4;
    const int c = static_cast<int>(i - row * f4) << 2;
    float4 v = __ldg(reinterpret_cast<const float4*>(x + row * ld_in + c));
    const bool sel = mask ? (mask[row] != 0) : philox_row_selected(seed, row0 + row, ratio);
    if (sel) {
      float4 z;
      if (zsel) {
        z = __ldg(reinterpret_cast<const float4*>(zsel + static_cast<long long>(selpos[row]) * F + c));
      } else {
        const unsigned long long e = static_cast<unsigned long long>(row0 + row) * F + c;   // global element index
        const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(e >> 2), static_cast<uint32_t>(e >> 34), 0u, 2u),
                                      make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
        const float2 a = box_muller(r.x, r.y), b = box_muller(r.z, r.w);
        z = make_float4(a.x, a.y, b.x, b.y);
      }
      const float4 m = __ldg(reinterpret_cast<const float4*>(mean + c));
      const float4 s = __ldg(reinterpret_cast<const float4*>(stdv + c));
      v.x = __fadd_rn(__fmul_rn(keep, v.x), __fmul_rn(rho, __fadd_rn(m.x, __fmul_rn(s.x, z.x))));
      v.y = __fadd_rn(__fmul_rn(keep, v.y), __fmul_rn(rho, __fadd_rn(m.y, __fmul_rn(s.y, z.y))));
      v.z = __fadd_rn(__fmul_rn(keep, v.z), __fmul_rn(rho, __fadd_rn(m.z, __fmul_rn(s.z, z.z))));
      v.w = __fadd_rn(__fmul_rn(keep, v.w), __fmul_rn(rho, __fadd_rn(m.w, __fmul_rn(s.w, z.w))));
    }
    *reinterpret_cast<float4*>(out + row * ld_out + c) = v;
  }
}

// writes the Philox row selection as a uint8 mask (entity_noise_mask of update_noise, SNAG.py:98)
__global__ void philox_rowmask_kernel(uint8_t* mask, long long N, float ratio, unsigned long long seed, long long row0) {
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (i < N) mask[i] = philox_row_selected(seed, row0 + i, ratio) ? 1 : 0;
}

// out[i,:] = mean + std * z(i,:)   (entity_noise of update_noise, SNAG.py:96), z from Philox stream 3
__global__ void __launch_bounds__(256) gauss_fill_kernel(float* __restrict__ out, const float* __restrict__ mean,
                                                         const float* __restrict__ stdv, long long N, int F,
                                                         long long ld, unsigned long long seed, long long row0) {
  const int f4 = F >> 2;
  const long long total = N * f4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / f4;
    const int c = static_cast<int>(i - row * f4) << 2;
    const unsigned long long e = static_cast<unsigned long long>(row0 + row) * F + c;
    const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(e >> 2), static_cast<uint32_t>(e >> 34), 0u, 3u),
                                  make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
    const float2 a = box_muller(r.x, r.y), b = box_muller(r.z, r.w);
    const float4 m = __ldg(reinterpret_cast<const float4*>(mean + c));
    const float4 s = __ldg(reinterpret_cast<const float4*>(stdv + c));
    float4 v;
    v.x = __fadd_rn(m.x, __fmul_rn(s.x, a.x));
    v.y = __fadd_rn(m.y, __fmul_rn(s.y, a.y));
    v.z = __fadd_rn(m.z, __fmul_rn(s.z, b.x));
    v.w = __fadd_rn(m.w, __fmul_rn(s.w, b.y));
    *reinterpret_cast<float4*>(out + row * ld + c) = v;
  }
}

// ------------------------------------------------------------------------------------------------
// a2/a3  column mean and unbiased std over (optionally a subset of) rows  (SNAG.py:77-84, 94-95)
// pass 1: per-(row slab, column) partial sum / sum of squares in fp64 -> atomics into acc[2][F]
// pass 2: mean = S/n, std = sqrt((SS - S*S/n)/(n-1))
// threads map to consecutive columns, so each warp reads 128 contiguous bytes of a row.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) col_stats_partial_kernel(const float* __restrict__ x, const uint8_t* __restrict__ valid,
                                                                long long N, int F, long long ld, int rows_per_slab,
                                                                double* __restrict__ acc, unsigned long long* __restrict__ cnt) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  const long long r0 = static_cast<long long>(blockIdx.y) * rows_per_slab;
  const long long r1 = min(r0 + rows_per_slab, N);
  double s = 0.0, ss = 0.0;
  unsigned long long n = 0;
  if (col < F) {
    for (long long r = r0; r < r1; ++r) {
      if (valid && !valid[r]) continue;
      const double v = static_cast<double>(__ldg(x + r * ld + col));
      s += v;
      ss += v * v;
      ++n;
    }
    atomicAdd(acc + col, s);
    atomicAdd(acc + F + col, ss);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (valid == nullptr) n = static_cast<unsigned long long>(r1 - r0);
    atomicAdd(cnt, n);
  }
}
// float4 variant (F % 4 == 0, 16-byte aligned rows): 4 columns per thread, 8 rows in flight per thread
__global__ void __launch_bounds__(256) col_stats_partial4_kernel(const float* __restrict__ x, const uint8_t* __restrict__ valid,
                                                                 long long N, int F, long long ld, int rows_per_slab,
                                                                 double* __restrict__ acc, unsigned long long* __restrict__ cnt) {
  const int col = (blockIdx.x * blockDim.x + threadIdx.x) << 2;
  const long long r0 = static_cast<long long>(blockIdx.y) * rows_per_slab;
  const long long r1 = min(r0 + rows_per_slab, N);
  double s[4] = {0, 0, 0, 0}, ss[4] = {0, 0, 0, 0};
  unsigned long long n = 0;
  if (col < F) {
    const float* base = x + col;
    long long r = r0;
    for (; r + 8 <= r1; r += 8) {                     // 8 rows (128 bytes per thread) in flight: the kernel is latency bound
      float4 v[8];
      bool ok[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        ok[u] = !valid || valid[r + u];
        v[u] = ok[u] ? __ldg(reinterpret_cast<const float4*>(base + (r + u) * ld)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const double a = v[u].x, b = v[u].y, c = v[u].z, d = v[u].w;
        s[0] += a; s[1] += b; s[2] += c; s[3] += d;
        ss[0] += a * a; ss[1] += b * b; ss[2] += c * c; ss[3] += d * d;
        n += ok[u] ? 1 : 0;
      }
    }
    for (; r < r1; ++r) {
      if (valid && !valid[r]) continue;
      const float4 v = __ldg(reinterpret_cast<const float4*>(base + r * ld));
      const double a = v.x, b = v.y, c = v.z, d = v.w;
      s[0] += a; s[1] += b; s[2] += c; s[3] += d;
      ss[0] += a * a; ss[1] += b * b; ss[2] += c * c; ss[3] += d * d;
      ++n;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      atomicAdd(acc + col + u, s[u]);
      atomicAdd(acc + F + col + u, ss[u]);
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(cnt, n);
}
__global__ void col_stats_final_kernel(const double* __restrict__ acc, const unsigned long long* __restrict__ cnt, int F,
                                       float* __restrict__ mean, float* __restrict__ stdv) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= F) return;
  const double n = static_cast<double>(*cnt);
  const double s = acc[col], ss = acc[F + col];
  const double m = s / n;
  double var = (ss - s * m) / (n - 1.0);
  if (var < 0.0) var = 0.0;
  mean[col] = static_cast<float>(m);
  stdv[col] = static_cast<float>(sqrt(var));
}

// ------------------------------------------------------------------------------------------------
// a4  entity-embedding blend inside MultiModalEncoder.forward (model/SNAG_tools.py:127-128)
//   fwd: out = mask ? a*e + c*noise : e        bwd: grad_e = mask ? a*g : g
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rowblend_fwd_kernel(const float* __restrict__ e, const float* __restrict__ noise,
                                                           const uint8_t* __restrict__ mask, float* __restrict__ out,
                                                           long long N, int D, float a, float c) {
  const int d4 = D >> 2;
  const long long total = N * d4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / d4;
    float4 v = __ldg(reinterpret_cast<const float4*>(e) + i);
    if (mask[row]) {
      const float4 z = __ldg(reinterpret_cast<const float4*>(noise) + i);
      v.x = __fadd_rn(__fmul_rn(a, v.x), __fmul_rn(c, z.x));
      v.y = __fadd_rn(__fmul_rn(a, v.y), __fmul_rn(c, z.y));
      v.z = __fadd_rn(__fmul_rn(a, v.z), __fmul_rn(c, z.z));
      v.w = __fadd_rn(__fmul_rn(a, v.w), __fmul_rn(c, z.w));
    }
    reinterpret_cast<float4*>(out)[i] = v;
  }
}
__global__ void __launch_bounds__(256) rowblend_bwd_kernel(const float* __restrict__ g, const uint8_t* __restrict__ mask,
                                                           float* __restrict__ gin, long long N, int D, float a) {
  const int d4 = D >> 2;
  const long long total = N * d4;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = i / d4;
    float4 v = __ldg(reinterpret_cast<const float4*>(g) + i);
    if (mask[row]) { v.x = __fmul_rn(a, v.x); v.y = __fmul_rn(a, v.y); v.z = __fmul_rn(a, v.z); v.w = __fmul_rn(a, v.w); }
    reinterpret_cast<float4*>(gin)[i] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// prologue: (gather) -> (L2 normalise, F.normalize eps 1e-12) -> round to bf16 -> zero-pad to Dpad,
// plus ||row||^2 of the ROUNDED row (fp64 accumulate, rounded once to fp32): the xn/yn of
// pairwise_distances (src/utils.py:210-212) on exactly the values the tensor cores will see.
// One warp per row; lanes stride the row so loads/stores are coalesced.
// ------------------------------------------------------------------------------------------------
constexpr int PREP_NARROW_MAX_D = 512;            // rows up to this width fit 4 float4 per lane
// One row (warp-cooperative): normalise (optional), round to bf16, zero pad to Dpad, return the fp64 sum of squares of the
// rounded values (valid on every lane; only when WANT_SS). Rows whose width is a multiple of 4 and whose storage is 16-byte
// aligned take the float4 path: the row is read ONCE (up to KEEP float4 per lane stay in registers between the norm and
// the rounding; wider rows re-read the tail from L1), 8-byte stores. The scalar path handles everything else. Both kernels
// below use it, and every lane adds its elements in increasing column order whatever KEEP is, so their outputs are
// bit-identical. KEEP = 4 (D <= 512, the per-modality tables) needs ~40 registers instead of ~100 for KEEP = 16
// (D <= 2048): the kernels are gathers whose only latency hiding is the number of resident warps. dst2 (or null): a second
// copy of the row (the repeated part of the stacked ICL operand).
template <int KEEP, bool WANT_SS>
__device__ __forceinline__ double prep_row(const float* __restrict__ src, int D, int Dpad, int normalize,
                                           __nv_bfloat16* __restrict__ dst, __nv_bfloat16* __restrict__ dst2, int lane,
                                           bool vec4) {
  double acc = 0.0;
  if (vec4) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
    const int n4 = D >> 2, np4 = Dpad >> 2;
    float4 v[KEEP];
    float ss = 0.f;
#pragma unroll
    for (int u = 0; u < KEEP; ++u) {
      const int c4 = lane + 32 * u;
      v[u] = c4 < n4 ? __ldg(s4 + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
      ss = __fmaf_rn(v[u].x, v[u].x, ss); ss = __fmaf_rn(v[u].y, v[u].y, ss);
      ss = __fmaf_rn(v[u].z, v[u].z, ss); ss = __fmaf_rn(v[u].w, v[u].w, ss);
    }
    for (int c4 = lane + 32 * KEEP; c4 < n4; c4 += 32) {
      const float4 t = __ldg(s4 + c4);
      ss = __fmaf_rn(t.x, t.x, ss); ss = __fmaf_rn(t.y, t.y, ss); ss = __fmaf_rn(t.z, t.z, ss); ss = __fmaf_rn(t.w, t.w, ss);
    }
    float denom = 1.0f;
    if (normalize) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
      denom = fmaxf(sqrtf(ss), 1e-12f);
    }
    auto emit = [&](int c4, float4 t) {
      if (normalize) { t.x = __fdiv_rn(t.x, denom); t.y = __fdiv_rn(t.y, denom); t.z = __fdiv_rn(t.z, denom); t.w = __fdiv_rn(t.w, denom); }
      const __nv_bfloat162 lo = __floats2bfloat162_rn(t.x, t.y), hi = __floats2bfloat162_rn(t.z, t.w);
      const uint2 packed = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
      *reinterpret_cast<uint2*>(dst + 4 * c4) = packed;
      if (dst2) *reinterpret_cast<uint2*>(dst2 + 4 * c4) = packed;
      if (WANT_SS) {
        const double a = __bfloat162float(lo.x), b = __bfloat162float(lo.y), c = __bfloat162float(hi.x), d = __bfloat162float(hi.y);
        acc += a * a; acc += b * b; acc += c * c; acc += d * d;
      }
    };
#pragma unroll
    for (int u = 0; u < KEEP; ++u) {
      const int c4 = lane + 32 * u;
      if (c4 < np4) emit(c4, v[u]);                   // beyond n4 the registers hold zeros: the padding
    }
    for (int c4 = lane + 32 * KEEP; c4 < np4; c4 += 32)
      emit(c4, c4 < n4 ? __ldg(s4 + c4) : make_float4(0.f, 0.f, 0.f, 0.f));
  } else {
    float denom = 1.0f;
    if (normalize) {
      float ss = 0.f;
      for (int c = lane; c < D; c += 32) { const float v = __ldg(src + c); ss = __fmaf_rn(v, v, ss); }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
      denom = fmaxf(sqrtf(ss), 1e-12f);
    }
    for (int c = lane; c < Dpad; c += 32) {
      float v = 0.f;
      if (c < D) v = normalize ? __fdiv_rn(__ldg(src + c), denom) : __ldg(src + c);
      const __nv_bfloat16 b = __float2bfloat16_rn(v);
      dst[c] = b;
      if (dst2) dst2[c] = b;
      if (WANT_SS) {
        const double w = static_cast<double>(__bfloat162float(b));
        acc += w * w;
      }
    }
  }
  if (WANT_SS) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  }
  return acc;
}

template <int KEEP>
__global__ void __launch_bounds__(256) prep_bf16_kernel(const float* __restrict__ emb, long long ld,
                                                        const long long* __restrict__ idx, int n, int D, int normalize,
                                                        __nv_bfloat16* __restrict__ out, int Dpad,
                                                        float* __restrict__ norm2) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n) return;
  const float* src = emb + (idx ? idx[warp] : static_cast<long long>(warp)) * ld;
  const bool vec4 = (D % 4 == 0) && (ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(emb) & 15) == 0);
  const double acc = prep_row<KEEP, true>(src, D, Dpad, normalize, out + static_cast<long long>(warp) * Dpad, nullptr, lane, vec4);
  if (lane == 0 && norm2) norm2[warp] = static_cast<float>(acc);
}

// Prologue of the fp32 evaluation: the rows prep_bf16 rounds, kept in fp32 (the canonical re-scores read them), and a
// three-term bf16 split of them for the tensor-core sweeps: h = bf16(x), m = bf16(x - h) (x - h is exact in fp32), laid
// out as [m | h | h] for sources (side 0) and [h | m | h] for targets (side 1), so that one bf16 contraction of width
// 3 Dpad forms m_x h_y + h_x m_y + h_x h_y in either operand order. The normalisation repeats prep_row's arithmetic
// step for step — each lane's fp32 sum of squares over its columns (float4 path or scalar path under the same
// condition), the same butterfly, the same __fdiv_rn — so x is bit for bit what prep_bf16 rounds and h is its output.
__global__ void __launch_bounds__(256) prep_split_kernel(const float* __restrict__ emb, long long ld,
                                                         const long long* __restrict__ idx, int n, int D, int normalize,
                                                         int side, float* __restrict__ rows, __nv_bfloat16* __restrict__ split,
                                                         int Dpad) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n) return;
  const float* src = emb + (idx ? idx[warp] : static_cast<long long>(warp)) * ld;
  float denom = 1.0f;
  if (normalize) {
    const bool vec4 = (D % 4 == 0) && (ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(emb) & 15) == 0);
    float ss = 0.f;
    if (vec4) {
      const float4* s4 = reinterpret_cast<const float4*>(src);
      for (int c4 = lane; c4 < (D >> 2); c4 += 32) {
        const float4 t = __ldg(s4 + c4);
        ss = __fmaf_rn(t.x, t.x, ss); ss = __fmaf_rn(t.y, t.y, ss); ss = __fmaf_rn(t.z, t.z, ss); ss = __fmaf_rn(t.w, t.w, ss);
      }
    } else {
      for (int c = lane; c < D; c += 32) { const float v = __ldg(src + c); ss = __fmaf_rn(v, v, ss); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    denom = fmaxf(sqrtf(ss), 1e-12f);
  }
  float* row = rows + static_cast<long long>(warp) * Dpad;
  __nv_bfloat16* sp = split + static_cast<long long>(warp) * 3 * Dpad;
  __nv_bfloat16* h0 = sp + (side ? 0 : Dpad);
  __nv_bfloat16* m0 = sp + (side ? Dpad : 0);
  __nv_bfloat16* h1 = sp + 2 * Dpad;
  for (int c = lane; c < Dpad; c += 32) {
    float v = 0.f;
    if (c < D) v = normalize ? __fdiv_rn(__ldg(src + c), denom) : __ldg(src + c);
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const __nv_bfloat16 m = __float2bfloat16_rn(__fsub_rn(v, __bfloat162float(h)));
    row[c] = v;
    h0[c] = h;
    m0[c] = m;
    h1[c] = h;
  }
}

// ------------------------------------------------------------------------------------------------
// Batched prologue / epilogue of the loss layer: the 2 + 2M icl_loss calls of a step share the batch of links, so the
// stacked operands of ALL calls are built by one launch and the gradients of all calls go back through one launch
// (at the reference's batch of 3500 the per-call launches of these two small kernels were 20 % of the step).
//   stack_prep : S3_p = [ z_p[idx_l] ; z_p[idx_r] ; z_p[idx_l] ], z = F.normalize(emb_p) rounded to bf16, every part
//                zero padded to Bp rows and Dpad_p columns (side a sweeps rows [Bp, 3Bp), side b rows [0, 2Bp))
//   scatter_many : normalize_bwd_scatter for both sides of every problem
// grid.y = problem (x side); one warp per row.
// ------------------------------------------------------------------------------------------------
constexpr int MANY_MAX = 16;
struct StackPrepArgs {
  const float* emb[MANY_MAX];
  long long ld[MANY_MAX];
  __nv_bfloat16* out[MANY_MAX];
  int D[MANY_MAX];
  int Dpad[MANY_MAX];
};
// One warp per row of [a ; b]; the warp of row i of part a also writes row i of the third part (the repeated a), so every
// source row is read and normalised once.
template <int KEEP>
__global__ void __launch_bounds__(256) icl_stack_prep_kernel(const __grid_constant__ StackPrepArgs a,
                                                             const long long* __restrict__ idx_l,
                                                             const long long* __restrict__ idx_r, int B, int Bp,
                                                             int normalize) {
  const int p = blockIdx.y;
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;       // row of the first two parts of S3_p
  const int lane = threadIdx.x & 31;
  if (r >= 2 * Bp) return;
  const int part = r >= Bp ? 1 : 0, i = r - part * Bp;
  const int D = a.D[p], Dpad = a.Dpad[p];
  __nv_bfloat16* dst = a.out[p] + static_cast<long long>(r) * Dpad;
  __nv_bfloat16* dst2 = part == 0 ? dst + 2ll * Bp * Dpad : nullptr;
  if (i >= B) {
    for (int c = lane; c < Dpad; c += 32) {
      dst[c] = __float2bfloat16_rn(0.f);
      if (dst2) dst2[c] = __float2bfloat16_rn(0.f);
    }
    return;
  }
  const float* src = a.emb[p] + (part == 1 ? idx_r[i] : idx_l[i]) * a.ld[p];
  const bool vec4 = (D % 4 == 0) && (a.ld[p] % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.emb[p]) & 15) == 0);
  prep_row<KEEP, false>(src, D, Dpad, normalize, dst, dst2, lane, vec4);
}

// Split stacks of the fp32 loss route: row r of [a ; b ; a] as [m | h | h | m | h] (5 Dpad bf16 per row), h = bf16(z),
// m = bf16(z - h), z normalised with prep_split_kernel's arithmetic step for step (so h is bit for bit what
// icl_stack_prep_kernel writes and m what prep_split_kernel writes). The side-0 window (columns [0, 3 Dpad)) is
// [m | h | h], the side-1 window (columns [2 Dpad, 5 Dpad)) is [h | m | h]: a contraction of a side-0 row with a side-1
// row forms m_i h_j + h_i m_j + h_i h_j. One warp per row of [a ; b]; the warp of row i of part a also writes the repeated
// row 2 Bp + i. a.Dpad[p] is the width of one block (Dpad of the table).
__global__ void __launch_bounds__(256) icl_stack_prep_split_kernel(const __grid_constant__ StackPrepArgs a,
                                                                   const long long* __restrict__ idx_l,
                                                                   const long long* __restrict__ idx_r, int B, int Bp,
                                                                   int normalize) {
  const int p = blockIdx.y;
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= 2 * Bp) return;
  const int part = r >= Bp ? 1 : 0, i = r - part * Bp;
  const int D = a.D[p], Dpad = a.Dpad[p];
  const long long ld = 5ll * Dpad;
  __nv_bfloat16* dst = a.out[p] + static_cast<long long>(r) * ld;
  __nv_bfloat16* dst2 = part == 0 ? dst + 2ll * Bp * ld : nullptr;
  const float* src = i < B ? a.emb[p] + (part == 1 ? idx_r[i] : idx_l[i]) * a.ld[p] : nullptr;
  float denom = 1.0f;
  if (src && normalize) {
    const bool vec4 = (D % 4 == 0) && (a.ld[p] % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.emb[p]) & 15) == 0);
    float ss = 0.f;
    if (vec4) {
      const float4* s4 = reinterpret_cast<const float4*>(src);
      for (int c4 = lane; c4 < (D >> 2); c4 += 32) {
        const float4 t = __ldg(s4 + c4);
        ss = __fmaf_rn(t.x, t.x, ss); ss = __fmaf_rn(t.y, t.y, ss); ss = __fmaf_rn(t.z, t.z, ss); ss = __fmaf_rn(t.w, t.w, ss);
      }
    } else {
      for (int c = lane; c < D; c += 32) { const float v = __ldg(src + c); ss = __fmaf_rn(v, v, ss); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    denom = fmaxf(sqrtf(ss), 1e-12f);
  }
  for (int c = lane; c < Dpad; c += 32) {
    float v = 0.f;
    if (src && c < D) v = normalize ? __fdiv_rn(__ldg(src + c), denom) : __ldg(src + c);
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const __nv_bfloat16 m = __float2bfloat16_rn(__fsub_rn(v, __bfloat162float(h)));
    dst[c] = m; dst[Dpad + c] = h; dst[2 * Dpad + c] = h; dst[3 * Dpad + c] = m; dst[4 * Dpad + c] = h;
    if (dst2) {
      dst2[c] = m; dst2[Dpad + c] = h; dst2[2 * Dpad + c] = h; dst2[3 * Dpad + c] = m; dst2[4 * Dpad + c] = h;
    }
  }
}

struct ScatterManyArgs {
  const float* emb[MANY_MAX];
  long long ld[MANY_MAX];
  int D[MANY_MAX];
  const float* dz[2 * MANY_MAX];          // [2 p + side]
  long long ld_dz[MANY_MAX];
  int n_parts[MANY_MAX];
  long long part_stride[MANY_MAX];
  float* demb[MANY_MAX];
  long long ld_demb[MANY_MAX];
  int vec4[MANY_MAX];                     // rows of emb / dz / demb are 16-byte aligned and D % 4 == 0: float4 path
};
// one 128-bit reduction instead of four 32-bit ones (sm_90+): the scatter is bound by the number of atomic operations
__device__ __forceinline__ void red_add_v4(float* addr, const float4& v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__global__ void __launch_bounds__(256) normalize_bwd_scatter_many_kernel(const __grid_constant__ ScatterManyArgs a,
                                                                         const long long* __restrict__ idx_l,
                                                                         const long long* __restrict__ idx_r, int n,
                                                                         int normalize) {
  const int p = blockIdx.y >> 1, side = blockIdx.y & 1;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n) return;
  const long long row = side ? idx_r[warp] : idx_l[warp];
  const int D = a.D[p], n_parts = a.n_parts[p];
  const long long part_stride = a.part_stride[p];
  const float* src = a.emb[p] + row * a.ld[p];
  const float* g0 = a.dz[2 * p + side] + static_cast<long long>(warp) * a.ld_dz[p];
  float* dst = a.demb[p] + row * a.ld_demb[p];
  auto g_at = [&](int c) {
    float v = __ldg(g0 + c);
    for (int q = 1; q < n_parts; ++q) v += __ldg(g0 + q * part_stride + c);
    return v;
  };
  if (a.vec4[p]) {
    const int D4 = D >> 2;
    const float4* src4 = reinterpret_cast<const float4*>(src);
    auto g4_at = [&](int c4) {
      float4 v = __ldg(reinterpret_cast<const float4*>(g0) + c4);
      for (int q = 1; q < n_parts; ++q) {
        const float4 w = __ldg(reinterpret_cast<const float4*>(g0 + q * part_stride) + c4);
        v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
      }
      return v;
    };
    if (!normalize) {
      for (int c4 = lane; c4 < D4; c4 += 32) red_add_v4(dst + 4 * c4, g4_at(c4));
      return;
    }
    float ss = 0.f, eg = 0.f;
    for (int c4 = lane; c4 < D4; c4 += 32) {
      const float4 v = __ldg(src4 + c4), gq = g4_at(c4);
      ss = __fmaf_rn(v.x, v.x, ss); ss = __fmaf_rn(v.y, v.y, ss); ss = __fmaf_rn(v.z, v.z, ss); ss = __fmaf_rn(v.w, v.w, ss);
      eg = __fmaf_rn(v.x, gq.x, eg); eg = __fmaf_rn(v.y, gq.y, eg); eg = __fmaf_rn(v.z, gq.z, eg); eg = __fmaf_rn(v.w, gq.w, eg);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      ss += __shfl_xor_sync(0xffffffffu, ss, o);
      eg += __shfl_xor_sync(0xffffffffu, eg, o);
    }
    const float nrm = sqrtf(ss);
    const bool ok = nrm > 1e-12f;
    const float inv = ok ? 1.0f / nrm : 1e12f;
    const float k = ok ? eg * inv * inv * inv : 0.f;
    for (int c4 = lane; c4 < D4; c4 += 32) {
      const float4 v = __ldg(src4 + c4), gq = g4_at(c4);
      red_add_v4(dst + 4 * c4, make_float4(__fmaf_rn(-v.x, k, gq.x * inv), __fmaf_rn(-v.y, k, gq.y * inv),
                                           __fmaf_rn(-v.z, k, gq.z * inv), __fmaf_rn(-v.w, k, gq.w * inv)));
    }
    return;
  }
  if (!normalize) {
    for (int c = lane; c < D; c += 32) atomicAdd(dst + c, g_at(c));
    return;
  }
  float ss = 0.f, eg = 0.f;
  for (int c = lane; c < D; c += 32) {
    const float v = __ldg(src + c);
    ss = __fmaf_rn(v, v, ss);
    eg = __fmaf_rn(v, g_at(c), eg);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    eg += __shfl_xor_sync(0xffffffffu, eg, o);
  }
  const float nrm = sqrtf(ss);
  if (nrm > 1e-12f) {
    const float inv = 1.0f / nrm;
    const float k = eg * inv * inv * inv;
    for (int c = lane; c < D; c += 32) atomicAdd(dst + c, __fmaf_rn(-__ldg(src + c), k, g_at(c) * inv));
  } else {
    for (int c = lane; c < D; c += 32) atomicAdd(dst + c, g_at(c) * 1e12f);
  }
}

// ------------------------------------------------------------------------------------------------
// f2  Joint (fusion-output) embeddings, model/SNAG_tools.py:44-49:
//   joint   [i, off_m + c] = w_ent[i, m] * e_m[i, c] / max(||e_m[i]||, 1e-12)      (per-entity attention weights)
//   joint_fz[i, off_m + c] = w_glob[m]   * e_m[i, c] / max(||e_m[i]||, 1e-12)      (softmax(weight_raw))
// for the M present modalities, concatenated along the row. One warp per (entity, modality): the reference's
// 2M normalise + 2M scale + 2 cat kernels become one pass that reads every table once and writes both outputs.
// Backward (same grid): with G = w_ent*dJ + w_glob*dJfz, z = e/||e||:
//   de = (G - z (z.G)) / ||e||,   dw_ent[i,m] = z.dJ,   dw_glob[m] += z.dJfz  (block-reduced, one atomic per block)
// ------------------------------------------------------------------------------------------------
struct JointTabs {
  const float* e[SNAG_MAX_MODAL];
  float* de[SNAG_MAX_MODAL];
  int width[SNAG_MAX_MODAL];
  int off[SNAG_MAX_MODAL];
};

__global__ void __launch_bounds__(256) joint_fuse_fwd_kernel(JointTabs tabs, long long N, const float* __restrict__ w_ent,
                                                             long long ldw, const float* __restrict__ w_glob,
                                                             float* __restrict__ joint, float* __restrict__ joint_fz,
                                                             long long ld_out) {
  const int m = blockIdx.y;
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= N) return;
  const int D = tabs.width[m];
  const float* src = tabs.e[m] + i * D;
  float ss = 0.f;
  for (int c = lane; c < D; c += 32) { const float v = __ldg(src + c); ss = __fmaf_rn(v, v, ss); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float denom = fmaxf(sqrtf(ss), 1e-12f);
  const float w1 = (joint && w_ent) ? w_ent[i * ldw + m] : 0.f;
  const float w2 = (joint_fz && w_glob) ? w_glob[m] : 0.f;
  const long long o0 = i * ld_out + tabs.off[m];
  for (int c = lane; c < D; c += 32) {
    const float z = __fdiv_rn(__ldg(src + c), denom);
    if (joint) joint[o0 + c] = __fmul_rn(w1, z);
    if (joint_fz) joint_fz[o0 + c] = __fmul_rn(w2, z);
  }
}

__global__ void __launch_bounds__(256) joint_fuse_bwd_kernel(JointTabs tabs, long long N, const float* __restrict__ w_ent,
                                                             long long ldw, const float* __restrict__ w_glob,
                                                             const float* __restrict__ d_joint,
                                                             const float* __restrict__ d_joint_fz, long long ld_out,
                                                             float* __restrict__ d_w_ent, float* __restrict__ d_w_glob) {
  __shared__ float red[8];
  const int m = blockIdx.y;
  const int wib = threadIdx.x >> 5;
  const long long i = blockIdx.x * static_cast<long long>(blockDim.x >> 5) + wib;
  const int lane = threadIdx.x & 31;
  float a2n = 0.f;                       // this warp's contribution to dw_glob[m]
  if (i < N) {
    const int D = tabs.width[m];
    const float* src = tabs.e[m] + i * D;
    const long long o0 = i * ld_out + tabs.off[m];
    float ss = 0.f, a1 = 0.f, a2 = 0.f;
    for (int c = lane; c < D; c += 32) {
      const float v = __ldg(src + c);
      ss = __fmaf_rn(v, v, ss);
      if (d_joint) a1 = __fmaf_rn(v, __ldg(d_joint + o0 + c), a1);
      if (d_joint_fz) a2 = __fmaf_rn(v, __ldg(d_joint_fz + o0 + c), a2);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      ss += __shfl_xor_sync(0xffffffffu, ss, o);
      a1 += __shfl_xor_sync(0xffffffffu, a1, o);
      a2 += __shfl_xor_sync(0xffffffffu, a2, o);
    }
    const float nrm = sqrtf(ss);
    const bool clamped = !(nrm > 1e-12f);
    const float inv = clamped ? 1e12f : 1.0f / nrm;
    const float w1 = (d_joint && w_ent) ? w_ent[i * ldw + m] : 0.f;
    const float w2 = (d_joint_fz && w_glob) ? w_glob[m] : 0.f;
    if (lane == 0 && d_w_ent) d_w_ent[i * ldw + m] = a1 * inv;
    a2n = a2 * inv;
    // z.G / ||e|| = (w1 a1 + w2 a2) inv^2 ; with a clamped denominator z = e * 1e12 is linear in e: de = G * 1e12
    const float k = clamped ? 0.f : (w1 * a1 + w2 * a2) * inv * inv * inv;
    float* dst = tabs.de[m] + i * D;
    for (int c = lane; c < D; c += 32) {
      float G = 0.f;
      if (d_joint) G = __fmaf_rn(w1, __ldg(d_joint + o0 + c), G);
      if (d_joint_fz) G = __fmaf_rn(w2, __ldg(d_joint_fz + o0 + c), G);
      dst[c] = __fmaf_rn(-__ldg(src + c), k, G * inv);
    }
  }
  if (d_w_glob) {
    if (lane == 0) red[wib] = a2n;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) t += red[w];
      atomicAdd(d_w_glob + m, t);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Backward of (gather ->) F.normalize, scattered into the embedding gradient (model/SNAG_loss.py:60-64 seen from
// autograd): for z = e / max(||e||, 1e-12) and upstream g = dL/dz,
//   dL/de = g / ||e|| - e (e.g) / ||e||^3        accumulated into demb[idx[r]] (atomic: a row may be linked twice)
// One warp per gathered row; replaces torch's normalize-backward chain + index_select backward.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) normalize_bwd_scatter_kernel(const float* __restrict__ emb, long long ld,
                                                                    const long long* __restrict__ idx, int n, int D,
                                                                    int normalize, const float* __restrict__ dz,
                                                                    long long ld_dz, int n_parts, long long part_stride,
                                                                    float* __restrict__ demb, long long ld_demb) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n) return;
  const long long row = idx ? idx[warp] : static_cast<long long>(warp);
  const float* src = emb + row * ld;
  const float* g0 = dz + static_cast<long long>(warp) * ld_dz;
  // dz may arrive as n_parts partial sums (column splits of the fused backward), part_stride floats apart: they are
  // added in split order, so the result does not depend on how the splits were scheduled
  auto g_at = [&](int c) {
    float v = __ldg(g0 + c);
    for (int q = 1; q < n_parts; ++q) v += __ldg(g0 + q * part_stride + c);
    return v;
  };
  if (!normalize) {                                 // plain gather: its backward is the scatter-add alone
    float* d0 = demb + row * ld_demb;
    for (int c = lane; c < D; c += 32) atomicAdd(d0 + c, g_at(c));
    return;
  }
  float ss = 0.f, eg = 0.f;
  for (int c = lane; c < D; c += 32) {
    const float v = __ldg(src + c);
    ss = __fmaf_rn(v, v, ss);
    eg = __fmaf_rn(v, g_at(c), eg);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    eg += __shfl_xor_sync(0xffffffffu, eg, o);
  }
  const float nrm = sqrtf(ss);
  float* dst = demb + row * ld_demb;
  if (nrm > 1e-12f) {
    const float inv = 1.0f / nrm;
    const float k = eg * inv * inv * inv;
    for (int c = lane; c < D; c += 32) atomicAdd(dst + c, __fmaf_rn(-__ldg(src + c), k, g_at(c) * inv));
  } else {                                         // clamped denominator: z = e / eps is linear in e
    for (int c = lane; c < D; c += 32) atomicAdd(dst + c, g_at(c) * 1e12f);
  }
}

// ------------------------------------------------------------------------------------------------
// CSLS neighbourhood means: merge the per-chunk ascending KT-lists of every row, keep the KT largest,
// nv[row] = (sum of the k largest, accumulated largest-first in fp32) / k     (src/utils.py:431-432)
// Optionally also emits the merged KT-list (descending) for the cross-GPU candidate exchange.
// ------------------------------------------------------------------------------------------------
// canonical dot product of two bf16 rows: fp64 accumulation in index order, rounded once to fp32 (the oracle's s_ij)
// Dpad is a multiple of 64: every trip fetches 64 contiguous bytes of each row with four 16-byte loads issued back to
// back (whole 32-byte sectors; with one 16-byte load per trip the second half of every sector had usually left L1
// before its turn came — the re-scores are gathers of whole rows and bandwidth bound), then accumulates in index order.
__device__ __forceinline__ float canonical_dot(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ y, int Dpad) {
  const uint4* xr = reinterpret_cast<const uint4*>(x);
  const uint4* yr = reinterpret_cast<const uint4*>(y);
  const int n = Dpad / 8;                        // 16-byte words per row; a multiple of 8
  double acc = 0.0;
  // software pipelined: the 64 bytes of the NEXT trip are requested before the 32 dependent fp64 FMAs of this one run
  // (ncu, profiles/r03o: the re-score kernels issue on 10 % of the cycles and wait on loads for the rest — one trip's
  // loads in flight per thread are not enough to cover the latency of a gather of whole rows)
  uint4 a[4], b[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) { a[u] = __ldg(xr + u); b[u] = __ldg(yr + u); }
  for (int c = 0; c < n; c += 4) {
    uint4 na[4], nb[4];
    const int cn = c + 4 < n ? c + 4 : c;        // the last trip re-requests its own (cached) words: no branch in the loop
#pragma unroll
    for (int u = 0; u < 4; ++u) { na[u] = __ldg(xr + cn + u); nb[u] = __ldg(yr + cn + u); }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t aw[4] = {a[u].x, a[u].y, a[u].z, a[u].w}, bw[4] = {b[u].x, b[u].y, b[u].z, b[u].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float a0 = __uint_as_float(aw[e] << 16), a1 = __uint_as_float(aw[e] & 0xffff0000u);
        const float b0 = __uint_as_float(bw[e] << 16), b1 = __uint_as_float(bw[e] & 0xffff0000u);
        acc = fma(static_cast<double>(a0), static_cast<double>(b0), acc);
        acc = fma(static_cast<double>(a1), static_cast<double>(b1), acc);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) { a[u] = na[u]; b[u] = nb[u]; }
  }
  return static_cast<float>(acc);
}
// The same for fp32 rows (the fp32 evaluation): an fp32 x fp32 product is exact in fp64 as well, so fma(double, double,
// acc) in index order is still the oracle's arithmetic. Same pipelining: 64 bytes of each row per trip (16 elements).
__device__ __forceinline__ float canonical_dot(const float* __restrict__ x, const float* __restrict__ y, int Dpad) {
  const float4* xr = reinterpret_cast<const float4*>(x);
  const float4* yr = reinterpret_cast<const float4*>(y);
  const int n = Dpad / 4;                        // 16-byte words per row; a multiple of 16
  double acc = 0.0;
  float4 a[4], b[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) { a[u] = __ldg(xr + u); b[u] = __ldg(yr + u); }
  for (int c = 0; c < n; c += 4) {
    float4 na[4], nb[4];
    const int cn = c + 4 < n ? c + 4 : c;
#pragma unroll
    for (int u = 0; u < 4; ++u) { na[u] = __ldg(xr + cn + u); nb[u] = __ldg(yr + cn + u); }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      acc = fma(static_cast<double>(a[u].x), static_cast<double>(b[u].x), acc);
      acc = fma(static_cast<double>(a[u].y), static_cast<double>(b[u].y), acc);
      acc = fma(static_cast<double>(a[u].z), static_cast<double>(b[u].z), acc);
      acc = fma(static_cast<double>(a[u].w), static_cast<double>(b[u].w), acc);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) { a[u] = na[u]; b[u] = nb[u]; }
  }
  return static_cast<float>(acc);
}
// the reference's fp32 chain from s to the (CSLS) distance, one rounding per op (simgemm.cuh has the same two helpers)
__device__ __forceinline__ float canonical_dist(float s, float xn, float yn, float nv1, float nv2, int use_csls) {
  const float d = fmaxf(__fmaf_rn(-2.0f, s, __fadd_rn(xn, yn)), 0.0f);
  if (!use_csls) return d;
  const float c = __fsub_rn(1.0f, d);
  return __fsub_rn(1.0f, __fsub_rn(__fmaf_rn(2.0f, c, -nv1), nv2));
}

template <bool kIdx>
__device__ __forceinline__ void topk_pair_insert(float (&top)[KT_LIST], int (&topi)[kIdx ? KT_LIST : 1], float v, int id) {
  // ascending list, top[0] = admission threshold; ties: the entry met first stays (callers feed ids in ascending order
  // within a list, lists in ascending column order)
  if (!(v > top[0])) return;
  top[0] = v;
  if (kIdx) topi[0] = id;
#pragma unroll
  for (int t = 0; t < KT_LIST - 1; ++t) {
    const bool sw = top[t] > top[t + 1];
    const float a = top[t], b = top[t + 1];
    top[t] = sw ? b : a;
    top[t + 1] = sw ? a : b;
    if (kIdx) {
      const int ia = topi[t], ib = topi[t + 1];
      topi[t] = sw ? ib : ia;
      topi[t + 1] = sw ? ia : ib;
    }
  }
}

template <bool kIdx>
__global__ void __launch_bounds__(128) topk_merge_mean_kernel(const float* __restrict__ part, const int* __restrict__ part_idx,
                                                              int n_lists, long long n_rows, int k, float* __restrict__ nv,
                                                              float* __restrict__ cand_out, int* __restrict__ cand_idx_out) {
  const long long row = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (row >= n_rows) return;
  float top[KT_LIST];
  int topi[kIdx ? KT_LIST : 1];
#pragma unroll
  for (int t = 0; t < KT_LIST; ++t) top[t] = -INFINITY;
  if (kIdx) {
#pragma unroll
    for (int t = 0; t < KT_LIST; ++t) topi[t] = -1;
  }
  for (int l = 0; l < n_lists; ++l) {
    const long long o0 = (static_cast<long long>(l) * n_rows + row) * KT_LIST;
    const float4* src = reinterpret_cast<const float4*>(part + o0);
    const int4* srci = reinterpret_cast<const int4*>(part_idx + (kIdx ? o0 : 0));
#pragma unroll
    for (int q = 0; q < KT_LIST / 4; ++q) {
      const float4 v4 = __ldg(src + q);
      const float vv[4] = {v4.x, v4.y, v4.z, v4.w};
      int ii[4] = {0, 0, 0, 0};
      if (kIdx) {
        const int4 i4 = __ldg(srci + q);
        ii[0] = i4.x; ii[1] = i4.y; ii[2] = i4.z; ii[3] = i4.w;
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) topk_pair_insert<kIdx>(top, topi, vv[e], ii[e]);
    }
  }
  if (nv) {
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < KT_LIST; ++t)
      if (t < k) s = __fadd_rn(s, top[KT_LIST - 1 - t]);
    nv[row] = __fdiv_rn(s, static_cast<float>(k));
  }
  if (cand_out) {
    float4* o = reinterpret_cast<float4*>(cand_out + row * KT_LIST);
#pragma unroll
    for (int q = 0; q < KT_LIST / 4; ++q) o[q] = make_float4(top[4 * q], top[4 * q + 1], top[4 * q + 2], top[4 * q + 3]);
  }
  if (kIdx && cand_idx_out) {
    int4* o = reinterpret_cast<int4*>(cand_idx_out + row * KT_LIST);
#pragma unroll
    for (int q = 0; q < KT_LIST / 4; ++q) o[q] = make_int4(topi[4 * q], topi[4 * q + 1], topi[4 * q + 2], topi[4 * q + 3]);
  }
}

// ------------------------------------------------------------------------------------------------
// Canonical CSLS neighbourhood means. cand_idx[row][KT] are the rows of B that the tensor-core sweep ranked highest
// for row `row` of A (cand_val their tensor-core scores c = 1 - d, ascending, -inf / -1 padded). Every candidate is
// re-scored with the canonical arithmetic (fp64 index-order dot, fp32 chain); nv = mean of the k largest, summed
// largest-first in fp32 (src/utils.py:431-432). The result equals the oracle's whenever no column outside the list
// can belong to the true top-k: every outsider's tensor-core score is <= the list's smallest, so its canonical score
// is <= that + delta; the row is verified if its k-th canonical score clears that bound (or the list is not full).
// Unverified rows (plateaus of near-equal scores wider than KT - k) are appended to `flagged` for the exhaustive
// pass below. One warp handles two rows: 16 lanes per row, one candidate per lane.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) topk_rescore_kernel(const T* __restrict__ A, const T* __restrict__ B,
                                                           int Dpad, long long n_rows, const float* __restrict__ an,
                                                           const float* __restrict__ bn, const int* __restrict__ cand_idx,
                                                           const float* __restrict__ cand_val, int k, float delta,
                                                           const float* __restrict__ outsider_bound,
                                                           float* __restrict__ nv, int* __restrict__ flagged,
                                                           int* __restrict__ flagged_cnt, int flagged_cap,
                                                           float* __restrict__ best_d, int* __restrict__ best_idx) {
  const long long gt = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  const long long row = gt >> 4;
  const int sub = threadIdx.x & 15;
  const bool live = row < n_rows;
  const long long r = live ? row : n_rows - 1;
  const int id = cand_idx[r * KT_LIST + sub];
  const float tc = cand_val[r * KT_LIST + sub];
  float c = -INFINITY, d = INFINITY;
  if (id >= 0) {
    const float s = canonical_dot(A + r * Dpad, B + static_cast<long long>(id) * Dpad, Dpad);
    d = fmaxf(__fmaf_rn(-2.0f, s, __fadd_rn(an[r], bn[id])), 0.0f);
    c = __fsub_rn(1.0f, d);
  }
  // rank of this lane's candidate among the 16: by distance ascending (= score descending), lower id first on equal
  // distances (torch.argmin / a stable sort), empty slots last — a permutation of 0..15
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
  if (live && rank == 0 && best_idx) {
    best_idx[row] = id;
    best_d[row] = d;
  }
  // largest-first fp32 sum of the k largest: lane with rank t contributes at step t
  float sum = 0.f, ck = 0.f;
#pragma unroll
  for (int t = 0; t < KT_LIST; ++t) {
    const unsigned who = __ballot_sync(gmask, rank == t) & gmask;
    const float v = __shfl_sync(gmask, c, __ffs(who) - 1);
    if (t < k) { sum = __fadd_rn(sum, v); ck = v; }
  }
  if (live && sub == 0) {
    nv[row] = __fdiv_rn(sum, static_cast<float>(k));
    // What bounds the tensor-core score of every row of B that is NOT in the list: the list's smallest entry when all
    // KT slots are taken; otherwise the admission threshold the list was collected under (outsider_bound: the two-sweep
    // path only streams elements at or above the column's sample-derived threshold, so a short list says nothing about
    // what lies just below that threshold), or nothing at all (-inf: the list saw every row of B).
    const bool full = tc_min > -INFINITY;                 // all KT slots hold a real candidate
    const float ob = full ? tc_min : (outsider_bound ? outsider_bound[row] : -INFINITY);
    if (ob > -INFINITY && !(ck >= ob + delta)) {
      const int slot = atomicAdd(flagged_cnt, 1);
      if (slot < flagged_cap) flagged[slot] = static_cast<int>(row);
    }
  }
}

// Exhaustive canonical neighbourhood of the flagged rows: one block per flagged row, threads stride over all rows of
// B keeping their own k largest canonical scores; lists are merged through shared memory.
template <typename T>
__global__ void __launch_bounds__(256) topk_exhaustive_kernel(const T* __restrict__ A, const T* __restrict__ B,
                                                              int Dpad, long long n_b, const float* __restrict__ an,
                                                              const float* __restrict__ bn, const int* __restrict__ flagged,
                                                              const int* __restrict__ flagged_cnt, int flagged_cap, int k,
                                                              float* __restrict__ nv, float* __restrict__ best_d,
                                                              int* __restrict__ best_idx) {
  __shared__ float lists[256 * KT_LIST];
  __shared__ float bd_s[256];
  __shared__ int bi_s[256];
  const int total = min(*flagged_cnt, flagged_cap);
  for (int f = blockIdx.x; f < total; f += gridDim.x) {
    const long long row = flagged[f];
    const float a = an[row];
    float top[KT_LIST];
    int dummy[1];
#pragma unroll
    for (int t = 0; t < KT_LIST; ++t) top[t] = -INFINITY;
    float bd = INFINITY;
    int bi = 0x7fffffff;
    for (long long j = threadIdx.x; j < n_b; j += blockDim.x) {
      const float s = canonical_dot(A + row * Dpad, B + j * Dpad, Dpad);
      const float dd = fmaxf(__fmaf_rn(-2.0f, s, __fadd_rn(a, bn[j])), 0.0f);
      if (dd < bd) { bd = dd; bi = static_cast<int>(j); }               // j ascending per thread: strict keeps the first
      topk_pair_insert<false>(top, dummy, __fsub_rn(1.0f, dd), 0);
    }
#pragma unroll
    for (int t = 0; t < KT_LIST; ++t) lists[threadIdx.x * KT_LIST + t] = top[t];
    bd_s[threadIdx.x] = bd;
    bi_s[threadIdx.x] = bi;
    __syncthreads();
    if (threadIdx.x == 0 && best_idx) {
      for (int o = 1; o < static_cast<int>(blockDim.x); ++o)
        if (bd_s[o] < bd || (bd_s[o] == bd && bi_s[o] < bi)) { bd = bd_s[o]; bi = bi_s[o]; }
      best_d[row] = bd;
      best_idx[row] = bi;
    }
    if (threadIdx.x == 0) {
      for (int o = 1; o < static_cast<int>(blockDim.x); ++o)
        for (int t = 0; t < KT_LIST; ++t) topk_pair_insert<false>(top, dummy, lists[o * KT_LIST + t], 0);
      float s = 0.f;
#pragma unroll
      for (int t = 0; t < KT_LIST; ++t)
        if (t < k) s = __fadd_rn(s, top[KT_LIST - 1 - t]);
      nv[row] = __fdiv_rn(s, static_cast<float>(k));
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// ground-truth scores: g[p] = CSLS distance of pair p = (x_p, y_p), with the dot product accumulated
// in fp64 in index order and rounded once to fp32 (the oracle's definition of s_pp), then the same
// fp32 chain as the fused epilogue. One thread per pair; 16-byte loads.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) pair_score_kernel(const T* __restrict__ X, const T* __restrict__ Y,
                                                         int Dpad, long long n, const float* __restrict__ xn,
                                                         const float* __restrict__ yn, const float* __restrict__ nv1,
                                                         const float* __restrict__ nv2, int use_csls, float* __restrict__ g,
                                                         float* __restrict__ s_out) {
  const long long p = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (p >= n) return;
  float s;
  if constexpr (std::is_same<T, float>::value) {
    s = canonical_dot(X + p * Dpad, Y + p * Dpad, Dpad);
  } else {
    const uint4* xr = reinterpret_cast<const uint4*>(X + p * Dpad);
    const uint4* yr = reinterpret_cast<const uint4*>(Y + p * Dpad);
    double acc = 0.0;
    for (int c = 0; c < Dpad / 8; ++c) {
      const uint4 a = __ldg(xr + c), b = __ldg(yr + c);
      const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        // bf16 -> fp32 is a 16-bit shift; low half first (little endian = lower column index)
        const float a0 = __uint_as_float(aw[e] << 16), a1 = __uint_as_float(aw[e] & 0xffff0000u);
        const float b0 = __uint_as_float(bw[e] << 16), b1 = __uint_as_float(bw[e] & 0xffff0000u);
        acc = fma(static_cast<double>(a0), static_cast<double>(b0), acc);
        acc = fma(static_cast<double>(a1), static_cast<double>(b1), acc);
      }
    }
    s = static_cast<float>(acc);
  }
  if (s_out) s_out[p] = s;
  const float t = __fadd_rn(xn[p], yn[p]);
  const float d = fmaxf(__fmaf_rn(-2.0f, s, t), 0.0f);
  if (!use_csls) { g[p] = d; return; }
  const float c = __fsub_rn(1.0f, d);
  const float u = __fmaf_rn(2.0f, c, -nv1[p]);
  g[p] = __fsub_rn(1.0f, __fsub_rn(u, nv2[p]));
}

// ------------------------------------------------------------------------------------------------
// Deferred elements of the rank sweep (EpiRankBand): every (row, column) whose margin to a ground-truth score was
// inside the band is judged here with the canonical arithmetic and the stable-sort tie-break (main.py:400-429 with
// torch.sort(stable=True)): one thread per element.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) band_rescore_kernel(const T* __restrict__ X, const T* __restrict__ Y,
                                                           int Dpad, const float* __restrict__ xn, const float* __restrict__ yn,
                                                           const float* __restrict__ nv1, const float* __restrict__ nv2,
                                                           const float* __restrict__ g_row, const float* __restrict__ g_col,
                                                           int row_gid0, int col_gid0, int use_csls,
                                                           const uint2* __restrict__ band, const unsigned int* __restrict__ band_cnt,
                                                           unsigned int band_cap, int* __restrict__ cnt_row, int* __restrict__ cnt_col,
                                                           const int* __restrict__ row_gids, int swapped) {
  // row_gids: the rows of X are a gathered subset (global pair ids listed); swapped: X holds TARGETS and Y sources (the
  // recount of selected targets runs the sweep with the operands exchanged) — the fp32 CSLS chain subtracts the SOURCE's
  // neighbourhood mean first, so the roles must be put back before it is evaluated
  const unsigned int total = min(*band_cnt, band_cap);
  for (unsigned int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const uint2 it = band[e];
    const int i = static_cast<int>(it.x & 0x3fffffffu), j = static_cast<int>(it.y);
    const uint32_t flags = it.x >> 30;
    const float s = canonical_dot(X + static_cast<long long>(i) * Dpad, Y + static_cast<long long>(j) * Dpad, Dpad);
    const float dist = swapped ? canonical_dist(s, yn[j], xn[i], use_csls ? nv2[j] : 0.f, use_csls ? nv1[i] : 0.f, use_csls)
                               : canonical_dist(s, xn[i], yn[j], use_csls ? nv1[i] : 0.f, use_csls ? nv2[j] : 0.f, use_csls);
    const int ig = row_gids != nullptr ? row_gids[i] : row_gid0 + i, jg = col_gid0 + j;
    if (ig == jg) continue;
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

// ------------------------------------------------------------------------------------------------
// One-pass evaluation (EpiOnePass in simgemm.cuh): the rank verdicts of main.py:400-429 are taken on the elements the
// single sweep streamed out, against thresholds known only after the sweep.
//   spec_bounds     : from the sample pre-pass lists (KT per entity, ascending, tensor-core c) and the canonical c of
//                     the entity's own pair:  lo = mean of the k largest of the sample - delta  (a LOWER bound of the
//                     final neighbourhood mean: every order statistic of the full population dominates the sample's),
//                     hi = a GUESS of an upper bound: the sample's order statistics shifted by `shift` times their
//                     tail scale (exponential-tail extrapolation from the sample to the population: an order statistic
//                     of rank r in a sample of m of n entities sits at population rank r n / m, i.e. ln(n/m) tail scales
//                     lower than the population's rank-r value), the own pair merged in.
//                     A guess that turns out too low is detected after the sweep and costs an exhaustive recount of that
//                     entity — never a wrong rank.
//   rank_judge      : every streamed element against the final constants of EpiRankBand: outside the band -> counted,
//                     inside -> deferred to band_rescore (canonical arithmetic + stable tie-break), exactly like sweep 2.
//   rank_exhaustive : canonical recount of listed rows of A against all rows of B (fp64 index-order dots).
// ------------------------------------------------------------------------------------------------
__global__ void spec_bounds_kernel(const float* __restrict__ cand, long long n, int k, const float* __restrict__ cdiag,
                                   float shift, float delta, float* __restrict__ lo, float* __restrict__ hi) {
  const long long j = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (j >= n) return;
  float v[KT_LIST];
#pragma unroll
  for (int t = 0; t < KT_LIST; ++t) v[t] = cand[j * KT_LIST + t];
  float sl = 0.f;
#pragma unroll
  for (int t = 0; t < KT_LIST; ++t)
    if (t < k) sl += v[KT_LIST - 1 - t];
  lo[j] = sl / static_cast<float>(k) - delta;
  // tail scale of the sample: mean exceedance of the 15 largest over the 16th (the maximum-likelihood estimate for an
  // exponential tail; far less noisy than the range v_1 - v_16). +inf when the sample list is not full.
  float exc = 0.f;
#pragma unroll
  for (int t = 1; t < KT_LIST; ++t) exc += v[t] - v[0];
  const float sh = shift * (exc / static_cast<float>(KT_LIST - 1));
  // merged top-k of {v_t + sh} and the own pair
  const float cd = cdiag[j];
  float sh_sum = 0.f;
  bool used = false;
  int taken = 0;
#pragma unroll
  for (int t = KT_LIST - 1; t >= 0; --t) {
    if (taken >= k) break;
    const float x = v[t] + sh;
    if (!used && cd > x) { sh_sum += cd; used = true; ++taken; if (taken >= k) break; }
    sh_sum += x;
    ++taken;
  }
  hi[j] = sh_sum / static_cast<float>(k) + delta;
}

__global__ void __launch_bounds__(256) rank_judge_kernel(const uint2* __restrict__ rk_stream, const int* __restrict__ rk_stream_row,
                                                         const int* __restrict__ rk_cnt, int rk_cap, const float* __restrict__ R,
                                                         const float* __restrict__ Rp, const float* __restrict__ C,
                                                         const float* __restrict__ Cp, const unsigned char* __restrict__ row_ok,
                                                         const unsigned char* __restrict__ col_ok, float eps, int row_gid0,
                                                         int col_gid0, int* __restrict__ cnt_row, int* __restrict__ cnt_col,
                                                         uint2* __restrict__ band, unsigned int* __restrict__ band_cnt,
                                                         unsigned int band_cap, int* __restrict__ overflow) {
  const int cta = blockIdx.y;
  int cnt = rk_cnt[cta];
  if (cnt > rk_cap) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(overflow, 1);
    cnt = rk_cap;
  }
  const uint2* sp = rk_stream + static_cast<long long>(cta) * rk_cap;
  const int* rp = rk_stream_row + static_cast<long long>(cta) * rk_cap;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < cnt; e += gridDim.x * blockDim.x) {
    const uint2 it = sp[e];
    const int j = static_cast<int>(it.x), i = rp[e];
    if (row_gid0 + i == col_gid0 + j) continue;          // the ground-truth pair never competes with itself
    const float s = __uint_as_float(it.y);
    uint32_t flags = 0;
    if (row_ok[i]) {
      const float x = __fsub_rn(s, C[j]), r = R[i];
      if (x > r + eps) atomicAdd(cnt_row + i, 1);
      else if (x > r - eps) flags |= 1u;
    }
    if (col_ok[j]) {
      const float y = __fsub_rn(s, Rp[i]), c = Cp[j];
      if (y > c + eps) atomicAdd(cnt_col + j, 1);
      else if (y > c - eps) flags |= 2u;
    }
    if (flags) {
      const unsigned int slot = atomicAdd(band_cnt, 1u);
      if (slot < band_cap) band[slot] = make_uint2(static_cast<uint32_t>(i) | (flags << 30), static_cast<uint32_t>(j));
    }
  }
}

constexpr int RX_ROWS = 8;       // listed rows one block of rank_exhaustive handles together (B is read once for all of them)
template <typename T>
__global__ void __launch_bounds__(256) rank_exhaustive_kernel(const T* __restrict__ A, const T* __restrict__ B,
                                                              int Dpad, long long n_b, const float* __restrict__ an,
                                                              const float* __restrict__ bn, const float* __restrict__ nva,
                                                              const float* __restrict__ nvb, const float* __restrict__ g,
                                                              const int* __restrict__ rows, int n_rows, int a_gid0, int b_gid0,
                                                              int use_csls, int swapped, int* __restrict__ cnt) {
  extern __shared__ float a_s[];                          // [RX_ROWS][Dpad] fp32 copies of the listed rows
  __shared__ int cnt_s[RX_ROWS];
  const int r0 = blockIdx.x * RX_ROWS;
  const int nr = min(RX_ROWS, n_rows - r0);
  for (int t = threadIdx.x; t < RX_ROWS * Dpad; t += blockDim.x) {
    const int r = t / Dpad, c = t - r * Dpad;
    a_s[t] = r < nr ? static_cast<float>(A[static_cast<long long>(rows[r0 + r]) * Dpad + c]) : 0.f;
  }
  if (threadIdx.x < RX_ROWS) cnt_s[threadIdx.x] = 0;
  __syncthreads();
  float a_n[RX_ROWS], a_nv[RX_ROWS], a_g[RX_ROWS];
  int a_id[RX_ROWS], my[RX_ROWS];
#pragma unroll
  for (int r = 0; r < RX_ROWS; ++r) {
    const int row = r < nr ? rows[r0 + r] : rows[r0];
    a_n[r] = an[row];
    a_nv[r] = use_csls ? nva[row] : 0.f;
    a_g[r] = g[row];
    a_id[r] = a_gid0 + row;
    my[r] = 0;
  }
  const long long per = (n_b + gridDim.y - 1) / gridDim.y;
  const long long j0 = blockIdx.y * per, j1 = min(n_b, j0 + per);
  for (long long j = j0 + threadIdx.x; j < j1; j += blockDim.x) {
    double acc[RX_ROWS];
#pragma unroll
    for (int r = 0; r < RX_ROWS; ++r) acc[r] = 0.0;
    for (int c = 0; c < Dpad / 8; ++c) {
      float bf[8];
      if constexpr (std::is_same<T, float>::value) {
        const float4* br = reinterpret_cast<const float4*>(B + j * Dpad);
        const float4 b0 = __ldg(br + 2 * c), b1 = __ldg(br + 2 * c + 1);
        bf[0] = b0.x; bf[1] = b0.y; bf[2] = b0.z; bf[3] = b0.w; bf[4] = b1.x; bf[5] = b1.y; bf[6] = b1.z; bf[7] = b1.w;
      } else {
        const uint4 b = __ldg(reinterpret_cast<const uint4*>(B + j * Dpad) + c);
        const uint32_t bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          bf[2 * e] = __uint_as_float(bw[e] << 16);
          bf[2 * e + 1] = __uint_as_float(bw[e] & 0xffff0000u);
        }
      }
#pragma unroll
      for (int r = 0; r < RX_ROWS; ++r) {
        const float4 a0 = *reinterpret_cast<const float4*>(a_s + r * Dpad + c * 8);
        const float4 a1 = *reinterpret_cast<const float4*>(a_s + r * Dpad + c * 8 + 4);
        const float af[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          if constexpr (std::is_same<T, float>::value)
            acc[r] = fma(static_cast<double>(af[e]), static_cast<double>(bf[e]), acc[r]);   // exact product in fp64
          else   // a bf16 x bf16 product is exact in fp32, so exact product + one fp64 rounding == fma(double a, double b, acc)
            acc[r] = __dadd_rn(acc[r], static_cast<double>(__fmul_rn(af[e], bf[e])));
        }
      }
    }
    const float b_n = bn[j], b_nv = use_csls ? nvb[j] : 0.f;
    const int b_id = b_gid0 + static_cast<int>(j);
#pragma unroll
    for (int r = 0; r < RX_ROWS; ++r) {
      const float sdot = static_cast<float>(acc[r]);
      const float dist = swapped ? canonical_dist(sdot, b_n, a_n[r], b_nv, a_nv[r], use_csls)
                                 : canonical_dist(sdot, a_n[r], b_n, a_nv[r], b_nv, use_csls);
      if (b_id != a_id[r] && (dist < a_g[r] || (dist == a_g[r] && b_id < a_id[r]))) ++my[r];
    }
  }
#pragma unroll
  for (int r = 0; r < RX_ROWS; ++r) {
    int v = my[r];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v != 0) atomicAdd(cnt_s + r, v);
  }
  __syncthreads();
  if (threadIdx.x < nr && cnt_s[threadIdx.x] != 0) atomicAdd(cnt + rows[r0 + threadIdx.x], cnt_s[threadIdx.x]);
}

// canonical dot products of an explicit list of (row of X, row of Y) pairs — the re-score of the similarity entries a
// thresholded sweep collected (unsupervised seed induction, src/data.py:367-375)
template <typename T>
__global__ void __launch_bounds__(128) pairs_dot_kernel(const T* __restrict__ X, const T* __restrict__ Y,
                                                        int Dpad, const int* __restrict__ rows, const int* __restrict__ cols,
                                                        long long n_pairs, float* __restrict__ s_out) {
  const long long p = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (p >= n_pairs) return;
  s_out[p] = canonical_dot(X + static_cast<long long>(rows[p]) * Dpad, Y + static_cast<long long>(cols[p]) * Dpad, Dpad);
}

// ||row||^2 of fp32 rows in fp64, in index order, rounded once (oracle_norm2): the canonical dot of the row with itself.
// (prep_row adds lane-strided partial sums: in that order fp64 sums of fp32 squares round differently now and then.)
__global__ void __launch_bounds__(128) row_norm2_kernel(const float* __restrict__ rows, int Dpad, long long n,
                                                        float* __restrict__ norm2) {
  const long long p = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (p >= n) return;
  norm2[p] = canonical_dot(rows + p * Dpad, rows + p * Dpad, Dpad);
}

// merge per-list top-4 candidate lists of each row (x descending = nearest first, column id ascending on ties)
__global__ void __launch_bounds__(128) top4_merge_kernel(const float* __restrict__ val, const int* __restrict__ idx, int n_lists,
                                                         long long n_rows, float* __restrict__ oval, int* __restrict__ oidx) {
  const long long row = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (row >= n_rows) return;
  float v[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
  int id[4] = {0x7fffffff, 0x7fffffff, 0x7fffffff, 0x7fffffff};
  for (int l = 0; l < n_lists; ++l) {
    const float4 cv = __ldg(reinterpret_cast<const float4*>(val + (static_cast<long long>(l) * n_rows + row) * 4));
    const int4 ci = __ldg(reinterpret_cast<const int4*>(idx + (static_cast<long long>(l) * n_rows + row) * 4));
    const float cvv[4] = {cv.x, cv.y, cv.z, cv.w};
    const int cii[4] = {ci.x, ci.y, ci.z, ci.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (cii[e] == 0x7fffffff) continue;
      if (cvv[e] > v[3] || (cvv[e] == v[3] && cii[e] < id[3])) {
        v[3] = cvv[e]; id[3] = cii[e];
#pragma unroll
        for (int t = 3; t > 0; --t) {
          if (v[t] > v[t - 1] || (v[t] == v[t - 1] && id[t] < id[t - 1])) {
            const float tv = v[t]; v[t] = v[t - 1]; v[t - 1] = tv;
            const int ti = id[t]; id[t] = id[t - 1]; id[t - 1] = ti;
          }
        }
      }
    }
  }
  *reinterpret_cast<float4*>(oval + row * 4) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<int4*>(oidx + row * 4) = make_int4(id[0], id[1], id[2], id[3]);
}

// canonical distances of each row's (up to) four nearest candidates, sorted ascending (column id ascending on ties):
// entries 0..2 are ret1..ret3 of the prediction file (main.py:411)
template <typename T>
__global__ void __launch_bounds__(128) top3_rescore_kernel(const T* __restrict__ X, const T* __restrict__ Y,
                                                           int Dpad, long long n_rows, const float* __restrict__ xn,
                                                           const float* __restrict__ yn, const float* __restrict__ nv1,
                                                           const float* __restrict__ nv2, int use_csls,
                                                           const int* __restrict__ cand, float* __restrict__ oval,
                                                           int* __restrict__ oidx) {
  const long long row = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (row >= n_rows) return;
  const int4 ci = __ldg(reinterpret_cast<const int4*>(cand + row * 4));
  int id[4] = {ci.x, ci.y, ci.z, ci.w};
  float v[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    if (id[e] == 0x7fffffff) { v[e] = INFINITY; continue; }
    const float s = canonical_dot(X + row * Dpad, Y + static_cast<long long>(id[e]) * Dpad, Dpad);
    v[e] = canonical_dist(s, xn[row], yn[id[e]], use_csls ? nv1[row] : 0.f, use_csls ? nv2[id[e]] : 0.f, use_csls);
  }
#pragma unroll
  for (int a = 1; a < 4; ++a) {           // insertion sort on (dist, id)
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
}

// merge per-chunk top-3 (value asc, index asc on ties) lists of each row

// ICL forward finalize: lse = log(sum over chunks) + 1/tau ; nll = lse - pos/tau
__global__ void icl_finalize_kernel(const float* __restrict__ rowsum_part, int n_chunks, int B, int Bp,
                                    const float* __restrict__ pos, float inv_tau, float* __restrict__ lse,
                                    float* __restrict__ nll) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  float s = 0.f;
  for (int c = 0; c < n_chunks; ++c) s += rowsum_part[static_cast<long long>(c) * Bp + i];
  const float l = logf(s) + inv_tau;
  lse[i] = l;
  nll[i] = l - pos[i] * inv_tau;
}

// ------------------------------------------------------------------------------------------------
// a9  csls_sim on a MATERIALISED similarity matrix (src/utils.py:417-435) — the drop-in that must take and
// return an [n1, n2] fp32 matrix. Three bandwidth passes:
//   rows : one warp per row, lanes stride the row (coalesced); each lane keeps its KT largest -> part_r[32][n1][KT]
//   cols : one thread per column per row slab (consecutive threads = consecutive columns, coalesced)
//          -> part_c[slabs][n2][KT]
//   (topk_merge_mean_kernel reduces both to nv1 / nv2, largest-first fp32 sum / k)
//   apply: out = (2*sim - nv1[i]) - nv2[j], float4 wide
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void topk_insert(float (&top)[KT_LIST], float v) {
  if (v > top[0]) {
    top[0] = v;
#pragma unroll
    for (int t = 0; t < KT_LIST - 1; ++t) {
      const float lo = fminf(top[t], top[t + 1]), hi = fmaxf(top[t], top[t + 1]);
      top[t] = lo;
      top[t + 1] = hi;
    }
  }
}
__global__ void __launch_bounds__(256) matrix_row_topk_kernel(const float* __restrict__ sim, long long n1, long long n2,
                                                              long long ld, float* __restrict__ part) {
  const long long row = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n1) return;
  float top[KT_LIST];
#pragma unroll
  for (int t = 0; t < KT_LIST; ++t) top[t] = -INFINITY;
  const float* r = sim + row * ld;
  for (long long j = lane; j < n2; j += 32) topk_insert(top, __ldg(r + j));
  float4* o = reinterpret_cast<float4*>(part + (static_cast<long long>(lane) * n1 + row) * KT_LIST);
#pragma unroll
  for (int q = 0; q < KT_LIST / 4; ++q) o[q] = make_float4(top[4 * q], top[4 * q + 1], top[4 * q + 2], top[4 * q + 3]);
}
__global__ void __launch_bounds__(128) matrix_col_topk_kernel(const float* __restrict__ sim, long long n1, long long n2,
                                                              long long ld, int rows_per_slab, float* __restrict__ part) {
  const long long col = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (col >= n2) return;
  const long long r0 = static_cast<long long>(blockIdx.y) * rows_per_slab;
  const long long r1 = min(r0 + rows_per_slab, n1);
  float top[KT_LIST];
#pragma unroll
  for (int t = 0; t < KT_LIST; ++t) top[t] = -INFINITY;
  for (long long i = r0; i < r1; ++i) topk_insert(top, __ldg(sim + i * ld + col));
  float4* o = reinterpret_cast<float4*>(part + (static_cast<long long>(blockIdx.y) * n2 + col) * KT_LIST);
#pragma unroll
  for (int q = 0; q < KT_LIST / 4; ++q) o[q] = make_float4(top[4 * q], top[4 * q + 1], top[4 * q + 2], top[4 * q + 3]);
}
__global__ void __launch_bounds__(256) csls_apply_kernel(const float* __restrict__ sim, const float* __restrict__ nv1,
                                                         const float* __restrict__ nv2, float* __restrict__ out, long long n1,
                                                         long long n2, long long ld, long long ld_out) {
  const long long total = n1 * n2;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long i = e / n2, j = e - i * n2;
    const float u = __fmaf_rn(2.0f, __ldg(sim + i * ld + j), -__ldg(nv1 + i));
    out[i * ld_out + j] = __fsub_rn(u, __ldg(nv2 + j));
  }
}

// ------------------------------------------------------------------------------------------------
// Column neighbourhoods of the two-sweep evaluation (see EpiRowColTopK in simgemm.cuh)
//   col_threshold : from the merged sample lists (ascending, KT per column) take the k-th largest c as the
//                   admission threshold, lowered by 2e-6 so that a last-bit difference between the sample
//                   pre-pass and the main sweep can never drop a true neighbour; b_j is its s-space form.
//   col_cand_finalize : nv[j] = mean of the k largest candidates of column j (largest-first fp32 sum / k);
//                   sets *overflow if a column received more candidates than its buffer holds.
// ------------------------------------------------------------------------------------------------
__global__ void col_threshold_kernel(const float* __restrict__ cand, long long n, int k, const float* __restrict__ yn,
                                     float* __restrict__ colthr, float* __restrict__ colb) {
  const long long j = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (j >= n) return;
  const float kth = cand[j * KT_LIST + (KT_LIST - k)];      // lists are ascending: index KT-k is the k-th largest
  const float thr = kth - 2e-6f;                             // -inf stays -inf: everything is admitted
  colthr[j] = thr;
  colb[j] = __fmaf_rn(0.5f, __fadd_rn(__fadd_rn(yn[j], -1.0f), thr), -4e-6f);
}
// The fused sweep leaves one candidate stream per CTA: (column, c) pairs in arrival order. Three bandwidth passes
// turn them into per-column segments (CSR) and reduce each segment to the column's neighbourhood mean:
//   hist    : hist[col] += 1 per entry (RED, no return value)            -> host: offs = exclusive cumsum(hist)
//   scatter : slot = cursor[col]++ ; vals[offs[col] + slot] = c
//   finalize: nv[col] = mean of the k largest of the segment (largest-first fp32 sum / k)
__global__ void __launch_bounds__(256) cand_hist_kernel(const uint2* __restrict__ stream, const int* __restrict__ stream_cnt,
                                                        int cta_cap, int* __restrict__ hist, int* __restrict__ overflow) {
  const int cta = blockIdx.y;
  int cnt = stream_cnt[cta];
  if (cnt > cta_cap) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(overflow, 1);
    cnt = cta_cap;
  }
  const uint2* sp = stream + static_cast<long long>(cta) * cta_cap;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < cnt; e += gridDim.x * blockDim.x) atomicAdd(hist + sp[e].x, 1);
}
__global__ void __launch_bounds__(256) cand_scatter_kernel(const uint2* __restrict__ stream, const int* __restrict__ stream_row,
                                                           const int* __restrict__ stream_cnt, int cta_cap,
                                                           const long long* __restrict__ offs, int* __restrict__ cursor,
                                                           float* __restrict__ vals, int* __restrict__ rows) {
  const int cta = blockIdx.y;
  const int cnt = min(stream_cnt[cta], cta_cap);
  const uint2* sp = stream + static_cast<long long>(cta) * cta_cap;
  const int* rp = stream_row ? stream_row + static_cast<long long>(cta) * cta_cap : nullptr;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < cnt; e += gridDim.x * blockDim.x) {
    const uint2 ent = sp[e];
    const int slot = atomicAdd(cursor + ent.x, 1);
    vals[offs[ent.x] + slot] = __uint_as_float(ent.y);
    if (rows) rows[offs[ent.x] + slot] = rp[e];
  }
}
// per column: the KT largest candidates of its segment (value ascending, source row alongside) and, optionally, the
// tensor-core neighbourhood mean. Segment order is arbitrary (atomics), so equal values are ordered by row id to keep
// the emitted list deterministic.
__global__ void __launch_bounds__(128) col_cand_finalize_kernel(const long long* __restrict__ offs, const int* __restrict__ hist,
                                                                const float* __restrict__ vals, const int* __restrict__ rows,
                                                                long long n, int k, float* __restrict__ nv,
                                                                float* __restrict__ cand_val, int* __restrict__ cand_idx,
                                                                int* __restrict__ overflow) {
  const long long j = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (j >= n) return;
  const int cnt = hist[j];
  if (cnt < k) atomicOr(overflow, 1);     // cannot happen with a valid threshold and no dropped entries
  float top[KT_LIST];
  int topi[KT_LIST];
#pragma unroll
  for (int t = 0; t < KT_LIST; ++t) { top[t] = -INFINITY; topi[t] = -1; }
  const float* v = vals + offs[j];
  const int* r = rows ? rows + offs[j] : nullptr;
  for (int e = 0; e < cnt; ++e) {
    const float x = v[e];
    const int id = r ? r[e] : 0;
    // admit on (value, then lower row id): a strict total order, independent of the arrival order
    if (x > top[0] || (r && x == top[0] && id < topi[0])) {
      top[0] = x; topi[0] = id;
#pragma unroll
      for (int t = 0; t < KT_LIST - 1; ++t) {
        const bool sw = top[t] > top[t + 1] || (top[t] == top[t + 1] && topi[t] < topi[t + 1]);
        const float a = top[t], b = top[t + 1];
        const int ia = topi[t], ib = topi[t + 1];
        top[t] = sw ? b : a; top[t + 1] = sw ? a : b;
        topi[t] = sw ? ib : ia; topi[t + 1] = sw ? ia : ib;
      }
    }
  }
  if (nv) {
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < KT_LIST; ++t)
      if (t < k) s = __fadd_rn(s, top[KT_LIST - 1 - t]);
    nv[j] = __fdiv_rn(s, static_cast<float>(k));
  }
  if (cand_val) {
#pragma unroll
    for (int t = 0; t < KT_LIST; ++t) { cand_val[j * KT_LIST + t] = top[t]; cand_idx[j * KT_LIST + t] = topi[t]; }
  }
}

// ================================================================================================
// host launchers
// ================================================================================================
int launch_col_threshold(const float* cand, long long n, int k, const float* yn, float* colthr, float* colb, cudaStream_t st) {
  if (!cand || !yn || !colthr || !colb || n <= 0) return SNAG_ERR_ARG;
  if (k < 1 || k > KT_LIST) return SNAG_ERR_SHAPE;
  col_threshold_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, st>>>(cand, n, k, yn, colthr, colb);
  return static_cast<int>(cudaGetLastError());
}
int launch_cand_hist(const uint2* stream, const int* stream_cnt, int n_ctas, int cta_cap, int* hist, int* overflow,
                     cudaStream_t st) {
  if (!stream || !stream_cnt || !hist || !overflow || n_ctas < 1 || cta_cap < 1) return SNAG_ERR_ARG;
  cand_hist_kernel<<<dim3(64, n_ctas), 256, 0, st>>>(stream, stream_cnt, cta_cap, hist, overflow);
  return static_cast<int>(cudaGetLastError());
}
int launch_cand_scatter(const uint2* stream, const int* stream_row, const int* stream_cnt, int n_ctas, int cta_cap,
                        const long long* offs, int* cursor, float* vals, int* rows, cudaStream_t st) {
  if (!stream || !stream_cnt || !offs || !cursor || !vals || n_ctas < 1 || cta_cap < 1) return SNAG_ERR_ARG;
  if ((rows != nullptr) != (stream_row != nullptr)) return SNAG_ERR_ARG;
  cand_scatter_kernel<<<dim3(64, n_ctas), 256, 0, st>>>(stream, stream_row, stream_cnt, cta_cap, offs, cursor, vals, rows);
  return static_cast<int>(cudaGetLastError());
}
int launch_col_cand_finalize(const long long* offs, const int* hist, const float* vals, const int* rows, long long n, int k,
                             float* nv, float* cand_val, int* cand_idx, int* overflow, cudaStream_t st) {
  if (!offs || !hist || !vals || !overflow || n <= 0 || (!nv && !cand_val)) return SNAG_ERR_ARG;
  if ((cand_val != nullptr) != (cand_idx != nullptr) || (cand_val && !rows)) return SNAG_ERR_ARG;
  if (k < 1 || k > KT_LIST) return SNAG_ERR_SHAPE;
  col_cand_finalize_kernel<<<static_cast<int>((n + 127) / 128), 128, 0, st>>>(offs, hist, vals, rows, n, k, nv, cand_val,
                                                                             cand_idx, overflow);
  return static_cast<int>(cudaGetLastError());
}
template <typename T>
int launch_topk_rescore(const T* A, const T* B, int Dpad, long long n_rows, const float* an,
                        const float* bn, const int* cand_idx, const float* cand_val, int k, float delta,
                        const float* outsider_bound, float* nv, int* flagged, int* flagged_cnt, int flagged_cap,
                        float* best_d, int* best_idx, cudaStream_t st) {
  if (!A || !B || !an || !bn || !cand_idx || !cand_val || !nv || !flagged || !flagged_cnt || n_rows <= 0 || flagged_cap < 1)
    return SNAG_ERR_ARG;
  if ((best_d == nullptr) != (best_idx == nullptr)) return SNAG_ERR_ARG;
  if (k < 1 || k > KT_LIST || (Dpad % 64)) return SNAG_ERR_SHAPE;
  const long long threads = n_rows * 16;
  topk_rescore_kernel<T><<<static_cast<unsigned>((threads + 127) / 128), 128, 0, st>>>(A, B, Dpad, n_rows, an, bn, cand_idx,
                                                                                   cand_val, k, delta, outsider_bound, nv, flagged,
                                                                                   flagged_cnt, flagged_cap, best_d, best_idx);
  return static_cast<int>(cudaGetLastError());
}
template <typename T>
int launch_topk_exhaustive(const T* A, const T* B, int Dpad, long long n_b, const float* an,
                           const float* bn, const int* flagged, const int* flagged_cnt, int flagged_cap, int k, float* nv,
                           float* best_d, int* best_idx, cudaStream_t st) {
  if (!A || !B || !an || !bn || !flagged || !flagged_cnt || !nv || n_b <= 0 || flagged_cap < 1) return SNAG_ERR_ARG;
  if ((best_d == nullptr) != (best_idx == nullptr)) return SNAG_ERR_ARG;
  if (k < 1 || k > KT_LIST || (Dpad % 64)) return SNAG_ERR_SHAPE;
  const int grid = flagged_cap < num_sms() * 4 ? flagged_cap : num_sms() * 4;
  topk_exhaustive_kernel<T><<<grid, 256, 0, st>>>(A, B, Dpad, n_b, an, bn, flagged, flagged_cnt, flagged_cap, k, nv, best_d, best_idx);
  return static_cast<int>(cudaGetLastError());
}
static inline int grid_for(long long work_items, int block, int num_sms, int ctas_per_sm);
// k > KT_LIST (the reference takes any k, src/utils.py:431): one block per row (or, with strides swapped, per column).
// A 4-pass radix select on the order-preserving integer image of the floats finds the k-th largest value; the values
// above it are collected in shared memory, sorted (bitonic, descending) and summed largest-first together with the
// needed copies of the k-th value — the oracle's arithmetic (mean_desc). k <= CSLS_ANYK_MAX.
constexpr int CSLS_ANYK_MAX = 1024;
__device__ __forceinline__ uint32_t float_order_key(float v) {
  const uint32_t u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__global__ void __launch_bounds__(256) vec_topk_mean_any_kernel(const float* __restrict__ sim, long long n_vec, long long len,
                                                                long long vec_stride, long long elem_stride, int k,
                                                                float* __restrict__ nv) {
  __shared__ int hist[256];
  __shared__ float buf[CSLS_ANYK_MAX];
  __shared__ uint32_t sh_prefix;
  __shared__ int sh_remaining, sh_cnt;
  for (long long v = blockIdx.x; v < n_vec; v += gridDim.x) {
    const float* base = sim + v * vec_stride;
    uint32_t prefix = 0, mask = 0;
    int remaining = k;                                   // rank (from the top) of the wanted value among keys matching prefix
    for (int shift = 24; shift >= 0; shift -= 8) {
      hist[threadIdx.x] = 0;
      __syncthreads();
      for (long long j = threadIdx.x; j < len; j += 256) {
        const uint32_t key = float_order_key(__ldg(base + j * elem_stride));
        if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1);
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        int cum = 0, d = 255;
        for (; d > 0; --d) {
          if (cum + hist[d] >= remaining) break;
          cum += hist[d];
        }
        sh_prefix = prefix | (static_cast<uint32_t>(d) << shift);
        sh_remaining = remaining - cum;
        sh_cnt = 0;
      }
      __syncthreads();
      prefix = sh_prefix;
      remaining = sh_remaining;
      mask |= 255u << shift;
    }
    // prefix = key of the k-th largest value; `remaining` copies of it belong to the top k, after the c = k - remaining
    // strictly larger values
    for (long long j = threadIdx.x; j < len; j += 256) {
      const float x = __ldg(base + j * elem_stride);
      if (float_order_key(x) > prefix) buf[atomicAdd(&sh_cnt, 1)] = x;
    }
    __syncthreads();
    const int c = sh_cnt;                                // == k - remaining
    int P = 1;
    while (P < c) P <<= 1;
    for (int t = c + threadIdx.x; t < P; t += 256) buf[t] = -INFINITY;
    __syncthreads();
    for (int size = 2; size <= P; size <<= 1)
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int t = threadIdx.x; t < P; t += 256) {
          const int partner = t ^ stride;
          if (partner > t) {
            const bool desc = (t & size) == 0;
            const float a = buf[t], b = buf[partner];
            if (desc ? (a < b) : (a > b)) { buf[t] = b; buf[partner] = a; }
          }
        }
        __syncthreads();
      }
    if (threadIdx.x == 0) {
      const uint32_t u = (prefix & 0x80000000u) ? (prefix & 0x7FFFFFFFu) : ~prefix;
      const float kth = __uint_as_float(u);
      float acc = 0.f;
      for (int t = 0; t < c; ++t) acc = __fadd_rn(acc, buf[t]);
      for (int t = 0; t < remaining; ++t) acc = __fadd_rn(acc, kth);
      nv[v] = __fdiv_rn(acc, static_cast<float>(k));
    }
    __syncthreads();
  }
}

static int csls_col_slabs(long long n1) {
  long long s = (n1 + 255) / 256;          // >= 256 rows per slab
  if (s > 64) s = 64;
  if (s < 1) s = 1;
  return static_cast<int>(s);
}
long long csls_workspace_floats(long long n1, long long n2) {
  return (32 * n1 + csls_col_slabs(n1) * n2) * KT_LIST;
}
int launch_csls_sim(const float* sim, long long n1, long long n2, long long ld, int k, float* out, long long ld_out,
                    float* nv1, float* nv2, float* workspace, cudaStream_t st) {
  if (!sim || !nv1 || !nv2 || !workspace || n1 <= 0 || n2 <= 0 || ld < n2) return SNAG_ERR_ARG;
  if (k < 1 || k > CSLS_ANYK_MAX || k > n1 || k > n2) return SNAG_ERR_SHAPE;
  if (reinterpret_cast<uintptr_t>(workspace) & 15) return SNAG_ERR_ALIGN;
  if (k > KT_LIST) {
    const int g1 = static_cast<int>(n1 < 8ll * num_sms() ? n1 : 8ll * num_sms());
    const int g2 = static_cast<int>(n2 < 8ll * num_sms() ? n2 : 8ll * num_sms());
    vec_topk_mean_any_kernel<<<g1, 256, 0, st>>>(sim, n1, n2, ld, 1, k, nv1);       // rows
    vec_topk_mean_any_kernel<<<g2, 256, 0, st>>>(sim, n2, n1, 1, ld, k, nv2);       // columns (strided reads)
    if (out) {
      const int g = grid_for(n1 * n2, 256, num_sms(), 8);
      csls_apply_kernel<<<g, 256, 0, st>>>(sim, nv1, nv2, out, n1, n2, ld, ld_out);
    }
    return static_cast<int>(cudaGetLastError());
  }
  float* part_r = workspace;
  float* part_c = workspace + 32 * n1 * KT_LIST;
  const int slabs = csls_col_slabs(n1);
  const int rows_per_slab = static_cast<int>((n1 + slabs - 1) / slabs);
  matrix_row_topk_kernel<<<static_cast<unsigned>((n1 * 32 + 255) / 256), 256, 0, st>>>(sim, n1, n2, ld, part_r);
  matrix_col_topk_kernel<<<dim3(static_cast<unsigned>((n2 + 127) / 128), slabs), 128, 0, st>>>(sim, n1, n2, ld, rows_per_slab, part_c);
  topk_merge_mean_kernel<false><<<static_cast<int>((n1 + 127) / 128), 128, 0, st>>>(part_r, nullptr, 32, n1, k, nv1, nullptr, nullptr);
  topk_merge_mean_kernel<false><<<static_cast<int>((n2 + 127) / 128), 128, 0, st>>>(part_c, nullptr, slabs, n2, k, nv2, nullptr, nullptr);
  if (out) {
    const int g = grid_for(n1 * n2, 256, num_sms(), 8);
    csls_apply_kernel<<<g, 256, 0, st>>>(sim, nv1, nv2, out, n1, n2, ld, ld_out);
  }
  return static_cast<int>(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------
// --distance 1 (main.py:387-390): the reference moves the embeddings to the host and calls
// scipy.spatial.distance.cdist(..., metric="cityblock"), whose result (float64) torch.FloatTensor rounds to fp32.
//   out[i,j] = fl32( sum_k | (double)x_ik - (double)y_jk | )      accumulated in fp64 in index order
// Not a contraction (no tensor cores): 32 x 32 output tile per block, x / y tiles staged in shared memory 32 k at a time.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) l1_distance_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                          long long n1, long long n2, int D, long long ldx, long long ldy,
                                                          float* __restrict__ out, long long ldo) {
  __shared__ float xs[32][33];
  __shared__ float ys[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 8 warps: warp ty owns rows ty, ty+8, ty+16, ty+24
  const long long i0 = static_cast<long long>(blockIdx.y) * 32, j0 = static_cast<long long>(blockIdx.x) * 32;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (int k0 = 0; k0 < D; k0 += 32) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int row = ty + 8 * r;
      const int kk = k0 + tx;
      xs[row][tx] = (i0 + row < n1 && kk < D) ? __ldg(x + (i0 + row) * ldx + kk) : 0.f;
      ys[row][tx] = (j0 + row < n2 && kk < D) ? __ldg(y + (j0 + row) * ldy + kk) : 0.f;
    }
    __syncthreads();
    const int kmax = min(32, D - k0);
    for (int kk = 0; kk < kmax; ++kk) {
      const double yv = static_cast<double>(ys[tx][kk]);
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[r] += fabs(static_cast<double>(xs[ty + 8 * r][kk]) - yv);
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const long long i = i0 + ty + 8 * r, j = j0 + tx;
    if (i < n1 && j < n2) out[i * ldo + j] = static_cast<float>(acc[r]);
  }
}

// Ranks of the ground truth on a MATERIALISED distance matrix (the two loops of main.py:400-411, 422-429 as counts):
//   cnt_row[i] = #{ j : d_ij < d_ii  or (d_ij == d_ii and j < i) },   cnt_col[j] = #{ i : d_ij < d_jj or (== and i < j) }
// one warp per row for the row counts; column counts by 32-row slabs with one atomic per (slab, column).
__global__ void __launch_bounds__(256) matrix_rank_kernel(const float* __restrict__ d, long long n, long long ld,
                                                          int* __restrict__ cnt_row, int* __restrict__ cnt_col) {
  const long long warp = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const long long n_slabs = (n + 31) / 32;
  if (warp < n) {                                          // rows
    const long long i = warp;
    const float g = __ldg(d + i * ld + i);
    int c = 0;
    for (long long j = lane; j < n; j += 32) {
      const float v = __ldg(d + i * ld + j);
      c += (v < g) || (v == g && j < i);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) cnt_row[i] = c;
  } else if (warp < n + n_slabs * ((n + 31) / 32)) {       // columns: (row slab, column group of 32)
    const long long t = warp - n;
    const long long slab = t / ((n + 31) / 32), cg = t % ((n + 31) / 32);
    const long long j = cg * 32 + lane;
    if (j < n) {
      const float g = __ldg(d + j * ld + j);
      int c = 0;
      const long long i1 = min(n, (slab + 1) * 32);
      for (long long i = slab * 32; i < i1; ++i) {
        const float v = __ldg(d + i * ld + j);
        c += (v < g) || (v == g && i < j);
      }
      if (c) atomicAdd(cnt_col + j, c);
    }
  }
}

static inline int grid_for(long long work_items, int block, int num_sms, int ctas_per_sm) {
  long long g = (work_items + block - 1) / block;
  const long long cap = static_cast<long long>(num_sms) * ctas_per_sm;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

int launch_l1_distance(const float* x, const float* y, long long n1, long long n2, int D, long long ldx, long long ldy,
                       float* out, long long ldo, cudaStream_t st) {
  if (!x || !y || !out || n1 <= 0 || n2 <= 0 || D <= 0 || ldx < D || ldy < D || ldo < n2) return SNAG_ERR_ARG;
  const dim3 grid(static_cast<unsigned>((n2 + 31) / 32), static_cast<unsigned>((n1 + 31) / 32));
  if (grid.y > 65535) return SNAG_ERR_SHAPE;
  l1_distance_kernel<<<grid, 256, 0, st>>>(x, y, n1, n2, D, ldx, ldy, out, ldo);
  return static_cast<int>(cudaGetLastError());
}
int launch_matrix_rank(const float* d, long long n, long long ld, int* cnt_row, int* cnt_col, cudaStream_t st) {
  if (!d || !cnt_row || !cnt_col || n <= 0 || ld < n) return SNAG_ERR_ARG;
  const long long groups = (n + 31) / 32;
  const long long warps = n + groups * groups;
  const cudaError_t e = cudaMemsetAsync(cnt_col, 0, sizeof(int) * static_cast<size_t>(n), st);
  if (e != cudaSuccess) return static_cast<int>(e);
  matrix_rank_kernel<<<static_cast<unsigned>((warps * 32 + 255) / 256), 256, 0, st>>>(d, n, ld, cnt_row, cnt_col);
  return static_cast<int>(cudaGetLastError());
}

int launch_noise_mask(const float* x, float* out, const float* mean, const float* stdv, const uint8_t* mask,
                      const float* zsel, const int* selpos, long long N, int F, long long ld_in, long long ld_out,
                      float ratio, float keep, float rho, unsigned long long seed, long long row0, cudaStream_t st) {
  if (!x || !out || !mean || !stdv || N <= 0 || F <= 0) return SNAG_ERR_ARG;
  if ((F & 3) || (ld_in & 3) || (ld_out & 3)) return SNAG_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(mean) |
       reinterpret_cast<uintptr_t>(stdv) | reinterpret_cast<uintptr_t>(zsel)) & 15) return SNAG_ERR_ALIGN;
  if (zsel && (!selpos || !mask)) return SNAG_ERR_ARG;
  const int g = grid_for(N * (F >> 2), 256, num_sms(), 8);
  noise_mask_kernel<<<g, 256, 0, st>>>(x, out, mean, stdv, mask, zsel, selpos, N, F, ld_in, ld_out, ratio, keep, rho, seed, row0);
  return static_cast<int>(cudaGetLastError());
}

int launch_philox_rowmask(uint8_t* mask, long long N, float ratio, unsigned long long seed, long long row0, cudaStream_t st) {
  if (!mask || N <= 0) return SNAG_ERR_ARG;
  philox_rowmask_kernel<<<static_cast<int>((N + 255) / 256), 256, 0, st>>>(mask, N, ratio, seed, row0);
  return static_cast<int>(cudaGetLastError());
}

int launch_gauss_fill(float* out, const float* mean, const float* stdv, long long N, int F, long long ld,
                      unsigned long long seed, long long row0, cudaStream_t st) {
  if (!out || !mean || !stdv || N <= 0 || F <= 0) return SNAG_ERR_ARG;
  if ((F & 3) || (ld & 3)) return SNAG_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(mean) | reinterpret_cast<uintptr_t>(stdv)) & 15)
    return SNAG_ERR_ALIGN;
  const int g = grid_for(N * (F >> 2), 256, num_sms(), 8);
  gauss_fill_kernel<<<g, 256, 0, st>>>(out, mean, stdv, N, F, ld, seed, row0);
  return static_cast<int>(cudaGetLastError());
}

int launch_col_mean_std(const float* x, const uint8_t* valid, long long N, int F, long long ld, float* mean, float* stdv,
                        void* workspace, cudaStream_t st) {
  if (!x || !mean || !stdv || !workspace || N <= 1 || F <= 0) return SNAG_ERR_ARG;
  double* acc = reinterpret_cast<double*>(workspace);
  unsigned long long* cnt = reinterpret_cast<unsigned long long*>(acc + 2 * static_cast<long long>(F));
  cudaError_t e = cudaMemsetAsync(workspace, 0, (2 * static_cast<size_t>(F) + 1) * 8, st);
  if (e != cudaSuccess) return static_cast<int>(e);
  const bool vec4 = (F % 4 == 0) && (ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  const int bx = vec4 ? (F / 4 + 255) / 256 : (F + 255) / 256;
  // enough row slabs to fill the machine a few times over, at least 64 rows each (every slab ends in 2 F fp64 atomics:
  // 32-row slabs measured slower at N = 39.6k)
  long long slabs = (static_cast<long long>(num_sms()) * 8 + bx - 1) / bx;
  long long rows_per_slab = (N + slabs - 1) / slabs;
  if (rows_per_slab < 64) rows_per_slab = 64;
  slabs = (N + rows_per_slab - 1) / rows_per_slab;
  if (vec4)
    col_stats_partial4_kernel<<<dim3(bx, static_cast<unsigned>(slabs)), 256, 0, st>>>(x, valid, N, F, ld, static_cast<int>(rows_per_slab), acc, cnt);
  else
    col_stats_partial_kernel<<<dim3(bx, static_cast<unsigned>(slabs)), 256, 0, st>>>(x, valid, N, F, ld, static_cast<int>(rows_per_slab), acc, cnt);
  col_stats_final_kernel<<<(F + 255) / 256, 256, 0, st>>>(acc, cnt, F, mean, stdv);
  return static_cast<int>(cudaGetLastError());
}

int launch_rowblend_fwd(const float* e, const float* noise, const uint8_t* mask, float* out, long long N, int D, float a,
                        float c, cudaStream_t st) {
  if (!e || !noise || !mask || !out || N <= 0 || D <= 0) return SNAG_ERR_ARG;
  if (D & 3) return SNAG_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(e) | reinterpret_cast<uintptr_t>(noise) | reinterpret_cast<uintptr_t>(out)) & 15)
    return SNAG_ERR_ALIGN;
  const int g = grid_for(N * (D >> 2), 256, num_sms(), 8);
  rowblend_fwd_kernel<<<g, 256, 0, st>>>(e, noise, mask, out, N, D, a, c);
  return static_cast<int>(cudaGetLastError());
}
int launch_rowblend_bwd(const float* g_out, const uint8_t* mask, float* g_in, long long N, int D, float a, cudaStream_t st) {
  if (!g_out || !mask || !g_in || N <= 0 || D <= 0) return SNAG_ERR_ARG;
  if (D & 3) return SNAG_ERR_ALIGN;
  if ((reinterpret_cast<uintptr_t>(g_out) | reinterpret_cast<uintptr_t>(g_in)) & 15) return SNAG_ERR_ALIGN;
  const int g = grid_for(N * (D >> 2), 256, num_sms(), 8);
  rowblend_bwd_kernel<<<g, 256, 0, st>>>(g_out, mask, g_in, N, D, a);
  return static_cast<int>(cudaGetLastError());
}

int launch_prep_bf16(const float* emb, long long ld, const long long* idx, int n, int D, int normalize,
                     __nv_bfloat16* out, int Dpad, float* norm2, cudaStream_t st) {
  if (!emb || !out || n <= 0 || D <= 0) return SNAG_ERR_ARG;
  if (Dpad < D || (Dpad % 64) != 0) return SNAG_ERR_SHAPE;
  const long long threads = static_cast<long long>(n) * 32;
  const int grid = static_cast<int>((threads + 255) / 256);
  if (D <= PREP_NARROW_MAX_D)
    prep_bf16_kernel<4><<<grid, 256, 0, st>>>(emb, ld, idx, n, D, normalize, out, Dpad, norm2);
  else
    prep_bf16_kernel<16><<<grid, 256, 0, st>>>(emb, ld, idx, n, D, normalize, out, Dpad, norm2);
  return static_cast<int>(cudaGetLastError());
}

int launch_prep_split(const float* emb, long long ld, const long long* idx, int n, int D, int normalize, int side,
                      float* rows, __nv_bfloat16* split, int Dpad, float* norm2, cudaStream_t st) {
  if (!emb || !rows || !split || !norm2 || n <= 0 || D <= 0 || (side != 0 && side != 1)) return SNAG_ERR_ARG;
  if (Dpad < D || (Dpad % 64) != 0) return SNAG_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(rows) & 15) || (reinterpret_cast<uintptr_t>(split) & 127)) return SNAG_ERR_ALIGN;
  const long long threads = static_cast<long long>(n) * 32;
  prep_split_kernel<<<static_cast<int>((threads + 255) / 256), 256, 0, st>>>(emb, ld, idx, n, D, normalize, side, rows, split, Dpad);
  row_norm2_kernel<<<static_cast<unsigned>((n + 127) / 128), 128, 0, st>>>(rows, Dpad, n, norm2);
  return static_cast<int>(cudaGetLastError());
}

int launch_icl_stack_prep(int n_prob, const float* const* emb, const long long* ld, const int* D, __nv_bfloat16* const* out,
                          const int* Dpad, const long long* idx_l, const long long* idx_r, int B, int Bp, int normalize,
                          cudaStream_t st) {
  if (n_prob < 1 || n_prob > MANY_MAX || !emb || !ld || !D || !out || !Dpad || !idx_l || !idx_r) return SNAG_ERR_ARG;
  if (B <= 0 || Bp < B || (Bp % 256) != 0) return SNAG_ERR_ARG;
  // narrow tables (the per-modality embeddings) and wide ones (the joint embeddings) go to different instantiations: the
  // narrow one keeps 4 float4 per lane and runs at more than twice the occupancy
  StackPrepArgs narrow{}, wide{};
  int n_narrow = 0, n_wide = 0;
  for (int p = 0; p < n_prob; ++p) {
    if (!emb[p] || !out[p] || D[p] <= 0 || ld[p] < D[p]) return SNAG_ERR_ARG;
    if (Dpad[p] < D[p] || (Dpad[p] % 64) != 0) return SNAG_ERR_SHAPE;
    StackPrepArgs& a = D[p] <= PREP_NARROW_MAX_D ? narrow : wide;
    const int q = D[p] <= PREP_NARROW_MAX_D ? n_narrow++ : n_wide++;
    a.emb[q] = emb[p]; a.ld[q] = ld[p]; a.out[q] = out[p]; a.D[q] = D[p]; a.Dpad[q] = Dpad[p];
  }
  const unsigned gx = static_cast<unsigned>((2ll * Bp * 32 + 255) / 256);
  if (n_narrow) icl_stack_prep_kernel<4><<<dim3(gx, static_cast<unsigned>(n_narrow)), 256, 0, st>>>(narrow, idx_l, idx_r, B, Bp, normalize);
  if (n_wide) icl_stack_prep_kernel<16><<<dim3(gx, static_cast<unsigned>(n_wide)), 256, 0, st>>>(wide, idx_l, idx_r, B, Bp, normalize);
  return static_cast<int>(cudaGetLastError());
}
int launch_icl_stack_prep_split(int n_prob, const float* const* emb, const long long* ld, const int* D, __nv_bfloat16* const* out,
                                const int* Dpad, const long long* idx_l, const long long* idx_r, int B, int Bp, int normalize,
                                cudaStream_t st) {
  if (n_prob < 1 || n_prob > MANY_MAX || !emb || !ld || !D || !out || !Dpad || !idx_l || !idx_r) return SNAG_ERR_ARG;
  if (B <= 0 || Bp < B || (Bp % 256) != 0) return SNAG_ERR_ARG;
  StackPrepArgs a{};
  for (int p = 0; p < n_prob; ++p) {
    if (!emb[p] || !out[p] || D[p] <= 0 || ld[p] < D[p]) return SNAG_ERR_ARG;
    if (Dpad[p] < D[p] || (Dpad[p] % 64) != 0) return SNAG_ERR_SHAPE;
    if (reinterpret_cast<uintptr_t>(out[p]) & 127) return SNAG_ERR_ALIGN;
    a.emb[p] = emb[p]; a.ld[p] = ld[p]; a.out[p] = out[p]; a.D[p] = D[p]; a.Dpad[p] = Dpad[p];
  }
  const unsigned gx = static_cast<unsigned>((2ll * Bp * 32 + 255) / 256);
  icl_stack_prep_split_kernel<<<dim3(gx, static_cast<unsigned>(n_prob)), 256, 0, st>>>(a, idx_l, idx_r, B, Bp, normalize);
  return static_cast<int>(cudaGetLastError());
}
int launch_normalize_bwd_scatter_many(int n_prob, const float* const* emb, const long long* ld, const int* D,
                                      const float* const* dz_a, const float* const* dz_b, const long long* ld_dz,
                                      const int* n_parts, const long long* part_stride, float* const* demb,
                                      const long long* ld_demb, const long long* idx_l, const long long* idx_r, int n,
                                      int normalize, cudaStream_t st) {
  if (n_prob < 1 || n_prob > MANY_MAX || !emb || !ld || !D || !dz_a || !dz_b || !ld_dz || !n_parts || !part_stride ||
      !demb || !ld_demb || !idx_l || !idx_r || n <= 0)
    return SNAG_ERR_ARG;
  ScatterManyArgs a{};
  for (int p = 0; p < n_prob; ++p) {
    if (!emb[p] || !dz_a[p] || !dz_b[p] || !demb[p] || D[p] <= 0 || ld[p] < D[p] || ld_dz[p] < D[p] || ld_demb[p] < D[p] ||
        n_parts[p] < 1)
      return SNAG_ERR_ARG;
    a.emb[p] = emb[p]; a.ld[p] = ld[p]; a.D[p] = D[p]; a.dz[2 * p] = dz_a[p]; a.dz[2 * p + 1] = dz_b[p];
    a.ld_dz[p] = ld_dz[p]; a.n_parts[p] = n_parts[p]; a.part_stride[p] = part_stride[p]; a.demb[p] = demb[p];
    a.ld_demb[p] = ld_demb[p];
    const uintptr_t ptrs = reinterpret_cast<uintptr_t>(emb[p]) | reinterpret_cast<uintptr_t>(dz_a[p]) |
                           reinterpret_cast<uintptr_t>(dz_b[p]) | reinterpret_cast<uintptr_t>(demb[p]);
    a.vec4[p] = (D[p] % 4 == 0) && (ptrs % 16 == 0) && (ld[p] % 4 == 0) && (ld_dz[p] % 4 == 0) && (ld_demb[p] % 4 == 0) &&
                (n_parts[p] == 1 || part_stride[p] % 4 == 0);
  }
  const dim3 grid(static_cast<unsigned>((static_cast<long long>(n) * 32 + 255) / 256), static_cast<unsigned>(2 * n_prob));
  normalize_bwd_scatter_many_kernel<<<grid, 256, 0, st>>>(a, idx_l, idx_r, n, normalize);
  return static_cast<int>(cudaGetLastError());
}

static int fill_tabs(JointTabs* t, const float* const* embs, float* const* d_embs, const int* widths, int M) {
  if (!embs || !widths || M < 1 || M > SNAG_MAX_MODAL) return SNAG_ERR_ARG;
  int off = 0;
  for (int m = 0; m < SNAG_MAX_MODAL; ++m) {
    t->e[m] = nullptr; t->de[m] = nullptr; t->width[m] = 0; t->off[m] = 0;
  }
  for (int m = 0; m < M; ++m) {
    if (!embs[m] || widths[m] <= 0) return SNAG_ERR_ARG;
    if (d_embs && !d_embs[m]) return SNAG_ERR_ARG;
    t->e[m] = embs[m];
    t->de[m] = d_embs ? d_embs[m] : nullptr;
    t->width[m] = widths[m];
    t->off[m] = off;
    off += widths[m];
  }
  return off;
}
int launch_joint_fuse_fwd(const float* const* embs, const int* widths, int M, long long N, const float* w_ent, long long ldw,
                          const float* w_glob, float* joint, float* joint_fz, long long ld_out, cudaStream_t st) {
  JointTabs t;
  const int tot = fill_tabs(&t, embs, nullptr, widths, M);
  if (tot < 0) return tot;
  if (N <= 0 || ld_out < tot || (!joint && !joint_fz) || (joint && (!w_ent || ldw < M)) || (joint_fz && !w_glob)) return SNAG_ERR_ARG;
  joint_fuse_fwd_kernel<<<dim3(static_cast<unsigned>((N + 7) / 8), M), 256, 0, st>>>(t, N, w_ent, ldw, w_glob, joint, joint_fz, ld_out);
  return static_cast<int>(cudaGetLastError());
}
int launch_joint_fuse_bwd(const float* const* embs, float* const* d_embs, const int* widths, int M, long long N,
                          const float* w_ent, long long ldw, const float* w_glob, const float* d_joint, const float* d_joint_fz,
                          long long ld_out, float* d_w_ent, float* d_w_glob, cudaStream_t st) {
  JointTabs t;
  if (!d_embs) return SNAG_ERR_ARG;
  const int tot = fill_tabs(&t, embs, d_embs, widths, M);
  if (tot < 0) return tot;
  if (N <= 0 || ld_out < tot || (!d_joint && !d_joint_fz) || (d_joint && (!w_ent || ldw < M)) || (d_joint_fz && !w_glob))
    return SNAG_ERR_ARG;
  joint_fuse_bwd_kernel<<<dim3(static_cast<unsigned>((N + 7) / 8), M), 256, 0, st>>>(t, N, w_ent, ldw, w_glob, d_joint, d_joint_fz,
                                                                                    ld_out, d_w_ent, d_w_glob);
  return static_cast<int>(cudaGetLastError());
}

int launch_normalize_bwd_scatter(const float* emb, long long ld, const long long* idx, int n, int D, int normalize,
                                 const float* dz, long long ld_dz, int n_parts, long long part_stride, float* demb,
                                 long long ld_demb, cudaStream_t st) {
  if (!emb || !dz || !demb || n <= 0 || D <= 0 || ld < D || ld_dz < D || ld_demb < D || n_parts < 1) return SNAG_ERR_ARG;
  const long long threads = static_cast<long long>(n) * 32;
  normalize_bwd_scatter_kernel<<<static_cast<int>((threads + 255) / 256), 256, 0, st>>>(emb, ld, idx, n, D, normalize, dz,
                                                                                       ld_dz, n_parts, part_stride, demb,
                                                                                       ld_demb);
  return static_cast<int>(cudaGetLastError());
}

int launch_topk_merge_mean(const float* part, const int* part_idx, int n_lists, long long n_rows, int k, float* nv,
                           float* cand_out, int* cand_idx_out, cudaStream_t st) {
  if (!part || n_lists <= 0 || n_rows <= 0 || (!nv && !cand_out)) return SNAG_ERR_ARG;
  if (cand_idx_out && (!part_idx || !cand_out)) return SNAG_ERR_ARG;
  if (k < 1 || k > KT_LIST) return SNAG_ERR_SHAPE;
  if (reinterpret_cast<uintptr_t>(part) & 15) return SNAG_ERR_ALIGN;
  const int grid = static_cast<int>((n_rows + 127) / 128);
  if (cand_idx_out)
    topk_merge_mean_kernel<true><<<grid, 128, 0, st>>>(part, part_idx, n_lists, n_rows, k, nv, cand_out, cand_idx_out);
  else
    topk_merge_mean_kernel<false><<<grid, 128, 0, st>>>(part, nullptr, n_lists, n_rows, k, nv, cand_out, nullptr);
  return static_cast<int>(cudaGetLastError());
}

template <typename T>
int launch_pair_score(const T* X, const T* Y, int Dpad, long long n, const float* xn, const float* yn,
                      const float* nv1, const float* nv2, int use_csls, float* g, float* s_out, cudaStream_t st) {
  if (!X || !Y || !xn || !yn || !g || n <= 0) return SNAG_ERR_ARG;
  if (use_csls && (!nv1 || !nv2)) return SNAG_ERR_ARG;
  if (Dpad % 64) return SNAG_ERR_SHAPE;
  pair_score_kernel<T><<<static_cast<int>((n + 127) / 128), 128, 0, st>>>(X, Y, Dpad, n, xn, yn, nv1, nv2, use_csls, g, s_out);
  return static_cast<int>(cudaGetLastError());
}

template <typename T>
int launch_band_rescore(const T* X, const T* Y, int Dpad, const float* xn, const float* yn,
                        const float* nv1, const float* nv2, const float* g_row, const float* g_col, int row_gid0, int col_gid0,
                        int use_csls, const uint2* band, const unsigned int* band_cnt, unsigned int band_cap, int* cnt_row,
                        int* cnt_col, cudaStream_t st, const int* row_gids, int swapped) {
  if (!X || !Y || !xn || !yn || !g_row || !g_col || !band || !band_cnt || !cnt_row || !cnt_col) return SNAG_ERR_ARG;
  if (use_csls && (!nv1 || !nv2)) return SNAG_ERR_ARG;
  if (Dpad % 64) return SNAG_ERR_SHAPE;
  // grid-stride over the device-side count: no host round trip
  band_rescore_kernel<T><<<num_sms() * 16, 128, 0, st>>>(X, Y, Dpad, xn, yn, nv1, nv2, g_row, g_col, row_gid0, col_gid0, use_csls,
                                                      band, band_cnt, band_cap, cnt_row, cnt_col, row_gids, swapped);
  return static_cast<int>(cudaGetLastError());
}

int launch_spec_bounds(const float* cand, long long n, int k, const float* cdiag, float shift, float delta, float* lo,
                       float* hi, cudaStream_t st) {
  if (!cand || !cdiag || !lo || !hi || n <= 0 || k < 1 || k > KT_LIST) return SNAG_ERR_ARG;
  spec_bounds_kernel<<<static_cast<int>((n + 255) / 256), 256, 0, st>>>(cand, n, k, cdiag, shift, delta, lo, hi);
  return static_cast<int>(cudaGetLastError());
}

int launch_rank_judge(const uint2* rk_stream, const int* rk_stream_row, const int* rk_cnt, int n_ctas, int rk_cap,
                      const float* R, const float* Rp, const float* C, const float* Cp, const unsigned char* row_ok,
                      const unsigned char* col_ok, float eps, int row_gid0, int col_gid0, int* cnt_row, int* cnt_col,
                      uint2* band, unsigned int* band_cnt, unsigned int band_cap, int* overflow, cudaStream_t st) {
  if (!rk_stream || !rk_stream_row || !rk_cnt || !R || !Rp || !C || !Cp || !row_ok || !col_ok || !cnt_row || !cnt_col ||
      !band || !band_cnt || !overflow || n_ctas < 1 || rk_cap < 1)
    return SNAG_ERR_ARG;
  rank_judge_kernel<<<dim3(64, n_ctas), 256, 0, st>>>(rk_stream, rk_stream_row, rk_cnt, rk_cap, R, Rp, C, Cp, row_ok, col_ok, eps,
                                                      row_gid0, col_gid0, cnt_row, cnt_col, band, band_cnt, band_cap, overflow);
  return static_cast<int>(cudaGetLastError());
}

template <typename T>
int launch_rank_exhaustive(const T* A, const T* B, int Dpad, long long n_b, const float* an,
                           const float* bn, const float* nva, const float* nvb, const float* g, const int* rows, int n_rows,
                           int a_gid0, int b_gid0, int use_csls, int swapped, int* cnt, cudaStream_t st) {
  if (!A || !B || !an || !bn || !g || !rows || !cnt || n_rows < 1 || n_b < 1) return SNAG_ERR_ARG;
  if (use_csls && (!nva || !nvb)) return SNAG_ERR_ARG;
  if (Dpad % 64) return SNAG_ERR_SHAPE;
  const int smem = RX_ROWS * Dpad * static_cast<int>(sizeof(float));
  if (smem > 200 * 1024) return SNAG_ERR_SHAPE;
  static std::once_flag once;
  std::call_once(once, [] {
    cudaFuncSetAttribute(rank_exhaustive_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  });
  const int gx = (n_rows + RX_ROWS - 1) / RX_ROWS;
  int gy = (num_sms() * 4 + gx - 1) / gx;                  // enough blocks to fill the machine when few rows are listed
  const long long max_gy = (n_b + 255) / 256;
  if (gy > max_gy) gy = static_cast<int>(max_gy);
  if (gy < 1) gy = 1;
  rank_exhaustive_kernel<T><<<dim3(gx, gy), 256, smem, st>>>(A, B, Dpad, n_b, an, bn, nva, nvb, g, rows, n_rows, a_gid0, b_gid0,
                                                          use_csls, swapped, cnt);
  return static_cast<int>(cudaGetLastError());
}

template <typename T>
int launch_pairs_dot(const T* X, const T* Y, int Dpad, const int* rows, const int* cols,
                     long long n_pairs, float* s_out, cudaStream_t st) {
  if (!X || !Y || !rows || !cols || !s_out || n_pairs <= 0) return SNAG_ERR_ARG;
  if (Dpad % 64) return SNAG_ERR_SHAPE;
  pairs_dot_kernel<T><<<static_cast<unsigned>((n_pairs + 127) / 128), 128, 0, st>>>(X, Y, Dpad, rows, cols, n_pairs, s_out);
  return static_cast<int>(cudaGetLastError());
}

int launch_top4_merge(const float* val, const int* idx, int n_lists, long long n_rows, float* oval, int* oidx, cudaStream_t st) {
  if (!val || !idx || !oval || !oidx || n_lists <= 0 || n_rows <= 0) return SNAG_ERR_ARG;
  top4_merge_kernel<<<static_cast<int>((n_rows + 127) / 128), 128, 0, st>>>(val, idx, n_lists, n_rows, oval, oidx);
  return static_cast<int>(cudaGetLastError());
}

template <typename T>
int launch_top3_rescore(const T* X, const T* Y, int Dpad, long long n_rows, const float* xn,
                        const float* yn, const float* nv1, const float* nv2, int use_csls, const int* cand, float* oval,
                        int* oidx, cudaStream_t st) {
  if (!X || !Y || !xn || !yn || !cand || !oval || !oidx || n_rows <= 0) return SNAG_ERR_ARG;
  if (use_csls && (!nv1 || !nv2)) return SNAG_ERR_ARG;
  if (Dpad % 64) return SNAG_ERR_SHAPE;
  top3_rescore_kernel<T><<<static_cast<int>((n_rows + 127) / 128), 128, 0, st>>>(X, Y, Dpad, n_rows, xn, yn, nv1, nv2, use_csls,
                                                                            cand, oval, oidx);
  return static_cast<int>(cudaGetLastError());
}


int launch_icl_finalize(const float* rowsum_part, int n_chunks, int B, int Bp, const float* pos, float inv_tau, float* lse,
                        float* nll, cudaStream_t st) {
  icl_finalize_kernel<<<(B + 255) / 256, 256, 0, st>>>(rowsum_part, n_chunks, B, Bp, pos, inv_tau, lse, nll);
  return static_cast<int>(cudaGetLastError());
}

// the canonical kernels for both row types: bf16 operands (default evaluation) and fp32 rows (precision="fp32")
#define SNAG_CANONICAL_INSTANTIATE(T)                                                                                       \
  template int launch_topk_rescore<T>(const T*, const T*, int, long long, const float*, const float*, const int*,         \
                                      const float*, int, float, const float*, float*, int*, int*, int, float*, int*,        \
                                      cudaStream_t);                                                                        \
  template int launch_topk_exhaustive<T>(const T*, const T*, int, long long, const float*, const float*, const int*,      \
                                         const int*, int, int, float*, float*, int*, cudaStream_t);                         \
  template int launch_pair_score<T>(const T*, const T*, int, long long, const float*, const float*, const float*,        \
                                    const float*, int, float*, float*, cudaStream_t);                                       \
  template int launch_band_rescore<T>(const T*, const T*, int, const float*, const float*, const float*, const float*,   \
                                      const float*, const float*, int, int, int, const uint2*, const unsigned int*,         \
                                      unsigned int, int*, int*, cudaStream_t, const int*, int);                             \
  template int launch_rank_exhaustive<T>(const T*, const T*, int, long long, const float*, const float*, const float*,   \
                                         const float*, const float*, const int*, int, int, int, int, int, int*,             \
                                         cudaStream_t);                                                                     \
  template int launch_pairs_dot<T>(const T*, const T*, int, const int*, const int*, long long, float*, cudaStream_t);    \
  template int launch_top3_rescore<T>(const T*, const T*, int, long long, const float*, const float*, const float*,      \
                                      const float*, int, const int*, float*, int*, cudaStream_t);
SNAG_CANONICAL_INSTANTIATE(__nv_bfloat16)
SNAG_CANONICAL_INSTANTIATE(float)
#undef SNAG_CANONICAL_INSTANTIATE

}  // namespace snag
