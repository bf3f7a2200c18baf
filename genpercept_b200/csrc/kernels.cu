#include "kernels.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "launch.h"
#include "ptx.cuh"

namespace gp {
namespace {

template <bool BF16>
__device__ __forceinline__ float f16_to_f32(uint16_t v) {
  if constexpr (BF16) return __bfloat162float(__ushort_as_bfloat16(v));
  else return __half2float(__ushort_as_half(v));
}
template <bool BF16>
__device__ __forceinline__ uint16_t f32_to_f16(float v) {
  if constexpr (BF16) return __bfloat16_as_ushort(__float2bfloat16_rn(v));
  else return __half_as_ushort(__float2half_rn(v));
}
template <bool BF16>
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    f[2 * e] = f16_to_f32<BF16>((uint16_t)(w[e] & 0xFFFF));
    f[2 * e + 1] = f16_to_f32<BF16>((uint16_t)(w[e] >> 16));
  }
}
template <bool BF16>
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int e = 0; e < 4; ++e)
    w[e] = (uint32_t)f32_to_f16<BF16>(f[2 * e]) | ((uint32_t)f32_to_f16<BF16>(f[2 * e + 1]) << 16);
  return make_uint4(w[0], w[1], w[2], w[3]);
}
// SiLU with ONE special-function op per element: x*sigmoid(x) = h + h*tanh(h), h = x/2.  tanh.approx.f32 has
// ~2^-11 relative error, i.e. below the fp16 rounding of the stored result; exp + reciprocal (2 MUFU ops
// per element) made the normalise+SiLU pass special-function-bound at 16 ops/clk/SM (r1d).
__device__ __forceinline__ float silu_f(float x) {
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
// High-precision (split) layout: a tensor with C logical channels is stored with 2C physical channels per pixel,
// [hi C | lo C], value = hi + lo (two fp16: ~22 mantissa bits).  `lo` = element offset of the lo plane (0 = plain).
template <bool BF16>
__device__ __forceinline__ void load8(const uint16_t* p, int lo, float (&f)[8]) {
  unpack8<BF16>(__ldg(reinterpret_cast<const uint4*>(p)), f);
  if (lo) {
    float g[8];
    unpack8<BF16>(__ldg(reinterpret_cast<const uint4*>(p + lo)), g);
#pragma unroll
    for (int e = 0; e < 8; ++e) f[e] += g[e];
  }
}
template <bool BF16>
__device__ __forceinline__ void store8(uint16_t* p, int lo, const float (&f)[8]) {
  const uint4 h = pack8<BF16>(f);
  *reinterpret_cast<uint4*>(p) = h;
  if (lo) {
    float hf[8], r[8];
    unpack8<BF16>(h, hf);
#pragma unroll
    for (int e = 0; e < 8; ++e) r[e] = f[e] - hf[e];
    *reinterpret_cast<uint4*>(p + lo) = pack8<BF16>(r);
  }
}
template <bool BF16>
__device__ __forceinline__ float load1(const uint16_t* p, int lo) {
  float v = f16_to_f32<BF16>(*p);
  if (lo) v += f16_to_f32<BF16>(p[lo]);
  return v;
}
template <bool BF16>
__device__ __forceinline__ void store1(uint16_t* p, int lo, float v) {
  const uint16_t h = f32_to_f16<BF16>(v);
  *p = h;
  if (lo) p[lo] = f32_to_f16<BF16>(v - f16_to_f32<BF16>(h));
}
// fp32-class SiLU for the high-precision mode (tanh.approx carries only ~11 bits)
__device__ __forceinline__ float silu_precise(float x) { return __fdividef(x, 1.f + __expf(-x)); }
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ------------------------------------------------------------------------------ direct conv
template <bool BF16>
__global__ void direct_conv_kernel(const DirectConvParams p) {
  const long long total = (long long)p.N * p.Ho * p.Wo * p.Cout;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int co = (int)(idx % p.Cout);
  long long r = idx / p.Cout;
  const int ox = (int)(r % p.Wo);
  r /= p.Wo;
  const int oy = (int)(r % p.Ho);
  const int n = (int)(r / p.Ho);
  const bool up = (p.flags & DC_UP2X) != 0;
  const int He = up ? 2 * p.H : p.H, We = up ? 2 * p.W : p.W;
  const uint16_t* in = reinterpret_cast<const uint16_t*>(p.in);
  float acc = p.bias ? p.bias[co] : 0.f;
  for (int ky = 0; ky < p.ks; ++ky) {
    int iy = oy * p.stride + ky - p.pad;
    if (iy < 0 || iy >= He) continue;
    if (up) iy >>= 1;
    for (int kx = 0; kx < p.ks; ++kx) {
      int ix = ox * p.stride + kx - p.pad;
      if (ix < 0 || ix >= We) continue;
      if (up) ix >>= 1;
      const uint16_t* xp = in + (((long long)n * p.H + iy) * p.W + ix) * p.in_cstride;
      const float* wp = p.w + ((long long)(ky * p.ks + kx) * p.Cin) * p.Cout + co;
      for (int ci = 0; ci < p.Cin; ++ci) acc += load1<BF16>(xp + ci, p.in_lo) * wp[(long long)ci * p.Cout];
    }
  }
  const long long opix = ((long long)n * p.Ho + oy) * p.Wo + ox;
  if (p.res) acc += load1<BF16>(reinterpret_cast<const uint16_t*>(p.res) + opix * p.out_cstride + co, p.out_lo);
  if (p.flags & DC_RELU) acc = fmaxf(acc, 0.f);
  if (p.flags & DC_AFFINE_CLAMP01) acc = fminf(fmaxf((acc + 1.f) * 0.5f, 0.f), 1.f);
  if (p.flags & DC_OUT_F32_NCHW) {
    reinterpret_cast<float*>(p.out)[(((long long)n * p.Cout + co) * p.Ho + oy) * p.Wo + ox] = acc;
  } else {
    store1<BF16>(reinterpret_cast<uint16_t*>(p.out) + opix * p.out_cstride + co, p.out_lo, acc);
  }
}

// ------------------------------------------------------------------------------ GroupNorm
// Deterministic two-level reduction (no atomics, fixed summation order => bit-reproducible runs):
//   gn_stats   : block (C/8 vectors x PIX pixel lanes) reduces its pixel chunk -> partial[n][chunk][c][2]
//   gn_finalize: one warp per (n, group) sums the partials in a fixed order -> scale/shift per channel
template <bool BF16>
__global__ void gn_stats_kernel(const uint16_t* __restrict__ x, long long HW, int C, float* __restrict__ partial,
                                int Ctot, int coff, int pix_per_block, int xs, int lo) {
  extern __shared__ float sh[];   // [PIX][C][2]
  const int n = blockIdx.y;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int nthr = blockDim.x * blockDim.y;
  const long long p0 = (long long)blockIdx.x * pix_per_block;
  long long p1 = p0 + pix_per_block;
  if (p1 > HW) p1 = HW;
  float s[8], q[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { s[e] = 0.f; q[e] = 0.f; }
  const uint16_t* base = x + ((long long)n * HW) * xs + threadIdx.x * 8;
  const int step = blockDim.y;
  long long p = p0 + threadIdx.y;
  for (; p + 3 * step < p1 && !lo; p += 4 * step) {      // four independent 16-byte loads in flight
    uint4 u[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) u[k] = __ldg(reinterpret_cast<const uint4*>(base + (p + (long long)k * step) * xs));
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float f[8];
      unpack8<BF16>(u[k], f);
#pragma unroll
      for (int e = 0; e < 8; ++e) { s[e] += f[e]; q[e] += f[e] * f[e]; }
    }
  }
  for (; p < p1; p += step) {
    float f[8];
    load8<BF16>(base + p * xs, lo, f);
#pragma unroll
    for (int e = 0; e < 8; ++e) { s[e] += f[e]; q[e] += f[e] * f[e]; }
  }
  float* mine = sh + ((size_t)threadIdx.y * C + threadIdx.x * 8) * 2;
#pragma unroll
  for (int e = 0; e < 8; ++e) { mine[2 * e] = s[e]; mine[2 * e + 1] = q[e]; }
  __syncthreads();
  float* dst = partial + (((long long)n * gridDim.x + blockIdx.x) * Ctot + coff) * 2;
  for (int i = tid; i < 2 * C; i += nthr) {
    float a = 0.f;
    for (int y = 0; y < (int)blockDim.y; ++y) a += sh[(size_t)y * C * 2 + i];
    dst[i] = a;
  }
}

// One CTA of 256 threads per (image, group): the partial sums (one slot per producing CTA or pixel chunk, up to
// 256 x channels-per-group entries) are read with all 8 warps in flight and reduced in a fixed order (thread ->
// warp shuffle -> 8 warp totals), so the result does not depend on scheduling.  (One WARP per group left the
// kernel latency-bound on 32 SMs: 113 launches x 16 us = 1.8 ms of a 95 ms step, ncu r1_final.)
__global__ void __launch_bounds__(256) gn_finalize_kernel(GnSrc s0, GnSrc s1, int nsrc, const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, int N, int Ctot, int groups,
                                                          float inv_count, float eps, float* __restrict__ ss) {
  __shared__ float red[2][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = blockIdx.x / groups, g = blockIdx.x % groups;
  const int cpg = Ctot / groups;
  const int glo = g * cpg, ghi = glo + cpg;
  float s = 0.f, q = 0.f;
  int cbase = 0;
  for (int si = 0; si < nsrc; ++si) {
    const GnSrc src = si == 0 ? s0 : s1;
    const int lo = max(glo, cbase), hi = min(ghi, cbase + src.C);   // this group's channels inside the source
    const int w = hi - lo;
    if (w > 0) {
      const int entries = w * src.chunks;
      for (int i = threadIdx.x; i < entries; i += 256) {
        const int ch = i / w, c = lo - cbase + (i - ch * w);
        const float2 v = *reinterpret_cast<const float2*>(src.partial + (((long long)n * src.chunks + ch) * src.C + c) * 2);
        s += v.x; q += v.y;
      }
    }
    cbase += src.C;
  }
  s = warp_sum(s); q = warp_sum(q);
  if (lane == 0) { red[0][warp] = s; red[1][warp] = q; }
  __syncthreads();
  s = ((red[0][0] + red[0][1]) + (red[0][2] + red[0][3])) + ((red[0][4] + red[0][5]) + (red[0][6] + red[0][7]));
  q = ((red[1][0] + red[1][1]) + (red[1][2] + red[1][3])) + ((red[1][4] + red[1][5]) + (red[1][6] + red[1][7]));
  const float mean = s * inv_count;
  const float var = fmaxf(q * inv_count - mean * mean, 0.f);
  const float rstd = rsqrtf(var + eps);
  for (int i = threadIdx.x; i < cpg; i += 256) {
    const int c = glo + i;
    const float sc = rstd * gamma[c];
    ss[((long long)n * Ctot + c) * 2] = sc;
    ss[((long long)n * Ctot + c) * 2 + 1] = beta[c] - mean * sc;
  }
}

template <bool BF16, bool SILU>
__global__ void gn_apply_kernel(const uint16_t* __restrict__ x, long long HW, int C, const float* __restrict__ ss,
                                int Ctot, int coff, uint16_t* __restrict__ y, int y_cstride, int pix_per_block, int xs,
                                int lo_x, int lo_y) {
  // blockDim = (C/8 channel vectors, PIX pixel lanes); grid = (pixel chunks, N).  The thread's 8
  // (scale, shift) pairs live in registers for its whole pixel strip.
  const int n = blockIdx.y;
  float sc[8], sh[8];
  {
    const float4* sp = reinterpret_cast<const float4*>(ss + ((long long)n * Ctot + coff + threadIdx.x * 8) * 2);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float4 a = __ldg(sp + e);
      sc[2 * e] = a.x; sh[2 * e] = a.y; sc[2 * e + 1] = a.z; sh[2 * e + 1] = a.w;
    }
  }
  const long long p0 = (long long)blockIdx.x * pix_per_block;
  long long p1 = p0 + pix_per_block;
  if (p1 > HW) p1 = HW;
  const uint16_t* xb = x + ((long long)n * HW) * xs + threadIdx.x * 8;
  uint16_t* yb = y + ((long long)n * HW) * y_cstride + coff + threadIdx.x * 8;
  const int step = blockDim.y;
  long long p = p0 + threadIdx.y;
  for (; p + 3 * step < p1 && !lo_y; p += 4 * step) {
    uint4 u[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) u[k] = __ldg(reinterpret_cast<const uint4*>(xb + (p + (long long)k * step) * xs));
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float f[8];
      unpack8<BF16>(u[k], f);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float v = f[e] * sc[e] + sh[e];
        f[e] = SILU ? silu_f(v) : v;
      }
      *reinterpret_cast<uint4*>(yb + (p + (long long)k * step) * y_cstride) = pack8<BF16>(f);
    }
  }
  for (; p < p1; p += step) {
    float f[8];
    load8<BF16>(xb + p * xs, lo_x, f);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float v = f[e] * sc[e] + sh[e];
      f[e] = SILU ? (lo_y ? silu_precise(v) : silu_f(v)) : v;
    }
    store8<BF16>(yb + p * y_cstride, lo_y, f);
  }
}

// ------------------------------------------------------------------------------ LayerNorm
constexpr int kLnMaxVec = 5;   // C <= 1280
// One warp per token; KV = 8-channel vectors per lane (2 for C <= 512, 3 for C <= 768, 5 for C <= 1280).  Sized to
// the channel count the kernel keeps ~35 registers at C = 320 instead of 64 (r1_final: 1.2 TB/s at half occupancy).
template <bool BF16, int KV, int TOK>
__global__ void __launch_bounds__(256) layernorm_kernel(const uint16_t* __restrict__ x, uint16_t* __restrict__ y, long long tokens,
                                                        int C, const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        float eps, int lo) {
  const int lane = threadIdx.x & 31;
  const long long tok0 = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * TOK;
  if (tok0 >= tokens) return;
  const int nvec = C / 8;
  const int xs = lo ? 2 * C : C;
  float f[TOK][KV][8];
#pragma unroll
  for (int t = 0; t < TOK; ++t) {
#pragma unroll
    for (int i = 0; i < KV; ++i) {
      const int v = lane + 32 * i;
      if (v < nvec && tok0 + t < tokens) {
        load8<BF16>(x + (tok0 + t) * xs + v * 8, lo, f[t][i]);
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) f[t][i][e] = 0.f;
      }
    }
  }
  float mean[TOK], rstd[TOK];
#pragma unroll
  for (int t = 0; t < TOK; ++t) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < KV; ++i) {
      if (lane + 32 * i < nvec) {
#pragma unroll
        for (int e = 0; e < 8; ++e) s += f[t][i][e];
      }
    }
    mean[t] = warp_sum(s) / C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < KV; ++i) {
      if (lane + 32 * i < nvec) {
#pragma unroll
        for (int e = 0; e < 8; ++e) { const float d = f[t][i][e] - mean[t]; q += d * d; }
      }
    }
    rstd[t] = rsqrtf(warp_sum(q) / C + eps);
  }
#pragma unroll
  for (int i = 0; i < KV; ++i) {
    const int v = lane + 32 * i;
    if (v < nvec) {
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + v * 8)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + v * 8 + 4));
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + v * 8)), b1 = __ldg(reinterpret_cast<const float4*>(beta + v * 8 + 4));
      const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int t = 0; t < TOK; ++t) {
        if (tok0 + t < tokens) {
          float o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = (f[t][i][e] - mean[t]) * rstd[t] * gg[e] + bb[e];
          store8<BF16>(y + (tok0 + t) * xs + v * 8, lo, o);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------ row softmax
constexpr int kSmMaxVec = 8;   // T <= 256 threads * 8 vec * 8 = 16384
template <bool BF16>
__global__ void softmax_rows_small_kernel(uint16_t* __restrict__ s, long long rows, int T, int Tp, int lo) {
  const int lane = threadIdx.x & 31;
  const long long r = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  uint16_t* row = s + r * (lo ? 2 * Tp : Tp);
  float m = -INFINITY;
  for (int i = lane; i < T; i += 32) m = fmaxf(m, load1<BF16>(row + i, lo));
  m = warp_max(m);
  float sum = 0.f;
  for (int i = lane; i < T; i += 32) sum += __expf(load1<BF16>(row + i, lo) - m);
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  for (int i = lane; i < T; i += 32) store1<BF16>(row + i, lo, __expf(load1<BF16>(row + i, lo) - m) * inv);
}

// MV = 8-column vectors per thread: 8 (any T up to 16384, 256 threads) or 3 with 512 threads for T <= 12288 — the
// VAE mid-block rows (T = 9216) then hold 24 values per thread instead of 64 (r1_final: 2.5 TB/s at low occupancy).
template <bool BF16, int MV>
__global__ void softmax_rows_kernel(uint16_t* __restrict__ s, int T, int Tp, int lo) {
  __shared__ float red[32];
  uint16_t* row = s + (long long)blockIdx.x * (lo ? 2 * Tp : Tp);
  const int nvec = T / 8;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  float f[MV][8];
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < MV; ++i) {
    const int v = threadIdx.x + i * blockDim.x;
    if (v < nvec) {
      load8<BF16>(row + v * 8, lo, f[i]);
#pragma unroll
      for (int e = 0; e < 8; ++e) m = fmaxf(m, f[i][e]);
    }
  }
  m = warp_max(m);
  if (lane == 0) red[warp] = m;
  __syncthreads();
  m = red[0];
  for (int w = 1; w < nwarp; ++w) m = fmaxf(m, red[w]);
  __syncthreads();
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < MV; ++i) {
    if (threadIdx.x + i * blockDim.x < nvec) {
#pragma unroll
      for (int e = 0; e < 8; ++e) { f[i][e] = __expf(f[i][e] - m); sum += f[i][e]; }
    }
  }
  sum = warp_sum(sum);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  sum = 0.f;
  for (int w = 0; w < nwarp; ++w) sum += red[w];
  const float inv = 1.f / sum;
#pragma unroll
  for (int i = 0; i < MV; ++i) {
    const int v = threadIdx.x + i * blockDim.x;
    if (v < nvec) {
#pragma unroll
      for (int e = 0; e < 8; ++e) f[i][e] *= inv;
      store8<BF16>(row + v * 8, lo, f[i]);
    }
  }
}

// Long rows (the VAE mid-block attention, T = 9216: 18 KiB per row, 73 728 rows per step and attention): a persistent
// CTA streams its rows through a 3-slot shared-memory ring with bulk async copies — slot k + 2 is loading and slot
// k - 1 is draining to global memory while row k is reduced in registers — so each SM keeps several rows in flight in
// both directions.  The one-row-per-CTA kernel above has its loads, two block reductions and stores back to back
// (r2: 2.4 TB/s, 1.1 ms per attention; this one is bound by the copy rate).
constexpr int kSmPipeThreads = 384;
constexpr int kSmPipeSlots = 3;
template <bool BF16, int MV>
__global__ void __launch_bounds__(kSmPipeThreads) softmax_rows_pipe_kernel(uint16_t* __restrict__ s, long long rows, int T, int Tp) {
  extern __shared__ __align__(128) uint8_t sm_raw[];
  __shared__ float red[2][kSmPipeThreads / 32];
  __shared__ __align__(8) uint64_t full[kSmPipeSlots];
  const int row_bytes = T * 2;
  const int slot_bytes = (row_bytes + 127) & ~127;
  const int nvec = T / 8;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = kSmPipeThreads / 32;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kSmPipeSlots; ++i) mbar_init(&full[i], 1);
    fence_barrier_init();
  }
  __syncthreads();
  auto issue_load = [&](long long k) {            // thread 0 only
    const long long r = (long long)blockIdx.x + k * gridDim.x;
    if (r >= rows) return;
    const int slot = (int)(k % kSmPipeSlots);
    mbar_expect_tx(&full[slot], (uint32_t)row_bytes);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(sm_raw + (size_t)slot * slot_bytes)),
                 "l"(reinterpret_cast<uint64_t>(s + r * Tp)), "r"(row_bytes), "r"(smem_u32(&full[slot]))
                 : "memory");
  };
  if (threadIdx.x == 0) { issue_load(0); issue_load(1); }
  long long k = 0;
  for (long long r = blockIdx.x; r < rows; r += gridDim.x, ++k) {
    const int slot = (int)(k % kSmPipeSlots);
    uint8_t* buf = sm_raw + (size_t)slot * slot_bytes;
    mbar_wait(&full[slot], (uint32_t)((k / kSmPipeSlots) & 1), 30);
    float f[MV][8];
    float m = -INFINITY;
#pragma unroll
    for (int i = 0; i < MV; ++i) {
      const int v = threadIdx.x + i * kSmPipeThreads;
      if (v < nvec) {
        unpack8<BF16>(*reinterpret_cast<const uint4*>(buf + v * 16), f[i]);
#pragma unroll
        for (int e = 0; e < 8; ++e) m = fmaxf(m, f[i][e]);
      }
    }
    m = warp_max(m);
    if (lane == 0) red[0][warp] = m;
    __syncthreads();
    m = red[0][0];
#pragma unroll
    for (int w = 1; w < NW; ++w) m = fmaxf(m, red[0][w]);
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < MV; ++i) {
      if (threadIdx.x + i * kSmPipeThreads < nvec) {
#pragma unroll
        for (int e = 0; e < 8; ++e) { f[i][e] = __expf(f[i][e] - m); sum += f[i][e]; }
      }
    }
    sum = warp_sum(sum);
    if (lane == 0) red[1][warp] = sum;
    __syncthreads();
    sum = 0.f;
#pragma unroll
    for (int w = 0; w < NW; ++w) sum += red[1][w];
    const float inv = 1.f / sum;
#pragma unroll
    for (int i = 0; i < MV; ++i) {
      const int v = threadIdx.x + i * kSmPipeThreads;
      if (v < nvec) {
#pragma unroll
        for (int e = 0; e < 8; ++e) f[i][e] *= inv;
        *reinterpret_cast<uint4*>(buf + v * 16) = pack8<BF16>(f[i]);
      }
    }
    fence_proxy_async_shared();                   // the generic-proxy writes above are visible to the bulk store
    __syncthreads();                              // (also: red[] is free for the next row)
    if (threadIdx.x == 0) {
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(reinterpret_cast<uint64_t>(s + r * Tp)),
                   "r"(smem_u32(buf)), "r"(row_bytes)
                   : "memory");
      tma_store_commit();
      // slot of row k + 2 == slot of row k - 1: its store (the group before the one just committed) has read the slot
      asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      issue_load(k + 2);
    }
  }
  if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ------------------------------------------------------------------------------ 2-token cross attention
// y = x + c0 + sigmoid(LN(x).U + u0).M : one warp handles TOK tokens at once so every U / M / c0 vector
// fetched from L1/L2 is reused TOK times (the single-token version re-read ~2*heads*C*4 bytes per token).
template <bool BF16, int KV, int TOK>
__global__ void xattn2_kernel(const uint16_t* __restrict__ x, uint16_t* __restrict__ y, long long tokens, int C,
                              int heads, const float* __restrict__ U, const float* __restrict__ u0,
                              const float* __restrict__ M, const float* __restrict__ c0, float eps, int lo) {
  const int lane = threadIdx.x & 31;
  const long long tok0 = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * TOK;
  if (tok0 >= tokens) return;
  const int nvec = C / 8;
  const int xs = lo ? 2 * C : C;
  float f[TOK][KV][8];
  float mean[TOK], rstd[TOK];
#pragma unroll
  for (int t = 0; t < TOK; ++t) {
    const bool tv = tok0 + t < tokens;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < KV; ++i) {
      const int v = lane + 32 * i;
      if (v < nvec && tv) {
        load8<BF16>(x + (tok0 + t) * xs + v * 8, lo, f[t][i]);
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) f[t][i][e] = 0.f;
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) s += f[t][i][e];
    }
    mean[t] = warp_sum(s) / C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < KV; ++i) {
      if (lane + 32 * i < nvec) {
#pragma unroll
        for (int e = 0; e < 8; ++e) { const float d = f[t][i][e] - mean[t]; q += d * d; }
      }
    }
    rstd[t] = rsqrtf(warp_sum(q) / C + eps);
  }
  float acc[TOK][KV][8];
#pragma unroll
  for (int i = 0; i < KV; ++i) {
    const int v = lane + 32 * i;
    if (v < nvec) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(c0 + v * 8));
      const float4 b = __ldg(reinterpret_cast<const float4*>(c0 + v * 8 + 4));
#pragma unroll
      for (int t = 0; t < TOK; ++t) {
        acc[t][i][0] = f[t][i][0] + a.x; acc[t][i][1] = f[t][i][1] + a.y; acc[t][i][2] = f[t][i][2] + a.z; acc[t][i][3] = f[t][i][3] + a.w;
        acc[t][i][4] = f[t][i][4] + b.x; acc[t][i][5] = f[t][i][5] + b.y; acc[t][i][6] = f[t][i][6] + b.z; acc[t][i][7] = f[t][i][7] + b.w;
      }
    }
  }
  for (int h = 0; h < heads; ++h) {
    float d[TOK];
#pragma unroll
    for (int t = 0; t < TOK; ++t) d[t] = 0.f;
#pragma unroll
    for (int i = 0; i < KV; ++i) {
      const int v = lane + 32 * i;
      if (v < nvec) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(U + (long long)h * C + v * 8));
        const float4 b = __ldg(reinterpret_cast<const float4*>(U + (long long)h * C + v * 8 + 4));
#pragma unroll
        for (int t = 0; t < TOK; ++t) {
          const float mt = mean[t];
          d[t] += (f[t][i][0] - mt) * a.x + (f[t][i][1] - mt) * a.y + (f[t][i][2] - mt) * a.z + (f[t][i][3] - mt) * a.w +
                  (f[t][i][4] - mt) * b.x + (f[t][i][5] - mt) * b.y + (f[t][i][6] - mt) * b.z + (f[t][i][7] - mt) * b.w;
        }
      }
    }
    float pr[TOK];
    const float u0h = __ldg(u0 + h);
#pragma unroll
    for (int t = 0; t < TOK; ++t) pr[t] = 1.f / (1.f + __expf(-(warp_sum(d[t]) * rstd[t] + u0h)));
#pragma unroll
    for (int i = 0; i < KV; ++i) {
      const int v = lane + 32 * i;
      if (v < nvec) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(M + (long long)h * C + v * 8));
        const float4 b = __ldg(reinterpret_cast<const float4*>(M + (long long)h * C + v * 8 + 4));
#pragma unroll
        for (int t = 0; t < TOK; ++t) {
          acc[t][i][0] += pr[t] * a.x; acc[t][i][1] += pr[t] * a.y; acc[t][i][2] += pr[t] * a.z; acc[t][i][3] += pr[t] * a.w;
          acc[t][i][4] += pr[t] * b.x; acc[t][i][5] += pr[t] * b.y; acc[t][i][6] += pr[t] * b.z; acc[t][i][7] += pr[t] * b.w;
        }
      }
    }
  }
#pragma unroll
  for (int t = 0; t < TOK; ++t) {
    if (tok0 + t < tokens) {
#pragma unroll
      for (int i = 0; i < KV; ++i) {
        const int v = lane + 32 * i;
        if (v < nvec) store8<BF16>(y + (tok0 + t) * xs + v * 8, lo, acc[t][i]);
      }
    }
  }
}

// Same operator with the folded weights resident in shared memory.  The kernel above re-reads U and M (2 * heads * C
// floats: 12.8 / 51 / 205 KB at C = 320 / 640 / 1280) through L1 for every warp's tokens — 0.94 GB of L2 traffic per
// launch at every level, 100-160 us for a 6-94 MB activation (r2 per-op events).  Here a persistent CTA loads them once,
// its warps loop over token groups, and the heads are taken five at a time so that the five warp reductions and
// sigmoids of a batch are independent chains instead of one serial chain per head.
constexpr int kXaHB = 5;
template <bool BF16, int KV, int TOK>
__global__ void __launch_bounds__(KV >= 5 ? 512 : 256) xattn2_smem_kernel(const uint16_t* __restrict__ x, uint16_t* __restrict__ y, long long tokens,
                                                          int C, int heads, const float* __restrict__ U,
                                                          const float* __restrict__ u0, const float* __restrict__ M,
                                                          const float* __restrict__ c0, float eps, int lo) {
  extern __shared__ __align__(16) float xa_sm[];
  float* sU = xa_sm;
  float* sM = sU + heads * C;
  float* sc0 = sM + heads * C;
  float* su0 = sc0 + C;
  {
    const int n4 = heads * C / 4;
    const float4* gU = reinterpret_cast<const float4*>(U);
    const float4* gM = reinterpret_cast<const float4*>(M);
    // four loads of each matrix in flight per thread (one per iteration left the 205 KB fill of C = 1280 latency-bound: 25 us)
    int i = threadIdx.x;
    for (; i + 3 * (int)blockDim.x < n4; i += 4 * blockDim.x) {
      float4 a[4], b[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) { a[k] = __ldg(gU + i + k * blockDim.x); b[k] = __ldg(gM + i + k * blockDim.x); }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        reinterpret_cast<float4*>(sU)[i + k * blockDim.x] = a[k];
        reinterpret_cast<float4*>(sM)[i + k * blockDim.x] = b[k];
      }
    }
    for (; i < n4; i += blockDim.x) {
      reinterpret_cast<float4*>(sU)[i] = __ldg(gU + i);
      reinterpret_cast<float4*>(sM)[i] = __ldg(gM + i);
    }
    for (int i = threadIdx.x; i < C; i += blockDim.x) sc0[i] = __ldg(c0 + i);
    for (int i = threadIdx.x; i < heads; i += blockDim.x) su0[i] = __ldg(u0 + i);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int nvec = C / 8;
  const int xs = lo ? 2 * C : C;
  for (long long tok0 = ((long long)blockIdx.x * nwarp + warp) * TOK; tok0 < tokens; tok0 += (long long)gridDim.x * nwarp * TOK) {
    float g[TOK][KV][8], acc[TOK][KV][8];
    float rstd[TOK];
#pragma unroll
    for (int t = 0; t < TOK; ++t) {
      const bool tv = tok0 + t < tokens;
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < KV; ++i) {
        const int v = lane + 32 * i;
        if (v < nvec && tv) {
          load8<BF16>(x + (tok0 + t) * xs + v * 8, lo, g[t][i]);
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) g[t][i][e] = 0.f;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) s += g[t][i][e];
      }
      const float mean = warp_sum(s) / C;
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < KV; ++i) {
        const int v = lane + 32 * i;
        if (v < nvec) {
          const float4 a = *reinterpret_cast<const float4*>(sc0 + v * 8), b = *reinterpret_cast<const float4*>(sc0 + v * 8 + 4);
          const float cc[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            acc[t][i][e] = g[t][i][e] + cc[e];
            g[t][i][e] -= mean;
            q += g[t][i][e] * g[t][i][e];
          }
        }
      }
      rstd[t] = rsqrtf(warp_sum(q) / C + eps);
    }
    for (int h0 = 0; h0 < heads; h0 += kXaHB) {
      float d[kXaHB][TOK];
#pragma unroll
      for (int hh = 0; hh < kXaHB; ++hh) {
#pragma unroll
        for (int t = 0; t < TOK; ++t) d[hh][t] = 0.f;
#pragma unroll
        for (int i = 0; i < KV; ++i) {
          const int v = lane + 32 * i;
          if (v < nvec) {
            const float* up = sU + (h0 + hh) * C + v * 8;
            const float4 a = *reinterpret_cast<const float4*>(up), b = *reinterpret_cast<const float4*>(up + 4);
#pragma unroll
            for (int t = 0; t < TOK; ++t)
              d[hh][t] += g[t][i][0] * a.x + g[t][i][1] * a.y + g[t][i][2] * a.z + g[t][i][3] * a.w + g[t][i][4] * b.x +
                          g[t][i][5] * b.y + g[t][i][6] * b.z + g[t][i][7] * b.w;
          }
        }
      }
#pragma unroll
      for (int hh = 0; hh < kXaHB; ++hh)
#pragma unroll
        for (int t = 0; t < TOK; ++t) d[hh][t] = 1.f / (1.f + __expf(-(warp_sum(d[hh][t]) * rstd[t] + su0[h0 + hh])));
#pragma unroll
      for (int hh = 0; hh < kXaHB; ++hh) {
#pragma unroll
        for (int i = 0; i < KV; ++i) {
          const int v = lane + 32 * i;
          if (v < nvec) {
            const float* mp = sM + (h0 + hh) * C + v * 8;
            const float4 a = *reinterpret_cast<const float4*>(mp), b = *reinterpret_cast<const float4*>(mp + 4);
#pragma unroll
            for (int t = 0; t < TOK; ++t) {
              const float pr = d[hh][t];
              acc[t][i][0] += pr * a.x; acc[t][i][1] += pr * a.y; acc[t][i][2] += pr * a.z; acc[t][i][3] += pr * a.w;
              acc[t][i][4] += pr * b.x; acc[t][i][5] += pr * b.y; acc[t][i][6] += pr * b.z; acc[t][i][7] += pr * b.w;
            }
          }
        }
      }
    }
#pragma unroll
    for (int t = 0; t < TOK; ++t) {
      if (tok0 + t < tokens) {
#pragma unroll
        for (int i = 0; i < KV; ++i) {
          const int v = lane + 32 * i;
          if (v < nvec) store8<BF16>(y + (tok0 + t) * xs + v * 8, lo, acc[t][i]);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------ elementwise
template <bool BF16>
__global__ void geglu_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, long long total_vec, int C4) {
  const int nvec = C4 / 8;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec;
       i += (long long)gridDim.x * blockDim.x) {
    const long long tok = i / nvec;
    const int v = (int)(i % nvec);
    float a[8], g[8];
    unpack8<BF16>(__ldg(reinterpret_cast<const uint4*>(in + tok * 2 * C4 + v * 8)), a);
    unpack8<BF16>(__ldg(reinterpret_cast<const uint4*>(in + tok * 2 * C4 + C4 + v * 8)), g);
#pragma unroll
    for (int e = 0; e < 8; ++e) a[e] *= 0.5f * g[e] * (1.f + erff(g[e] * 0.70710678118654752f));
    *reinterpret_cast<uint4*>(out + tok * C4 + v * 8) = pack8<BF16>(a);
  }
}

template <bool BF16>
__global__ void relu_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, long long total_vec, int nvec,
                            int lo) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec;
       i += (long long)gridDim.x * blockDim.x) {
    const long long off = lo ? (i / nvec) * (2LL * lo) + (i % nvec) * 8 : i * 8;   // [pixel][hi C | lo C]
    float a[8];
    load8<BF16>(in + off, lo, a);
#pragma unroll
    for (int e = 0; e < 8; ++e) a[e] = fmaxf(a[e], 0.f);
    store8<BF16>(out + off, lo, a);
  }
}

template <bool BF16>
__global__ void bilinear_up2x_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, int N, int H, int W,
                                     int C, float sy, float sx, long long total_vec, int lo) {
  const int nvec = C / 8;
  const int Ho = 2 * H, Wo = 2 * W;
  const int xs = lo ? 2 * C : C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % nvec);
    long long r = i / nvec;
    const int ox = (int)(r % Wo);
    r /= Wo;
    const int oy = (int)(r % Ho);
    const int n = (int)(r / Ho);
    const float fy = sy * oy, fx = sx * ox;
    const int y0 = (int)fy, x0 = (int)fx;
    const int y1 = y0 + (y0 < H - 1 ? 1 : 0), x1 = x0 + (x0 < W - 1 ? 1 : 0);
    const float h1 = fy - y0, w1 = fx - x0, h0 = 1.f - h1, w0 = 1.f - w1;
    const uint16_t* b = in + ((long long)n * H * W) * xs + v * 8;
    float a00[8], a01[8], a10[8], a11[8], o[8];
    load8<BF16>(b + ((long long)y0 * W + x0) * xs, lo, a00);
    load8<BF16>(b + ((long long)y0 * W + x1) * xs, lo, a01);
    load8<BF16>(b + ((long long)y1 * W + x0) * xs, lo, a10);
    load8<BF16>(b + ((long long)y1 * W + x1) * xs, lo, a11);
#pragma unroll
    for (int e = 0; e < 8; ++e) o[e] = h0 * (w0 * a00[e] + w1 * a01[e]) + h1 * (w0 * a10[e] + w1 * a11[e]);
    store8<BF16>(out + (((long long)n * Ho + oy) * Wo + ox) * xs + v * 8, lo, o);
  }
}

template <bool BF16>
__global__ void preprocess_kernel(const void* __restrict__ in, int kind, uint16_t* __restrict__ out, int N,
                                  long long HW, int lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * HW) return;
  const int n = (int)(i / HW);
  const long long p = i % HW;
  float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const long long off = ((long long)n * 3 + c) * HW + p;
    if (kind == 0) f[c] = (float)reinterpret_cast<const uint8_t*>(in)[off] / 255.0f * 2.0f - 1.0f;
    else if (kind == 1) f[c] = f16_to_f32<false>(reinterpret_cast<const uint16_t*>(in)[off]);
    else f[c] = reinterpret_cast<const float*>(in)[off];
  }
  store8<BF16>(out + i * (lo ? 16 : 8), lo, f);
}

// K-packed stem: the 3x3 neighbourhood of every pixel laid out along the channel axis, NHWC32 =
// [centre tap (3 ch) | the other 8 taps in row-major order (24 ch) | 5 zeros], so that AutoencoderKL.encoder.conv_in
// (3 -> 128, 3x3) becomes a 1x1 GEMM with K = 27 (one 64-channel chunk) instead of nine 64-wide chunks of which 3
// channels are real (1177 us -> one pass bound by the 1.2 GB output write at 8 x 768^2).  Out-of-image taps are zero.
template <bool BF16>
__global__ void preprocess_im2col_kernel(const void* __restrict__ in, int kind, uint16_t* __restrict__ out, int N, int H, int W,
                                         int lo) {
  const long long HW = (long long)H * W;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * HW) return;
  const int n = (int)(i / HW);
  const long long p = i % HW;
  const int y = (int)(p / W), x = (int)(p % W);
  float f[32];
#pragma unroll
  for (int k = 0; k < 32; ++k) f[k] = 0.f;
  auto fetch = [&](int yy, int xx, int c) -> float {
    if ((unsigned)yy >= (unsigned)H || (unsigned)xx >= (unsigned)W) return 0.f;
    const long long off = ((long long)n * 3 + c) * HW + (long long)yy * W + xx;
    if (kind == 0) return (float)reinterpret_cast<const uint8_t*>(in)[off] / 255.0f * 2.0f - 1.0f;
    if (kind == 1) return f16_to_f32<false>(reinterpret_cast<const uint16_t*>(in)[off]);
    return reinterpret_cast<const float*>(in)[off];
  };
  int slot = 1;
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const int k = (r == 1 && q == 1) ? 0 : slot++;
#pragma unroll
      for (int c = 0; c < 3; ++c) f[k * 3 + c] = fetch(y + r - 1, x + q - 1, c);
    }
  uint16_t* o = out + i * (lo ? 64 : 32);
#pragma unroll
  for (int v = 0; v < 4; ++v) {
    float g[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) g[e] = f[v * 8 + e];
    store8<BF16>(o + v * 8, lo, g);
  }
}

__device__ __forceinline__ unsigned int f2ord(float f) {
  unsigned int u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned int u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}
__global__ void minmax_init_kernel(unsigned int* s, int N) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) { s[2 * i] = 0xFFFFFFFFu; s[2 * i + 1] = 0u; }
}
__global__ void minmax_reduce_kernel(const float* __restrict__ x, long long HW, unsigned int* s) {
  const int n = blockIdx.y;
  float mn = INFINITY, mx = -INFINITY;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += (long long)gridDim.x * blockDim.x) {
    const float v = x[(long long)n * HW + i];
    mn = fminf(mn, v); mx = fmaxf(mx, v);
  }
  mn = -warp_max(-mn); mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) { atomicMin(&s[2 * n], f2ord(mn)); atomicMax(&s[2 * n + 1], f2ord(mx)); }
}
__global__ void minmax_apply_kernel(float* __restrict__ x, long long HW, const unsigned int* __restrict__ s, float dmin, int zero_min) {
  const int n = blockIdx.y;
  const float mn = zero_min ? 0.f : ord2f(s[2 * n]), mx = ord2f(s[2 * n + 1]);
  const float d = fmaxf(mx - mn, dmin);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += (long long)gridDim.x * blockDim.x)
    x[(long long)n * HW + i] = (x[(long long)n * HW + i] - mn) / d;
}

inline int blocks_for(long long total, int threads, int cap = 148 * 16) {
  long long b = (total + threads - 1) / threads;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace

#define GP_DISPATCH_BF16(bf16, ...) \
  do {                              \
    if (bf16) {                     \
      constexpr bool BF = true;     \
      __VA_ARGS__;                  \
    } else {                        \
      constexpr bool BF = false;    \
      __VA_ARGS__;                  \
    }                               \
  } while (0)

cudaError_t direct_conv(const DirectConvParams& p, bool bf16, cudaStream_t s) {
  const long long total = (long long)p.N * p.Ho * p.Wo * p.Cout;
  if (total <= 0) return cudaSuccess;
  const int threads = 256;
  const long long blocks = (total + threads - 1) / threads;
  GP_DISPATCH_BF16(bf16, (launch(direct_conv_kernel<BF>, (unsigned)blocks, threads, 0, s, p)));
  return cudaGetLastError();
}

int gn_chunks(int N, long long HW) {
  (void)N;   // independent of the batch size: a batch of B equals B batches of 1 bit for bit
  long long c = (HW + 63) / 64;
  if (c > 256) c = 256;
  if (c < 1) c = 1;
  return (int)c;
}

cudaError_t gn_stats(const void* x, int N, long long HW, int C, float* partial, int chunks, int Ctot, int coff,
                     bool bf16, cudaStream_t s, bool split) {
  const int nvec = C / 8;
  int pix = 256 / nvec;
  if (pix < 1) pix = 1;
  if (pix > 32) pix = 32;
  const int pix_per_block = (int)((HW + chunks - 1) / chunks);
  dim3 block(nvec, pix);
  dim3 grid((unsigned)chunks, N);
  const size_t smem = (size_t)pix * C * 2 * sizeof(float);
  GP_DISPATCH_BF16(bf16, (launch(gn_stats_kernel<BF>, grid, block, smem, s, reinterpret_cast<const uint16_t*>(x), HW, C,
                                                                         partial, Ctot, coff, pix_per_block,
                                                                         split ? 2 * C : C, split ? C : 0)));
  return cudaGetLastError();
}

cudaError_t gn_finalize(const GnSrc* srcs, int nsrc, const float* gamma, const float* beta, int N, int Ctot,
                        int groups, long long HW, float eps, float* ss, cudaStream_t s) {
  if (nsrc < 1 || nsrc > 2) return cudaErrorInvalidValue;
  const float inv_count = 1.0f / ((float)HW * (float)(Ctot / groups));
  launch(gn_finalize_kernel, N * groups, 256, 0, s, srcs[0], nsrc > 1 ? srcs[1] : srcs[0], nsrc, gamma, beta, N, Ctot,
                                                       groups, inv_count, eps, ss);
  return cudaGetLastError();
}

cudaError_t gn_apply(const void* x, int N, long long HW, int C, const float* ss, int Ctot, int coff, void* y,
                     int y_cstride, bool silu, bool bf16, cudaStream_t s, bool split) {
  // split: x carries [hi C | lo C] per pixel; y has y_cstride LOGICAL channels, i.e. [hi y_cstride | lo y_cstride]
  const int xs = split ? 2 * C : C, lo_x = split ? C : 0, lo_y = split ? y_cstride : 0;
  if (split) y_cstride *= 2;
  const int nvec = C / 8;
  int pix = 256 / nvec;
  if (pix < 1) pix = 1;
  if (pix > 32) pix = 32;
  // (a software-pipelined variant — next four loads in flight during the arithmetic, 72 registers — and 4x longer pixel
  //  strips per block measured 97.9 / 98.0 ms per step against 96.3-96.9 for this form, r2o)
  const int pix_per_block = pix * 16;
  dim3 block(nvec, pix);
  dim3 grid((unsigned)((HW + pix_per_block - 1) / pix_per_block), N);
  const uint16_t* xi = reinterpret_cast<const uint16_t*>(x);
  uint16_t* yo = reinterpret_cast<uint16_t*>(y);
  if (silu)
    GP_DISPATCH_BF16(bf16, (launch(gn_apply_kernel<BF, true>, grid, block, 0, s, xi, HW, C, ss, Ctot, coff, yo, y_cstride, pix_per_block, xs, lo_x, lo_y)));
  else
    GP_DISPATCH_BF16(bf16, (launch(gn_apply_kernel<BF, false>, grid, block, 0, s, xi, HW, C, ss, Ctot, coff, yo, y_cstride, pix_per_block, xs, lo_x, lo_y)));
  return cudaGetLastError();
}

cudaError_t layernorm(const void* x, void* y, long long tokens, int C, const float* gamma, const float* beta,
                      float eps, bool bf16, cudaStream_t s, bool split) {
  const int lo = split ? C : 0;
  if (C % 8 || C / 8 > 32 * kLnMaxVec) return cudaErrorInvalidValue;
  const int tpb = 8;
  const uint16_t* xi = reinterpret_cast<const uint16_t*>(x);
  uint16_t* yo = reinterpret_cast<uint16_t*>(y);
  const int kv = (C / 8 + 31) / 32;
  // one token per warp; two per warp (all loads up front) measured slower: 80 registers, 0.87 -> 1.08 ms per step (r2m)
  const int tok = 1;
  const long long blocks = (tokens + tpb * tok - 1) / (tpb * tok);
  if (kv <= 2)
    GP_DISPATCH_BF16(bf16, (launch(layernorm_kernel<BF, 2, 1>, (unsigned)blocks, tpb * 32, 0, s, xi, yo, tokens, C, gamma, beta, eps, lo)));
  else if (kv <= 3)
    GP_DISPATCH_BF16(bf16, (launch(layernorm_kernel<BF, 3, 1>, (unsigned)blocks, tpb * 32, 0, s, xi, yo, tokens, C, gamma, beta, eps, lo)));
  else
    GP_DISPATCH_BF16(bf16, (launch(layernorm_kernel<BF, 5, 1>, (unsigned)blocks, tpb * 32, 0, s, xi, yo, tokens, C, gamma, beta, eps, lo)));
  return cudaGetLastError();
}

cudaError_t softmax_rows(void* sio, long long rows, int T, int Tp, bool bf16, cudaStream_t s, bool split) {
  const int lo = split ? Tp : 0;
  if (T % 8 || Tp % 8 || T < 64) {
    const int wpb = 8;
    GP_DISPATCH_BF16(bf16, (launch(softmax_rows_small_kernel<BF>, (unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, s, 
                               reinterpret_cast<uint16_t*>(sio), rows, T, Tp, lo)));
    return cudaGetLastError();
  }
  if (T / 8 > 256 * kSmMaxVec) return cudaErrorInvalidValue;
  if (!split && T >= 2048 && T / 8 <= kSmPipeThreads * 6 && rows >= 1024) {
    const int slot_bytes = (T * 2 + 127) & ~127;
    const int smem = kSmPipeSlots * slot_bytes;
    if (smem <= 200 * 1024) {
      static int sms[64] = {0};
      int dev = 0;
      cudaGetDevice(&dev);
      if (!sms[dev & 63]) {
        cudaDeviceGetAttribute(&sms[dev & 63], cudaDevAttrMultiProcessorCount, dev);
        GP_DISPATCH_BF16(bf16, (cudaFuncSetAttribute(softmax_rows_pipe_kernel<BF, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)));
        GP_DISPATCH_BF16(bf16, (cudaFuncSetAttribute(softmax_rows_pipe_kernel<BF, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)));
      }
      int per_sm = (220 * 1024) / (smem + 1024);
      if (per_sm > 5) per_sm = 5;                 // 5 x 384 threads
      if (per_sm < 1) per_sm = 1;
      long long grid = (long long)sms[dev & 63] * per_sm;
      if (grid > rows) grid = rows;
      if (T / 8 <= kSmPipeThreads * 3) {
        GP_DISPATCH_BF16(bf16, (launch(softmax_rows_pipe_kernel<BF, 3>, (unsigned)grid, kSmPipeThreads, smem, s, reinterpret_cast<uint16_t*>(sio), rows, T, Tp)));
      } else {
        GP_DISPATCH_BF16(bf16, (launch(softmax_rows_pipe_kernel<BF, 6>, (unsigned)grid, kSmPipeThreads, smem, s, reinterpret_cast<uint16_t*>(sio), rows, T, Tp)));
      }
      return cudaGetLastError();
    }
  }
  int threads = ((T / 8 + 31) / 32) * 32;
  if (threads > 256) threads = 256;
  if (threads < 32) threads = 32;
  if (T / 8 > 256 && T / 8 <= 512 * 3) {
    GP_DISPATCH_BF16(bf16, (launch(softmax_rows_kernel<BF, 3>, (unsigned)rows, 512, 0, s, reinterpret_cast<uint16_t*>(sio), T, Tp, lo)));
    return cudaGetLastError();
  }
  GP_DISPATCH_BF16(bf16, (launch(softmax_rows_kernel<BF, kSmMaxVec>, (unsigned)rows, threads, 0, s, reinterpret_cast<uint16_t*>(sio), T, Tp, lo)));
  return cudaGetLastError();
}

template <bool BF, int KV, int TOK>
static cudaError_t xattn2_launch(const void* x, void* y, long long tokens, int C, int heads, const float* U, const float* u0,
                                 const float* M, const float* c0, float eps, cudaStream_t s, int lo) {
  const int wpb = 8;
  const long long per_block = (long long)wpb * TOK;
  const long long blocks = (tokens + per_block - 1) / per_block;
  launch(xattn2_kernel<BF, KV, TOK>, (unsigned)blocks, wpb * 32, 0, s, reinterpret_cast<const uint16_t*>(x),
                                                                    reinterpret_cast<uint16_t*>(y), tokens, C, heads, U, u0, M,
                                                                    c0, eps, lo);
  return cudaGetLastError();
}

cudaError_t xattn2(const void* x, void* y, long long tokens, int C, int heads, const float* U, const float* u0,
                   const float* M, const float* c0, float eps, bool bf16, cudaStream_t s, bool split) {
  const int lo = split ? C : 0;
  if (C % 8 || C / 8 > 32 * kLnMaxVec) return cudaErrorInvalidValue;
  const int kv = (C / 8 + 31) / 32;
  cudaError_t e = cudaSuccess;
  const size_t smem = ((size_t)2 * heads * C + C + heads) * sizeof(float);
  if (heads % kXaHB == 0 && C % 32 == 0 && smem <= 226 * 1024) {
    static int sms[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!sms[dev & 63]) {
      const int big = 226 * 1024;
      GP_DISPATCH_BF16(bf16, (cudaFuncSetAttribute(xattn2_smem_kernel<BF, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)));
      GP_DISPATCH_BF16(bf16, (cudaFuncSetAttribute(xattn2_smem_kernel<BF, 3, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)));
      GP_DISPATCH_BF16(bf16, (cudaFuncSetAttribute(xattn2_smem_kernel<BF, 5, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, big)));
      cudaDeviceGetAttribute(&sms[dev & 63], cudaDevAttrMultiProcessorCount, dev);
    }
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (per_sm > 2) per_sm = 2;                       // 256 threads at <= 128 registers
    if (per_sm < 1) per_sm = 1;
    const int tok = kv <= 3 ? 2 : 1;
    const int threads = kv <= 3 ? 256 : 512;          // C = 1280 leaves room for one CTA per SM: 16 warps instead of 8
    if (kv > 3) per_sm = 1;
    long long grid = (tokens + (threads / 32) * tok - 1) / ((threads / 32) * tok);
    if (grid > (long long)sms[dev & 63] * per_sm) grid = (long long)sms[dev & 63] * per_sm;
    const uint16_t* xi = reinterpret_cast<const uint16_t*>(x);
    uint16_t* yo = reinterpret_cast<uint16_t*>(y);
    if (kv <= 2)
      GP_DISPATCH_BF16(bf16, (launch(xattn2_smem_kernel<BF, 2, 2>, (unsigned)grid, 256, smem, s, xi, yo, tokens, C, heads, U, u0, M, c0, eps, lo)));
    else if (kv <= 3)
      GP_DISPATCH_BF16(bf16, (launch(xattn2_smem_kernel<BF, 3, 2>, (unsigned)grid, 256, smem, s, xi, yo, tokens, C, heads, U, u0, M, c0, eps, lo)));
    else
      GP_DISPATCH_BF16(bf16, (launch(xattn2_smem_kernel<BF, 5, 1>, (unsigned)grid, threads, smem, s, xi, yo, tokens, C, heads, U, u0, M, c0, eps, lo)));
    return cudaGetLastError();
  }
  if (kv <= 2)
    GP_DISPATCH_BF16(bf16, (e = xattn2_launch<BF, 2, 2>(x, y, tokens, C, heads, U, u0, M, c0, eps, s, lo)));
  else if (kv <= 3)
    GP_DISPATCH_BF16(bf16, (e = xattn2_launch<BF, 3, 1>(x, y, tokens, C, heads, U, u0, M, c0, eps, s, lo)));
  else
    GP_DISPATCH_BF16(bf16, (e = xattn2_launch<BF, 5, 1>(x, y, tokens, C, heads, U, u0, M, c0, eps, s, lo)));
  return e;
}

cudaError_t geglu(const void* in, void* out, long long tokens, int C4, bool bf16, cudaStream_t s) {
  const long long total_vec = tokens * (C4 / 8);
  GP_DISPATCH_BF16(bf16, (launch(geglu_kernel<BF>, blocks_for(total_vec, 256), 256, 0, s, 
                             reinterpret_cast<const uint16_t*>(in), reinterpret_cast<uint16_t*>(out), total_vec, C4)));
  return cudaGetLastError();
}

cudaError_t relu16(const void* in, void* out, long long n, bool bf16, cudaStream_t s, int split_c) {
  const long long total_vec = n / 8;        // n = pixels * C logical elements
  GP_DISPATCH_BF16(bf16, (launch(relu_kernel<BF>, blocks_for(total_vec, 256), 256, 0, s, 
                             reinterpret_cast<const uint16_t*>(in), reinterpret_cast<uint16_t*>(out), total_vec,
                             split_c ? split_c / 8 : 1, split_c)));
  return cudaGetLastError();
}

cudaError_t bilinear_up2x(const void* in, void* out, int N, int H, int W, int C, bool bf16, cudaStream_t s, bool split) {
  const long long total_vec = (long long)N * 4 * H * W * (C / 8);
  const float sy = H > 1 ? (float)(H - 1) / (float)(2 * H - 1) : 0.f;
  const float sx = W > 1 ? (float)(W - 1) / (float)(2 * W - 1) : 0.f;
  GP_DISPATCH_BF16(bf16, (launch(bilinear_up2x_kernel<BF>, blocks_for(total_vec, 256), 256, 0, s, 
                             reinterpret_cast<const uint16_t*>(in), reinterpret_cast<uint16_t*>(out), N, H, W, C, sy,
                             sx, total_vec, split ? C : 0)));
  return cudaGetLastError();
}

cudaError_t preprocess_rgb(const void* in, int in_kind, void* out, int N, int H, int W, bool bf16, cudaStream_t s, bool split) {
  const long long HW = (long long)H * W;
  const long long total = (long long)N * HW;
  GP_DISPATCH_BF16(bf16, (launch(preprocess_kernel<BF>, (unsigned)((total + 255) / 256), 256, 0, s, 
                             in, in_kind, reinterpret_cast<uint16_t*>(out), N, HW, split ? 8 : 0)));
  return cudaGetLastError();
}

namespace {
// 16-bit NHWC8 (first `c` channels) -> fp32 NCHW [N, c, H, W]
template <bool BF16>
__global__ void nhwc8_to_nchw_kernel(const uint16_t* __restrict__ in, float* __restrict__ out, int N, long long HW, int c, int lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * HW) return;
  const int n = (int)(i / HW);
  const long long p = i % HW;
  float f[8];
  load8<BF16>(in + i * (lo ? 16 : 8), lo, f);
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (k < c) out[((long long)n * c + k) * HW + p] = f[k];
}
// fp32 NCHW [N, 4, H, W] -> y = M (x * pre) + b per pixel -> 16-bit NHWC8 (channels 4..7 zero).  m: [4][4] row-major
// (null = identity), b: [4] (null = 0).
template <bool BF16>
__global__ void nchw4_affine_to_nhwc8_kernel(const float* __restrict__ in, uint16_t* __restrict__ out, int N, long long HW,
                                             float pre, const float* __restrict__ m, const float* __restrict__ b, int lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * HW) return;
  const int n = (int)(i / HW);
  const long long p = i % HW;
  float x[4], f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < 4; ++k) x[k] = in[((long long)n * 4 + k) * HW + p] * pre;
#pragma unroll
  for (int o = 0; o < 4; ++o) {
    if (m) {
      float a = b ? b[o] : 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) a = fmaf(m[o * 4 + k], x[k], a);
      f[o] = a;
    } else {
      f[o] = x[o];
    }
  }
  store8<BF16>(out + i * (lo ? 16 : 8), lo, f);
}
}  // namespace

namespace {
// Latent-space glue of the multi-step archs (SURVEY.md §8 f4), all on 16-bit NHWC8 latents (4 real channels).
// unet_input = cat([rgb_latent, pred_latent]) for the 8-channel conv_in (genpercept_pipeline.py:446-449), else pred_latent.
template <bool BF16>
__global__ void latent_pack_kernel(const uint16_t* __restrict__ lat, const uint16_t* __restrict__ smp, uint16_t* __restrict__ xin,
                                   long long npx, int in_ch, int lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npx) return;
  const long long o = i * (lo ? 16 : 8);
  float a[8], b[8], f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  load8<BF16>(smp + o, lo, b);
  if (in_ch == 8) {
    load8<BF16>(lat + o, lo, a);
#pragma unroll
    for (int k = 0; k < 4; ++k) { f[k] = a[k]; f[4 + k] = b[k]; }
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) f[k] = b[k];
  }
  store8<BF16>(xin + o, lo, f);
}
// DDIMScheduler.step with eta = 0: x0 = c0 * sample + c1 * model_output, prev_sample = c2 * sample + c3 * model_output
// (genpercept_b200/scheduler.py step_coefficients); prev_sample overwrites `smp`.
template <bool BF16>
__global__ void ddim_step_kernel(const uint16_t* __restrict__ mo, uint16_t* __restrict__ smp, uint16_t* __restrict__ x0, long long npx,
                                 float c0, float c1, float c2, float c3, int lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npx) return;
  const long long o = i * (lo ? 16 : 8);
  float m[8], x[8], p0[8], pv[8];
  load8<BF16>(mo + o, lo, m);
  load8<BF16>(smp + o, lo, x);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    p0[k] = k < 4 ? c0 * x[k] + c1 * m[k] : 0.f;
    pv[k] = k < 4 ? c2 * x[k] + c3 * m[k] : 0.f;
  }
  store8<BF16>(x0 + o, lo, p0);
  store8<BF16>(smp + o, lo, pv);
}
// z = M (x * pre) + b on NHWC8 latents (post_quant_conv(pred_latent / 0.18215), genpercept_pipeline.py:519-521)
template <bool BF16>
__global__ void latent_affine_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, long long npx, float pre,
                                     const float* __restrict__ mat, const float* __restrict__ bias, int lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npx) return;
  const long long o = i * (lo ? 16 : 8);
  float x[8], f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  load8<BF16>(in + o, lo, x);
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    float a = bias ? bias[r] : 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) a = fmaf(mat[r * 4 + k], x[k] * pre, a);
    f[r] = a;
  }
  store8<BF16>(out + o, lo, f);
}
}  // namespace

cudaError_t latent_pack(const void* lat, const void* smp, void* xin, long long npx, int in_ch, bool bf16, cudaStream_t s, bool split) {
  GP_DISPATCH_BF16(bf16, (launch(latent_pack_kernel<BF>, (unsigned)((npx + 255) / 256), 256, 0, s, 
                             reinterpret_cast<const uint16_t*>(lat), reinterpret_cast<const uint16_t*>(smp),
                             reinterpret_cast<uint16_t*>(xin), npx, in_ch, split ? 8 : 0)));
  return cudaGetLastError();
}
cudaError_t ddim_step(const void* model_out, void* sample, void* x0, long long npx, const float c[4], bool bf16, cudaStream_t s, bool split) {
  GP_DISPATCH_BF16(bf16, (launch(ddim_step_kernel<BF>, (unsigned)((npx + 255) / 256), 256, 0, s, 
                             reinterpret_cast<const uint16_t*>(model_out), reinterpret_cast<uint16_t*>(sample),
                             reinterpret_cast<uint16_t*>(x0), npx, c[0], c[1], c[2], c[3], split ? 8 : 0)));
  return cudaGetLastError();
}
cudaError_t latent_affine(const void* in, void* out, long long npx, float pre, const float* mat, const float* bias, bool bf16,
                          cudaStream_t s, bool split) {
  GP_DISPATCH_BF16(bf16, (launch(latent_affine_kernel<BF>, (unsigned)((npx + 255) / 256), 256, 0, s, 
                             reinterpret_cast<const uint16_t*>(in), reinterpret_cast<uint16_t*>(out), npx, pre, mat, bias,
                             split ? 8 : 0)));
  return cudaGetLastError();
}

cudaError_t nhwc8_to_nchw_f32(const void* in, float* out, int N, int H, int W, int c, bool bf16, cudaStream_t s, bool split) {
  const long long HW = (long long)H * W, total = (long long)N * HW;
  GP_DISPATCH_BF16(bf16, (launch(nhwc8_to_nchw_kernel<BF>, (unsigned)((total + 255) / 256), 256, 0, s, 
                             reinterpret_cast<const uint16_t*>(in), out, N, HW, c, split ? 8 : 0)));
  return cudaGetLastError();
}

cudaError_t nchw4_affine_to_nhwc8(const float* in, void* out, int N, int H, int W, float pre, const float* m, const float* b,
                                  bool bf16, cudaStream_t s, bool split) {
  const long long HW = (long long)H * W, total = (long long)N * HW;
  GP_DISPATCH_BF16(bf16, (launch(nchw4_affine_to_nhwc8_kernel<BF>, (unsigned)((total + 255) / 256), 256, 0, s, 
                             in, reinterpret_cast<uint16_t*>(out), N, HW, pre, m, b, split ? 8 : 0)));
  return cudaGetLastError();
}

cudaError_t preprocess_rgb_im2col(const void* in, int in_kind, void* out, int N, int H, int W, bool bf16, cudaStream_t s, bool split) {
  const long long total = (long long)N * H * W;
  GP_DISPATCH_BF16(bf16, (launch(preprocess_im2col_kernel<BF>, (unsigned)((total + 127) / 128), 128, 0, s, 
                             in, in_kind, reinterpret_cast<uint16_t*>(out), N, H, W, split ? 32 : 0)));
  return cudaGetLastError();
}

cudaError_t minmax_normalize(float* x, int N, long long HW, unsigned int* scratch, cudaStream_t s, float dmin, bool zero_min) {
  launch(minmax_init_kernel, (N + 63) / 64, 64, 0, s, scratch, N);
  int bx = (int)((HW + 256 * 8 - 1) / (256 * 8));
  if (bx > 256) bx = 256;
  if (bx < 1) bx = 1;
  launch(minmax_reduce_kernel, dim3(bx, N), 256, 0, s, x, HW, scratch);
  launch(minmax_apply_kernel, dim3(bx, N), 256, 0, s, x, HW, scratch, dmin, zero_min ? 1 : 0);
  return cudaGetLastError();
}

namespace {
// Test-time ensembling (genpercept/util/ensemble.py:117-156,190-191): members aligned by (scale, shift), then the per-pixel
// median (torch.median: the LOWER middle value for an even count) or mean.
__global__ void ensemble_reduce_kernel(const float* __restrict__ d, int B, long long HW, const float* __restrict__ sc,
                                       const float* __restrict__ sh, int median, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= HW) return;
  float v[32];
  float sum = 0.f;
  for (int b = 0; b < B; ++b) {
    const float x = __fadd_rn(__fmul_rn(d[(long long)b * HW + i], sc[b]), sh[b]);   // torch: mul, then add (no FMA)
    sum += x;
    int j = b;                                   // insertion sort (B <= 32)
    while (j > 0 && v[j - 1] > x) { v[j] = v[j - 1]; --j; }
    v[j] = x;
  }
  out[i] = median ? v[(B - 1) / 2] : sum / (float)B;
}
}  // namespace

cudaError_t ensemble_reduce(const float* d, int B, long long HW, const float* scale_dev, const float* shift_dev, bool median, float* out,
                            cudaStream_t s) {
  if (B < 1 || B > 32) return cudaErrorInvalidValue;
  launch(ensemble_reduce_kernel, (unsigned)((HW + 255) / 256), 256, 0, s, d, B, HW, scale_dev, shift_dev, median ? 1 : 0, out);
  return cudaGetLastError();
}

namespace {
__global__ void nearest_resize_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int N, int H, int W, int OH,
                                      int OW, int nvec, float sy, float sx, long long total_vec) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % nvec);
    long long r = i / nvec;
    const int ox = (int)(r % OW);
    r /= OW;
    const int oy = (int)(r % OH);
    const int n = (int)(r / OH);
    const int iy = min((int)floorf(oy * sy), H - 1), ix = min((int)floorf(ox * sx), W - 1);   // ATen nearest index
    out[i] = __ldg(in + (((long long)n * H + iy) * W + ix) * nvec + v);
  }
}
}  // namespace

namespace {
template <bool BF16>
__global__ void softmax_groups_kernel(uint16_t* __restrict__ x, long long rows, int ld, int groups, int n, int lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * groups) return;
  uint16_t* p = x + (i / groups) * (lo ? 2 * ld : ld) + (i % groups) * n;
  float m = -INFINITY;
  for (int j = 0; j < n; ++j) m = fmaxf(m, load1<BF16>(p + j, lo));
  float s = 0.f;
  for (int j = 0; j < n; ++j) s += __expf(load1<BF16>(p + j, lo) - m);
  const float inv = 1.f / s;
  for (int j = 0; j < n; ++j) store1<BF16>(p + j, lo, __expf(load1<BF16>(p + j, lo) - m) * inv);
}
}  // namespace

cudaError_t softmax_groups(void* x, long long rows, int ld, int groups, int n, bool bf16, cudaStream_t s, bool split) {
  if (groups < 1 || n < 1 || groups * n > ld) return cudaErrorInvalidValue;
  const long long total = rows * groups;
  GP_DISPATCH_BF16(bf16, (launch(softmax_groups_kernel<BF>, (unsigned)((total + 127) / 128), 128, 0, s, 
                             reinterpret_cast<uint16_t*>(x), rows, ld, groups, n, split ? ld : 0)));
  return cudaGetLastError();
}

namespace {
// F.interpolate(size=(OH,OW), mode="bilinear", align_corners=False): src = max((dst + 0.5) * in/out - 0.5, 0)
template <bool BF16>
__global__ void bilinear_resize_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, int N, int H, int W, int OH,
                                       int OW, int C, float sy, float sx, long long total_vec, int lo) {
  const int nvec = C / 8;
  const int xs = lo ? 2 * C : C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % nvec);
    long long r = i / nvec;
    const int ox = (int)(r % OW);
    r /= OW;
    const int oy = (int)(r % OH);
    const int n = (int)(r / OH);
    const float fy = fmaxf((oy + 0.5f) * sy - 0.5f, 0.f), fx = fmaxf((ox + 0.5f) * sx - 0.5f, 0.f);
    const int y0 = min((int)fy, H - 1), x0 = min((int)fx, W - 1);
    const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
    const float h1 = fy - y0, w1 = fx - x0, h0 = 1.f - h1, w0 = 1.f - w1;
    const uint16_t* b = in + ((long long)n * H * W) * xs + v * 8;
    float a00[8], a01[8], a10[8], a11[8], o[8];
    load8<BF16>(b + ((long long)y0 * W + x0) * xs, lo, a00);
    load8<BF16>(b + ((long long)y0 * W + x1) * xs, lo, a01);
    load8<BF16>(b + ((long long)y1 * W + x0) * xs, lo, a10);
    load8<BF16>(b + ((long long)y1 * W + x1) * xs, lo, a11);
#pragma unroll
    for (int e = 0; e < 8; ++e) o[e] = h0 * (w0 * a00[e] + w1 * a01[e]) + h1 * (w0 * a10[e] + w1 * a11[e]);
    store8<BF16>(out + (((long long)n * OH + oy) * OW + ox) * xs + v * 8, lo, o);
  }
}
}  // namespace

cudaError_t bilinear_resize(const void* in, void* out, int N, int H, int W, int OH, int OW, int C, bool bf16, cudaStream_t s,
                            bool split) {
  if (C % 8) return cudaErrorInvalidValue;
  const long long total_vec = (long long)N * OH * OW * (C / 8);
  GP_DISPATCH_BF16(bf16, (launch(bilinear_resize_kernel<BF>, blocks_for(total_vec, 256), 256, 0, s, 
                             reinterpret_cast<const uint16_t*>(in), reinterpret_cast<uint16_t*>(out), N, H, W, OH, OW, C,
                             (float)H / (float)OH, (float)W / (float)OW, total_vec, split ? C : 0)));
  return cudaGetLastError();
}

cudaError_t nearest_resize(const void* in, void* out, int N, int H, int W, int OH, int OW, int C, cudaStream_t s) {
  if (C % 8) return cudaErrorInvalidValue;
  const long long total_vec = (long long)N * OH * OW * (C / 8);
  launch(nearest_resize_kernel, blocks_for(total_vec, 256), 256, 0, s, reinterpret_cast<const uint4*>(in),
                                                                  reinterpret_cast<uint4*>(out), N, H, W, OH, OW, C / 8,
                                                                  (float)H / (float)OH, (float)W / (float)OW, total_vec);
  return cudaGetLastError();
}

}  // namespace gp
