// Device code shared by the two tcgen05 implicit-GEMM kernels (tap-streaming: igemm.cu, patch-resident:
// igemm_patch.cu): tile decoding, 16-bit helpers, the exact-erf GELU and the two epilogues.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "igemm.h"
#include "ptx.cuh"

namespace gp {
namespace {

constexpr int kABytes = kBM * kBK * 2;       // 16 KiB per 128-row tile
constexpr int kTmemCols = 512;
constexpr int kAccStride = 256;              // TMEM columns between the two accumulator buffers
constexpr int kMaxSmem = 227 * 1024;

struct TileCoord {
  int n_tile, tx, ty, z0, z1;
};

__device__ __forceinline__ TileCoord decode_tile(const IgemmParams& p, int tile) {
  TileCoord t;
  t.n_tile = tile % p.n_tiles_n;
  int r = tile / p.n_tiles_n;
  t.tx = r % p.tiles_x;
  r /= p.tiles_x;
  t.ty = r % p.tiles_y;
  r /= p.tiles_y;
  t.z0 = r % p.Z0;
  t.z1 = r / p.Z0;
  return t;
}

template <bool BF16>
__device__ __forceinline__ float cvt16(uint16_t v) {
  if constexpr (BF16) {
    return __bfloat162float(__ushort_as_bfloat16(v));
  } else {
    return __half2float(__ushort_as_half(v));
  }
}
template <bool BF16>
__device__ __forceinline__ uint32_t pack16(float a, float b) {
  if constexpr (BF16) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
}
template <bool BF16>
__device__ __forceinline__ void add8(float* v, const uint4& u) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    v[2 * e] += cvt16<BF16>((uint16_t)(w[e] & 0xFFFF));
    v[2 * e + 1] += cvt16<BF16>((uint16_t)(w[e] >> 16));
  }
}

// 8 consecutive channels -> one 16-byte store; in the high-precision layout (lo != 0) the rounding residual
// v - float(hi) goes to the lo plane `lo` elements further.
template <bool BF16>
__device__ __forceinline__ void store8_hl(uint16_t* op, long long lo, const float* v) {
  uint4 u;
  u.x = pack16<BF16>(v[0], v[1]);
  u.y = pack16<BF16>(v[2], v[3]);
  u.z = pack16<BF16>(v[4], v[5]);
  u.w = pack16<BF16>(v[6], v[7]);
  *reinterpret_cast<uint4*>(op) = u;
  if (lo) {
    const uint32_t hw[4] = {u.x, u.y, u.z, u.w};
    uint32_t lw[4];
#pragma unroll
    for (int e = 0; e < 4; ++e)
      lw[e] = pack16<BF16>(v[2 * e] - cvt16<BF16>((uint16_t)(hw[e] & 0xFFFF)), v[2 * e + 1] - cvt16<BF16>((uint16_t)(hw[e] >> 16)));
    *reinterpret_cast<uint4*>(op + lo) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
  }
}

// gelu(g) = g * Phi(g), exact-erf form (what diffusers' GEGLU uses), with erf from Abramowitz-Stegun 7.1.26
// (|error| <= 1.5e-7): one MUFU.RCP, one MUFU.EX2 and a degree-5 Horner instead of erff()'s two-branch
// polynomial — the GEGLU projection is bound by its epilogue (tensor pipe 33 %, ncu r1_final).
//   1 - erf(z) = (a1 t + ... + a5 t^5) e^{-z^2},  t = 1 / (1 + p z),  z = |g| / sqrt(2)
__device__ __forceinline__ float gelu_erf(float g) {
  const float z = fabsf(g) * 0.70710678118654752f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.f)));
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z * z * -1.4426950408889634f));
  float q = fmaf(1.061405429f, t, -1.453152027f);
  q = fmaf(q, t, 1.421413741f);
  q = fmaf(q, t, -0.284496736f);
  q = fmaf(q, t, 0.254829592f);
  q = q * t * e * 0.5f;                                   // = (1 - erf(z)) / 2 = Phi(-|g|)
  return g * (g >= 0.f ? 1.f - q : q);
}

// NW epilogue warps (4 or 8).  With 8, warps w and w + 4 read the same TMEM lane quadrant (lanes 32 * (w % 4) ...) and split the
// tile's 64-channel groups between them: one epilogue warp per sub-partition is stalled ~78 % of the time (TMEM / shared
// memory latency, instruction fetch: ncu r2, the K = 1 stem GEMM), a second one fills those slots.
template <int NW>
__device__ __forceinline__ void epi_sync() {   // the epilogue threads only
  asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");
}

// The bias of the CTA's current N tile lives in shared memory (kBiasSlots floats, zero beyond Cout): every 32-column piece
// of the epilogue used to fetch it with eight dependent 16-byte global loads — with almost all of L1 configured as shared
// memory those miss to L2 (~600 cycles), in front of every piece (ncu r2: the K = 1 stem GEMM, nothing but epilogue, ran
// with the epilogue warps issuing 22 % of the time and no unit above 25 %).
constexpr int kBiasSlots = 288;
// A layer with several N tiles changes tile column on every tile of a CTA (tiles are numbered N-fastest and taken with a
// stride of gridDim.x), i.e. two barriers of all epilogue warps plus an L2 round trip per tile: when the padded Cout fits
// (p.bias_all, igemm_finalize) the whole bias vector is loaded once instead.
template <int NW>
__device__ __forceinline__ void load_bias_tile(const IgemmParams& p, float* sbias, int n_base, int etid) {
  epi_sync<NW>();                              // nobody still reads the previous tile's values
  const int count = p.bias_all ? p.bias_slots : kBiasSlots;
  for (int i = etid; i < count; i += NW * 32) {
    const int n = n_base + i;
    sbias[i] = (p.bias != nullptr && n < p.Cout) ? __ldg(p.bias + n) : 0.f;
  }
  epi_sync<NW>();
}
__device__ __forceinline__ void bias32(const float* sbias, int c, float (&bz)[32]) {
#pragma unroll
  for (int q = 0; q < 32; q += 4) {
    const float4 b4 = *reinterpret_cast<const float4*>(sbias + c + q);
    bz[q] = b4.x; bz[q + 1] = b4.y; bz[q + 2] = b4.z; bz[q + 3] = b4.w;
  }
}

// Staged epilogue (shared by the tap-streaming and the patch-resident main loops): TMEM -> registers
// (bias / residuals / ReLU) -> 16-bit rows in a SWIZZLE_128B shared tile -> one TMA store per
// (warp, 64-channel group), plus the GroupNorm partial sums read back column-wise from the tile.
// SPLIT / RES are compile-time: with run-time flags one 32 x 64 piece executed ~830 warp instructions, 97 of them MOVs
// and 27 branches around the variants not taken (ncu source page, r2q: the 320 -> 2560 linear issues 13.4 k warp
// instructions per 128 x 256 tile against 2560 tensor cycles).  RES: 0 none, 1 residual tile through TMA, 2 per-thread rows.
template <bool BF16, int NW, bool SPLIT, int RES>
__device__ __forceinline__ void epilogue_staged(const IgemmParams& p, uint8_t* stg_base, float* sacc, float* sbias, uint64_t* tfull_bar,
                                                uint64_t* tempty_bar, uint64_t* res_bar, uint32_t tmem_base, int warp, int lane) {
  // ===================================================================== epilogue, staged + TMA store
  // TMEM -> registers (bias / residuals / ReLU) -> 16-bit rows in a SWIZZLE_128B shared tile ->
  // one TMA store per (warp, 64-channel group): full-line writes instead of 16-byte pieces at a
  // 2C-byte stride, and image-edge clipping for free.  GroupNorm partial sums are read back
  // column-wise from the staged tile (conflict-free), in a fixed order.
  const int wq = warp & 3;                   // epilogue warps are warps 0..NW-1; warp % 4 -> TMEM lanes [32*wq, +32)
  const int half = warp >> 2;                // NW == 8: which of the tile's 64-channel groups this warp takes (parity)
  uint8_t* stg = stg_base + warp * 4096;
  const uint32_t stg_addr = smem_u32(stg);
  const uint32_t my_row = stg_addr + lane * 128;
  constexpr bool split = SPLIT;              // high-precision mode: a second staged tile (+NW * 4 KiB) takes the lo plane
  const uint32_t my_row_lo = my_row + NW * 4096;
  // 64-channel groups of the N tile go to the two halves by parity; a tile with one group only is done by half 0
  // (statistics: the halves then never accumulate the same channel into sacc[wq])
  const bool two_groups = NW == 8 && (p.BN >> 6) >= 2;
  auto mine = [&](int c0) { return NW == 4 || (two_groups ? ((c0 >> 6) & 1) == half : half == 0); };
  const int sw = lane & 7;
  int acc = 0;
  uint32_t acc_phase = 0, res_phase = 0;
  const bool relu = (p.flags & IG_RELU) != 0;
  const bool do_stats = p.stats != nullptr;
  const int etid = threadIdx.x;
  int cur_img = -1;
  int cur_nt = -1;
  // sum the four warp-private accumulators in a fixed order, publish this CTA's slot, reset
  auto flush_stats = [&](int img) {
    epi_sync<NW>();
    float* dst = p.stats + ((long long)img * p.stats_slots + blockIdx.x) * p.Cout * 2;
    for (int i = etid; i < 2 * p.Cout; i += NW * 32) {
      const float tot = (sacc[i] + sacc[2 * p.Cout + i]) + (sacc[4 * p.Cout + i] + sacc[6 * p.Cout + i]);
      dst[i] = tot;
      sacc[i] = 0.f; sacc[2 * p.Cout + i] = 0.f; sacc[4 * p.Cout + i] = 0.f; sacc[6 * p.Cout + i] = 0.f;
    }
    epi_sync<NW>();
  };
  if (do_stats) {
    for (int i = etid; i < 8 * p.Cout; i += NW * 32) sacc[i] = 0.f;
    epi_sync<NW>();
  }
  if (p.bias_all) load_bias_tile<NW>(p, sbias, 0, etid);
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    const TileCoord t = decode_tile(p, tile);
    const int cls = p.cls_from_z0 ? t.z0 : 0;
    const int n_base = t.n_tile * p.BN;
    bool waited = false;
    if (t.n_tile != cur_nt && !p.bias_all) {
      load_bias_tile<NW>(p, sbias, n_base, etid);
      cur_nt = t.n_tile;
    }
    const int bias_origin = p.bias_all ? 0 : n_base;
    // The residual boxes of this CTA's NEXT tile are pulled into L2 now, a whole tile period before their TMA loads:
    // those loads sit serially in front of every 32 x 64 piece of the epilogue, and with DRAM latency (1.5 us under
    // load) four of them per warp outlast the main loop of the short-K (Cout = 128) layers (r2: residual convs 20-30 %
    // slower than plain ones; the main loop of a 128->128 tile is 6 us).
    if (RES == 1 && lane == 0 && tile + (int)gridDim.x < p.total_tiles) {
      const TileCoord tn = decode_tile(p, tile + gridDim.x);
      const int ncls = p.cls_from_z0 ? tn.z0 : 0;
      for (int h = 0; h < p.MT; ++h) {
        const int r0 = h * 128 + wq * 32;
        const int psx = tn.tx * p.TW + (r0 & (p.TW - 1)), psy = tn.ty * p.TH + (r0 >> p.tw_shift);
        for (int c0 = 0; c0 < p.BN && tn.n_tile * p.BN + c0 < p.Cout; c0 += 64)
          if (mine(c0)) tma_prefetch_l2_4d(&p.tmRes[ncls], tn.n_tile * p.BN + c0, psx, psy, tn.z1);
      }
    }
    if (do_stats) {
      const int img = p.stats_hw ? (t.tx * p.TW) / p.stats_hw : t.z1;
      if (img != cur_img) {
        if (cur_img >= 0) flush_stats(cur_img);
        cur_img = img;
      }
    }
    for (int h = 0; h < p.MT; ++h) {
      const int r0 = h * 128 + wq * 32;                       // first tile row of this warp
      const int row = r0 + lane;
      const int ti = row >> p.tw_shift, tj = row & (p.TW - 1);
      const int gy = t.ty * p.TH + ti, gx = t.tx * p.TW + tj;
      const bool valid = gy < p.gridH && gx < p.gridW;
      const int oy = gy * p.out_sy + p.cls_py[cls], ox = gx * p.out_sx + p.cls_px[cls];
      const long long pix_off = t.z1 * p.out_z1 + (long long)oy * p.out_row_stride + (long long)ox * p.out_pix_stride;
      const int sx = t.tx * p.TW + (r0 & (p.TW - 1)), sy = t.ty * p.TH + (r0 >> p.tw_shift);   // store box origin
      const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + acc * kAccStride + h * 128;
      for (int c0 = 0; c0 < p.BN; c0 += 64) {
        const int n0 = n_base + c0;
        if (n0 >= p.Cout) break;
        if (!mine(c0)) continue;
        if (lane == 0) tma_store_wait_read0();                // the previous store has finished reading the tile
        __syncwarp();
        uint4 rt[8];                                          // this thread's residual row (64 channels), res_tma only
        if constexpr (RES == 1) {
          if (lane == 0) {
            mbar_expect_tx(&res_bar[warp], 4096);
            tma_load_4d(stg, &p.tmRes[cls], &res_bar[warp], n0, sx, sy, t.z1);
          }
          mbar_wait(&res_bar[warp], res_phase, 7);
          res_phase ^= 1;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(rt[i].x), "=r"(rt[i].y), "=r"(rt[i].z), "=r"(rt[i].w)
                         : "r"(my_row + ((i ^ sw) << 4)));
          __syncwarp();                                       // every row is in registers before the tile is overwritten
        }
        float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
        for (int sub = 0; sub < 2; ++sub) {
          const int ns = n0 + sub * 32;
          const long long off = pix_off + ns;
          float bz[32];
          bias32(sbias, ns - bias_origin, bz);
          uint4 r1[4], r2[4];
          const bool has1 = RES == 1 || (RES == 2 && valid && p.res1 != nullptr), has2 = RES == 2 && valid && p.res2 != nullptr;
          if constexpr (RES == 1) {
#pragma unroll
            for (int q = 0; q < 4; ++q) r1[q] = rt[sub * 4 + q];
          } else if (has1) {
            const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(p.res1) + off);
#pragma unroll
            for (int q = 0; q < 4; ++q) r1[q] = rp[q];
          }
          if (has2) {
            const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(p.res2) + off);
#pragma unroll
            for (int q = 0; q < 4; ++q) r2[q] = rp[q];
          }
          if (!waited) {
            mbar_wait(&tfull_bar[acc], acc_phase, 4);
            tc_fence_after();
            waited = true;
          }
          uint32_t r[32];
          tmem_ld_32x32(taddr + c0 + sub * 32, r);
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int q = 0; q < 32; ++q) v[q] = __uint_as_float(r[q]) + bz[q];
          if (has1) {
#pragma unroll
            for (int q = 0; q < 4; ++q) add8<BF16>(&v[q * 8], r1[q]);
          }
          if (has2) {
#pragma unroll
            for (int q = 0; q < 4; ++q) add8<BF16>(&v[q * 8], r2[q]);
          }
          if (split) {       // lo planes of the residuals
            if (has1) {
              const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(p.res1) + off + p.out_lo);
#pragma unroll
              for (int q = 0; q < 4; ++q) add8<BF16>(&v[q * 8], rp[q]);
            }
            if (has2) {
              const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(p.res2) + off + p.out_lo);
#pragma unroll
              for (int q = 0; q < 4; ++q) add8<BF16>(&v[q * 8], rp[q]);
            }
          }
          if (relu) {
#pragma unroll
            for (int q = 0; q < 32; ++q) v[q] = fmaxf(v[q], 0.f);
          }
          if (!valid) {      // rows outside the image are clipped by the TMA store; zero them for the statistics
#pragma unroll
            for (int q = 0; q < 32; ++q) v[q] = 0.f;
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t a = my_row + (((sub * 4 + i) ^ sw) << 4);
            const uint32_t h0 = pack16<BF16>(v[8 * i], v[8 * i + 1]), h1 = pack16<BF16>(v[8 * i + 2], v[8 * i + 3]);
            const uint32_t h2 = pack16<BF16>(v[8 * i + 4], v[8 * i + 5]), h3 = pack16<BF16>(v[8 * i + 6], v[8 * i + 7]);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(h0), "r"(h1), "r"(h2), "r"(h3) : "memory");
            if (split) {     // lo = v - float(hi), rounded to 16 bit
              const uint32_t hw[4] = {h0, h1, h2, h3};
              uint32_t lw[4];
#pragma unroll
              for (int e = 0; e < 4; ++e)
                lw[e] = pack16<BF16>(v[8 * i + 2 * e] - cvt16<BF16>((uint16_t)(hw[e] & 0xFFFF)),
                                     v[8 * i + 2 * e + 1] - cvt16<BF16>((uint16_t)(hw[e] >> 16)));
              const uint32_t al = my_row_lo + (((sub * 4 + i) ^ sw) << 4);
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(al), "r"(lw[0]), "r"(lw[1]), "r"(lw[2]), "r"(lw[3]) : "memory");
            }
          }
        }
        fence_proxy_async_shared();
        __syncwarp();
        if (lane == 0) {
          tma_store_4d(&p.tmOut[cls], stg_addr, n0, sx, sy, t.z1);
          if (split) tma_store_4d(&p.tmOutLo[cls], stg_addr + NW * 4096, n0, sx, sy, t.z1);
          tma_store_commit();
        }
        if (do_stats) {
          // lane l owns channels n0 + 2l, n0 + 2l + 1: one 32-bit word per staged row
          const uint32_t col = stg_addr + (lane & 3) * 4;
          const int chunk = lane >> 2;
#pragma unroll 8
          for (int rr = 0; rr < 32; ++rr) {
            uint32_t w;
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(w) : "r"(col + rr * 128 + ((chunk ^ (rr & 7)) << 4)));
            const float a = cvt16<BF16>((uint16_t)(w & 0xFFFF)), b = cvt16<BF16>((uint16_t)(w >> 16));
            s0 += a; q0 += a * a; s1 += b; q1 += b * b;
          }
          float* d = sacc + ((size_t)wq * p.Cout + n0 + 2 * lane) * 2;
          d[0] += s0; d[1] += q0; d[2] += s1; d[3] += q1;
        }
      }
    }
    if (!waited) {
      mbar_wait(&tfull_bar[acc], acc_phase, 4);
      tc_fence_after();
    }
    tc_fence_before();
    mbar_arrive(&tempty_bar[acc]);
    acc ^= 1;
    if (acc == 0) acc_phase ^= 1;
  }
  if (lane == 0) tma_store_wait_read0();
  if (do_stats && cur_img >= 0) flush_stats(cur_img);
}


// Run-time flags -> the specialised staged epilogue.  LEAN (the patch-resident kernel): no (hi, lo) layout.
template <bool BF16, int NW, bool LEAN>
__device__ __forceinline__ void run_epilogue_staged(const IgemmParams& p, uint8_t* stg_base, float* sacc, float* sbias, uint64_t* tfull_bar,
                                                    uint64_t* tempty_bar, uint64_t* res_bar, uint32_t tmem_base, int warp, int lane) {
  const int rm = p.res_tma ? 1 : ((p.res1 != nullptr || p.res2 != nullptr) ? 2 : 0);
  if constexpr (!LEAN) {
    if (p.out_lo != 0) {
      if (rm == 2) epilogue_staged<BF16, NW, true, 2>(p, stg_base, sacc, sbias, tfull_bar, tempty_bar, res_bar, tmem_base, warp, lane);
      else epilogue_staged<BF16, NW, true, 0>(p, stg_base, sacc, sbias, tfull_bar, tempty_bar, res_bar, tmem_base, warp, lane);
      return;
    }
  }
  if (rm == 1) epilogue_staged<BF16, NW, false, 1>(p, stg_base, sacc, sbias, tfull_bar, tempty_bar, res_bar, tmem_base, warp, lane);
  else if (rm == 2) epilogue_staged<BF16, NW, false, 2>(p, stg_base, sacc, sbias, tfull_bar, tempty_bar, res_bar, tmem_base, warp, lane);
  else epilogue_staged<BF16, NW, false, 0>(p, stg_base, sacc, sbias, tfull_bar, tempty_bar, res_bar, tmem_base, warp, lane);
}

// Direct epilogue: TMEM -> registers (bias / residuals / ReLU / affine clamp / GEGLU) -> global stores straight from
// the registers: fp32 NCHW maps, odd channel counts, GEGLU, the high-precision (hi, lo) layout.
// LEAN = the GEGLU projection of the default mode (full 32-column chunks, no residual, 16-bit output, no (hi, lo) planes): every
// other variant is compiled out of its loop (same reasoning as the staged epilogue's template parameters).
template <bool BF16, int NW, bool LEAN>
__device__ __forceinline__ void epilogue_direct(const IgemmParams& p, float* sbias, uint64_t* tfull_bar, uint64_t* tempty_bar,
                                                uint32_t tmem_base, int warp, int lane) {
  // ===================================================================== epilogue
  const int wq = warp & 3;                 // warp % 4 -> TMEM lanes [32*wq, 32*wq+32)
  const int half = warp >> 2;              // NW == 8: the tile's 32-column chunks go to the two halves by parity
  const bool two_chunks = NW == 8 && p.BN > 32;
  int acc = 0;
  uint32_t acc_phase = 0;
  const bool f32out = !LEAN && (p.flags & IG_OUT_F32_NCHW) != 0;
  const bool relu = !LEAN && (p.flags & IG_RELU) != 0;
  const bool aff = !LEAN && (p.flags & IG_AFFINE_CLAMP01) != 0;
  const bool geglu = LEAN || (p.flags & IG_GEGLU) != 0;
  const void* const res1 = LEAN ? nullptr : p.res1;
  const void* const res2 = LEAN ? nullptr : p.res2;
  const long long out_lo = LEAN ? 0 : p.out_lo;
  const int etid = threadIdx.x;              // 0..127 among the epilogue threads
  int cur_nt = -1;
  if (p.bias_all) load_bias_tile<NW>(p, sbias, 0, etid);
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    const TileCoord t = decode_tile(p, tile);
    const int cls = p.cls_from_z0 ? t.z0 : 0;
    const int n_base = t.n_tile * p.BN;
    bool waited = false;
    if (t.n_tile != cur_nt && !p.bias_all) {
      load_bias_tile<NW>(p, sbias, n_base, etid);
      cur_nt = t.n_tile;
    }
    const int bias_origin = p.bias_all ? 0 : n_base;
    for (int h = 0; h < p.MT; ++h) {
      const int row = h * 128 + wq * 32 + lane;
      const int ti = row >> p.tw_shift, tj = row & (p.TW - 1);
      const int gy = t.ty * p.TH + ti, gx = t.tx * p.TW + tj;
      const bool valid = gy < p.gridH && gx < p.gridW;
      const int oy = gy * p.out_sy + p.cls_py[cls], ox = gx * p.out_sx + p.cls_px[cls];
      const long long pix_off = t.z1 * p.out_z1 + t.z0 * p.out_z0 + (long long)oy * p.out_row_stride +
                                (long long)ox * p.out_pix_stride;
      const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + acc * kAccStride + h * 128;
      for (int c0 = 0; c0 < p.BN; c0 += 32) {
        if (NW == 8 && (two_chunks ? ((c0 >> 5) & 1) != half : half != 0)) continue;
        const int ncols = (LEAN || p.BN - c0 >= 32) ? 32 : 16;
        const int n0 = n_base + c0;
        const int nvalid = LEAN ? 32 : min(ncols, p.Cout - n0);
        const bool live = valid && nvalid > 0;
        const long long off = pix_off + n0;
        const bool vec = !f32out && live && (nvalid == ncols) && ((off & 7) == 0);
        // operands that do not depend on the accumulator are fetched BEFORE waiting on it
        float bz[32];
        bias32(sbias, n_base - bias_origin + c0, bz);
        uint4 r1[4], r2[4];
        const bool has1 = vec && res1 != nullptr, has2 = vec && res2 != nullptr;
        if (has1) {
          const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(res1) + off);
#pragma unroll
          for (int q = 0; q < 4; ++q) if (q * 8 < ncols) r1[q] = rp[q];
        }
        if (has2) {
          const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(res2) + off);
#pragma unroll
          for (int q = 0; q < 4; ++q) if (q * 8 < ncols) r2[q] = rp[q];
        }
        if (!waited) {
          mbar_wait(&tfull_bar[acc], acc_phase, 4);
          tc_fence_after();
          waited = true;
        }
        uint32_t r[32];
        if (LEAN || ncols == 32) tmem_ld_32x32(taddr + c0, r); else tmem_ld_32x16(taddr + c0, r);
        tmem_ld_wait();
        if (!live) continue;
        float v[32];
#pragma unroll
        for (int q = 0; q < 32; ++q) v[q] = __uint_as_float(r[q]) + bz[q];
        if (f32out) {
          float* o = reinterpret_cast<float*>(p.out);
#pragma unroll
          for (int q = 0; q < 32; ++q) {
            if (q < nvalid) {
              float x = v[q];
              if (relu) x = fmaxf(x, 0.f);
              if (aff) x = fminf(fmaxf((x + 1.f) * 0.5f, 0.f), 1.f);
              o[(((long long)t.z1 * p.Cout + (n0 + q)) * p.outH + oy) * p.outW + ox] = x;
            }
          }
          continue;
        }
        if (has1) {
#pragma unroll
          for (int q = 0; q < 4; ++q) if (q * 8 < ncols) add8<BF16>(&v[q * 8], r1[q]);
        } else if (res1 != nullptr && live) {
          const uint16_t* rp = reinterpret_cast<const uint16_t*>(res1) + off;
#pragma unroll
          for (int q = 0; q < 32; ++q) if (q < nvalid) v[q] += cvt16<BF16>(rp[q]);
        }
        if (has2) {
#pragma unroll
          for (int q = 0; q < 4; ++q) if (q * 8 < ncols) add8<BF16>(&v[q * 8], r2[q]);
        } else if (res2 != nullptr && live) {
          const uint16_t* rp = reinterpret_cast<const uint16_t*>(res2) + off;
#pragma unroll
          for (int q = 0; q < 32; ++q) if (q < nvalid) v[q] += cvt16<BF16>(rp[q]);
        }
        if (out_lo) {      // high-precision layout: lo planes of the residuals
#pragma unroll
          for (int ri = 0; ri < 2; ++ri) {
            const void* rb = ri == 0 ? res1 : res2;
            if (rb == nullptr || !live) continue;
            const uint16_t* rp = reinterpret_cast<const uint16_t*>(rb) + off + out_lo;
            if (vec) {
#pragma unroll
              for (int q = 0; q < 4; ++q) if (q * 8 < ncols) add8<BF16>(&v[q * 8], reinterpret_cast<const uint4*>(rp)[q]);
            } else {
#pragma unroll
              for (int q = 0; q < 32; ++q) if (q < nvalid) v[q] += cvt16<BF16>(rp[q]);
            }
          }
        }
        if (relu) {
#pragma unroll
          for (int q = 0; q < 32; ++q) v[q] = fmaxf(v[q], 0.f);
        }
        if (geglu) {   // [16 values | 16 gates] -> 16 outputs at column n0/2 (weights are packed interleaved)
          uint16_t* og = reinterpret_cast<uint16_t*>(p.out) + pix_off + (n0 >> 1);
          float g[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) g[q] = v[q] * gelu_erf(v[16 + q]);
#pragma unroll
          for (int q = 0; q < 16; q += 8) store8_hl<BF16>(og + q, out_lo, &g[q]);
          continue;
        }
        uint16_t* op = reinterpret_cast<uint16_t*>(p.out) + off;
        if (vec) {
#pragma unroll
          for (int q = 0; q < 32; q += 8) {
            if (q < ncols) store8_hl<BF16>(op + q, out_lo, &v[q]);
          }
        } else if (live) {
#pragma unroll
          for (int q = 0; q < 32; ++q) {
            if (q < nvalid) {
              const uint16_t h = (uint16_t)(pack16<BF16>(v[q], 0.f) & 0xFFFF);
              op[q] = h;
              if (out_lo) op[q + out_lo] = (uint16_t)(pack16<BF16>(v[q] - cvt16<BF16>(h), 0.f) & 0xFFFF);
            }
          }
        }
      }
    }
    if (!waited) {   // unreachable (BN >= 16), kept so the barrier protocol can never desynchronise
      mbar_wait(&tfull_bar[acc], acc_phase, 4);
      tc_fence_after();
    }
    tc_fence_before();
    mbar_arrive(&tempty_bar[acc]);
    acc ^= 1;
    if (acc == 0) acc_phase ^= 1;
  }
}

template <bool BF16, int NW>
__device__ __forceinline__ void run_epilogue_direct(const IgemmParams& p, float* sbias, uint64_t* tfull_bar, uint64_t* tempty_bar,
                                                    uint32_t tmem_base, int warp, int lane) {
  const bool lean = (p.flags & IG_GEGLU) && !(p.flags & (IG_OUT_F32_NCHW | IG_RELU | IG_AFFINE_CLAMP01)) && p.out_lo == 0 &&
                    p.res1 == nullptr && p.res2 == nullptr && (p.BN % 32) == 0 && (p.Cout % p.BN) == 0;
  if (lean) epilogue_direct<BF16, NW, true>(p, sbias, tfull_bar, tempty_bar, tmem_base, warp, lane);
  else epilogue_direct<BF16, NW, false>(p, sbias, tfull_bar, tempty_bar, tmem_base, warp, lane);
}

}  // namespace
}  // namespace gp
