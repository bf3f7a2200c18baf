// Patch-resident tcgen05 implicit GEMM for 3x3 stride-1 convolutions over wide images (W % 128 == 0), with the
// producer-side GroupNorm(+SiLU) applied to the operand ON ITS WAY to the tensor core.
//
// Per 64-channel K chunk ONE (TH+2) x 130 pixel halo patch of the source lands in shared memory (a single TMA box,
// image borders zero-filled) and all nine filter taps are fed from it by row-offset SWIZZLE_128B descriptors: tap
// (dy,dx) of image row h starts ((h+dy+1)*130 + dx+1) rows into the patch (scripts/exp_baseoffset.cu: any 128-byte
// row is a valid descriptor start because the swizzle is a function of the absolute shared-memory address).
// Activation traffic L2 -> SM drops from 9 to (TH+2)*130 / (TH*128) reads per element.
//
// GroupNorm fusion (SURVEY.md §7 step 3, App. C.8; reference call sites: every `norm1 -> SiLU -> conv1` /
// `norm2 -> SiLU -> conv2` / `conv_norm_out -> SiLU -> conv_out` of the diffusers VAE blocks that
// /root/reference/genpercept/genpercept_pipeline.py:500,521 drive): the statistics of the source tensor come from
// its producer's epilogue (gn_finalize turns them into one (scale, shift) pair per (image, channel)); a transform
// warpgroup rewrites each landed patch in place, y = silu(x * scale + shift), leaving the zero-filled halo pixels
// outside the image at zero (the convolution pads the NORMALISED tensor with zeros), and only then hands the patch to
// the MMA issuers.  The normalised tensor never exists in HBM: one 2-byte read + one 2-byte write per element and
// one kernel launch less per GroupNorm.
//
// Extra K chunks for a fused 1x1 shortcut (ResnetBlock2D.conv_shortcut over the RAW block input): centre tap only,
// loaded through a second tensor map and passed through the transform stage untouched.
//
// Warp roles (384 threads, 1 CTA / SM, persistent).  Three builds: default (layers with a residual), NE4 (layers without:
// four epilogue warps, warps 8..11 idle, one more weight-ring stage) and XFORM.  Default (XFORM = false): warps 0..7 epilogue (as in igemm.cu),
// warp 8 patch producer (TMA), warps 9 (,10) MMA issuers — one per image row of the tile (MT = TH = 1 or 2), warp 10 also
// owns the TMEM allocation —, warp 11 weight producer (one TMA box per (chunk, tap)).  GroupNorm-transform build
// (XFORM = true, GP_GN_FUSE=1): warps 0..3 epilogue, 4..7 the same roles, 8..11 operand transform (GroupNorm scale/shift +
// SiLU in place); registers re-balanced with setmaxnreg.
#include "igemm_common.cuh"
#include "launch.h"

namespace gp {

namespace {

constexpr int kPatchThreads = 384;
constexpr int kPW = kBM + 2;      // patch width in pixels (TW = 128)
constexpr int kPP = kPW;          // patch row pitch in pixels (one TMA box per patch: rows are contiguous)

template <int N>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

__device__ __forceinline__ float silu_tanh(float x) {   // x * sigmoid(x) = h + h * tanh(h), h = x / 2 (kernels.cu silu_f)
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
// Two channels per special-function op: the transform of a 64-channel patch is bound by the MUFU (16 results / clk / SM
// with tanh.approx.f32: 520 x 64 / 16 = 2080 cycles per K chunk, against 4608 cycles of MMA per chunk and a TMA load
// that cannot start before the previous use of the slot retires).  tanh.approx.f16x2 has the same ~2^-11 relative
// error as the f32 form; h and the final h + h * tanh(h) stay in fp32.
__device__ __forceinline__ uint32_t silu_pair_f16(float ha, float hb) {     // inputs are already x / 2
  const __half2 h2 = __floats2half2_rn(ha, hb);
  uint32_t hi = *reinterpret_cast<const uint32_t*>(&h2), ti;
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(ti) : "r"(hi));
  const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&ti));
  const __half2 y = __floats2half2_rn(fmaf(ha, t.x, ha), fmaf(hb, t.y, hb));
  return *reinterpret_cast<const uint32_t*>(&y);
}

// XFORM = false: no transform warpgroup, eight epilogue warps; the MMA issuers wait for the landed patch directly.
// XFORM = true: four epilogue warps + the transform warpgroup, GroupNorm(+SiLU) in the operand path.  384 threads either way.
// NE4 (without XFORM): four epilogue warps, warps 8..11 idle — the layers WITHOUT a residual, where the 16 KiB of staging
// that eight warps need would cost the fourth weight-ring stage (igemm_finalize): round 1 ran them with 4 warps + 4 stages
// at 1011-1025 us, eight warps + three stages measured 1053-1195 us (r2v); the residual layers keep eight (1290 -> 1125 us).
template <bool BF16, bool XFORM, bool NE4>
__global__ void __launch_bounds__(kPatchThreads, 1) igemm_patch_kernel(const __grid_constant__ IgemmParams p) {
  // default: warps 0..7 epilogue, 8..11 roles.  XFORM / NE4: warps 0..3 epilogue, 4..7 roles, 8..11 transform / idle.
  constexpr int NE = (XFORM || NE4) ? 4 : 8;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int b_bytes = p.BN * 128;
  const int stages = p.stages;                       // depth of the weight ring
  uint8_t* sB = smem + 2 * p.a_slot_bytes;
  uint8_t* stg_base = sB + stages * b_bytes;
  uint64_t* a_full = reinterpret_cast<uint64_t*>(stg_base + (p.tma_store ? NE * 4096 : 0));   // [slot][4]: only [slot][0] is used
  uint64_t* a_ready = a_full + 8;
  uint64_t* a_empty = a_ready + 2;
  uint64_t* b_full = a_empty + 2;
  uint64_t* b_empty = b_full + stages;
  uint64_t* tfull_bar = b_empty + stages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* res_bar = tempty_bar + 2;                                  // [epilogue warps] residual tile landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + 8);
  float* sbias = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 15) & ~uintptr_t(15));   // [kBiasSlots]
  float* sacc = sbias + p.bias_slots;

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;
  const int prows = (p.TH + 2) * kPP;                // 128-byte rows of a patch slot (130 pixels + 6 unused per image row)
  const int kc_all = p.kc_count + p.kc_sc;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&p.tmPatch);
    tma_prefetch_desc(&p.tmPatch2);
    tma_prefetch_desc(&p.tmB);
    for (int i = 0; i < 8; ++i) mbar_init(&a_full[i], 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a_ready[i], 128);                   // the transform warpgroup
      mbar_init(&a_empty[i], p.MT);                  // one tcgen05.commit per MMA issuer
    }
    for (int i = 0; i < stages; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], p.MT); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], p.MT); mbar_init(&tempty_bar[i], NE * 32); }
    for (int i = 0; i < 8; ++i) mbar_init(&res_bar[i], 1);
    fence_barrier_init();
  }
  const int rw = warp - NE;                          // role index: 0 patch producer, 1 / 2 MMA issuers, 3 weight producer
  if (rw == 2) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < NE) {
    // ===================================================================== epilogue
    if constexpr (XFORM) setmaxnreg_inc<232>();
    if (p.tma_store) run_epilogue_staged<BF16, NE, true>(p, stg_base, sacc, sbias, tfull_bar, tempty_bar, res_bar, tmem_base, warp, lane);
    else epilogue_direct<BF16, NE, false>(p, sbias, tfull_bar, tempty_bar, tmem_base, warp, lane);
  } else if (rw < 4) {
    if constexpr (XFORM) setmaxnreg_dec<72>();
    if (rw == 0) {
      // =================================================================== patch producer
      const bool leader = elect_one();
      int slot = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const TileCoord t = decode_tile(p, tile);
        const int x0 = t.tx * p.TW - 1, y0 = t.ty * p.TH - 1;
        for (int kc = 0; kc < kc_all; ++kc) {
          const bool main = kc < p.kc_count;
          mbar_wait(&a_empty[slot], phase ^ 1, 1);
          if (leader) {
            // ONE box per patch.  (One box per patch row on its own barrier — so that the transform could start on the
            // first row — was tried in round 2: 902 us against 728 us for the plain 128->128 layer, tensor pipe 78 % vs
            // 92 %, +32 % DRAM reads: profiles/r2_igemm_ncu_set_full.txt.)
            mbar_expect_tx(&a_full[slot * 4], (uint32_t)((p.TH + 2) * kPW * 128));
            tma_load_4d(smem + slot * p.a_slot_bytes, main ? &p.tmPatch : &p.tmPatch2, &a_full[slot * 4],
                        (main ? kc : kc - p.kc_count) * kBK, x0, y0, t.z1);
          }
          __syncwarp();
          if (++slot == 2) { slot = 0; phase ^= 1; }
        }
      }
    } else if (rw == 3) {
      // =================================================================== weight producer
      const bool leader = elect_one();
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const TileCoord t = decode_tile(p, tile);
        const int b_row = t.n_tile * p.BN;
        for (int kc = 0; kc < kc_all; ++kc) {
          const bool main = kc < p.kc_count;
          const int ntap = main ? 9 : 1;
          for (int tap = 0; tap < ntap; ++tap) {
            // packed weights: [tap][main chunk] ... then the shortcut chunks
            const int kblk = main ? tap * p.kc_count + kc : 9 * p.kc_count + (kc - p.kc_count);
            mbar_wait(&b_empty[stage], phase ^ 1, 5);
            if (leader) {
              mbar_expect_tx(&b_full[stage], (uint32_t)b_bytes);
              tma_load_3d(sB + stage * b_bytes, &p.tmB, &b_full[stage], kblk * kBK, b_row, 0);
            }
            __syncwarp();
            if (++stage == stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    } else if (rw - 1 < p.MT) {
      // =================================================================== MMA issuers (one per image row h)
      const bool leader = elect_one();
      const uint32_t idesc = make_idesc_f16(kBM, p.BN, BF16 ? 1 : 0);
      const int h = rw - 1;
      int slot = 0, stage = 0;
      uint32_t a_phase = 0, b_phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int mma_n = 0;
      int tap_off[9];
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) tap_off[tap] = ((p.seg[0][tap].dy + 1 + h) * kPP + p.seg[0][tap].dx + 1) * 128;
      const int centre_off = ((1 + h) * kPP + 1) * 128;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1, 2);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * kAccStride + h * 128;
        for (int kc = 0; kc < kc_all; ++kc) {
          const bool trm = p.trace != nullptr && blockIdx.x == 0 && h == 0 && leader;
          const int mix = trm ? mma_n++ : 0;
          if (trm && mix < 60) p.trace[mix * 8 + 4] = clock64();
          if constexpr (XFORM) {
            mbar_wait(&a_ready[slot], a_phase, 3);
          } else {
            mbar_wait(&a_full[slot * 4], a_phase, 3);                                            // the patch has landed
          }
          tc_fence_after();
          if (trm && mix < 60) p.trace[mix * 8 + 5] = clock64();
          const uint32_t patch = smem_u32(smem + slot * p.a_slot_bytes);
          if (kc < p.kc_count) {
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              mbar_wait(&b_full[stage], b_phase, 6);
              tc_fence_after();
              const uint64_t b_desc = make_sw128_kmajor_desc(smem_u32(sB + stage * b_bytes));
              if (leader) {
                const uint64_t a_desc = make_sw128_kmajor_desc(patch + tap_off[tap]);
#pragma unroll
                for (int k = 0; k < kBK / 16; ++k)
                  umma_f16(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kc | tap | k) ? 1u : 0u);
                umma_commit(&b_empty[stage]);
              }
              __syncwarp();
              if (++stage == stages) { stage = 0; b_phase ^= 1; }
            }
          } else {                                   // shortcut chunk: centre tap only (kc >= 1 here, always accumulate)
            mbar_wait(&b_full[stage], b_phase, 6);
            tc_fence_after();
            const uint64_t b_desc = make_sw128_kmajor_desc(smem_u32(sB + stage * b_bytes));
            if (leader) {
              const uint64_t a_desc = make_sw128_kmajor_desc(patch + centre_off);
#pragma unroll
              for (int k = 0; k < kBK / 16; ++k) umma_f16(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, 1u);
              umma_commit(&b_empty[stage]);
            }
            __syncwarp();
            if (++stage == stages) { stage = 0; b_phase ^= 1; }
          }
          if (leader) umma_commit(&a_empty[slot]);
          __syncwarp();
          if (trm && mix < 60) p.trace[mix * 8 + 6] = clock64();
          if (++slot == 2) { slot = 0; a_phase ^= 1; }
        }
        if (leader) umma_commit(&tfull_bar[acc]);
        __syncwarp();
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if constexpr (XFORM) {
    // ===================================================================== operand transform (warps 8..11)
    setmaxnreg_dec<104>();
    const int tt = threadIdx.x - 256;                // 0..127
    const int cpos = tt & 7;                         // 16-byte position inside the 128-byte row
    const int rbase = tt >> 3;                       // rows rbase, rbase + 16, ...
    // SWIZZLE_128B: position = logical 16-byte chunk ^ (row & 7); rows advance by 16 and the pitch (136) is a multiple
    // of 8, so (row & 7) is fixed per thread
    const int jlog = cpos ^ (rbase & 7);             // this thread's logical channel group (8 channels) in every chunk
    const bool do_gn = p.gn_ss != nullptr;
    const bool do_silu = p.gn_silu != 0;
    int slot = 0;
    uint32_t phase = 0;
    int trace_n = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord t = decode_tile(p, tile);
      const int x0 = t.tx * p.TW - 1, y0 = t.ty * p.TH - 1;
      const float* ssn = p.gn_ss + (long long)t.z1 * p.gn_C * 2;
      for (int kc = 0; kc < kc_all; ++kc) {
        const bool xf = do_gn && kc < p.kc_count;
        float sc[8], sh[8];
        if (xf) {                                    // fetched before the patch lands
          const float4* sp = reinterpret_cast<const float4*>(ssn + (kc * kBK + jlog * 8) * 2);
          const float pre = (do_silu && !BF16) ? 0.5f : 1.f;   // the fp16 SiLU form takes h = x / 2: folded into the affine
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float4 a = __ldg(sp + e);
            sc[2 * e] = a.x * pre; sh[2 * e] = a.y * pre; sc[2 * e + 1] = a.z * pre; sh[2 * e + 1] = a.w * pre;
          }
        }
        const bool trx = p.trace != nullptr && blockIdx.x == 0 && tt == 0;
        const int tix = trx ? trace_n++ : 0;
        if (trx && tix < 60) p.trace[tix * 8 + 0] = clock64();
        mbar_wait(&a_full[slot * 4], phase, 8);
        if (trx && tix < 60) p.trace[tix * 8 + 1] = clock64();
        if (xf) {
          const uint32_t base = smem_u32(smem + slot * p.a_slot_bytes) + cpos * 16;
          int py = 0, px = rbase;                    // rbase < 16 < kPW
          for (int r = rbase; r < prows; r += 64) {  // four rows in flight per thread
            uint32_t w[4][4];
            bool ok[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int rr = r + 16 * u;
              ok[u] = rr < prows && px < kPW && (unsigned)(y0 + py) < (unsigned)p.gridH && (unsigned)(x0 + px) < (unsigned)p.gridW;
              if (ok[u])
                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(w[u][0]), "=r"(w[u][1]), "=r"(w[u][2]), "=r"(w[u][3]) : "r"(base + rr * 128));
              px += 16;
              if (px >= kPP) { px -= kPP; ++py; }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              if (!ok[u]) continue;
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                float a = fmaf(cvt16<BF16>((uint16_t)(w[u][e] & 0xFFFF)), sc[2 * e], sh[2 * e]);
                float b = fmaf(cvt16<BF16>((uint16_t)(w[u][e] >> 16)), sc[2 * e + 1], sh[2 * e + 1]);
                if constexpr (BF16) {
                  if (do_silu) { a = silu_tanh(a); b = silu_tanh(b); }
                  w[u][e] = pack16<BF16>(a, b);
                } else {
                  w[u][e] = do_silu ? silu_pair_f16(a, b) : pack16<BF16>(a, b);
                }
              }
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(base + (r + 16 * u) * 128), "r"(w[u][0]),
                           "r"(w[u][1]), "r"(w[u][2]), "r"(w[u][3]) : "memory");
            }
          }
          fence_proxy_async_shared();                // generic-proxy writes -> visible to the tensor core's reads
        }
        if (trx && tix < 60) p.trace[tix * 8 + 2] = clock64();
        mbar_arrive(&a_ready[slot]);
        if (++slot == 2) { slot = 0; phase ^= 1; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (rw == 2) {
    __syncwarp();          // reconverge before the .aligned dealloc
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace

static long long* g_patch_trace = nullptr;
void igemm_patch_set_trace(long long* dev_buf) { g_patch_trace = dev_buf; }

cudaError_t igemm_patch_launch(const IgemmParams& p_in, int grid, cudaStream_t stream) {
  IgemmParams p = p_in;
  p.trace = g_patch_trace;
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
  if (!attr_set[dev]) {
    const void* fns[6] = {(const void*)igemm_patch_kernel<false, false, false>, (const void*)igemm_patch_kernel<false, true, false>,
                          (const void*)igemm_patch_kernel<true, false, false>,  (const void*)igemm_patch_kernel<true, true, false>,
                          (const void*)igemm_patch_kernel<false, false, true>,  (const void*)igemm_patch_kernel<true, false, true>};
    for (const void* f : fns) {
      cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
      if (e != cudaSuccess) return e;
    }
    attr_set[dev] = true;
  }
  const bool xform = p.gn_ss != nullptr;
  const bool ne4 = !xform && p.epi_warps == 4;
  if (p.flags & IG_BF16) {
    if (xform) launch(igemm_patch_kernel<true, true, false>, grid, kPatchThreads, kMaxSmem, stream, p);
    else if (ne4) launch(igemm_patch_kernel<true, false, true>, grid, kPatchThreads, kMaxSmem, stream, p);
    else launch(igemm_patch_kernel<true, false, false>, grid, kPatchThreads, kMaxSmem, stream, p);
  } else {
    if (xform) launch(igemm_patch_kernel<false, true, false>, grid, kPatchThreads, kMaxSmem, stream, p);
    else if (ne4) launch(igemm_patch_kernel<false, false, true>, grid, kPatchThreads, kMaxSmem, stream, p);
    else launch(igemm_patch_kernel<false, false, false>, grid, kPatchThreads, kMaxSmem, stream, p);
  }
  return cudaGetLastError();
}

}  // namespace gp
