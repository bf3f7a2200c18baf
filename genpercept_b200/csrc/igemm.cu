// tcgen05 implicit-GEMM kernel (see igemm.h for the operand model).
//
// Warp roles (384 threads, 1 CTA / SM, persistent over a static round-robin tile list).  The single-thread
// producer / issuer roles sit in the HIGHEST warp ids (8..11): the SM sub-partition arbiter favours higher warp
// ids, and an issuer starved by the epilogue warps of its sub-partition stalls the tensor pipe (fattn trace, r1h).
// Each single-thread role is executed by its WHOLE warp (every lane walks the loop and waits on the barriers) and
// one elect.sync lane issues: coordinates and descriptors stay in uniform registers (back-to-back UTCHMMA).
//   warp 8         : TMA producer A (activation box per 64-channel K block, `stages`-deep ring)
//   warp 11        : TMA producer B (weight box per K block) — its own warp: one thread issuing
//                    both boxes plus the barrier traffic could not keep up with BN=128 tiles
//                    (ncu r1a: tensor pipe 45 % active on the 128->128 convs, DRAM/L2 not saturated)
//   warp 9 (and 10): MMA issuer(s), one per accumulator tile (4 tcgen05.mma 128xBNx16 per K block; commit frees the slot)
//   warp 10        : TMEM allocator (512 columns = 2 accumulator buffers x MT tiles)
//   warps 0..7     : epilogue, two per sub-partition: warps w and w + 4 read the same TMEM lane quadrant and split the
//                    tile's 64-channel groups (tcgen05.ld 32 lanes x 32 columns -> bias (from shared memory) / TMA-loaded
//                    residual / act -> staged tile -> TMA store, GroupNorm partial sums from the staged tile).  One
//                    epilogue warp per sub-partition was stalled 78 % of the time (ncu r2, the K = 1 stem GEMM).
// MT = 2 (a 256-pixel M tile per CTA, two accumulators sharing every weight box) when BN <= 128:
// halves the weight traffic and the per-byte barrier / TMA issue cost of the narrow-N layers.
#include "igemm.h"

#include <cstring>

#include "igemm_common.cuh"
#include "launch.h"

namespace gp {

namespace {

constexpr int kEpiWarps = 8;                         // epilogue warps 0..7; the single-thread roles are warps 8..11
constexpr int kTapThreads = (kEpiWarps + 4) * 32;    // 384

template <bool BF16>
__global__ void __launch_bounds__(kTapThreads, 1) igemm_kernel(const __grid_constant__ IgemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int a_bytes = kABytes * p.MT;
  const int stage_bytes = a_bytes + p.BN * 128;
  const int stages = p.stages;
  uint8_t* stg_base = smem + stages * stage_bytes;                     // one 4 KiB staging tile per epilogue warp (tma_store only)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(stg_base + (p.tma_store ? (p.out_lo ? 2 : 1) * p.epi_warps * 4096 : 0));
  uint64_t* empty_bar = full_bar + stages;
  uint64_t* tfull_bar = empty_bar + stages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* res_bar = tempty_bar + 2;                                  // [epilogue warps] residual tile landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + kEpiWarps);
  float* sbias = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 15) & ~uintptr_t(15));   // [kBiasSlots]
  float* sacc = sbias + p.bias_slots;   // [4 epilogue warps][Cout][2], only with p.stats

  const int warp = uniform_warp_id();
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < (p.npass > 1 ? 8 : 4); ++i) tma_prefetch_desc(&p.tmA[i]);
    tma_prefetch_desc(&p.tmB);
    for (int i = 0; i < stages; ++i) {
      mbar_init(&full_bar[i], 2);    // producer A + producer B
      mbar_init(&empty_bar[i], p.MT);  // one tcgen05.commit per MMA issuer
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], p.MT);
      mbar_init(&tempty_bar[i], p.epi_warps * 32);
    }
    for (int i = 0; i < kEpiWarps; ++i) mbar_init(&res_bar[i], 1);
    fence_barrier_init();
  }
  if (warp == kEpiWarps + 2) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Single-thread roles run warp-uniform (every lane walks the loop and waits on the barriers) and one
  // elected lane issues: the TMA coordinates / UMMA descriptors then stay in uniform registers.
  if (warp == kEpiWarps) {
    // ===================================================================== TMA producer A
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord t = decode_tile(p, tile);
      const int cls = p.cls_from_z0 ? t.z0 : 0;
      const int a_n = t.z1 * p.a_n_z1 + t.z0 * p.a_n_z0;
      const int a_k0 = t.z0 * p.a_k_z0;
      const int x0 = t.tx * p.TW, y0 = t.ty * p.TH;
      const int ns = p.nseg[cls];
      for (int pass = 0; pass < p.npass; ++pass) {
        const int moff = p.pass_amap[pass];
        for (int s = 0; s < ns; ++s) {
          const IgemmSeg sg = p.seg[cls][s];
          const CUtensorMap* tm = &p.tmA[sg.map + moff];
          const int xs = x0 + sg.dx, ys = y0 + sg.dy;
          for (int c = 0; c < sg.nchunks; ++c) {
            mbar_wait(&empty_bar[stage], phase ^ 1, 1);
            if (leader) {
              mbar_expect_tx(&full_bar[stage], (uint32_t)a_bytes);
              tma_load_4d(smem + stage * stage_bytes, tm, &full_bar[stage], a_k0 + c * kBK, xs, ys, a_n);
            }
            __syncwarp();
            if (++stage == stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == kEpiWarps + 3) {
    // ===================================================================== TMA producer B
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t b_bytes = (uint32_t)p.BN * 128;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord t = decode_tile(p, tile);
      const int cls = p.cls_from_z0 ? t.z0 : 0;
      const int b_z = t.z1 * p.b_z_z1 + t.z0 * p.b_z_z0;
      const int b_row = t.z0 * p.b_row_z0 + t.n_tile * p.BN;
      const int b_k0 = t.z0 * p.b_k_z0;
      const int nkb = p.nkb[cls];
      for (int pass = 0; pass < p.npass; ++pass) {
        const CUtensorMap* tmb = p.pass_bmap[pass] ? &p.tmB2 : &p.tmB;
        const int bk = b_k0 + p.pass_bk[pass];
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1, 5);
          if (leader) {
            mbar_expect_tx(&full_bar[stage], b_bytes);
            tma_load_3d(smem + stage * stage_bytes + a_bytes, tmb, &full_bar[stage], bk + kb * kBK, b_row, b_z);
          }
          __syncwarp();
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kEpiWarps + 1 || (warp == kEpiWarps + 2 && p.MT == 2)) {
    const bool leader = elect_one();
    // ===================================================================== MMA issuer(s)
    // With two accumulator tiles (MT = 2, BN <= 128) each tile gets its own issuing thread: a single
    // thread cannot issue one 64-cycle 128x128x16 MMA every 64 cycles once descriptor arithmetic and
    // barrier polls are added (ncu r1h: tensor pipe 57 % busy, issuer never blocked on a barrier).
    const uint32_t idesc = make_idesc_f16(kBM, p.BN, BF16 ? 1 : 0);
    const int h_lo = warp - (kEpiWarps + 1), h_hi = (p.MT == 2) ? warp - kEpiWarps : 1;
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord t = decode_tile(p, tile);
      const int cls = p.cls_from_z0 ? t.z0 : 0;
      const int nkb = p.nkb[cls] * p.npass;
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1, 2);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * kAccStride;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&full_bar[stage], phase, 3);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + stage * stage_bytes);
        const uint64_t b_desc = make_sw128_kmajor_desc(a_addr + a_bytes);
        if (leader) {
          for (int h = h_lo; h < h_hi; ++h) {
            const uint64_t a_desc = make_sw128_kmajor_desc(a_addr + h * kABytes);
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k) {
              // +32 bytes per UMMA_K inside the 128-byte swizzle row -> +2 in the (addr >> 4) field
              umma_f16(d_tmem + h * 128, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) ? 1u : 0u);
            }
          }
          umma_commit(&empty_bar[stage]);
        }
        __syncwarp();
        if (++stage == stages) { stage = 0; phase ^= 1; }
      }
      if (leader) umma_commit(&tfull_bar[acc]);
      __syncwarp();
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else if (warp < kEpiWarps && p.epi_warps == kEpiWarps) {
    if (p.tma_store) run_epilogue_staged<BF16, kEpiWarps, false>(p, stg_base, sacc, sbias, tfull_bar, tempty_bar, res_bar, tmem_base, warp, lane);
    else run_epilogue_direct<BF16, kEpiWarps>(p, sbias, tfull_bar, tempty_bar, tmem_base, warp, lane);
  } else if (warp < 4) {
    // four epilogue warps (warps 4..7 idle): the long-K BN = 256 layers, where eight 4 KiB staging tiles would cost the fourth
    // pipeline stage (igemm_finalize) and the epilogue is hidden behind an 18 k-cycle main loop anyway
    if (p.tma_store) run_epilogue_staged<BF16, 4, false>(p, stg_base, sacc, sbias, tfull_bar, tempty_bar, res_bar, tmem_base, warp, lane);
    else run_epilogue_direct<BF16, 4>(p, sbias, tfull_bar, tempty_bar, tmem_base, warp, lane);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kEpiWarps + 2) {
    __syncwarp();          // reconverge before the .aligned dealloc
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* f = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<PFN_encodeTiled>(f);
  return fn;
}

int g_num_sms = 0;

}  // namespace

cudaError_t make_tmap_a(CUtensorMap* m, const void* base, int C, int W, int H, int N, long long sW,
                        long long sH, long long sN, int TW, int TH, bool bf16) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return cudaErrorNotSupported;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)sW * 2, (cuuint64_t)sH * 2, (cuuint64_t)sN * 2};
  cuuint32_t box[4] = {(cuuint32_t)kBK, (cuuint32_t)TW, (cuuint32_t)TH, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

cudaError_t make_tmap_b(CUtensorMap* m, const void* base, long long K, long long rows, long long Z,
                        long long sRow, long long sZ, int BN, bool bf16) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return cudaErrorNotSupported;
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)Z};
  cuuint64_t strides[2] = {(cuuint64_t)sRow * 2, (cuuint64_t)sZ * 2};
  cuuint32_t box[3] = {(cuuint32_t)kBK, (cuuint32_t)BN, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

size_t igemm_smem_bytes(const IgemmParams& p) {
  return (size_t)p.stages * (kABytes * p.MT + p.BN * 128) + (2 * p.stages + 4) * 8 + 16 + 1024;
}

const char* igemm_finalize(IgemmParams* p) {
  if (p->MT == 0) p->MT = 1;
  if (p->npass == 0) p->npass = 1;
  if (p->npass != 1 && p->npass != 3) return "npass must be 1 or 3";
  if (p->npass == 1) { p->pass_amap[0] = 0; p->pass_bk[0] = 0; p->pass_bmap[0] = 0; }
  if (p->out_lo && (p->stats || p->res_tma || p->patch || (p->flags & IG_OUT_F32_NCHW)))
    return "the high-precision output layout excludes epilogue statistics, TMA residuals, the patch loop and fp32 maps";
  if (p->MT != 1 && p->MT != 2) return "MT must be 1 or 2";
  if (p->MT == 2 && p->BN > 128) return "MT=2 needs BN <= 128 (TMEM: 2 buffers x 2 tiles x BN columns)";
  if (p->TW * p->TH != kBM * p->MT) return "TW*TH must be 128*MT";
  if (p->TW > 256 || p->TH > 256) return "TMA box dims are limited to 256";
  if ((1 << p->tw_shift) != p->TW) return "TW must be a power of two";
  if (p->BN < 16 || p->BN > 256 || (p->BN % 16)) return "BN must be a multiple of 16 in [16,256]";
  if (p->Z0 < 1 || p->Z1 < 1) return "bad batch dims";
  p->tiles_x = (p->gridW + p->TW - 1) / p->TW;
  p->tiles_y = (p->gridH + p->TH - 1) / p->TH;
  p->n_tiles_n = (p->Cout + p->BN - 1) / p->BN;
  const int ncls = p->cls_from_z0 ? p->Z0 : 1;
  if (ncls > kMaxClasses) return "too many classes";
  for (int c = 0; c < ncls; ++c) {
    if (p->nseg[c] < 1 || p->nseg[c] > kMaxSegs) return "bad segment count";
    int n = 0;
    for (int s = 0; s < p->nseg[c]; ++s) n += p->seg[c][s].nchunks;
    p->nkb[c] = n;
    if (n < 1) return "empty K loop";
  }
  long long total = (long long)p->n_tiles_n * p->tiles_x * p->tiles_y * p->Z0 * p->Z1;
  if (total > 0x7fffffffLL) return "too many tiles";
  p->total_tiles = (int)total;
  const int stage_bytes = kABytes * p->MT + p->BN * 128;
  const int stats_bytes = p->stats ? 4 * p->Cout * 2 * (int)sizeof(float) : 0;
  if (p->tma_store && ((p->Cout % 64) || (p->BN % 64) || (p->flags & IG_OUT_F32_NCHW) || p->out_z0 != 0))
    return "staged epilogue needs Cout % 64 == 0, BN % 64 == 0, plain 16-bit NHWC output";
  if (p->tma_store && (p->flags & IG_GEGLU)) return "GEGLU needs the direct epilogue";
  if (p->stats && (!p->tma_store || p->Cout > 512 || (p->flags & IG_GEGLU))) return "statistics need the staged epilogue and Cout <= 512";
  // staging: one 4 KiB tile per epilogue warp (8; 4 in the patch kernel's GroupNorm-transform build), x2 for the (hi, lo) layout
  int epi_warps = (p->patch && p->gn_ss) ? 4 : 8;
  // patch-resident layers without a residual: four warps and the fourth 16 KiB weight-ring stage (see igemm_patch.cu, NE4)
  if (p->patch && !p->gn_ss && p->tma_store && !p->res_tma && p->res1 == nullptr && p->res2 == nullptr)
    epi_warps = 4;
  auto staging_of = [&](int ew) { return p->tma_store ? ew * 4096 * (p->out_lo ? 2 : 1) : 0; };
  int nkb_max = 0;
  for (int c = 0; c < ncls; ++c) nkb_max = p->nkb[c] > nkb_max ? p->nkb[c] : nkb_max;
  // Eight staging tiles + the statistics scratch leave the BN = 256 layers three 48 KiB stages instead of four (r2: the
  // 512- and 256-channel VAE convs ran 8-15 % slower than in round 1: 929 -> 1006..1069 us).  Their main loop is >= 16 K
  // blocks (18 k cycles per tile) and hides a four-warp epilogue, so those layers keep four warps and the fourth stage.
  if (!p->patch && epi_warps == 8 && nkb_max >= 16 &&
      (kMaxSmem - 3072 - stats_bytes - staging_of(4)) / stage_bytes > (kMaxSmem - 3072 - stats_bytes - staging_of(8)) / stage_bytes)
    epi_warps = 4;
  p->epi_warps = epi_warps;
  const int staging = staging_of(epi_warps);
  // bias: one N tile (288 floats, inside the 3072 reserved bytes) or the whole padded vector when it is small (<= 16 KiB)
  p->bias_slots = kBiasSlots;
  p->bias_all = 0;
  if (p->n_tiles_n > 1 && p->n_tiles_n * p->BN + 32 <= 4096) {
    p->bias_all = 1;
    p->bias_slots = p->n_tiles_n * p->BN + 32;
  }
  int bias_extra = (p->bias_slots - kBiasSlots) * (int)sizeof(float);
  int st = (kMaxSmem - 3072 - stats_bytes - staging - bias_extra) / stage_bytes;
  // ... but never at the price of a pipeline stage: the BN = 256 layers fit exactly four 48 KiB stages, and the UNet's deep
  // levels (L2-latency-bound) lost 25-30 % with three (r2r: 2560 -> 1280 on 8 x 12 x 12 pixels 134 -> 179 us)
  if (p->bias_all && !p->patch && st < (kMaxSmem - 3072 - stats_bytes - staging) / stage_bytes) {
    p->bias_all = 0;
    p->bias_slots = kBiasSlots;
    bias_extra = 0;
    st = (kMaxSmem - 3072 - stats_bytes - staging) / stage_bytes;
  }
  if (p->patch) {
    if (p->TW != 128 || p->TH != p->MT || p->Z0 != 1 || p->Z1 < 1 || p->nseg[0] != 9 + (p->kc_sc > 0 ? 1 : 0) || p->kc_count < 1 ||
        p->nkb[0] != 9 * p->kc_count + p->kc_sc || p->npass != 1 || p->gridW % 128 || p->gridH % p->TH)
      return "patch mode needs TW = 128, TH = MT, full tiles and a single-source 3x3 tap table (+ shortcut chunks)";
    if (p->gn_ss && p->gn_C != p->kc_count * 64) return "patch mode: GroupNorm channels must equal the source's";
    p->a_slot_bytes = ((p->TW + 2) * (p->TH + 2) * 128 + 1023) & ~1023;
    st = (kMaxSmem - 3072 - stats_bytes - staging - bias_extra - 2 * p->a_slot_bytes) / (p->BN * 128);
    if (p->bias_all && st < (kMaxSmem - 3072 - stats_bytes - staging - 2 * p->a_slot_bytes) / (p->BN * 128)) {
      p->bias_all = 0;
      p->bias_slots = kBiasSlots;
      st = (kMaxSmem - 3072 - stats_bytes - staging - 2 * p->a_slot_bytes) / (p->BN * 128);
    }
  }
  if (st > 8) st = 8;
  if (st < 2) return "tile too large for shared memory";
  p->stages = st;
  return nullptr;
}

static cudaError_t igemm_init();

int igemm_grid(const IgemmParams& p) {
  if (igemm_init() != cudaSuccess) return 0;
  return p.total_tiles < g_num_sms ? p.total_tiles : g_num_sms;
}

// Function attributes are per device: keyed by the current device so that engines on several GPUs of one process work.
static cudaError_t igemm_init() {
  static bool attr_set[64] = {};
  static int sms[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
  if (!attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(igemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(igemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return e;
    cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
    attr_set[dev] = true;
  }
  g_num_sms = sms[dev];
  return cudaSuccess;
}

cudaError_t igemm_launch(const IgemmParams& p, cudaStream_t stream) {
  cudaError_t ie = igemm_init();
  if (ie != cudaSuccess) return ie;
  if (p.total_tiles <= 0) return cudaSuccess;
  if (p.stats && p.stats_slots < (p.total_tiles < g_num_sms ? p.total_tiles : g_num_sms)) return cudaErrorInvalidValue;
  const int grid = p.total_tiles < g_num_sms ? p.total_tiles : g_num_sms;
  // always request the maximum so exactly one CTA (512 TMEM columns) is resident per SM
  const size_t smem = kMaxSmem;
  if (p.patch) return igemm_patch_launch(p, grid, stream);
  if (p.flags & IG_BF16) {
    launch(igemm_kernel<true>, grid, kTapThreads, smem, stream, p);
  } else {
    launch(igemm_kernel<false>, grid, kTapThreads, smem, stream, p);
  }
  return cudaGetLastError();
}

}  // namespace gp
