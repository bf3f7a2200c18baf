// Fused self-attention forward for head_dim 64 (the SD-2.1 UNet's BasicTransformerBlock.attn1):
//   O = softmax(Q K^T) V   per (image, head), non-causal, fp32 softmax state, 16-bit operands.
// (Softmax scale is folded into Wq at load.)  FlashAttention-style online softmax on tcgen05, with
// TWO 128-row query tiles per CTA that share every K/V block:
//
//   warp 8        : TMA producer  — both Q tiles once; K block [128 keys x 64] + V^T block
//                                   [64 x 128 keys] per iteration into a 4-stage ring
//   warps 9,10    : MMA issuers   — one per tile t, an event loop over two independent streams:
//                                   S_t,j+1 = Q_t K_{j+1}^T (128x128x64) as soon as the softmax warps have
//                                   pulled S_t,j into registers; O_t += P_t,j V_j (128x64x128, accumulated
//                                   IN TMEM across all key blocks) as soon as P_t,j is in shared memory
//   warp 11       : TMEM allocator (512 columns: S_A [0,128) S_B [128,256) O_A [256,320) O_B [320,384))
//   warps 0..3    : softmax of tile A, warps 4..7 : softmax of tile B — one query row per thread.
//                   Per key block: the 128 scores of the row are read from TMEM ONCE (four loads in
//                   flight) and S_t is released immediately, so the next score tile is computed
//                   under this block's exponentials; row max; P = 2^(s*c - m*c) written 16-bit into
//                   shared memory in the K-major SWIZZLE_128B operand layout.
//   Lazy rescaling: the running maximum m that scales P and O is only raised when some row of the warp
//   saw its maximum grow by more than 2^8 (P <= 256 stays exact enough in 16 bits, sums are fp32).  Only
//   then the warp rescales its 32 rows of O in TMEM (tcgen05.ld / st).  On most blocks the softmax warps
//   never touch O, which removes the per-block "wait for P.V, load O, rescale" chain of the first version
//   (git history, "fattn_v1": 4200 cycles per block, 1900 of them outside the exponential pass; profiles/README.md §4).
// One elected lane of each single-thread role issues, the whole warp walks the loop (uniform registers).
//
// S and P never touch HBM (the round-1 unfused path wrote both: 4 x T^2 x 2 bytes per head).
#include "fattn.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "launch.h"
#include "ptx.cuh"

namespace gp {
namespace {

constexpr int kThreads = 384;
constexpr int kStages = 4;
constexpr int kQBytes = 128 * 64 * 2;          // 16 KiB per tile
constexpr int kKBytes = 128 * 64 * 2;          // 16 KiB
constexpr int kVBytes = 64 * 128 * 2;          // 16 KiB (two 64-key sub-tiles of 8 KiB)
constexpr int kPBytes = 128 * 128 * 2;         // 32 KiB per tile (two 64-key sub-tiles of 16 KiB)
constexpr int kSmemBytes = 2 * kQBytes + kStages * (kKBytes + kVBytes) + 2 * kPBytes + 256 + 1024;
constexpr int kTmemCols = 512;
constexpr int kOCol = 256;                     // O_t at 256 + t*64
constexpr long long kWatchdog = 100000000000LL;

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
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
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

template <bool BF16>
__global__ void __launch_bounds__(kThreads, 1) fattn_kernel(const __grid_constant__ FattnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                               // [tile][16 KiB]
  uint8_t* sK = sQ + 2 * kQBytes;                   // [stage][16 KiB]
  uint8_t* sV = sK + kStages * kKBytes;             // [stage][16 KiB]
  uint8_t* sP = sV + kStages * kVBytes;             // [tile][32 KiB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * kPBytes);
  uint64_t* q_full = bars;
  uint64_t* kv_full = bars + 1;                     // [kStages]
  uint64_t* kv_empty = kv_full + kStages;           // [kStages]  one commit per tile
  uint64_t* s_full = kv_empty + kStages;            // [tile]  S_t,j is in TMEM              (tcgen05.commit)
  uint64_t* s_free = s_full + 2;                    // [tile]  S_t,j is in registers          (128 arrivals)
  uint64_t* p_full = s_free + 2;                    // [tile]  P_t,j is in shared memory, O_t rescaled if needed (128)
  uint64_t* o_full = p_full + 2;                    // [tile]  O_t += P_t,j V_j has completed  (tcgen05.commit)
  uint64_t* pp = o_full + 2;                        // [tile]  the other tile has finished an exponential pass (128)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pp + 2);

  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const int pairs = (p.q_tiles + 1) >> 1;
  const int qp = blockIdx.x % pairs;
  const int bh = blockIdx.x / pairs;
  const int head = bh % p.heads, b = bh / p.heads;
  const int T = p.T;
  const int nblk = (T + 127) >> 7;
  const int ntile = (2 * qp + 1 < p.q_tiles) ? 2 : 1;   // the last pair of an odd tile count is half empty

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&p.tmQ);
    tma_prefetch_desc(&p.tmK);
    tma_prefetch_desc(&p.tmV);
    mbar_init(q_full, 1);
    for (int i = 0; i < kStages; ++i) { mbar_init(&kv_full[i], 1); mbar_init(&kv_empty[i], ntile); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_free[i], 128);
      mbar_init(&p_full[i], 128);
      mbar_init(&o_full[i], 1);
      mbar_init(&pp[i], 128);
    }
    fence_barrier_init();
  }
  if (warp == 11) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 8) {
    // ------------------------------------------------------------------ TMA producer (whole warp waits, one lane issues)
    const bool leader = elect_one();
    if (leader) {
      mbar_expect_tx(q_full, (uint32_t)(ntile * kQBytes));
      for (int t = 0; t < ntile; ++t) tma_load_3d(sQ + t * kQBytes, &p.tmQ, q_full, head * 64, (2 * qp + t) * 128, b);
    }
    for (int j = 0; j < nblk; ++j) {
      const int st = j % kStages;
      mbar_wait(&kv_empty[st], ((j / kStages) & 1) ^ 1, 10);
      if (leader) {
        mbar_expect_tx(&kv_full[st], kKBytes + kVBytes);
        tma_load_3d(sK + st * kKBytes, &p.tmK, &kv_full[st], head * 64, j * 128, b);
        tma_load_3d(sV + st * kVBytes, &p.tmV, &kv_full[st], j * 128, head * 64, b);
        tma_load_3d(sV + st * kVBytes + 8192, &p.tmV, &kv_full[st], j * 128 + 64, head * 64, b);
      }
      __syncwarp();
    }
  } else if ((warp == 9 || warp == 10) && (warp - 9) < ntile) {
    // ------------------------------------------------------------------ MMA issuer of tile t (event loop)
    const int t = warp - 9;
    const bool leader = elect_one();
    const uint32_t idesc_s = make_idesc_f16(128, 128, BF16 ? 1 : 0);
    const uint32_t idesc_o = make_idesc_f16(128, 64, BF16 ? 1 : 0);
    const uint64_t q_desc = make_sw128_kmajor_desc(smem_u32(sQ + t * kQBytes));
    const uint64_t p_desc = make_sw128_kmajor_desc(smem_u32(sP + t * kPBytes));
    const uint64_t k_desc0 = make_sw128_kmajor_desc(smem_u32(sK));
    const uint64_t v_desc0 = make_sw128_kmajor_desc(smem_u32(sV));
    const uint32_t s_tmem = tmem_base + t * 128;
    const uint32_t o_tmem = tmem_base + kOCol + t * 64;
    const bool trm = p.trace != nullptr && blockIdx.x == 0 && t == 0 && leader;
    auto issue_s = [&](int j) {               // S_t = Q_t K_j^T
      mbar_wait(&kv_full[j % kStages], (j / kStages) & 1, 11);
      tc_fence_after();
      const uint64_t k_desc = k_desc0 + (uint64_t)((j % kStages) * (kKBytes >> 4));
      if (leader) {
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16(s_tmem, q_desc + 2 * k, k_desc + 2 * k, idesc_s, k ? 1u : 0u);
        umma_commit(&s_full[t]);
      }
      __syncwarp();
      if (trm && j < 64) p.trace[512 + j * 4 + 0] = clock64();
    };
    auto issue_pv = [&](int j) {              // O_t (+)= P_t,j V_j
      const int st = j % kStages;
      const uint64_t v_desc = v_desc0 + (uint64_t)(st * (kVBytes >> 4));
      if (trm && j < 64) p.trace[512 + j * 4 + 1] = clock64();
      if (leader) {
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          umma_f16(o_tmem, p_desc + (uint64_t)((kk >> 2) * (16384 >> 4) + 2 * (kk & 3)),
                   v_desc + (uint64_t)((kk >> 2) * (8192 >> 4) + 2 * (kk & 3)), idesc_o, (j | kk) ? 1u : 0u);
        umma_commit(&o_full[t]);
        umma_commit(&kv_empty[st]);           // this tile has issued every use of block j (barrier counts both tiles)
      }
      __syncwarp();
      if (trm && j < 64) p.trace[512 + j * 4 + 2] = clock64();
    };
    mbar_wait(q_full, 0, 12);
    issue_s(0);
    int js = 1, jp = 0;
    long long t_progress = clock64();
    while (jp < nblk) {
      bool s_ok = js < nblk && mbar_test_wait(&s_free[t], (js - 1) & 1);
      s_ok = __all_sync(0xffffffffu, s_ok);
      if (s_ok) {                             // the softmax warps hold S_t,js-1 in registers
        tc_fence_after();
        issue_s(js);
        ++js;
        t_progress = clock64();
        continue;
      }
      bool p_ok = mbar_test_wait(&p_full[t], jp & 1);
      p_ok = __all_sync(0xffffffffu, p_ok);
      if (p_ok) {                             // P_t,jp is in shared memory (and O_t rescaled if it had to be)
        tc_fence_after();
        issue_pv(jp);
        ++jp;
        t_progress = clock64();
      } else if (clock64() - t_progress > kWatchdog) {
        if (leader) printf("[gp] fattn issuer watchdog: block %d tile %d js %d jp %d\n", (int)blockIdx.x, t, js, jp);
        __trap();
      }
    }
  } else if (warp < 8 && (warp >> 2) < ntile) {
    // ------------------------------------------------------------------ softmax of tile t
    const int t = warp >> 2;
    const int wq = warp & 3;             // == warp % 4 -> TMEM lanes [32*wq, 32*wq+32)
    const int row = wq * 32 + lane;
    const uint32_t lane_off = (uint32_t)(wq * 32) << 16;
    const float c2 = p.scale_log2e;
    const float thr = 8.0f;              // lazy-rescale threshold in the log2 domain (P <= 2^8)
    float m = -INFINITY, l = 0.f;        // m: the maximum P and O are currently scaled by
    const uint32_t prow = smem_u32(sP + t * kPBytes) + row * 128;
    const int sw = row & 7;
    const uint32_t ts = tmem_base + lane_off + t * 128;
    const uint32_t to = tmem_base + lane_off + kOCol + t * 64;
    const bool tr = p.trace != nullptr && blockIdx.x == 0 && t == 0 && wq == 0 && lane == 0;
    // Phase relation of the two tiles.  Left alone they run in lock-step: both exponential passes share the
    // MUFU (2 x 128 x 8 cycles per sub-partition) and both idle it together during the rest of the block
    // (r1j: 3700 cycles per block).  With strict alternation (A_j, B_j, A_j+1, ...; two mbarriers) one
    // tile's load / max / wait phases run under the other's exponentials: 3200 cycles, 11.7 -> 9.8 ms
    // per step.  A start offset for tile B is the cheaper idea that did not hold the phase.
    const bool pingpong = ntile == 2;
    for (int j = 0; j < nblk; ++j) {
      if (tr && j < 64) p.trace[j * 8 + 0] = clock64();
      mbar_wait(&s_full[t], j & 1, 15);
      tc_fence_after();
      if (tr && j < 64) p.trace[j * 8 + 1] = clock64();
      const int kvalid = min(128, T - j * 128);
      uint32_t s[4][32];
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld_32x32(ts + c * 32, s[c]);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&s_free[t]);                     // S_t may be overwritten by S_t,j+1 from here on
      if (kvalid < 128) {
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int q = 0; q < 32; ++q)
            if (c * 32 + q >= kvalid) s[c][q] = 0xff800000u;   // -inf: max ignores it, exp2 gives 0
      }
      float mx0 = m, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int q = 0; q < 32; q += 4) {
          mx0 = fmaxf(mx0, __uint_as_float(s[c][q]));
          mx1 = fmaxf(mx1, __uint_as_float(s[c][q + 1]));
          mx2 = fmaxf(mx2, __uint_as_float(s[c][q + 2]));
          mx3 = fmaxf(mx3, __uint_as_float(s[c][q + 3]));
        }
      const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
      const bool raise = __any_sync(0xffffffffu, (mx - m) * c2 > thr);   // j == 0: m = -inf -> true
      if (tr && j < 64) p.trace[j * 8 + 2] = clock64();
      if (j > 0) {                                 // P_t,j-1 V_j-1 done: the P buffer is reusable, O_t is stable
        mbar_wait(&o_full[t], (j - 1) & 1, 16);
        tc_fence_after();
      }
      if (tr && j < 64) p.trace[j * 8 + 3] = clock64();
      if (raise) {                                 // warp-uniform
        const float alpha = ex2((m - mx) * c2);    // j == 0: 0 (and l == 0, O not yet written)
        if (j > 0) {
#pragma unroll 1
          for (int c = 0; c < 64; c += 8) {
            uint32_t r[8];
            tmem_ld_32x8(to + c, r);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 8; ++q) r[q] = __float_as_uint(__uint_as_float(r[q]) * alpha);
            tmem_st_32x8(to + c, r);
          }
          tmem_st_wait();
        }
        l *= alpha;
        m = mx;
      }
      if (pingpong) {                              // A_j after B_j-1, B_j after A_j
        if (t == 0) { if (j > 0) mbar_wait(&pp[0], (j - 1) & 1, 18); }
        else mbar_wait(&pp[1], j & 1, 18);
      }
      if (tr && j < 64) p.trace[j * 8 + 4] = clock64();
      // probabilities -> shared memory (A operand of P.V), row sum (8 partial sums)
      const float mb = m * c2;
      float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f, l4 = 0.f, l5 = 0.f, l6 = 0.f, l7 = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float pv[32];
#pragma unroll
        for (int q = 0; q < 32; ++q) {
          const float x = __uint_as_float(s[c][q]) * c2 - mb;      // <= thr
          pv[q] = ex2(x);
        }
        // hand the MUFU to the other tile once the exponentials of chunk 1 are issued: its wake-up latency and the first
        // FFMAs of its pass run under this tile's remaining sums / packs / stores (r1l trace, block period in cycles by
        // hand-over chunk: 3440 (0) / 3180 (1) / 3290 (2) / 3350 (3) / 3560 (after the pass))
        if (pingpong && c == 1) mbar_arrive(&pp[1 - t]);
#pragma unroll
        for (int q = 0; q < 32; q += 8) {
          l0 += pv[q]; l1 += pv[q + 1]; l2 += pv[q + 2]; l3 += pv[q + 3];
          l4 += pv[q + 4]; l5 += pv[q + 5]; l6 += pv[q + 6]; l7 += pv[q + 7];
        }
        const uint32_t dst = prow + (c >> 1) * 16384;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          st_shared_v4(dst + ((((c & 1) * 4 + i) ^ sw) << 4), pack16<BF16>(pv[8 * i + 0], pv[8 * i + 1]),
                       pack16<BF16>(pv[8 * i + 2], pv[8 * i + 3]), pack16<BF16>(pv[8 * i + 4], pv[8 * i + 5]),
                       pack16<BF16>(pv[8 * i + 6], pv[8 * i + 7]));
      }
      l += ((l0 + l1) + (l2 + l3)) + ((l4 + l5) + (l6 + l7));
      if (tr && j < 64) p.trace[j * 8 + 5] = clock64();
      tc_fence_before();                          // the O_t rescale (if any) is ordered before the next P.V
      fence_proxy_async_smem();                   // P_t visible to the tensor core (async proxy)
      mbar_arrive(&p_full[t]);
      if (tr && j < 64) p.trace[j * 8 + 6] = clock64();
    }
    // normalise, store
    mbar_wait(&o_full[t], (nblk - 1) & 1, 17);
    tc_fence_after();
    const float inv = 1.f / l;
    uint32_t o[2][32];
    tmem_ld_32x32(to, o[0]);
    tmem_ld_32x32(to + 32, o[1]);
    tmem_ld_wait();
    const int qrow = (2 * qp + t) * 128 + row;
    if (qrow < T) {
      uint16_t* op = reinterpret_cast<uint16_t*>(p.out) + (long long)b * p.out_b_stride +
                     (long long)qrow * p.out_row_stride + head * 64;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t* r = &o[i >> 2][(i & 3) * 8];
        uint4 u;
        u.x = pack16<BF16>(__uint_as_float(r[0]) * inv, __uint_as_float(r[1]) * inv);
        u.y = pack16<BF16>(__uint_as_float(r[2]) * inv, __uint_as_float(r[3]) * inv);
        u.z = pack16<BF16>(__uint_as_float(r[4]) * inv, __uint_as_float(r[5]) * inv);
        u.w = pack16<BF16>(__uint_as_float(r[6]) * inv, __uint_as_float(r[7]) * inv);
        *reinterpret_cast<uint4*>(op + 8 * i) = u;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 11) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace

static long long* g_trace = nullptr;
void fattn_set_trace(long long* dev_buf) { g_trace = dev_buf; }
long long* fattn_get_trace() { return g_trace; }

cudaError_t fattn_launch(const FattnParams& p, cudaStream_t stream) {
  static bool attr_dev[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
  bool& attr_set = attr_dev[dev];      // function attributes are per device
  if (!attr_set) {
    for (const void* f : {(const void*)fattn_kernel<false>, (const void*)fattn_kernel<true>}) {
      cudaError_t e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
      if (e != cudaSuccess) return e;
    }
    attr_set = true;
  }
  const int grid = p.B * p.heads * ((p.q_tiles + 1) / 2);
  if (grid <= 0) return cudaSuccess;
  if (p.bf16) launch(fattn_kernel<true>, grid, kThreads, kSmemBytes, stream, p);
  else launch(fattn_kernel<false>, grid, kThreads, kSmemBytes, stream, p);
  return cudaGetLastError();
}

}  // namespace gp
