// Persistent warp-specialised tcgen05 implicit-GEMM: the one tensor-core kernel behind every 3x3
// convolution (stride 1, stride 2, nearest-2x-upsample-fused), 1x1 convolution / linear layer
// and batched attention GEMM of the hot path.
//
//   D[pixel, n] = sum over K-segments s, channels c :  A_s[pixel + (dy_s, dx_s), c] * B[n, k(s, c)]
//
// A operand: up to 4 NHWC activation views, each a 4-D TMA tensor map (C, W, H, N); a CTA's
// 128-row M tile is a TW x TH spatial patch, loaded per K-chunk of 64 channels as one TMA box whose
// start coordinate carries the filter-tap offset (halo/padding = TMA out-of-bounds zero fill).
// B operand: K-major [rows, K] matrix (packed weights, or activations for attention), 3-D map.
// Accumulators: fp32 in TMEM, double buffered (2 x 256 columns) so the epilogue of tile i overlaps
// the main loop of tile i+1.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace gp {

constexpr int kMaxSegs = 20;
constexpr int kMaxClasses = 4;
constexpr int kBM = 128;      // UMMA M (TMEM lanes)
constexpr int kBK = 64;       // channels per pipeline stage (= one 128-byte swizzle row of fp16)

struct IgemmSeg {
  int8_t map;        // index into tmA
  int8_t dy, dx;     // tap offset in the map's pixel grid
  uint16_t nchunks;  // ceil(C / 64)  (up to 256 for the P.V product over 16384 keys)
};

enum IgemmFlags : int {
  IG_RELU = 1,            // max(v, 0) after bias/residual
  IG_OUT_F32_NCHW = 2,    // write fp32 planar [Z1, Cout, outH, outW] instead of 16-bit NHWC
  IG_AFFINE_CLAMP01 = 4,  // v = clamp((v + 1) / 2, 0, 1)   (genpercept_pipeline.py:470-472)
  IG_BF16 = 8,            // operands / 16-bit outputs are bf16 instead of fp16
  IG_GEGLU = 16,          // columns come in chunks of 32 = [16 values | 16 gates]: out = value * gelu_erf(gate),
                          // 16 outputs per chunk at column n/2 (ff.net.0 of BasicTransformerBlock)
};

struct IgemmParams {
  CUtensorMap tmA[8];            // [0..3]: the (hi) planes of up to 4 sources; [4..7]: their lo planes (high-precision mode)
  CUtensorMap tmB;
  CUtensorMap tmB2;              // lo plane of an ACTIVATION B operand (attention GEMMs, high-precision mode)
  // High-precision mode (gp_config::precision = 1): every operand is an fp16 (hi, lo) pair and the K loop runs
  // three passes over the segment table, accumulating hi*hi + lo*hi + hi*lo in the same fp32 TMEM accumulator.
  // Packed weights carry both planes along K: [.. ktot hi .. | .. ktot lo ..].
  int npass;                     // 1, or 3
  int pass_amap[3];              // added to IgemmSeg::map          {0, 4, 0}
  int pass_bk[3];                // added to the B K coordinate      {0, 0, ktot}
  int pass_bmap[3];              // 0: tmB, 1: tmB2                  {0, 0, 0 or 1}
  long long out_lo;              // element offset of the output's lo plane inside a pixel (0: plain 16-bit output);
                                 // residuals share the output's layout
  CUtensorMap tmOutLo[kMaxClasses];
  IgemmSeg seg[kMaxClasses][kMaxSegs];
  int nseg[kMaxClasses];
  int nkb[kMaxClasses];          // total K blocks per class
  int8_t cls_py[kMaxClasses], cls_px[kMaxClasses];
  int out_sy, out_sx;            // output pixel = tile-grid pixel * s + (py, px)
  int MT;                        // 128-row accumulator tiles per CTA tile: 1, or 2 when BN <= 128
  int TW, TH, tw_shift;          // M tile = TH rows x TW cols, TW*TH == 128*MT, TW = 1 << tw_shift
  int tiles_x, tiles_y, n_tiles_n, BN;
  int gridW, gridH;              // valid extent of the tile grid (pixels)
  int Z1, Z0;                    // batch dims (z1 outer: image; z0 inner: parity class / head)
  int cls_from_z0;
  int a_n_z1, a_n_z0, a_k_z0;                    // A coords: n = z1*a_n_z1 + z0*a_n_z0 ; k0 = z0*a_k_z0
  int b_z_z1, b_z_z0, b_row_z0, b_k_z0;          // B coords
  long long out_z1, out_z0;                      // output element offsets per batch index
  void* out;
  int outW, outH;
  long long out_pix_stride;      // elements between consecutive pixels of a row (16-bit NHWC mode)
  long long out_row_stride;      // elements between rows
  int Cout;                      // valid output columns
  const float* bias;             // [Cout] or null
  const void* res1;              // same addressing as out, or null
  const void* res2;
  int flags;
  int stages;
  int total_tiles;
  // Optional GroupNorm statistics of the (rounded) output, produced by the epilogue: per image and
  // per CTA slot, per-channel sum / sum of squares, fp32, fixed summation order (deterministic):
  //   stats[((image * stats_slots + blockIdx.x) * Cout + c) * 2 + {0, 1}]
  // Pre-zeroed by the caller (CTAs that see no tile of an image do not write its slot).
  float* stats;
  int stats_slots;               // >= gridDim.x (igemm_grid())
  int stats_hw;                  // tokens mode (Z1 == 1, gridH == 1): pixels per image; else 0
  // Staged epilogue: each epilogue warp writes its 32 rows x 64 channels (16-bit) into a swizzled
  // shared-memory tile and issues one TMA store (full 128-byte lines, image-edge clipping by the
  // tensor map).  Needs Cout % 64 == 0, BN % 64 == 0, plain 16-bit NHWC output.  One map per class.
  int tma_store;
  CUtensorMap tmOut[kMaxClasses];   // (C, W, H, N) views of the output, box (64, min(TW,32), 32/min(TW,32), 1)
  // Residual through TMA (staged epilogue, res1 only): the same boxes of the residual tensor are LOADED into the
  // staging tile before the accumulator is read.  Row-per-thread global loads of a residual cost 32 L1 sector
  // look-ups per warp request (ncu r1k: 58 % tensor pipe with a residual vs 92 % without, same layer).
  int res_tma;
  int bias_slots;                // floats of shared memory holding the bias: 288 (one N tile, reloaded per tile) or, when the
                                 // layer has several N tiles and Cout is small enough, all of them (loaded once: bias_all)
  int bias_all;
  int epi_warps;                 // epilogue warps of the tap-streaming kernel: 8, or 4 where 8 would cost a pipeline stage (igemm_finalize)
  CUtensorMap tmRes[kMaxClasses];
  // Patch-resident main loop (igemm_patch.cu; 3x3 stride-1, one source, TW = 128, TH = MT = 1 or 2): per
  // 64-channel K chunk ONE (TH+2) x (TW+2) halo patch is loaded and all nine taps are fed from it by
  // row-offset descriptors (tap (dy,dx) starts (h+dy+1)*(TW+2) + dx+1 rows into the patch), instead of
  // nine shifted boxes.  Cuts the activation L2->SM traffic 9 -> 2.03 reads per element: the narrow-N
  // (Cout = 128) layers are bound by exactly that traffic (~42 B/clk/SM of unique data).
  int patch;
  int kc_count;                  // 64-channel K chunks per tap (packed weights are tap-major, kc_count*64 wide per tap)
  int kc_sc;                     // extra centre-tap-only chunks from tmPatch2 (fused 1x1 shortcut over the raw block input)
  int a_slot_bytes;              // bytes reserved per patch slot (2 slots), multiple of 1024
  CUtensorMap tmPatch;           // (C, W, H, N) view of the source, box (64, TW+2, TH+2, 1)
  CUtensorMap tmPatch2;          // same box over the shortcut source
  // GroupNorm(+SiLU) of the patch source applied in shared memory before the MMA reads it (patch mode only):
  // y = silu(x * scale + shift), (scale, shift) = gn_ss[(image * gn_C + channel) * 2 + {0, 1}] (gn_finalize's output).
  long long* trace;              // debug (gp_debug_patch_trace): CTA 0 stamps clock64() per K chunk; null = off
  const float* gn_ss;            // null: the source is used as it is
  int gn_C;                      // channels of the normalised tensor (= the patch source's)
  int gn_silu;
};

cudaError_t igemm_patch_launch(const IgemmParams& p, int grid, cudaStream_t stream);   // igemm_patch.cu
void igemm_patch_set_trace(long long* dev_buf);   // applies to subsequent launches (debug only)

int igemm_grid(const IgemmParams& p);   // CTAs that igemm_launch will use for p (after igemm_finalize)

// host helpers ----------------------------------------------------------------------------------
// Encode a 4-D NHWC view (C, W, H, N) with element strides (sW, sH, sN) and box (64, TW, TH, 1).
cudaError_t make_tmap_a(CUtensorMap* m, const void* base, int C, int W, int H, int N, long long sW,
                        long long sH, long long sN, int TW, int TH, bool bf16);
// Encode a 3-D K-major matrix view (K, rows, Z) with element strides (sRow, sZ) and box (64, BN, 1).
cudaError_t make_tmap_b(CUtensorMap* m, const void* base, long long K, long long rows, long long Z,
                        long long sRow, long long sZ, int BN, bool bf16);
// Fill tile counts / stage count and validate; returns nullptr or an error string.
const char* igemm_finalize(IgemmParams* p);
cudaError_t igemm_launch(const IgemmParams& p, cudaStream_t stream);
size_t igemm_smem_bytes(const IgemmParams& p);

}  // namespace gp
