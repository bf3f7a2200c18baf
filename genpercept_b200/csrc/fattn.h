// Fused (FlashAttention-style) self-attention forward for head_dim 64 on tcgen05; see fattn.cu.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

namespace gp {

struct FattnParams {
  CUtensorMap tmQ;   // (C, T, B)  box (64, 128, 1) over the q part of the packed qk tensor
  CUtensorMap tmK;   // (C, T, B)  box (64, 128, 1) over the k part
  CUtensorMap tmV;   // (T, C, B)  box (64, 64, 1)  over V^T  [B][C][Tp]
  void* out;         // 16-bit [B, T, heads*64]
  long long out_b_stride;
  int out_row_stride;
  int T, heads, B, q_tiles;
  float scale_log2e;
  int bf16;
  long long* trace;   // debug: CTA 0 records clock64() at phase boundaries (null = off); see scripts/fattn_trace.py
};

void fattn_set_trace(long long* dev_buf);   // applies to subsequently built FattnParams (debug only)
long long* fattn_get_trace();

cudaError_t fattn_launch(const FattnParams& p, cudaStream_t stream);

}  // namespace gp
