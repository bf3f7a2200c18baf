// Internal C++ types of the engine: host weight store, packed device weights, the plan-time
// activation arena and op list builder.  The public surface is include/genpercept_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <functional>
#include <map>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/genpercept_b200.h"
#include "igemm.h"
#include "kernels.h"

namespace gp {

struct GpError : std::runtime_error {
  gp_status st;
  GpError(gp_status s, const std::string& m) : std::runtime_error(m), st(s) {}
};
#define GP_CUDA(call)                                                                           \
  do {                                                                                          \
    cudaError_t e__ = (call);                                                                   \
    if (e__ != cudaSuccess)                                                                     \
      throw ::gp::GpError(GP_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));    \
  } while (0)
#define GP_REQUIRE(cond, msg)                                             \
  do {                                                                    \
    if (!(cond)) throw ::gp::GpError(GP_ERR_INVALID, std::string(msg));   \
  } while (0)

struct HostT {
  std::vector<float> d;
  std::vector<int64_t> shape;
  int64_t numel() const { int64_t n = 1; for (auto s : shape) n *= s; return n; }
};

// K-major 16-bit matrix [nz][rows][ktot] (+ fp32 bias[rows]) on the device.
struct PackedW {
  uint16_t* w = nullptr;
  int rows = 0, ktot = 0, nz = 1;
  int planes = 1;            // 2 in the high-precision mode: every row is [ktot hi | ktot lo] (value = hi + lo)
  float* bias = nullptr;
};
struct NormW { float* gamma = nullptr; float* beta = nullptr; int C = 0; };
struct XattnW { float* U = nullptr; float* u0 = nullptr; float* M = nullptr; float* c0 = nullptr; int C = 0, heads = 0; };
struct DirectW { float* w = nullptr; float* bias = nullptr; int Cin = 0, Cout = 0, ks = 0; };

// value(co, c) = sum_t coef_t * p_t[co * sco_t + c * sc_t]
struct Term { const float* p; long long sco, sc; float coef; };
struct SegSpec { std::vector<Term> terms; int C; };

// dense 16-bit NHWC activation; `off` is a byte offset into the arena (or an absolute address
// when the builder's base is null).
// High-precision mode: planes == 2, a pixel holds [hi C | lo C] (two fp16 planes, value = hi + lo).
struct T4 {
  long long off = -1;
  int N = 0, H = 0, W = 0, C = 0;
  int planes = 1;
  size_t bytes() const { return (size_t)N * H * W * C * 2 * planes; }
  long long pixels() const { return (long long)N * H * W; }
  long long ps() const { return (long long)C * planes; }      // elements between consecutive pixels
};

class Arena {
 public:
  size_t alloc(size_t bytes);
  void release(size_t off);
  size_t high_water() const { return high_; }
 private:
  struct Blk { size_t off, size; bool free; };
  std::vector<Blk> blks_;
  size_t high_ = 0;
};

struct Op {
  std::string name;
  int stage = 0;
  int variant = 0;            // 0: always; 1 / 3: only when out_channels matches
  int launches = 1;
  int kind = 0;               // 1: tcgen05 implicit-GEMM launch, 0: anything else
  double flops = 0, bytes = 0;   // algorithmic work (SURVEY.md 8d): what the reference's op costs
  double flops_exec = -1;        // MMA work actually issued when it differs (upsample-fused convs run 4 of 9 taps); -1: = flops
  float usec = 0;
  std::function<cudaError_t(cudaStream_t)> run;
};

struct ConvArgs {
  std::vector<T4> srcs;       // concatenated sources of the main taps
  int ks = 3;
  int mode = 0;               // 0 s1, 1 s2 pad 1, 2 s2 pad (0,1,0,1), 3 nearest-2x then s1
  std::vector<T4> sc;         // raw sources of a fused 1x1 shortcut (extra K segments)
  const PackedW* w = nullptr;
  T4 out;                     // 16-bit NHWC destination (ignored when out_f32 != null)
  int cout_valid = -1;        // columns to store (default out.C)
  const T4* res1 = nullptr;
  const T4* res2 = nullptr;
  int flags = 0;
  float* out_f32 = nullptr;   // fp32 NCHW destination [N, cout_valid, Ho, Wo]
  int force_bn = 0;
  bool want_stats = false;    // let the epilogue emit GroupNorm partial sums of `out` (consumed by Builder::gn)
  // GroupNorm(+SiLU) over concat(srcs) in front of the convolution (norm1 / norm2 / conv_norm_out of the diffusers
  // blocks).  Where the patch-resident kernel applies, it is fused into the operand path (igemm_patch.cu); elsewhere
  // Builder::conv materialises the normalised tensor with Builder::gn and convolves that.
  const NormW* gn = nullptr;
  std::string gn_name;
  int gn_groups = 32;
  float gn_eps = 1e-6f;
  bool gn_silu = true;
};

class Builder {
 public:
  Builder(bool bf16, bool measuring, uint8_t* base, bool split = false);
  bool split() const { return split_; }
  T4 alloc(int N, int H, int W, int C);
  T4 external(const void* p, int N, int H, int W, int C) const;
  void release(const T4& t);
  void* ptr(const T4& t) const { return base_ + t.off; }
  size_t raw_alloc(size_t bytes) { return arena_.alloc(bytes); }
  void* raw_ptr(size_t off) const { return base_ + off; }

  void conv(const std::string& name, const ConvArgs& a);
  // generic batched GEMM pieces of attention; q/k/v views live inside `qk` / `l`
  void attention(const std::string& name, const T4& l, const PackedW& wqk, const PackedW& wv, const float* pv_bias,
                 int heads, const T4& out);
  void attention_qkv(const std::string& name, const void* q, const void* k, long long qk_cstride, const void* vT, int B,
                     int T, int heads, int d, const float* pv_bias, const T4& out, long long qk_lo = 0);
  void gn(const std::string& name, const std::vector<T4>& srcs, const NormW& nw, int groups, float eps, bool silu,
          const T4& out);
  // statistics -> per-(image, channel) scale / shift in gn_ss (the first half of gn(); the apply pass is the caller's)
  void gn_scale_shift(const std::string& name, const std::vector<T4>& srcs, const NormW& nw, int groups, float eps);
  void ln(const std::string& name, const T4& x, const NormW& nw, float eps, const T4& out);
  void xattn(const std::string& name, const T4& x, const XattnW& w, float eps, const T4& out);
  void geglu_op(const std::string& name, const T4& in, const T4& out);
  void relu_op(const std::string& name, const T4& in, const T4& out);
  void bilinear(const std::string& name, const T4& in, const T4& out);
  void direct(const std::string& name, const T4& in, int cin, const DirectW& w, const T4& out, int flags,
              float* out_f32, int up);
  void custom(const std::string& name, int launches, double bytes, std::function<cudaError_t(cudaStream_t)> fn);

  struct StatsInfo { size_t off; int slots; int C; };
  std::map<long long, StatsInfo> stats;   // live tensors (by arena offset) whose producer emitted GN partial sums
  int num_sms = 148;

  std::vector<Op> ops;
  int stage = 0;
  int variant = 0;
  bool bf16() const { return bf16_; }
  bool measuring() const { return measuring_; }
  size_t arena_bytes() const { return arena_.high_water(); }
  float* gn_sums = nullptr;   // [N][Cmax][2]
  float* gn_ss = nullptr;
  // When set, ops that write the final fp32 map (ConvArgs::out_f32 / direct(..., out_f32)) read their destination from
  // *out_slot at LAUNCH time, so gp_infer can point them at the caller's device buffer (no copy of the result).
  float** out_slot = nullptr;

 private:
  void push(const std::string& name, int launches, double flops, double bytes,
            std::function<cudaError_t(cudaStream_t)> fn);
  bool bf16_, measuring_, split_ = false;
  uint8_t* base_;
  Arena arena_;
};

// builder.cu: (BN, MT) of a stride-1 implicit-GEMM layer (default policy + the waves / L2-traffic model)
void tile_shape_for(int cout, double k_elems, bool tokens_mode, int images, int gw, int gh, int num_sms, int* bn, int* mt);

}  // namespace gp
