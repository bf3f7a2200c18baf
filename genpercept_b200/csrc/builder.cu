// Plan-time arena and op-list builder: turns layer-level calls (conv, attention, norms ...) into
// fully parameterised kernel launches (tensor maps encoded once, at plan time).
#include <algorithm>
#include <cmath>
#include <cstring>

#include <cstdlib>

#include "engine.h"
#include "fattn.h"

namespace gp {

// ------------------------------------------------------------------------------------ Arena
size_t Arena::alloc(size_t bytes) {
  bytes = (bytes + 1023) & ~size_t(1023);
  if (bytes == 0) bytes = 1024;
  for (size_t i = 0; i < blks_.size(); ++i) {
    if (blks_[i].free && blks_[i].size >= bytes) {
      if (blks_[i].size > bytes) {
        Blk rest{blks_[i].off + bytes, blks_[i].size - bytes, true};
        blks_[i].size = bytes;
        blks_.insert(blks_.begin() + i + 1, rest);
      }
      blks_[i].free = false;
      return blks_[i].off;
    }
  }
  size_t off = blks_.empty() ? 0 : blks_.back().off + blks_.back().size;
  if (!blks_.empty() && blks_.back().free) {   // grow the trailing free block
    off = blks_.back().off;
    blks_.back().size = bytes;
    blks_.back().free = false;
  } else {
    blks_.push_back(Blk{off, bytes, false});
  }
  high_ = std::max(high_, off + bytes);
  return off;
}

void Arena::release(size_t off) {
  for (size_t i = 0; i < blks_.size(); ++i) {
    if (blks_[i].off == off && !blks_[i].free) {
      blks_[i].free = true;
      if (i + 1 < blks_.size() && blks_[i + 1].free) {
        blks_[i].size += blks_[i + 1].size;
        blks_.erase(blks_.begin() + i + 1);
      }
      if (i > 0 && blks_[i - 1].free) {
        blks_[i - 1].size += blks_[i].size;
        blks_.erase(blks_.begin() + i);
      }
      return;
    }
  }
  throw GpError(GP_ERR_STATE, "arena: release of unknown block");
}

// ------------------------------------------------------------------------------------ Builder
Builder::Builder(bool bf16, bool measuring, uint8_t* base, bool split)
    : bf16_(bf16), measuring_(measuring), split_(split), base_(base) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
    num_sms = n;
}
T4 Builder::alloc(int N, int H, int W, int C) {
  T4 t;
  t.N = N; t.H = H; t.W = W; t.C = C;
  t.planes = split_ ? 2 : 1;
  t.off = (long long)arena_.alloc(t.bytes());
  return t;
}
T4 Builder::external(const void* p, int N, int H, int W, int C) const {
  T4 t;
  t.N = N; t.H = H; t.W = W; t.C = C;
  t.planes = split_ ? 2 : 1;
  t.off = (long long)(reinterpret_cast<const uint8_t*>(p) - base_);
  return t;
}
void Builder::release(const T4& t) {
  auto it = stats.find(t.off);
  if (it != stats.end()) {
    arena_.release(it->second.off);
    stats.erase(it);
  }
  arena_.release((size_t)t.off);
}

void Builder::push(const std::string& name, int launches, double flops, double bytes,
                   std::function<cudaError_t(cudaStream_t)> fn) {
  Op o;
  o.name = name;
  o.stage = stage;
  o.variant = variant;
  o.launches = launches;
  o.flops = flops;
  o.bytes = bytes;
  o.run = std::move(fn);
  ops.push_back(std::move(o));
}
void Builder::custom(const std::string& name, int launches, double bytes, std::function<cudaError_t(cudaStream_t)> fn) {
  if (measuring_) return;
  push(name, launches, 0, bytes, std::move(fn));
}

static int ceil_div(int a, int b) { return (a + b - 1) / b; }
static int choose_bn(int cout, int force) {
  if (force) return force;
  const int c16 = ceil_div(cout, 16) * 16;
  if (c16 <= 256) return c16;
  // Cout = 320 / 640 (the SD-2.1 UNet's first two levels): an exact divisor (160) is not a multiple of 64 and forces the
  // direct epilogue (16-byte stores at a 2*Cout-byte stride, per-thread residual rows, no GroupNorm statistics).  A
  // multiple of 64 keeps the staged TMA-store epilogue even if the last N tile is partly empty: 640 = 5 x 128 exactly,
  // 320 -> 2 x 192 (64 idle columns).
  if ((cout % 64) == 0) {
    for (int bn : {256, 192, 128})
      if (cout % bn == 0) return bn;
    int best = 256, best_pad = 1 << 30;
    for (int bn : {256, 192, 128}) {
      const int pad = ceil_div(cout, bn) * bn - cout;
      if (pad < best_pad) { best_pad = pad; best = bn; }
    }
    return best;
  }
  for (int bn = 256; bn >= 128; bn -= 16)
    if (cout % bn == 0) return bn;
  const int n = ceil_div(cout, 256);
  return ceil_div(ceil_div(cout, n), 16) * 16;
}
// pick the TW x TH = `rows` (128 or 256) patch with the least padding waste (ties: wider rows)
static void choose_tile(int gw, int gh, int rows, int* tw, int* th, int* shift) {
  double best = 1e30;
  for (int s = 7; s >= 0; --s) {
    const int w = 1 << s, h = rows >> s;
    if (h > 256) continue;
    const double waste = (double)ceil_div(gw, w) * w * ceil_div(gh, h) * h / ((double)gw * gh);
    if (waste < best - 1e-9) { best = waste; *tw = w; *th = h; *shift = s; }
  }
}

// Tile shape (BN, MT) for the layers that do not fill the GPU (the UNet's deep levels at any batch, everything at batch
// 1).  Two bounds per candidate: the tensor time of the longest-running SM — ceil(tiles / SMs) waves of tiles whose
// duration scales with the MMA width (a 128 x 64 x 16 MMA is bound by its 6 KB of operand fetch: 48 cycles, not 32) — and
// the L2 -> SM operand traffic, tiles x K x (128 MT + BN) x 2 bytes at an effective 7 TB/s (what such few-tile layers sustain; r2n: the
// 2560 -> 1280 conv on 8 x 12 x 12 pixels moves 796 MB with BN = 256 and 1062 MB with BN = 128: 152 vs 210 us, although
// BN = 128 doubles the number of busy SMs; at batch 1 the same level has 2 M tiles, BN = 256 keeps 10 SMs busy for 61 us
// and BN = 64 runs 40 tiles in ~25 us).  A candidate replaces the default only for a predicted gain above 10 %, so
// every layer with many waves stays where choose_bn put it.
struct TileShape { int bn, mt; };
template <class MTilesFn>
static TileShape choose_tile_shape(int cout, double k_elems, int num_sms, TileShape dflt, MTilesFn mtiles_of) {
  if (cout % 64 != 0 || cout < 128) return dflt;
  auto cost = [&](TileShape t) {
    const double tiles = (double)mtiles_of(t.mt) * ceil_div(cout, t.bn);
    const double waves = std::ceil(tiles / num_sms);
    const double cyc_per_kb = 4.0 * t.mt * (t.bn == 64 ? 48.0 : t.bn / 2.0);
    const double t_mma = waves * ((k_elems / 64.0) * cyc_per_kb / 1.5e9 + 3e-6);     // + epilogue / pipeline fill per wave
    const double t_l2 = tiles * k_elems * (128.0 * t.mt + t.bn) * 2.0 / 7.0e12;
    return std::max(t_mma, t_l2);
  };
  TileShape best = dflt;
  const double c0 = cost(dflt);
  double best_cost = c0;
  for (int bn : {256, 192, 128, 64})
    for (int mt : {1, 2}) {
      if (mt == 2 && bn > 128) continue;
      const double c = cost(TileShape{bn, mt});
      if (c < 0.9 * c0 && c < best_cost) { best_cost = c; best = TileShape{bn, mt}; }
    }
  return best;
}
// Default (choose_bn, two M tiles when the N tile is narrow and the layer fills the GPU) + the model above, for a stride-1
// layer of `images` maps of gw x gh output pixels (tokens_mode: one row of images * gw * gh tokens).  Host-only; exported
// as gp_tile_shape so that the decision table is pinned by a CPU test.
void tile_shape_for(int cout, double k_elems, bool tokens_mode, int images, int gw, int gh, int num_sms, int* bn, int* mt) {
  const long long work_px = (long long)images * gw * gh;
  const int bn0 = choose_bn(cout, 0);
  const int mt0 = (bn0 <= 128 && work_px >= 256LL * 148) ? 2 : 1;
  auto mtiles_of = [&](int m) -> long long {
    if (tokens_mode) return (work_px + 128 * m - 1) / (128 * m);
    int tw = 128, th = m, sh = 7;
    choose_tile(gw, gh, 128 * m, &tw, &th, &sh);
    return (long long)images * ceil_div(gw, tw) * ceil_div(gh, th);
  };
  const TileShape ts = choose_tile_shape(cout, k_elems, num_sms, TileShape{bn0, mt0}, mtiles_of);
  *bn = ts.bn;
  *mt = ts.mt;
}

static void check_cuda(cudaError_t e, const std::string& what) {
  if (e != cudaSuccess) throw GpError(GP_ERR_CUDA, what + ": " + cudaGetErrorString(e));
}
static void finalize_or_throw(IgemmParams* p, const std::string& name) {
  const char* err = igemm_finalize(p);
  if (err) throw GpError(GP_ERR_INVALID, name + ": " + err);
}

// The patch-resident kernel with the GroupNorm transform in its operand path (igemm_patch.cu) takes a convolution when:
// 3x3 stride 1, ONE normalised source (channels % 64 == 0), at most one raw shortcut source, W % 128 == 0, and either the
// staged epilogue (Cout % 64 == 0) or an fp32 map as output.  Opt-in (GP_GN_FUSE=1): it removes the GroupNorm passes over
// the big maps (-8 ms, -38 GB of DRAM traffic per step) but its shared-memory traffic competes with the tensor core's own
// operand fetch, which already uses the SM's whole shared-memory bandwidth on these layers: no net gain (DESIGN.md 4.1).
static bool gn_fusable(const ConvArgs& a, bool split) {
  const char* on = std::getenv("GP_GN_FUSE");        // read at plan time (tests toggle it)
  const bool off = on == nullptr || on[0] == '0';
  if (off || split || a.mode != 0 || a.ks != 3 || a.srcs.size() != 1 || a.sc.size() > 1) return false;
  const T4& s = a.srcs[0];
  if ((s.W % 128) || (s.C % 64) || (!a.sc.empty() && (a.sc[0].C % 64))) return false;
  const int Cout = a.cout_valid > 0 ? a.cout_valid : a.out.C;
  if (!a.out_f32 && (Cout != a.out.C || (Cout % 64))) return false;
  if (a.flags & IG_GEGLU) return false;
  return true;
}

void Builder::conv(const std::string& name, const ConvArgs& a) {
  GP_REQUIRE(!a.srcs.empty() && a.w != nullptr, name + ": bad conv args");
  const bool gn_fused = a.gn != nullptr && gn_fusable(a, split_);
  if (a.gn != nullptr && !gn_fused) {      // materialise GroupNorm(+SiLU)(concat(srcs)), then the plain convolution
    int ctot = 0;
    for (auto& s : a.srcs) ctot += s.C;
    T4 tmp = alloc(a.srcs[0].N, a.srcs[0].H, a.srcs[0].W, ctot);
    gn(a.gn_name, a.srcs, *a.gn, a.gn_groups, a.gn_eps, a.gn_silu, tmp);
    ConvArgs b = a;
    b.gn = nullptr;
    b.srcs = {tmp};
    conv(name, b);
    release(tmp);
    return;
  }
  if (gn_fused) gn_scale_shift(a.gn_name, a.srcs, *a.gn, a.gn_groups, a.gn_eps);
  const T4& s0 = a.srcs[0];
  const int N = s0.N, H = s0.H, W = s0.W;
  int Ho = H, Wo = W;
  if (a.mode == 1) { Ho = (H + 2 - 3) / 2 + 1; Wo = (W + 2 - 3) / 2 + 1; }
  if (a.mode == 2) { Ho = (H + 1 - 3) / 2 + 1; Wo = (W + 1 - 3) / 2 + 1; }
  if (a.mode == 3) { Ho = 2 * H; Wo = 2 * W; }
  const int PL = split_ ? 2 : 1;
  const int out_cl = a.out_f32 ? 0 : a.out.C;   // logical channels of the 16-bit output ...
  const int out_c = out_cl * PL;                // ... and its pixel stride in elements
  GP_REQUIRE(a.w->planes == PL, name + ": packed weights do not match the engine's precision mode");
  const int Cout = a.cout_valid > 0 ? a.cout_valid : a.out.C;
  int cin_total = 0;
  for (auto& s : a.srcs) cin_total += s.C;
  double flops = 2.0 * N * Ho * Wo * (double)Cout * cin_total * a.ks * a.ks;
  for (auto& s : a.sc) flops += 2.0 * N * Ho * Wo * (double)Cout * s.C;
  double bytes = (double)N * Ho * Wo * Cout * (a.out_f32 ? 4 : 2) + (double)a.w->rows * a.w->ktot * a.w->nz * 2;
  for (auto& s : a.srcs) bytes += (double)s.bytes();
  for (auto& s : a.sc) bytes += (double)s.bytes();
  if (a.res1) bytes += (double)a.res1->bytes();
  if (a.res2) bytes += (double)a.res2->bytes();
  if (!a.out_f32) GP_REQUIRE(a.out.N == N && a.out.H == Ho && a.out.W == Wo, name + ": output shape mismatch");
  // GroupNorm partial sums from the epilogue: same decision (and arena allocation) in both passes
  const bool tokens_mode = (a.ks == 1 && a.mode == 0 && a.sc.empty() && a.srcs.size() == 1 && !a.out_f32);
  const long long work_px = tokens_mode ? (long long)N * H * W
                                        : (long long)(a.mode == 3 ? W : Wo) * (a.mode == 3 ? H : Ho) * N * (a.mode == 3 ? 4 : 1);
  int bn_pre = choose_bn(Cout, a.force_bn);
  int mt_pre = gn_fused ? ((bn_pre <= 128 && (H % 2) == 0) ? 2 : 1) : (bn_pre <= 128 && work_px >= 256LL * 148) ? 2 : 1;
  if (!a.force_bn && !(a.flags & IG_GEGLU) && !gn_fused) {
    const double k_elems = flops / (2.0 * N * Ho * Wo * (double)Cout) * (a.mode == 3 ? 4.0 / 9.0 : 1.0);
    tile_shape_for(Cout, k_elems, tokens_mode, N * (a.mode == 3 ? 4 : 1), (a.mode == 3) ? W : Wo, (a.mode == 3) ? H : Ho, num_sms,
                   &bn_pre, &mt_pre);
  }
  const bool is_geglu = (a.flags & IG_GEGLU) != 0;
  // GEGLU keeps the direct epilogue: a staged GEGLU epilogue measured slower than the direct stores (r1g, r2p)
  const bool staged = !a.out_f32 && !is_geglu && Cout == a.out.C && (Cout % 64) == 0 && (bn_pre % 64) == 0;
  const bool patch_eligible = gn_fused || (staged && a.mode == 0 && a.ks == 3 && a.srcs.size() == 1 && a.sc.empty() && mt_pre == 2 &&
                                           (W % 128) == 0 && (H % 2) == 0 && !split_);
  bool emit_stats = a.want_stats && staged && Cout <= 512 && !split_;
  if (emit_stats && tokens_mode && ((long long)H * W) % (128 * mt_pre) != 0) emit_stats = false;
  size_t stats_off = 0;
  const size_t stats_bytes = (size_t)N * num_sms * Cout * 2 * sizeof(float);
  if (emit_stats) {
    GP_REQUIRE(stats.find(a.out.off) == stats.end(), name + ": output already has statistics");
    stats_off = arena_.alloc(stats_bytes);
    stats[a.out.off] = StatsInfo{stats_off, num_sms, Cout};
  }
  if (measuring_) return;

  IgemmParams p;
  std::memset(&p, 0, sizeof(p));
  p.flags = a.flags | (bf16_ ? IG_BF16 : 0) | (a.out_f32 ? IG_OUT_F32_NCHW : 0);
  p.bias = a.w->bias;
  p.res1 = a.res1 ? ptr(*a.res1) : nullptr;
  p.res2 = a.res2 ? ptr(*a.res2) : nullptr;
  p.out = a.out_f32 ? (void*)a.out_f32 : ptr(a.out);
  p.Cout = Cout;
  p.BN = bn_pre;
  p.Z1 = 1; p.Z0 = 1;
  p.out_sy = p.out_sx = 1;
  const bool tokens = tokens_mode;
  if (tokens) {
    const long long ntok = (long long)N * H * W;
    GP_REQUIRE(ntok < (1LL << 31), name + ": too many tokens");
    p.gridW = (int)ntok; p.gridH = 1;
    p.MT = mt_pre;
    p.TW = 128 * p.MT; p.TH = 1; p.tw_shift = p.MT == 2 ? 8 : 7;
    p.nseg[0] = 1;
    p.seg[0][0] = IgemmSeg{0, 0, 0, (uint16_t)ceil_div(s0.C, 64)};
    p.outW = (int)ntok; p.outH = 1;
    p.out_pix_stride = out_c; p.out_row_stride = 0;
    check_cuda(make_tmap_a(&p.tmA[0], ptr(s0), s0.C, (int)ntok, 1, 1, s0.ps(), ntok * s0.ps(), ntok * s0.ps(), p.TW, 1, bf16_),
               name + ": tmap A");
    for (int i = 1; i < 4; ++i) p.tmA[i] = p.tmA[0];
    if (split_) {
      check_cuda(make_tmap_a(&p.tmA[4], reinterpret_cast<const uint16_t*>(ptr(s0)) + s0.C, s0.C, (int)ntok, 1, 1, s0.ps(),
                             ntok * s0.ps(), ntok * s0.ps(), p.TW, 1, bf16_), name + ": tmap A lo");
      for (int i = 5; i < 8; ++i) p.tmA[i] = p.tmA[4];
    }
  } else {
    p.Z1 = N;
    p.a_n_z1 = 1;
    p.outW = Wo; p.outH = Ho;
    p.out_pix_stride = out_c;
    p.out_row_stride = (long long)Wo * out_c;
    p.out_z1 = (long long)Ho * Wo * out_c;
    p.gridW = (a.mode == 3) ? W : Wo;
    p.gridH = (a.mode == 3) ? H : Ho;
    // two accumulator tiles per CTA when the N tile is narrow and there is enough work to fill the GPU
    p.MT = mt_pre;
    if (patch_eligible) { p.TW = 128; p.TH = p.MT; p.tw_shift = 7; }
    else choose_tile(p.gridW, p.gridH, 128 * p.MT, &p.TW, &p.TH, &p.tw_shift);
    int nmap = 0;
    if (a.mode == 0 || a.mode == 3) {
      GP_REQUIRE(a.srcs.size() + a.sc.size() <= 4, name + ": too many sources");
      auto add_src = [&](const T4& s) {
        check_cuda(make_tmap_a(&p.tmA[nmap], ptr(s), s.C, W, H, N, s.ps(), (long long)W * s.ps(),
                               (long long)H * W * s.ps(), p.TW, p.TH, bf16_), name + ": tmap A");
        if (split_)
          check_cuda(make_tmap_a(&p.tmA[nmap + 4], reinterpret_cast<const uint16_t*>(ptr(s)) + s.C, s.C, W, H, N, s.ps(),
                                 (long long)W * s.ps(), (long long)H * W * s.ps(), p.TW, p.TH, bf16_), name + ": tmap A lo");
        ++nmap;
      };
      for (auto& s : a.srcs) {
        GP_REQUIRE(s.N == N && s.H == H && s.W == W, name + ": source shape mismatch");
        add_src(s);
      }
      for (auto& s : a.sc) {
        GP_REQUIRE(s.N == N && s.H == H && s.W == W && a.mode == 0, name + ": shortcut shape mismatch");
        add_src(s);
      }
    } else {
      GP_REQUIRE(a.srcs.size() == 1 && a.sc.empty() && H >= 2 && W >= 2, name + ": stride-2 needs one source");
      for (int hp = 0; hp < 2; ++hp)
        for (int wp = 0; wp < 2; ++wp) {
          const uint8_t* b = reinterpret_cast<const uint8_t*>(ptr(s0)) + ((long long)hp * W + wp) * s0.ps() * 2;
          check_cuda(make_tmap_a(&p.tmA[hp * 2 + wp], b, s0.C, (W - wp + 1) / 2, (H - hp + 1) / 2, N, 2LL * s0.ps(),
                                 2LL * W * s0.ps(), (long long)H * W * s0.ps(), p.TW, p.TH, bf16_), name + ": tmap A");
          if (split_)
            check_cuda(make_tmap_a(&p.tmA[4 + hp * 2 + wp], b + s0.C * 2, s0.C, (W - wp + 1) / 2, (H - hp + 1) / 2, N, 2LL * s0.ps(),
                                   2LL * W * s0.ps(), (long long)H * W * s0.ps(), p.TW, p.TH, bf16_), name + ": tmap A lo");
        }
      nmap = 4;
    }
    for (int i = nmap; i < 4; ++i) { p.tmA[i] = p.tmA[0]; if (split_) p.tmA[i + 4] = p.tmA[4]; }
    if (a.mode == 0) {
      int ns = 0;
      const int half = a.ks / 2;
      for (int r = 0; r < a.ks; ++r)
        for (int s = 0; s < a.ks; ++s)
          for (size_t i = 0; i < a.srcs.size(); ++i)
            p.seg[0][ns++] = IgemmSeg{(int8_t)i, (int8_t)(r - half), (int8_t)(s - half), (uint16_t)ceil_div(a.srcs[i].C, 64)};
      for (size_t j = 0; j < a.sc.size(); ++j)
        p.seg[0][ns++] = IgemmSeg{(int8_t)(a.srcs.size() + j), 0, 0, (uint16_t)ceil_div(a.sc[j].C, 64)};
      GP_REQUIRE(ns <= kMaxSegs, name + ": too many K segments");
      p.nseg[0] = ns;
    } else if (a.mode == 1 || a.mode == 2) {
      const int pad = (a.mode == 1) ? 1 : 0;
      int ns = 0;
      for (int r = 0; r < 3; ++r)
        for (int s = 0; s < 3; ++s) {
          const int ty = r - pad, tx = s - pad;
          const int hp = ((ty % 2) + 2) % 2, wp = ((tx % 2) + 2) % 2;
          p.seg[0][ns++] = IgemmSeg{(int8_t)(hp * 2 + wp), (int8_t)((ty - hp) / 2), (int8_t)((tx - wp) / 2),
                                    (uint16_t)ceil_div(s0.C, 64)};
        }
      p.nseg[0] = ns;
    } else {
      p.Z0 = 4;
      p.cls_from_z0 = 1;
      p.b_z_z0 = 1;
      p.out_sy = p.out_sx = 2;
      for (int c = 0; c < 4; ++c) {
        const int py = c >> 1, px = c & 1;
        p.cls_py[c] = (int8_t)py; p.cls_px[c] = (int8_t)px;
        int ns = 0;
        for (int aa = 0; aa < 2; ++aa)
          for (int bb = 0; bb < 2; ++bb)
            p.seg[c][ns++] = IgemmSeg{0, (int8_t)(py - 1 + aa), (int8_t)(px - 1 + bb), (uint16_t)ceil_div(s0.C, 64)};
        p.nseg[c] = ns;
      }
    }
  }
  check_cuda(make_tmap_b(&p.tmB, a.w->w, (long long)a.w->ktot * PL, a.w->rows, a.w->nz, (long long)a.w->ktot * PL,
                         (long long)a.w->rows * a.w->ktot * PL, p.BN, bf16_), name + ": tmap B");
  if (split_) {   // three passes: hi*hi, lo*hi, hi*lo (the weights' lo plane follows the hi plane along K)
    p.npass = 3;
    p.pass_amap[0] = 0; p.pass_amap[1] = 4; p.pass_amap[2] = 0;
    p.pass_bk[0] = 0; p.pass_bk[1] = 0; p.pass_bk[2] = a.w->ktot;
    if (!a.out_f32) p.out_lo = out_cl;
  }
  if (staged) {   // output tensor maps for the TMA-store epilogue (one per parity class)
    p.tma_store = 1;
    const int bw = p.TW < 32 ? p.TW : 32, bh = 32 / bw;
    for (int pl = 0; pl < PL; ++pl) {          // plane 0: tmOut, plane 1 (high-precision lo): tmOutLo
      CUtensorMap* tmo = pl == 0 ? p.tmOut : p.tmOutLo;
      const uint8_t* obase = reinterpret_cast<const uint8_t*>(ptr(a.out)) + (size_t)pl * out_cl * 2;
      if (tokens) {
        const long long ntok = (long long)N * H * W;
        check_cuda(make_tmap_a(&tmo[0], obase, out_cl, (int)ntok, 1, 1, out_c, ntok * out_c, ntok * out_c, bw, bh, bf16_),
                   name + ": tmap out");
        for (int i = 1; i < 4; ++i) tmo[i] = tmo[0];
      } else if (a.mode == 3) {
        for (int c = 0; c < 4; ++c) {
          const int py = c >> 1, px = c & 1;
          const uint8_t* ob = obase + ((long long)py * Wo + px) * out_c * 2;
          check_cuda(make_tmap_a(&tmo[c], ob, out_cl, W, H, N, 2LL * out_c, 2LL * Wo * out_c, (long long)Ho * Wo * out_c, bw, bh,
                                 bf16_), name + ": tmap out");
        }
      } else {
        check_cuda(make_tmap_a(&tmo[0], obase, out_cl, Wo, Ho, N, out_c, (long long)Wo * out_c, (long long)Ho * Wo * out_c,
                               bw, bh, bf16_), name + ": tmap out");
        for (int i = 1; i < 4; ++i) tmo[i] = tmo[0];
      }
    }
    // the residual has the output's shape and addressing: same maps over its base
    if (a.res1 && !a.res2 && !split_) {
      p.res_tma = 1;
      const void* rb = ptr(*a.res1);
      if (tokens) {
        const long long ntok = (long long)N * H * W;
        check_cuda(make_tmap_a(&p.tmRes[0], rb, out_c, (int)ntok, 1, 1, out_c, ntok * out_c, ntok * out_c, bw, bh, bf16_),
                   name + ": tmap res");
        for (int i = 1; i < 4; ++i) p.tmRes[i] = p.tmRes[0];
      } else if (a.mode == 3) {
        for (int c = 0; c < 4; ++c) {
          const int py = c >> 1, px = c & 1;
          const uint8_t* ob = reinterpret_cast<const uint8_t*>(rb) + ((long long)py * Wo + px) * out_c * 2;
          check_cuda(make_tmap_a(&p.tmRes[c], ob, out_c, W, H, N, 2LL * out_c, 2LL * Wo * out_c, (long long)Ho * Wo * out_c, bw, bh,
                                 bf16_), name + ": tmap res");
        }
      } else {
        check_cuda(make_tmap_a(&p.tmRes[0], rb, out_c, Wo, Ho, N, out_c, (long long)Wo * out_c, (long long)Ho * Wo * out_c,
                               bw, bh, bf16_), name + ": tmap res");
        for (int i = 1; i < 4; ++i) p.tmRes[i] = p.tmRes[0];
      }
    }
  }
  // patch-resident main loop for the wide-image, narrow-N 3x3 layers
  if (patch_eligible) {
    GP_REQUIRE(p.TW == 128 && p.TH == p.MT, name + ": patch tile");
    p.patch = 1;
    p.kc_count = ceil_div(s0.C, 64);
    check_cuda(make_tmap_a(&p.tmPatch, ptr(s0), s0.C, W, H, N, s0.C, (long long)W * s0.C, (long long)H * W * s0.C,
                           p.TW + 2, p.TH + 2, bf16_), name + ": tmap patch");
    p.tmPatch2 = p.tmPatch;
    if (!a.sc.empty()) {
      const T4& x = a.sc[0];
      p.kc_sc = ceil_div(x.C, 64);
      check_cuda(make_tmap_a(&p.tmPatch2, ptr(x), x.C, W, H, N, x.C, (long long)W * x.C, (long long)H * W * x.C,
                             p.TW + 2, p.TH + 2, bf16_), name + ": tmap patch (shortcut)");
    }
    if (gn_fused) {
      p.gn_ss = gn_ss;
      p.gn_C = s0.C;
      p.gn_silu = a.gn_silu ? 1 : 0;
    }
  }
  if (emit_stats) {
    p.stats = reinterpret_cast<float*>(raw_ptr(stats_off));
    p.stats_slots = num_sms;
    p.stats_hw = tokens ? H * W : 0;
  }
  finalize_or_throw(&p, name);
  GP_REQUIRE(p.MT == mt_pre && p.BN == bn_pre, name + ": tile pre-selection disagrees with the plan");
  const int ncls = p.cls_from_z0 ? p.Z0 : 1;
  for (int c = 0; c < ncls; ++c)
    GP_REQUIRE(p.nkb[c] * 64 == a.w->ktot, name + ": packed K (" + std::to_string(a.w->ktot) + ") != planned K (" +
                                              std::to_string(p.nkb[c] * 64) + ")");
  GP_REQUIRE(a.w->rows >= Cout || a.w->rows == Cout, name + ": packed rows < Cout");
  if (emit_stats) {
    float* sp = p.stats;
    push(name, 2, flops, bytes, [p, sp, stats_bytes](cudaStream_t s) {
      cudaError_t e = cudaMemsetAsync(sp, 0, stats_bytes, s);
      if (e != cudaSuccess) return e;
      return igemm_launch(p, s);
    });
  } else if (a.out_f32 && out_slot) {
    float** slot = out_slot;
    push(name, 1, flops, bytes, [p, slot](cudaStream_t s) {
      IgemmParams q = p;
      q.out = *slot;
      return igemm_launch(q, s);
    });
  } else {
    push(name, 1, flops, bytes, [p](cudaStream_t s) { return igemm_launch(p, s); });
  }
  ops.back().kind = 1;
  if (a.mode == 3) ops.back().flops_exec = flops * 4.0 / 9.0;      // four 2x2 parity convs instead of a 3x3 on the 2x grid
}

void Builder::attention_qkv(const std::string& name, const void* q, const void* k, long long cs, const void* vT, int B,
                            int T, int heads, int d, const float* pv_bias, const T4& out, long long qk_lo) {
  // High-precision mode: q / k carry their lo planes `qk_lo` elements further (same pixel stride cs), V^T rows are
  // [hi Tp | lo Tp], S / P rows likewise; the three GEMM passes of IgemmParams::npass do hi*hi + lo*hi + hi*lo.
  const int Tp = ceil_div(T, 8) * 8;
  const int C = heads * d;
  const int PL = split_ ? 2 : 1;
  const long long TpP = (long long)Tp * PL;   // physical row pitch of S and V^T
  auto set_passes = [&](IgemmParams& p) {
    if (!split_) return;
    p.npass = 3;
    p.pass_amap[0] = 0; p.pass_amap[1] = 4; p.pass_amap[2] = 0;
    p.pass_bmap[0] = 0; p.pass_bmap[1] = 0; p.pass_bmap[2] = 1;
  };
  if (d == 64 && !split_) {   // fused tcgen05 flash-attention kernel (S and P stay on chip)
    if (measuring_) return;
    FattnParams p;
    std::memset(&p, 0, sizeof(p));
    p.out = ptr(out);
    p.out_b_stride = (long long)T * C;
    p.out_row_stride = C;
    p.T = T; p.heads = heads; p.B = B; p.q_tiles = ceil_div(T, 128);
    p.scale_log2e = 1.4426950408889634f;
    p.bf16 = bf16_ ? 1 : 0;
    p.trace = fattn_get_trace();
    check_cuda(make_tmap_b(&p.tmQ, q, C, T, B, cs, (long long)T * cs, 128, bf16_), name + ": tmap Q");
    check_cuda(make_tmap_b(&p.tmK, k, C, T, B, cs, (long long)T * cs, 128, bf16_), name + ": tmap K");
    check_cuda(make_tmap_b(&p.tmV, vT, T, C, B, Tp, (long long)C * Tp, 64, bf16_), name + ": tmap Vt");
    push(name + ".fattn", 1, 4.0 * B * heads * (double)T * T * d, 4.0 * B * T * C * 2,
         [p](cudaStream_t s) { return fattn_launch(p, s); });
    ops.back().kind = 2;
    return;
  }
  const size_t s_bytes = (size_t)B * heads * T * TpP * 2;
  const size_t s_off = arena_.alloc(s_bytes);
  if (!measuring_) {
    void* S = raw_ptr(s_off);
    {  // S = Q K^T  (softmax scale is folded into Wq)
      IgemmParams p;
      std::memset(&p, 0, sizeof(p));
      p.flags = bf16_ ? IG_BF16 : 0;
      p.gridW = T; p.gridH = 1; p.TW = 128; p.TH = 1; p.tw_shift = 7;
      p.Z1 = B; p.Z0 = heads;
      p.a_n_z1 = 1; p.a_k_z0 = d;
      p.b_z_z1 = 1; p.b_k_z0 = d;
      p.nseg[0] = 1;
      p.seg[0][0] = IgemmSeg{0, 0, 0, (uint16_t)ceil_div(d, 64)};
      p.out = S; p.outW = T; p.outH = 1;
      p.out_pix_stride = TpP; p.out_row_stride = 0;
      p.out_z1 = (long long)heads * T * TpP; p.out_z0 = (long long)T * TpP;
      p.out_sy = p.out_sx = 1;
      p.Cout = T;
      p.BN = choose_bn(T, 0);
      check_cuda(make_tmap_a(&p.tmA[0], q, C, T, 1, B, cs, (long long)T * cs, (long long)T * cs, 128, 1, bf16_), name + ": tmap Q");
      for (int i = 1; i < 4; ++i) p.tmA[i] = p.tmA[0];
      check_cuda(make_tmap_b(&p.tmB, k, C, T, B, cs, (long long)T * cs, p.BN, bf16_), name + ": tmap K");
      if (split_) {
        const uint16_t* ql = reinterpret_cast<const uint16_t*>(q) + qk_lo;
        const uint16_t* kl = reinterpret_cast<const uint16_t*>(k) + qk_lo;
        check_cuda(make_tmap_a(&p.tmA[4], ql, C, T, 1, B, cs, (long long)T * cs, (long long)T * cs, 128, 1, bf16_), name + ": tmap Q lo");
        for (int i = 5; i < 8; ++i) p.tmA[i] = p.tmA[4];
        check_cuda(make_tmap_b(&p.tmB2, kl, C, T, B, cs, (long long)T * cs, p.BN, bf16_), name + ": tmap K lo");
        p.out_lo = Tp;
        set_passes(p);
      }
      finalize_or_throw(&p, name + ".qk");
      push(name + ".qk", 1, 2.0 * B * heads * (double)T * T * d, (double)s_bytes + 2.0 * B * T * C * 2,
           [p](cudaStream_t s) { return igemm_launch(p, s); });
      ops.back().kind = 1;
    }
    {
      const long long rows = (long long)B * heads * T;
      const bool bf = bf16_;
      const bool sp = split_;
      push(name + ".softmax", 1, 0, 2.0 * s_bytes, [S, rows, T, Tp, bf, sp](cudaStream_t s) { return softmax_rows(S, rows, T, Tp, bf, s, sp); });
    }
    {  // O = P V
      IgemmParams p;
      std::memset(&p, 0, sizeof(p));
      p.flags = bf16_ ? IG_BF16 : 0;
      p.gridW = T; p.gridH = 1; p.TW = 128; p.TH = 1; p.tw_shift = 7;
      p.Z1 = B; p.Z0 = heads;
      p.a_n_z1 = heads; p.a_n_z0 = 1;
      p.b_z_z1 = 1; p.b_row_z0 = d;
      p.nseg[0] = 1;
      p.seg[0][0] = IgemmSeg{0, 0, 0, (uint16_t)ceil_div(T, 64)};
      p.out = ptr(out); p.outW = T; p.outH = 1;
      p.out_pix_stride = out.ps(); p.out_row_stride = 0;
      p.out_z1 = (long long)T * out.ps(); p.out_z0 = d;
      p.out_sy = p.out_sx = 1;
      p.Cout = d;
      p.bias = pv_bias;
      p.BN = choose_bn(d, 0);
      check_cuda(make_tmap_a(&p.tmA[0], S, T, T, 1, B * heads, TpP, (long long)T * TpP, (long long)T * TpP, 128, 1, bf16_), name + ": tmap P");
      for (int i = 1; i < 4; ++i) p.tmA[i] = p.tmA[0];
      check_cuda(make_tmap_b(&p.tmB, vT, T, C, B, TpP, (long long)C * TpP, p.BN, bf16_), name + ": tmap Vt");
      if (split_) {
        check_cuda(make_tmap_a(&p.tmA[4], reinterpret_cast<const uint16_t*>(S) + Tp, T, T, 1, B * heads, TpP, (long long)T * TpP,
                               (long long)T * TpP, 128, 1, bf16_), name + ": tmap P lo");
        for (int i = 5; i < 8; ++i) p.tmA[i] = p.tmA[4];
        check_cuda(make_tmap_b(&p.tmB2, reinterpret_cast<const uint16_t*>(vT) + Tp, T, C, B, TpP, (long long)C * TpP, p.BN, bf16_),
                   name + ": tmap Vt lo");
        p.out_lo = out.C;
        set_passes(p);
      }
      finalize_or_throw(&p, name + ".pv");
      push(name + ".pv", 1, 2.0 * B * heads * (double)T * T * d, (double)s_bytes + 2.0 * B * T * C * 2,
           [p](cudaStream_t s) { return igemm_launch(p, s); });
      ops.back().kind = 1;
    }
  }
  arena_.release(s_off);
}

void Builder::attention(const std::string& name, const T4& l, const PackedW& wqk, const PackedW& wv,
                        const float* pv_bias, int heads, const T4& out) {
  const int B = l.N, T = l.H * l.W, C = l.C, d = C / heads;
  const int Tp = ceil_div(T, 8) * 8;
  T4 qk = alloc(B, l.H, l.W, 2 * C);
  {
    ConvArgs a;
    a.srcs = {l}; a.ks = 1; a.w = &wqk; a.out = qk;
    conv(name + ".to_qk", a);
  }
  const int PL = split_ ? 2 : 1;
  const long long TpP = (long long)Tp * PL;
  GP_REQUIRE(wv.planes == PL && wqk.planes == PL, name + ": packed weights do not match the engine's precision mode");
  const size_t vt_bytes = (size_t)B * C * TpP * 2;
  const size_t vt_off = arena_.alloc(vt_bytes);
  if (!measuring_) {   // V^T[b] = Wv . l[b]^T : A = weights (rows = channels), B = tokens
    IgemmParams p;
    std::memset(&p, 0, sizeof(p));
    p.flags = bf16_ ? IG_BF16 : 0;
    p.gridW = C; p.gridH = 1; p.TW = 128; p.TH = 1; p.tw_shift = 7;
    p.Z1 = B; p.Z0 = 1;
    p.b_z_z1 = 1;
    p.nseg[0] = 1;
    p.seg[0][0] = IgemmSeg{0, 0, 0, (uint16_t)(wv.ktot / 64)};
    p.out = raw_ptr(vt_off); p.outW = C; p.outH = 1;
    p.out_pix_stride = TpP; p.out_row_stride = 0;
    p.out_z1 = (long long)C * TpP;
    p.out_sy = p.out_sx = 1;
    p.Cout = T;
    p.BN = choose_bn(T, 0);
    const long long wrow = (long long)wv.ktot * PL;
    check_cuda(make_tmap_a(&p.tmA[0], wv.w, wv.ktot, C, 1, 1, wrow, (long long)C * wrow, (long long)C * wrow,
                           128, 1, bf16_), name + ": tmap Wv");
    for (int i = 1; i < 4; ++i) p.tmA[i] = p.tmA[0];
    check_cuda(make_tmap_b(&p.tmB, ptr(l), C, T, B, l.ps(), (long long)T * l.ps(), p.BN, bf16_), name + ": tmap l");
    if (split_) {
      check_cuda(make_tmap_a(&p.tmA[4], wv.w + wv.ktot, wv.ktot, C, 1, 1, wrow, (long long)C * wrow, (long long)C * wrow,
                             128, 1, bf16_), name + ": tmap Wv lo");
      for (int i = 5; i < 8; ++i) p.tmA[i] = p.tmA[4];
      check_cuda(make_tmap_b(&p.tmB2, reinterpret_cast<const uint16_t*>(ptr(l)) + C, C, T, B, l.ps(), (long long)T * l.ps(), p.BN, bf16_),
                 name + ": tmap l lo");
      p.npass = 3;
      p.pass_amap[0] = 0; p.pass_amap[1] = 4; p.pass_amap[2] = 0;
      p.pass_bmap[0] = 0; p.pass_bmap[1] = 0; p.pass_bmap[2] = 1;
      p.out_lo = Tp;
    }
    finalize_or_throw(&p, name + ".to_vT");
    push(name + ".to_vT", 1, 2.0 * B * (double)T * C * C, (double)vt_bytes + (double)l.bytes(),
         [p](cudaStream_t s) { return igemm_launch(p, s); });
    ops.back().kind = 1;
  }
  const uint16_t* qp = measuring_ ? nullptr : reinterpret_cast<const uint16_t*>(ptr(qk));
  attention_qkv(name, qp, qp ? qp + C : nullptr, qk.ps(), measuring_ ? nullptr : raw_ptr(vt_off), B, T, heads, d, pv_bias, out,
                split_ ? 2LL * C : 0);
  arena_.release(vt_off);
  release(qk);
}

void Builder::gn_scale_shift(const std::string& name, const std::vector<T4>& srcs, const NormW& nw, int groups, float eps) {
  int ctot = 0;
  for (auto& s : srcs) ctot += s.C;
  GP_REQUIRE(nw.C == ctot && ctot % groups == 0 && srcs.size() <= 2 && !srcs.empty(), name + ": GroupNorm channel mismatch");
  const int N = srcs[0].N;
  const long long HW = (long long)srcs[0].H * srcs[0].W;
  const int chunks = gn_chunks(N, HW);
  std::vector<size_t> own(srcs.size(), (size_t)-1);
  std::vector<GnSrc> gs(srcs.size());
  for (size_t i = 0; i < srcs.size(); ++i) {
    auto it = stats.find(srcs[i].off);
    if (it != stats.end() && it->second.C == srcs[i].C) {
      gs[i] = GnSrc{measuring_ ? nullptr : reinterpret_cast<const float*>(raw_ptr(it->second.off)), it->second.slots, srcs[i].C};
    } else {
      own[i] = arena_.alloc((size_t)N * chunks * srcs[i].C * 2 * sizeof(float));
      gs[i] = GnSrc{measuring_ ? nullptr : reinterpret_cast<const float*>(raw_ptr(own[i])), chunks, srcs[i].C};
    }
  }
  if (!measuring_) {
    float* ss = gn_ss;
    const bool bf = bf16_, sp = split_;
    std::vector<const void*> xs;
    std::vector<int> cs;
    std::vector<bool> need;
    int launches = 1;
    double bytes = 0;
    for (size_t i = 0; i < srcs.size(); ++i) {
      xs.push_back(ptr(srcs[i]));
      cs.push_back(srcs[i].C);
      need.push_back(own[i] != (size_t)-1);
      if (need[i]) { bytes += (double)srcs[i].bytes(); ++launches; }
    }
    const float* gamma = nw.gamma;
    const float* beta = nw.beta;
    push(name, launches, 0, bytes, [=](cudaStream_t s) {
      cudaError_t e;
      for (size_t i = 0; i < xs.size(); ++i) {
        if (!need[i]) continue;
        e = gn_stats(xs[i], N, HW, cs[i], const_cast<float*>(gs[i].partial), chunks, cs[i], 0, bf, s, sp);
        if (e != cudaSuccess) return e;
      }
      return gn_finalize(gs.data(), (int)gs.size(), gamma, beta, N, ctot, groups, HW, eps, ss, s);
    });
  }
  for (size_t i = 0; i < srcs.size(); ++i)
    if (own[i] != (size_t)-1) arena_.release(own[i]);
}

void Builder::gn(const std::string& name, const std::vector<T4>& srcs, const NormW& nw, int groups, float eps,
                 bool silu, const T4& out) {
  int ctot = 0;
  for (auto& s : srcs) ctot += s.C;
  GP_REQUIRE(ctot == out.C && nw.C == ctot && ctot % groups == 0 && srcs.size() <= 2, name + ": GroupNorm channel mismatch");
  const int N = out.N;
  const long long HW = (long long)out.H * out.W;
  const int chunks = gn_chunks(N, HW);
  // per source: partial sums either already produced by the conv that wrote it, or computed here
  std::vector<size_t> own(srcs.size(), (size_t)-1);
  std::vector<GnSrc> gs(srcs.size());
  for (size_t i = 0; i < srcs.size(); ++i) {
    auto it = stats.find(srcs[i].off);
    if (it != stats.end() && it->second.C == srcs[i].C) {
      gs[i] = GnSrc{measuring_ ? nullptr : reinterpret_cast<const float*>(raw_ptr(it->second.off)), it->second.slots, srcs[i].C};
    } else {
      own[i] = arena_.alloc((size_t)N * chunks * srcs[i].C * 2 * sizeof(float));
      gs[i] = GnSrc{measuring_ ? nullptr : reinterpret_cast<const float*>(raw_ptr(own[i])), chunks, srcs[i].C};
    }
  }
  if (!measuring_) {
    float* ss = gn_ss;
    const bool bf = bf16_;
    std::vector<const void*> xs;
    std::vector<int> cs;
    std::vector<bool> need;
    int launches = 1;
    double bytes = (double)out.bytes();
    for (size_t i = 0; i < srcs.size(); ++i) {
      xs.push_back(ptr(srcs[i]));
      cs.push_back(srcs[i].C);
      need.push_back(own[i] != (size_t)-1);
      bytes += (need[i] ? 2.0 : 1.0) * srcs[i].bytes();
      launches += need[i] ? 2 : 1;
    }
    void* y = ptr(out);
    const float* gamma = nw.gamma;
    const float* beta = nw.beta;
    const bool sp = split_;
    push(name, launches, 0, bytes, [=](cudaStream_t s) {
      cudaError_t e;
      for (size_t i = 0; i < xs.size(); ++i) {
        if (!need[i]) continue;
        e = gn_stats(xs[i], N, HW, cs[i], const_cast<float*>(gs[i].partial), chunks, cs[i], 0, bf, s, sp);
        if (e != cudaSuccess) return e;
      }
      e = gn_finalize(gs.data(), (int)gs.size(), gamma, beta, N, ctot, groups, HW, eps, ss, s);
      if (e != cudaSuccess) return e;
      int coff = 0;
      for (size_t i = 0; i < xs.size(); ++i) {
        e = gn_apply(xs[i], N, HW, cs[i], ss, ctot, coff, y, ctot, silu, bf, s, sp);
        if (e != cudaSuccess) return e;
        coff += cs[i];
      }
      return cudaSuccess;
    });
  }
  for (size_t i = 0; i < srcs.size(); ++i)
    if (own[i] != (size_t)-1) arena_.release(own[i]);
}

void Builder::ln(const std::string& name, const T4& x, const NormW& nw, float eps, const T4& out) {
  GP_REQUIRE(nw.C == x.C && out.C == x.C, name + ": LayerNorm channel mismatch");
  if (measuring_) return;
  const void* xi = ptr(x);
  void* yo = ptr(out);
  const long long tokens = x.pixels();
  const int C = x.C;
  const bool bf = bf16_;
  const float* g = nw.gamma;
  const float* b = nw.beta;
  const bool sp = split_;
  push(name, 1, 0, 2.0 * x.bytes(), [=](cudaStream_t s) { return layernorm(xi, yo, tokens, C, g, b, eps, bf, s, sp); });
}

void Builder::xattn(const std::string& name, const T4& x, const XattnW& w, float eps, const T4& out) {
  GP_REQUIRE(w.C == x.C, name + ": cross-attention channel mismatch");
  if (measuring_) return;
  const void* xi = ptr(x);
  void* yo = ptr(out);
  const long long tokens = x.pixels();
  const bool bf = bf16_, sp = split_;
  const XattnW ww = w;
  push(name, 1, 4.0 * tokens * (double)w.C * w.heads, 2.0 * x.bytes(), [=](cudaStream_t s) {
    return xattn2(xi, yo, tokens, ww.C, ww.heads, ww.U, ww.u0, ww.M, ww.c0, eps, bf, s, sp);
  });
}

void Builder::geglu_op(const std::string& name, const T4& in, const T4& out) {
  if (measuring_) return;
  const void* xi = ptr(in);
  void* yo = ptr(out);
  const long long tokens = in.pixels();
  const int c4 = out.C;
  const bool bf = bf16_;
  push(name, 1, 0, (double)in.bytes() + out.bytes(), [=](cudaStream_t s) { return geglu(xi, yo, tokens, c4, bf, s); });
}

void Builder::relu_op(const std::string& name, const T4& in, const T4& out) {
  if (measuring_) return;
  const void* xi = ptr(in);
  void* yo = ptr(out);
  const long long n = in.pixels() * in.C;
  const bool bf = bf16_;
  const int sc = split_ ? in.C : 0;
  push(name, 1, 0, 2.0 * in.bytes(), [=](cudaStream_t s) { return relu16(xi, yo, n, bf, s, sc); });
}

void Builder::bilinear(const std::string& name, const T4& in, const T4& out) {
  GP_REQUIRE(out.H == 2 * in.H && out.W == 2 * in.W && out.C == in.C, name + ": bilinear shape mismatch");
  if (measuring_) return;
  const void* xi = ptr(in);
  void* yo = ptr(out);
  const T4 t = in;
  const bool bf = bf16_;
  const bool sp = split_;
  push(name, 1, 0, (double)in.bytes() + out.bytes(), [=](cudaStream_t s) { return bilinear_up2x(xi, yo, t.N, t.H, t.W, t.C, bf, s, sp); });
}

void Builder::direct(const std::string& name, const T4& in, int cin, const DirectW& w, const T4& out, int flags,
                     float* out_f32, int up) {
  GP_REQUIRE(w.Cin == cin, name + ": direct conv channel mismatch");
  if (measuring_) return;
  DirectConvParams p;
  std::memset(&p, 0, sizeof(p));
  p.in = ptr(in);
  p.N = in.N; p.H = in.H; p.W = in.W; p.Cin = cin; p.in_cstride = (int)in.ps();
  p.in_lo = split_ ? in.C : 0;
  p.w = w.w; p.bias = w.bias;
  p.Ho = up ? 2 * in.H : in.H; p.Wo = up ? 2 * in.W : in.W;
  p.Cout = w.Cout;
  p.ks = w.ks; p.stride = 1; p.pad = w.ks / 2;
  p.flags = flags | (up ? DC_UP2X : 0) | (out_f32 ? DC_OUT_F32_NCHW : 0);
  if (out_f32) { p.out = out_f32; p.out_cstride = w.Cout; }
  else { p.out = ptr(out); p.out_cstride = (int)out.ps(); p.out_lo = split_ ? out.C : 0; }
  const bool bf = bf16_;
  const double flops = 2.0 * p.N * p.Ho * p.Wo * (double)p.Cout * cin * w.ks * w.ks;
  float** slot = out_f32 ? out_slot : nullptr;
  push(name, 1, flops, (double)in.bytes() + (double)p.N * p.Ho * p.Wo * p.Cout * (out_f32 ? 4 : 2),
       [p, bf, slot](cudaStream_t s) {
         if (!slot) return direct_conv(p, bf, s);
         DirectConvParams q = p;
         q.out = *slot;
         return direct_conv(q, bf, s);
       });
}

}  // namespace gp
