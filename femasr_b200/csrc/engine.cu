// Host-side engine: the FeMaSRNet inference graph (femasr_arch.py:311-385) as a fixed kernel sequence
// over a caller-provided device workspace.  No arithmetic happens here; every step is one of the
// exported operator kernels.  The graph is data-independent, so one forward = one launch list that a
// caller may capture in a CUDA graph.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <vector>

#include <cuda_fp16.h>

#include "common.cuh"

namespace femasr {

static thread_local std::string g_err;
thread_local long g_launches = 0;
void set_error(const std::string& msg) { g_err = msg; }
int fail(int code, const std::string& msg) { g_err = msg; return code; }

// ---------------------------------------------------------------------------------------------
// Offset allocator over the workspace (first fit + coalescing).  Deterministic, so a dry run with
// base == nullptr yields the exact high-water mark the real run needs.
struct Arena {
  struct Blk { size_t off, size; bool free; };
  std::vector<Blk> blks;
  char* base = nullptr;
  size_t top = 0, peak = 0, cap = 0;
  bool dry = true;
  bool overflow = false;      // real run only: an allocation ran past the caller's workspace (sizing bug) - never launch on it
  static size_t align(size_t n) { return (n + 255) & ~size_t(255); }
  size_t alloc_off(size_t bytes) {
    bytes = align(std::max<size_t>(bytes, 256));
    for (size_t i = 0; i < blks.size(); ++i) {
      if (blks[i].free && blks[i].size >= bytes) {
        if (blks[i].size > bytes) {
          Blk rest{blks[i].off + bytes, blks[i].size - bytes, true};
          blks[i].size = bytes;
          blks.insert(blks.begin() + i + 1, rest);
        }
        blks[i].free = false;
        return blks[i].off;
      }
    }
    Blk b{top, bytes, false};
    blks.push_back(b);
    top += bytes;
    peak = std::max(peak, top);
    if (!dry && top > cap) overflow = true;
    return b.off;
  }
  float* alloc(size_t nfloats) {
    size_t off = alloc_off(nfloats * sizeof(float));
    return reinterpret_cast<float*>(base + off);   // only dereferenced when !dry
  }
  void release(const void* p) {
    size_t off = (size_t)(reinterpret_cast<const char*>(p) - base);
    for (size_t i = 0; i < blks.size(); ++i) {
      if (blks[i].off == off && !blks[i].free) {
        blks[i].free = true;
        if (i + 1 < blks.size() && blks[i + 1].free) { blks[i].size += blks[i + 1].size; blks.erase(blks.begin() + i + 1); }
        if (i > 0 && blks[i - 1].free) { blks[i - 1].size += blks[i].size; blks.erase(blks.begin() + i); }
        while (!blks.empty() && blks.back().free) { top = blks.back().off; blks.pop_back(); }
        return;
      }
    }
  }
};

struct DevBuf {
  float* p = nullptr;
  size_t n = 0;
};

struct ParamInfo {
  size_t numel;
  int kind;  // 0 plain, 1 conv/linear weight [Cout,Cin,k,k], 2 rel-pos table, 3 codebook
  int Cout, Cin, k;
};

struct Tap { float* dst; size_t cap; };

struct ProfRec { const char* name; double flops; cudaEvent_t e0, e1; };

}  // namespace femasr

using namespace femasr;

struct femasr_net {
  femasr_net_config cfg;
  int depth;   // encode depth (1 for x4, 2 for x2, 3 for the HQ autoencoder)
  bool hq = false;   // scale_factor 1: LQ_stage=False graph (no Swin, no up branches, no skip adds)
  std::map<std::string, ParamInfo> spec;
  std::map<std::string, DevBuf> raw;      // fp32 copy in the reference layout
  std::map<std::string, DevBuf> packed;   // K-major GEMM operand / expanded rel bias / codebook^T
  std::map<std::string, DevBuf> packed_mma;   // rel-pos bias in the mma attention kernel's fragment order
  std::map<std::string, DevBuf> tcw;      // tensor-core operand (split fp16), gemm_path 1
  std::map<std::string, DevBuf> tcw_up;   // sub-pixel phase filters of the upsample-fused 3x3 convs
  std::map<std::string, DevBuf> tcw8, tcw_up8;   // the same two in the F8 cross-term packing (layers behind the VQ)
  std::map<std::string, DevBuf> esq;      // sum e^2 per codebook row, keyed by the codebook's parameter name
  struct Codebook { int scale, n_e, e_dim; };
  std::vector<Codebook> cbs;              // codebook_params rows; cbs[0].scale == 32
  int level_cb[3] = {0, -1, -1};          // decoder level i (resolution 32 << i) -> codebook index or -1
  int last_q_level = 0;                   // last decoder level that quantises (everything before it is index-critical)
  std::map<std::string, Tap> taps;
  int last_launches = 0;
  bool profile = false;
  bool f8_cross = true;                   // layers behind the VQ: the two cross products of the split as one fp8 product (FEMASR_F8_CROSS=0: three fp16 products)
  std::vector<ProfRec> prof;
  std::string prof_json;
  ~femasr_net() {
    for (auto& r : prof) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
    for (auto& kv : raw) cudaFree(kv.second.p);
    for (auto& kv : packed) cudaFree(kv.second.p);
    for (auto& kv : packed_mma) cudaFree(kv.second.p);
    for (auto& kv : tcw) cudaFree(kv.second.p);
    for (auto& kv : tcw_up) cudaFree(kv.second.p);
    for (auto& kv : tcw8) cudaFree(kv.second.p);
    for (auto& kv : tcw_up8) cudaFree(kv.second.p);
    for (auto& kv : esq) cudaFree(kv.second.p);
  }
};

namespace femasr {

// K-sliced accumulation of the tensor-core convs in front of the VQ: the truncating MMA accumulator is folded into an
// fp32 running sum every TC_SLICE_KB 64-wide k-blocks (256 of K)
constexpr int TC_SLICE_KB = 4;

static int chan(int res) {
  switch (res) { case 8: case 16: case 32: case 64: return 256; case 128: return 128; case 256: return 64; case 512: return 32; }
  return -1;
}

static void add_conv(femasr_net* n, const std::string& p, int ci, int co, int k) {
  n->spec[p + ".weight"] = ParamInfo{(size_t)co * ci * k * k, 1, co, ci, k};
  n->spec[p + ".bias"] = ParamInfo{(size_t)co, 0, 0, 0, 0};
}
static void add_vec(femasr_net* n, const std::string& name, size_t c) { n->spec[name] = ParamInfo{c, 0, 0, 0, 0}; }
static void add_resblock(femasr_net* n, const std::string& p, int c) {
  add_vec(n, p + ".conv.0.norm.weight", c); add_vec(n, p + ".conv.0.norm.bias", c);
  add_conv(n, p + ".conv.2", c, c, 3);
  add_vec(n, p + ".conv.3.norm.weight", c); add_vec(n, p + ".conv.3.norm.bias", c);
  add_conv(n, p + ".conv.5", c, c, 3);
}

static void build_spec(femasr_net* n) {
  const int scale = n->cfg.scale_factor;
  const int d = n->depth;
  int res = 256 / scale;
  const std::string enc = "multiscale_encoder";
  add_conv(n, enc + ".in_conv", n->cfg.in_channel, chan(res), 4);
  for (int i = 0; i < d; ++i) {
    const std::string b = enc + ".blocks." + std::to_string(i);
    add_conv(n, b + ".0", chan(res), chan(res / 2), 3);
    add_resblock(n, b + ".1", chan(res / 2));
    add_resblock(n, b + ".2", chan(res / 2));
    res /= 2;
  }
  const std::string sw = enc + ".blocks." + std::to_string(d) + ".swin_blks.";
  for (int r = 0; r < (n->hq ? 0 : 4); ++r) {
    for (int b = 0; b < 6; ++b) {
      const std::string p = sw + std::to_string(r) + ".residual_group.blocks." + std::to_string(b);
      add_vec(n, p + ".norm1.weight", 256); add_vec(n, p + ".norm1.bias", 256);
      n->spec[p + ".attn.relative_position_bias_table"] = ParamInfo{225 * 8, 2, 0, 0, 0};
      add_conv(n, p + ".attn.qkv", 256, 768, 1);
      add_conv(n, p + ".attn.proj", 256, 256, 1);
      add_vec(n, p + ".norm2.weight", 256); add_vec(n, p + ".norm2.bias", 256);
      add_conv(n, p + ".mlp.fc1", 256, 1024, 1);
      add_conv(n, p + ".mlp.fc2", 1024, 256, 1);
    }
    add_conv(n, sw + std::to_string(r) + ".conv", 256, 256, 3);
  }
  for (int j = d + 1; j <= (n->hq ? d : d + 2); ++j) {
    const std::string b = enc + ".blocks." + std::to_string(j);
    add_conv(n, b + ".1", chan(res), chan(res * 2), 3);
    add_resblock(n, b + ".2", chan(res * 2));
    add_resblock(n, b + ".3", chan(res * 2));
    res *= 2;
  }
  for (int i = 0; i < 3; ++i) {
    const int r = 32 << i;
    const std::string b = "decoder_group." + std::to_string(i) + ".block";
    add_conv(n, b + ".1", chan(r), chan(r * 2), 3);
    add_resblock(n, b + ".2", chan(r * 2));
    add_resblock(n, b + ".3", chan(r * 2));
  }
  add_conv(n, "out_conv", 64, 3, 3);
  for (size_t k = 0; k < n->cbs.size(); ++k) {           // femasr_arch.py:280-299
    const femasr_net::Codebook& cb = n->cbs[k];
    const std::string ks = std::to_string(k);
    const int ch = chan(cb.scale);
    n->spec["quantize_group." + ks + ".embedding.weight"] = ParamInfo{(size_t)cb.n_e * cb.e_dim, 3, cb.n_e, cb.e_dim, 1};
    add_conv(n, "before_quant_group." + ks, k == 0 ? ch : 2 * ch, cb.e_dim, 1);
    add_conv(n, "after_quant_group." + ks + ".conv", k == 0 ? cb.e_dim : n->cbs[k - 1].e_dim + cb.e_dim, ch, 3);
  }
}

// ---------------------------------------------------------------------------------------------
struct Ctx {
  femasr_net* net;
  Arena ar;
  cudaStream_t st;
  int status = FEMASR_OK;
  bool precise_region = false;   // true while emitting the layers in front of the VQ (index-critical)
  bool dry() const { return ar.dry; }
  bool ok() const { return status == FEMASR_OK; }
  void check(int s) { if (status == FEMASR_OK && s != FEMASR_OK) status = s; }

  // every kernel launch of the graph goes through here; in profile mode it is bracketed by CUDA events
  template <class F>
  void run(const char* name, double flops, F&& f) {
    if (dry() || !ok()) return;
    if (ar.overflow) { check(fail(FEMASR_ERR_STATE, "workspace plan mismatch: the graph needs more than femasr_net_workspace_bytes reported")); return; }
    if (net->profile) {
      ProfRec r{name, flops, nullptr, nullptr};
      cudaEventCreate(&r.e0); cudaEventCreate(&r.e1);
      cudaEventRecord(r.e0, st);
      check(f());
      cudaEventRecord(r.e1, st);
      net->prof.push_back(r);
    } else {
      check(f());
    }
  }

  // FEMASR_PROFILE_DETAIL=1: per-shape kernel labels in the profile ("tc_igemm:k3:64->64@512x512"); the strings are
  // interned for the life of the process because the profile records keep only the pointer
  const char* detail_name(const char* base, int k, int Cin, int Cout, int H, int W, int up, int stride, int slice) {
    static const bool detail = [] { const char* e = getenv("FEMASR_PROFILE_DETAIL"); return e && atoi(e) != 0; }();
    if (!detail || !net->profile) return base;
    static std::set<std::string> names;
    std::string s = std::string(base) + ":k" + std::to_string(k) + ":" + std::to_string(Cin) + "->" + std::to_string(Cout) + "@" +
                    std::to_string(H) + "x" + std::to_string(W) + (up ? ":up" : "") + (stride == 2 ? ":s2" : "") + (slice ? ":sliced" : "");
    return names.insert(s).first->c_str();
  }

  const float* P(const std::string& name) {      // packed (or raw when there is no packed form)
    if (dry()) return nullptr;
    auto it = net->packed.find(name);
    if (it != net->packed.end()) return it->second.p;
    auto jt = net->raw.find(name);
    if (jt == net->raw.end()) { check(fail(FEMASR_ERR_STATE, "parameter not set: " + name)); return nullptr; }
    return jt->second.p;
  }
  const void* TCW(const std::string& name) {
    auto it = net->tcw.find(name);
    return it == net->tcw.end() ? nullptr : it->second.p;
  }
  void tap(const char* stage, const float* src, size_t n) {
    if (dry() || !ok()) return;
    auto it = net->taps.find(stage);
    if (it == net->taps.end() || !it->second.dst) return;
    if (it->second.cap < n) { check(fail(FEMASR_ERR_ARG, std::string("tap buffer too small: ") + stage)); return; }
    cudaError_t e = cudaMemcpyAsync(it->second.dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) check(fail(FEMASR_ERR_CUDA, cudaGetErrorString(e)));
  }

  // y = conv(x) (+epilogue); wname is the conv's parameter prefix.
  void conv(const std::string& wname, const float* x, float* y, int B, int Hin, int Win, int Cin, int Cout, int ksize,
            int stride, int upsample, int prologue, const float* pa, const float* pb, const float* gamma,
            const float* beta, int act, const float* res1, const float* res2, bool has_bias = true) {
    if (has_bias && tc_eligible(wname, Cin, Cout, ksize, stride, upsample)) {
      conv_tc(wname, x, y, B, Hin, Win, Cin, Cout, ksize, upsample, prologue, pa, pb, gamma, beta, act, res1, res2,
              nullptr, nullptr, nullptr, nullptr, nullptr, stride);
      return;
    }
    if (dry() || !ok()) return;
    femasr_igemm_args a;
    memset(&a, 0, sizeof(a));
    a.x = x; a.w = P(wname + ".weight"); a.bias = has_bias ? P(wname + ".bias") : nullptr;
    a.res1 = res1; a.res2 = res2; a.y = y; a.pro_a = pa; a.pro_b = pb; a.gamma = gamma; a.beta = beta;
    a.B = B; a.Hin = Hin; a.Win = Win; a.Cin = Cin; a.Cout = Cout; a.ksize = ksize; a.stride = stride;
    a.upsample = upsample; a.prologue = prologue; a.act = act;
    if (!ok()) return;
    int Ho, Wo;
    if (ksize == 1) { Ho = Hin; Wo = Win; }
    else { const int He = upsample ? 2 * Hin : Hin, We = upsample ? 2 * Win : Win;
           Ho = stride == 1 ? He : (He - 1) / 2 + 1; Wo = stride == 1 ? We : (We - 1) / 2 + 1; }
    const double flops = 2.0 * B * Ho * Wo * (double)Cout * Cin * ksize * ksize;
    run("igemm_simt", flops, [&] { return femasr_igemm_simt(&a, st); });
  }

  bool tc_eligible(const std::string& wname, int Cin, int Cout, int ksize, int stride, int upsample) const {
    if (net->cfg.gemm_path != 1 || (ksize != 1 && ksize != 3) || Cin % 64 || Cout % 64) return false;
    if (stride != 1 && !(stride == 2 && ksize == 3 && !upsample)) return false;
    if (dry()) return true;
    return upsample ? net->tcw_up.count(wname + ".weight") != 0 : net->tcw.count(wname + ".weight") != 0;
  }

  // tensor-core variant of conv(): stage the activation operand (prologue + fp16 split) unless the producer
  // already wrote split planes (pre_hi/pre_lo), then the tcgen05 implicit GEMM; optionally the result is
  // emitted as split planes for the next GEMM (out_hi/out_lo) instead of fp32 y.  A fused nearest-x2 upsample
  // runs as four sub-pixel 2x2 convs on the low-res operand.  Allocation happens in dry runs too.
  void conv_tc(const std::string& wname, const float* x, float* y, int B, int Hin, int Win, int Cin, int Cout, int ksize,
               int upsample, int prologue, const float* pa, const float* pb, const float* gamma, const float* beta,
               int act, const float* res1, const float* res2, const void* pre_hi = nullptr, const void* pre_lo = nullptr,
               void* out_hi = nullptr, void* out_lo = nullptr, float* gn_partial = nullptr, int stride = 1,
               bool precise = false) {
    const size_t plane_halves = (size_t)B * Hin * Win * Cin;
    float *ahi = nullptr, *alo = nullptr;
    if (!pre_hi) {
      ahi = ar.alloc((plane_halves + 1) / 2);
      alo = ar.alloc((plane_halves + 1) / 2);
    }
    if (!dry() && ok()) {
      // behind the VQ (bar: 1e-3 on the output): approximate-unit SiLU, and the two cross products of the split as one
      // fp8 product (F8 mode: staging writes the interleaved e4m3 plane, the weights come from the F8 packing)
      const bool relaxed = !precise && !precise_region;
      const bool f8 = relaxed && net->f8_cross && !pre_hi && ksize == 3 && prologue != FEMASR_PRO_LN &&
                      (upsample ? net->tcw_up8.count(wname + ".weight") : net->tcw8.count(wname + ".weight")) != 0;
      if (!pre_hi) {
        const int pmode = (prologue == FEMASR_PRO_GN_SILU && relaxed) ? FEMASR_PRO_GN_SILU_FAST : prologue;
        run(detail_name(f8 ? "tc_prepare_f8" : "tc_prepare", pmode, Cin, Cin, Hin, Win, 0, 1, 0), 0.0, [&] {
          return f8 ? femasr_tc_prepare_f8(x, ahi, alo, pmode, pa, pb, B, Hin, Win, Cin, st)
                    : femasr_tc_prepare(x, ahi, alo, pmode, pa, pb, gamma, beta, B, Hin, Win, Cin, 0,
                                        prologue == FEMASR_PRO_LN ? 1e-5f : 1e-6f, st);
        });
      }
      femasr_tc_args t;
      memset(&t, 0, sizeof(t));
      t.a_hi = pre_hi ? pre_hi : ahi; t.a_lo = pre_hi ? pre_lo : alo;
      t.f8 = f8 ? 1 : 0;
      t.w_blob = f8 ? (upsample ? net->tcw_up8[wname + ".weight"].p : net->tcw8[wname + ".weight"].p)
                    : (upsample ? net->tcw_up[wname + ".weight"].p : net->tcw[wname + ".weight"].p);
      t.bias = P(wname + ".bias");
      t.res1 = res1; t.res2 = res2; t.y = y; t.out_hi = out_hi; t.out_lo = out_lo; t.gn_partial = gn_partial;
      t.B = B; t.H = Hin; t.W = Win; t.Cin = Cin; t.Cout = Cout; t.ksize = ksize; t.act = act; t.upsample = upsample;
      t.stride = stride; t.pair = -1; t.strip = -1;
      const int u = upsample ? 2 : 1;
      const int Ho = stride == 2 ? (Hin - 1) / 2 + 1 : Hin * u, Wo = stride == 2 ? (Win - 1) / 2 + 1 : Win * u;
      const double flops = 2.0 * B * Ho * (double)Wo * Cout * Cin * ksize * ksize;   // algorithmic (reference) count
      const int nkb = (upsample ? 4 : ksize * ksize) * (Cin / 64);
      if ((precise || precise_region) && nkb > TC_SLICE_KB) {
        // K-sliced accumulation (layers in front of the VQ): every 256 of K the tensor core's truncating accumulator
        // is folded into an fp32 round-to-nearest running sum held in TMEM (see femasr_tc_args.slice_kb)
        t.slice_kb = TC_SLICE_KB;
      }
      run(detail_name("tc_igemm", ksize, Cin, Cout, Hin, Win, upsample, stride, t.slice_kb), flops,
          [&] { return femasr_tc_igemm(&t, st); });
    }
    if (alo) ar.release(alo);
    if (ahi) ar.release(ahi);
  }

  // GroupNorm statistics of x folded into scale/shift tables (allocated by the caller)
  void gn(const std::string& norm, const float* x, float* sc, float* sh, float* scratch, int B, int HW, int C) {
    if (dry() || !ok()) return;
    const float *gw = P(norm + ".weight"), *gb = P(norm + ".bias");
    run("gn_stats", 0.0, [&] { return femasr_gn_stats(x, gw, gb, sc, sh, scratch, B, HW, C, 1e-6f, st); });
  }

  // GroupNorm partial sums produced by a tensor-core conv epilogue (see femasr_tc_args.gn_partial)
  struct Stats { float* partial = nullptr; int rows = 0; };
  // for the tensor-core conv [B,H,W,Cin] -> Cout (H,W: conv-input size, low-res if upsample) that will produce them
  Stats alloc_stats(int B, int H, int W, int Cin, int Cout, int upsample, int stride) {
    femasr_tc_args t;
    memset(&t, 0, sizeof(t));
    t.B = B; t.H = H; t.W = W; t.Cin = Cin; t.Cout = Cout; t.ksize = 3; t.upsample = upsample; t.stride = stride;
    t.pair = -1; t.strip = -1;
    t.slice_kb = (precise_region && (upsample ? 4 : 9) * (Cin / 64) > TC_SLICE_KB) ? TC_SLICE_KB : 0;
    Stats st_;
    st_.rows = femasr_tc_gn_partial_rows(&t);
    st_.partial = ar.alloc((size_t)B * st_.rows * 32 * 2);
    return st_;
  }
  bool tc_convs(int C) const { return net->cfg.gemm_path == 1 && C % 64 == 0; }

  // scale/shift tables for `norm` applied to x: from epilogue partials when available, else a stats pass over x
  void gn_tables(const std::string& norm, const float* x, const Stats& sx, float* sc, float* sh, int B, int HW, int C) {
    if (sx.partial) {
      if (dry() || !ok()) return;
      const float *gw = P(norm + ".weight"), *gb = P(norm + ".bias");
      run("gn_finalize_rows", 0.0, [&] { return femasr_gn_finalize_rows(sx.partial, gw, gb, sc, sh, B, sx.rows, HW, C, 1e-6f, st); });
    } else {
      float* scratch = ar.alloc(femasr_gn_scratch_floats(B, HW, C));
      gn(norm, x, sc, sh, scratch, B, HW, C);
      ar.release(scratch);
    }
  }

  // fema_utils.py:65-84, in place on x; optional extra residual added after the block (encoder skip).
  // sx: GroupNorm partials of x from its producer (consumed/released here); returns the partials of the block's
  // output when want_out (for the next ResBlock's first norm), which the caller releases after use.
  Stats resblock(const std::string& p, float* x, int B, int H, int W, int C, const float* extra, Stats sx, bool want_out) {
    const size_t n = (size_t)B * H * W * C;
    const bool tc = tc_convs(C);
    float* sc = ar.alloc((size_t)B * C);
    float* sh = ar.alloc((size_t)B * C);
    float* t = ar.alloc(n);
    gn_tables(p + ".conv.0.norm", x, sx, sc, sh, B, H * W, C);
    if (sx.partial) ar.release(sx.partial);
    Stats s1, s2;
    if (tc) s1 = alloc_stats(B, H, W, C, C, 0, 1);
    if (tc)
      conv_tc(p + ".conv.2", x, t, B, H, W, C, C, 3, 0, FEMASR_PRO_GN_SILU, sc, sh, nullptr, nullptr, 0, nullptr, nullptr,
              nullptr, nullptr, nullptr, nullptr, s1.partial);
    else
      conv(p + ".conv.2", x, t, B, H, W, C, C, 3, 1, 0, FEMASR_PRO_GN_SILU, sc, sh, nullptr, nullptr, 0, nullptr, nullptr);
    gn_tables(p + ".conv.3.norm", t, s1, sc, sh, B, H * W, C);
    if (s1.partial) ar.release(s1.partial);
    if (tc && want_out) s2 = alloc_stats(B, H, W, C, C, 0, 1);
    if (tc)
      conv_tc(p + ".conv.5", t, x, B, H, W, C, C, 3, 0, FEMASR_PRO_GN_SILU, sc, sh, nullptr, nullptr, 0, x, extra,
              nullptr, nullptr, nullptr, nullptr, s2.partial);
    else
      conv(p + ".conv.5", t, x, B, H, W, C, C, 3, 1, 0, FEMASR_PRO_GN_SILU, sc, sh, nullptr, nullptr, 0, x, extra);
    ar.release(t); ar.release(sh); ar.release(sc);
    return s2;
  }

  // nn.Upsample(2) -> conv3x3 -> ResBlock -> ResBlock  (femasr_arch.py:168-180, 195-211); returns new buffer
  float* up_block(const std::string& pconv, const std::string& prb1, const std::string& prb2, const float* x, int B,
                  int H, int W, int Cin, int Cout, const float* extra) {
    float* y = ar.alloc((size_t)B * 2 * H * 2 * W * Cout);
    Stats s0;
    if (tc_convs(Cin) && tc_convs(Cout) && (dry() || net->tcw_up.count(pconv + ".weight"))) {
      s0 = alloc_stats(B, H, W, Cin, Cout, 1, 1);
      conv_tc(pconv, x, y, B, H, W, Cin, Cout, 3, 1, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr,
              nullptr, nullptr, nullptr, nullptr, s0.partial);
    } else {
      conv(pconv, x, y, B, H, W, Cin, Cout, 3, 1, 1, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr);
    }
    Stats s1 = resblock(prb1, y, B, 2 * H, 2 * W, Cout, nullptr, s0, true);
    resblock(prb2, y, B, 2 * H, 2 * W, Cout, extra, s1, false);
    return y;
  }

  // SwinLayers (femasr_arch.py:126-132): 4 x RSTB on tokens X [B, H*W, 256], in place.
  void swin(const std::string& p, float* X, int B, int H, int W) {
    const int C = 256;
    const size_t M = (size_t)B * H * W;
    float* T = ar.alloc(M * C);
    float* qkv = ar.alloc(M * 3 * C);
    float* ao = ar.alloc(M * C);
    float* hid = ar.alloc(M * 4 * C);
    float* mu = ar.alloc(M);
    float* rs = ar.alloc(M);
    const bool tc = net->cfg.gemm_path == 1 && (dry() || net->tcw.count(p + ".swin_blks.0.conv.weight") != 0);
    for (int r = 0; r < 4; ++r) {
      const std::string rp = p + ".swin_blks." + std::to_string(r);
      for (int b = 0; b < 6; ++b) {
        const std::string bp = rp + ".residual_group.blocks." + std::to_string(b);
        const float* in = b == 0 ? X : T;
        const float* rb = P(bp + ".attn.relative_position_bias_table");
        const double attn_flops = 2.0 * 2.0 * 64 * C * (double)M;
        if (tc) {
          // operands travel between the kernels as split fp16 planes: `ao` and `hid` are reinterpreted as
          // [hi plane | lo plane] (same byte size as the fp32 tensors they replace)
          __half* ao_hi = reinterpret_cast<__half*>(ao);  __half* ao_lo = ao_hi + M * C;
          __half* hd_hi = reinterpret_cast<__half*>(hid); __half* hd_lo = hd_hi + M * 4 * C;
          conv_tc(bp + ".attn.qkv", in, qkv, B, H, W, C, 3 * C, 1, 0, FEMASR_PRO_LN, nullptr, nullptr, P(bp + ".norm1.weight"),
                  P(bp + ".norm1.bias"), 0, nullptr, nullptr);
          const float* rbm = dry() ? nullptr : net->packed_mma[bp + ".attn.relative_position_bias_table"].p;
          run("window_attention_mma", attn_flops, [&] {
            return femasr_window_attention_mma(qkv, rbm, nullptr, ao_hi, ao_lo, B, H, W, C, 8, (b & 1) ? 4 : 0, st);
          });
          conv_tc(bp + ".attn.proj", nullptr, T, B, H, W, C, C, 1, 0, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0,
                  in, nullptr, ao_hi, ao_lo);
          conv_tc(bp + ".mlp.fc1", T, nullptr, B, H, W, C, 4 * C, 1, 0, FEMASR_PRO_LN, nullptr, nullptr, P(bp + ".norm2.weight"),
                  P(bp + ".norm2.bias"), FEMASR_ACT_GELU, nullptr, nullptr, nullptr, nullptr, hd_hi, hd_lo);
          conv_tc(bp + ".mlp.fc2", nullptr, T, B, H, W, 4 * C, C, 1, 0, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0,
                  T, nullptr, hd_hi, hd_lo);
          continue;
        }
        run("ln_stats", 0.0, [&] { return femasr_ln_stats(in, mu, rs, (int)M, C, 1e-5f, st); });
        conv(bp + ".attn.qkv", in, qkv, B, H, W, C, 3 * C, 1, 1, 0, FEMASR_PRO_LN, mu, rs, P(bp + ".norm1.weight"),
             P(bp + ".norm1.bias"), 0, nullptr, nullptr);
        run("window_attention", attn_flops,
            [&] { return femasr_window_attention(qkv, rb, ao, B, H, W, C, 8, (b & 1) ? 4 : 0, st); });
        conv(bp + ".attn.proj", ao, T, B, H, W, C, C, 1, 1, 0, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0, in, nullptr);
        run("ln_stats", 0.0, [&] { return femasr_ln_stats(T, mu, rs, (int)M, C, 1e-5f, st); });
        conv(bp + ".mlp.fc1", T, hid, B, H, W, C, 4 * C, 1, 1, 0, FEMASR_PRO_LN, mu, rs, P(bp + ".norm2.weight"),
             P(bp + ".norm2.bias"), FEMASR_ACT_GELU, nullptr, nullptr);
        conv(bp + ".mlp.fc2", hid, T, B, H, W, 4 * C, C, 1, 1, 0, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0, T, nullptr);
      }
      conv(rp + ".conv", T, X, B, H, W, C, C, 3, 1, 0, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0, X, nullptr);
    }
    ar.release(rs); ar.release(mu); ar.release(hid); ar.release(ao); ar.release(qkv); ar.release(T);
  }

  // One quantiser (femasr_arch.py:337-342 + VectorQuantizer.forward :50-100): z = before_quant(src) [N,e], argmin over
  // codebook k, zq = z + (E[idx] - z); loss terms accumulate into cb_loss.  Returns z and zq (caller releases both).
  void quantise(int k, const float* src, int Cin, int B, int hh, int ww, int64_t* indices, float* cb_loss,
                const int64_t* gt, float** z_out, float** zq_out) {
    const femasr_net::Codebook& cb = net->cbs[k];
    const std::string ks = std::to_string(k);
    const size_t N = (size_t)B * hh * ww;
    const int e = cb.e_dim;
    float* z = ar.alloc(N * e);
    conv("before_quant_group." + ks, src, z, B, hh, ww, Cin, e, 1, 1, 0, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr);
    tap(k == 0 ? "z" : (k == 1 ? "z1" : "z2"), z, N * e);
    const std::string cname = "quantize_group." + ks + ".embedding.weight";
    const bool fused = net->cfg.gemm_path == 1 && (dry() || net->tcw.count(cname) != 0);
    // fused: tensor-core distances + in-kernel top-4 (no [N, n_e] tensor); else the fp32 SIMT product + vq_select
    float *zc = nullptr, *arow = nullptr, *zhi = nullptr, *zlo = nullptr, *cand = nullptr;
    if (fused) {
      arow = ar.alloc(N);
      zhi = ar.alloc((N * e + 1) / 2);
      zlo = ar.alloc((N * e + 1) / 2);
      cand = ar.alloc(N * 8);
    } else {
      zc = ar.alloc(N * cb.n_e);
      conv("quantize_group." + ks + ".embedding", z, zc, B, hh, ww, e, cb.n_e, 1, 1, 0, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, false);
    }
    float* zq = ar.alloc(N * e);
    float* lrows = ar.alloc(N);
    const bool gt_loss = gt && !net->hq;                 // :84: only the LQ stage uses gt_indices for the loss
    float *zq_gt = nullptr, *gpart = nullptr;
    const int gtiles = femasr_gram_diff_tiles(e);
    if (gt_loss) { zq_gt = ar.alloc(N * e); gpart = ar.alloc((size_t)B * gtiles); }
    if (!dry() && ok()) {
      const float* cbw = net->raw[cname].p;
      const float* esq = net->esq[cname].p;
      if (fused) {
        const void* cbt = net->tcw[cname].p;
        run("vq_row_sumsq", 0.0, [&] { return femasr_row_sumsq(z, arow, (int)N, e, st); });
        run("tc_prepare", 0.0, [&] { return femasr_tc_prepare(z, zhi, zlo, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, B, hh, ww, e, 0, 0.f, st); });
        run("vq_match_tc", 2.0 * (double)N * cb.n_e * e, [&] { return femasr_vq_match_tc(zhi, zlo, cbt, arow, esq, cand, (int)N, cb.n_e, e, st); });
        run("vq_finish", 0.0, [&] { return femasr_vq_finish(z, arow, cand, cbw, esq, indices, zq, lrows, nullptr, (int)N, cb.n_e, e, st); });
      } else {
        run("vq_select", 0.0, [&] { return femasr_vq_select(z, zc, cbw, esq, indices, zq, lrows, (int)N, cb.n_e, e, 0, st); });
      }
      if (cb_loss && !gt_loss) {
        const double s = 1.25 / ((double)N * e);         // q_latent + 0.25 * e_latent, :92
        run("sum_scaled", 0.0, [&] { return k == 0 ? femasr_sum_scaled(lrows, cb_loss, N, s, st) : femasr_sum_scaled_add(lrows, cb_loss, N, s, st); });
      } else if (cb_loss) {
        run("vq_gt_rows", 0.0, [&] { return femasr_vq_gt_rows(z, cbw, gt, zq_gt, lrows, (int)N, cb.n_e, e, st); });
        const double s = 0.25 / ((double)N * e);         // beta * mean((z_q_gt - z)^2), :87
        run("sum_scaled", 0.0, [&] { return k == 0 ? femasr_sum_scaled(lrows, cb_loss, N, s, st) : femasr_sum_scaled_add(lrows, cb_loss, N, s, st); });
        run("gram_diff", 4.0 * B * (double)hh * ww * e * e, [&] { return femasr_gram_diff(z, zq_gt, gpart, B, hh * ww, e, st); });
        run("sum_scaled", 0.0, [&] { return femasr_sum_scaled_add(gpart, cb_loss, (size_t)B * gtiles, 1.0 / ((double)B * e * e), st); });
      }
    }
    if (gt_loss) { ar.release(gpart); ar.release(zq_gt); }
    ar.release(lrows);
    if (fused) { ar.release(cand); ar.release(zlo); ar.release(zhi); ar.release(arow); }
    else ar.release(zc);
    if (k == 0) tap("zq", zq, N * e);
    *z_out = z; *zq_out = zq;
  }

  // The decoder loop of encode_and_decode (femasr_arch.py:327-369) from decoder level 0 on.
  //   feats[i]   enc_feats[i] (NHWC, level i = resolution 32 << i) or nullptr when that level needs none
  //   zq0_given  decode_indices: the gathered codebook-0 entries; no quantiser runs at any level (:376-385)
  void decode_loop(const float* const* feats, const float* zq0_given, float* y_nchw, int64_t* indices, float* cb_loss,
                   const int64_t* gt, int B, int h, int w) {
    const femasr_net_config& cfg = net->cfg;
    const bool lq = !net->hq;
    float* t = nullptr;                       // decoder stream
    float* prev_q = nullptr; int pq_h = 0, pq_w = 0, pq_e = 0;   // previous z_quant (:358)
    float* prev_z = nullptr;
    size_t idx_off = 0;
    int Cprev = 0;                            // channels of t
    for (int i = 0; i < 3; ++i) {
      const int hh = h << i, ww = w << i, ch = chan(32 << i), co = chan(64 << i);
      const int k = zq0_given ? (i == 0 ? 0 : -1) : net->level_cb[i];
      if (k >= 0) {
        const femasr_net::Codebook& cb = net->cbs[k];
        const size_t N = (size_t)B * hh * ww;
        const float* aq = zq0_given;
        float *z = nullptr, *zq = nullptr;
        if (!zq0_given) {
          precise_region = true;
          const float* src = feats[i];
          float* cat = nullptr;
          int Cin = ch;
          if (t) {                            // cat(enc_feats[i], prev_dec_feat), :332-333
            cat = ar.alloc(N * 2 * ch);
            if (!dry() && ok())
              run("concat_channels", 0.0, [&] { return femasr_concat_channels(feats[i], ch, t, hh, ww, ch, cat, B, hh, ww, st); });
            ar.release(t); t = nullptr;
            src = cat; Cin = 2 * ch;
          }
          quantise(k, src, Cin, B, hh, ww, indices ? indices + idx_off : nullptr, cb_loss,
                   gt ? gt + idx_off : nullptr, &z, &zq);
          idx_off += N;
          if (cat) ar.release(cat);
          aq = cfg.use_quantize ? zq : z;     // :349-350
          if (i >= net->last_q_level) precise_region = false;
        }
        int e_in = cb.e_dim;
        float* cat2 = nullptr;
        if (prev_q) {                         // CombineQuantBlock: cat(z_quant, interpolate(prev_quant)), fema_utils.py:92-99
          cat2 = ar.alloc(N * (cb.e_dim + pq_e));
          const float* a0 = aq; const int pe = pq_e, ph = pq_h, pw = pq_w; const float* pq = prev_q;
          if (!dry() && ok())
            run("concat_channels", 0.0, [&] { return femasr_concat_channels(a0, cb.e_dim, pq, ph, pw, pe, cat2, B, hh, ww, st); });
          aq = cat2; e_in += pq_e;
        }
        t = ar.alloc(N * ch);
        conv("after_quant_group." + std::to_string(k) + ".conv", aq, t, B, hh, ww, e_in, ch, 3, 1, 0, FEMASR_PRO_NONE,
             nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr);
        if (k == 0) tap("after_quant", t, N * ch);
        if (cat2) ar.release(cat2);
        if (prev_q) { ar.release(prev_q); ar.release(prev_z); }
        if (!zq0_given) {                     // prev_quant_feat = z_quant (after the use_quantize override), :358
          prev_q = cfg.use_quantize ? zq : z; prev_z = cfg.use_quantize ? z : zq;
          pq_h = hh; pq_w = ww; pq_e = cb.e_dim;
        }
      }
      (void)Cprev;
      // the skip add of the NEXT level (x = x + enc_feats[i+1], :361-362) rides on this block's last epilogue
      const bool next_quant = i + 1 < 3 && !zq0_given && net->level_cb[i + 1] >= 0;
      const float* extra = (i + 1 < 3 && !zq0_given && lq && cfg.use_residual && !next_quant) ? feats[i + 1] : nullptr;
      const std::string b = "decoder_group." + std::to_string(i) + ".block";
      float* nt = up_block(b + ".1", b + ".2", b + ".3", t, B, hh, ww, ch, co, extra);
      ar.release(t);
      t = nt;
      tap(i == 0 ? "dec0" : (i == 1 ? "dec1" : "dec2"), t, (size_t)B * 2 * hh * 2 * ww * co);
    }
    if (prev_q) { ar.release(prev_q); ar.release(prev_z); }
    {
      const float *ow = P("out_conv.weight"), *ob = P("out_conv.bias");
      const float* d2 = t;
      run("out_conv", 2.0 * 9 * 64 * 3 * (double)B * 64 * h * w,
          [&] { return net->cfg.gemm_path == 1 ? femasr_out_conv3x3_mma(d2, ow, ob, y_nchw, B, 8 * h, 8 * w, 64, st)
                                               : femasr_out_conv3x3(d2, ow, ob, y_nchw, B, 8 * h, 8 * w, 64, st); });
    }
    ar.release(t);
  }

  void forward(const float* x_nchw, float* y_nchw, int64_t* indices, float* cb_loss, const int64_t* gt, int B, int H, int W) {
    const femasr_net_config& cfg = net->cfg;
    const int d = net->depth;
    const std::string enc = "multiscale_encoder";
    int c = chan(256 / cfg.scale_factor);
    int h = H - 1, w = W - 1;
    const bool tc = tc_convs(c);
    precise_region = true;
    const float *iw = P(enc + ".in_conv.weight"), *ib = P(enc + ".in_conv.bias");
    const double in_flops = 2.0 * 16 * cfg.in_channel * c * (double)B * h * w;
    const bool want_in_tap = net->taps.count("in_conv") && net->taps["in_conv"].dst;
    float* cur = nullptr;                 // fp32 in_conv output (SIMT path, or when its tap is requested)
    float* in_hi = nullptr; float* in_lo = nullptr;   // tensor-core path: in_conv writes the split operand planes directly
    const size_t in_elems = (size_t)B * h * w * c;
    if (!tc || want_in_tap) {     // identical in the dry (sizing) run and the real run: taps are registered first
      cur = ar.alloc(in_elems);
      const int c0 = c;
      run("in_conv", in_flops, [&] { return femasr_in_conv4x4(x_nchw, iw, ib, cur, B, cfg.in_channel, H, W, c0, st); });
      tap("in_conv", cur, in_elems);
    }
    if (tc) {
      // K = 48 (-> 64) GEMM over im2col rows on the tensor cores, writing the down conv's split planes; set_param packs
      // its weight blob (#im2col) for every in_conv of the tensor-core path
      in_hi = ar.alloc((in_elems + 1) / 2);
      in_lo = ar.alloc((in_elems + 1) / 2);
      const size_t rows = (size_t)B * h * w;
      float* ic_hi = ar.alloc(rows * 64 / 2);
      float* ic_lo = ar.alloc(rows * 64 / 2);
      if (!dry() && ok()) {
        const std::string wkey = enc + ".in_conv.weight#im2col";
        const auto wt = net->tcw.find(wkey);
        if (wt == net->tcw.end() || !wt->second.p) check(fail(FEMASR_ERR_STATE, "tensor-core weight not packed: " + wkey));
        run("in_conv_im2col", 0.0, [&] { return femasr_in_conv_im2col(x_nchw, ic_hi, ic_lo, B, cfg.in_channel, H, W, st); });
        if (ok()) {
          femasr_tc_args t;
          memset(&t, 0, sizeof(t));
          t.a_hi = ic_hi; t.a_lo = ic_lo; t.w_blob = wt->second.p; t.bias = ib;
          t.out_hi = in_hi; t.out_lo = in_lo;
          t.B = B; t.H = h; t.W = w; t.Cin = 64; t.Cout = c; t.ksize = 1; t.stride = 1; t.pair = -1; t.strip = -1;
          run("in_conv", in_flops, [&] { return femasr_tc_igemm(&t, st); });
        }
      }
      ar.release(ic_lo); ar.release(ic_hi);
    }
    // which enc_feats the decoder loop reads: at quantising levels (before_quant input) and, in the LQ stage with
    // use_residual, at the other levels > 0 (skip adds)
    bool need[3];
    for (int i = 0; i < 3; ++i)
      need[i] = net->level_cb[i] >= 0 || (i > 0 && !net->hq && cfg.use_residual);
    float* feats[3] = {nullptr, nullptr, nullptr};
    for (int i = 0; i < d; ++i) {
      const std::string b = enc + ".blocks." + std::to_string(i);
      const int ho = (h + 2 - 3) / 2 + 1, wo = (w + 2 - 3) / 2 + 1, co = chan((256 / cfg.scale_factor) >> (i + 1));
      float* nxt = ar.alloc((size_t)B * ho * wo * co);
      Stats sd0;
      if (tc) {
        sd0 = alloc_stats(B, h, w, c, co, 0, 2);
        conv_tc(b + ".0", cur, nxt, B, h, w, c, co, 3, 0, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr,
                i == 0 ? in_hi : nullptr, i == 0 ? in_lo : nullptr, nullptr, nullptr, sd0.partial, 2);
      } else {
        conv(b + ".0", cur, nxt, B, h, w, c, co, 3, 2, 0, FEMASR_PRO_NONE, nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr);
      }
      if (i == 0 && in_lo) { ar.release(in_lo); ar.release(in_hi); in_lo = in_hi = nullptr; }
      // HQ stage: enc_feats = the down blocks' outputs reversed (:316); block i-1's output is level d-i
      if (cur) { if (net->hq && i > 0 && need[d - i]) feats[d - i] = cur; else ar.release(cur); }
      cur = nxt; h = ho; w = wo; c = co;
      Stats sd = resblock(b + ".1", cur, B, h, w, c, nullptr, sd0, true);
      resblock(b + ".2", cur, B, h, w, c, nullptr, sd, false);
    }
    tap("down", cur, (size_t)B * h * w * c);
    if (!net->hq) swin(enc + ".blocks." + std::to_string(d), cur, B, h, w);
    tap("swin", cur, (size_t)B * h * w * c);
    feats[0] = cur;
    // the up branches reach the decoder's skip adds (femasr_arch.py:361-362) and, in multi-scale nets, the later quantisers
    precise_region = net->last_q_level >= 1;
    if (!net->hq && (need[1] || need[2])) {
      const std::string b1 = enc + ".blocks." + std::to_string(d + 1), b2 = enc + ".blocks." + std::to_string(d + 2);
      feats[1] = up_block(b1 + ".1", b1 + ".2", b1 + ".3", cur, B, h, w, 256, 256, nullptr);
      tap("up1", feats[1], (size_t)B * 2 * h * 2 * w * 256);
      if (need[2]) {
        precise_region = net->last_q_level >= 2;
        feats[2] = up_block(b2 + ".1", b2 + ".2", b2 + ".3", feats[1], B, 2 * h, 2 * w, 256, 128, nullptr);
        tap("up2", feats[2], (size_t)B * 4 * h * 4 * w * 128);
      }
    }
    precise_region = false;
    decode_loop(feats, nullptr, y_nchw, indices, cb_loss, gt, B, h, w);
    for (int i = 2; i >= 0; --i) if (feats[i]) ar.release(feats[i]);
  }

  void decode_indices(const int64_t* idx, float* y_nchw, int B, int h, int w) {
    const femasr_net::Codebook& cb = net->cbs[0];
    const size_t N = (size_t)B * h * w;
    float* zq = ar.alloc(N * cb.e_dim);
    if (!dry() && ok()) {
      const float* cbw = net->raw["quantize_group.0.embedding.weight"].p;
      run("codebook_gather", 0.0, [&] { return femasr_codebook_gather(idx, cbw, zq, (int)N, cb.n_e, cb.e_dim, st); });
    }
    const float* none[3] = {nullptr, nullptr, nullptr};
    decode_loop(none, zq, y_nchw, nullptr, nullptr, nullptr, B, h, w);
    ar.release(zq);
  }
};

static int check_geometry(femasr_net* net, int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return fail(FEMASR_ERR_ARG, "forward: empty input");
  if (net->hq) {
    if (H % 8 || W % 8) return fail(FEMASR_ERR_ARG, "forward (HQ stage): H and W must be multiples of 8");
    return FEMASR_OK;
  }
  const int div = net->cfg.scale_factor == 4 ? 2 : 4;
  if (H % 2 || W % 2) return fail(FEMASR_ERR_ARG, "forward: H and W must be even");
  const int hs = H / div, ws = W / div;
  if (H % div || W % div || hs % 8 || ws % 8 || hs == 0 || ws == 0)
    return fail(FEMASR_ERR_ARG, "forward: Swin stage (H/" + std::to_string(div) + " x W/" + std::to_string(div) +
                                    ") must be a non-empty multiple of the 8x8 window");
  return FEMASR_OK;
}

}  // namespace femasr

extern "C" const char* femasr_last_error(void) { return g_err.c_str(); }
extern "C" int femasr_abi_version(void) { return 5; }   // 3: fused VQ + im2col in_conv entries; 4: femasr_tc_args.f8 + the F8 staging / packing entries; 5: femasr_in_conv4x4_split removed

extern "C" int femasr_device_cc(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(FEMASR_ERR_NO_DEVICE, "no CUDA device");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return fail(FEMASR_ERR_NO_DEVICE, "no CUDA device");
  return prop.major * 10 + prop.minor;
}

extern "C" int femasr_net_create(const femasr_net_config* cfg, femasr_net** out) {
  FEMASR_CHECK_ARG(cfg && out, "net_create: null pointer");
  FEMASR_CHECK_ARG(cfg->scale_factor == 1 || cfg->scale_factor == 2 || cfg->scale_factor == 4,
                   "net_create: scale_factor must be 4, 2 (LQ stage) or 1 (HQ autoencoder stage)");
  FEMASR_CHECK_ARG(cfg->in_channel == 3, "net_create: in_channel must be 3");
  FEMASR_CHECK_ARG(cfg->gemm_path == 0 || cfg->gemm_path == 1, "net_create: gemm_path must be 0 or 1");
  FEMASR_CHECK_ARG(cfg->n_codebooks >= 0 && cfg->n_codebooks <= FEMASR_MAX_CODEBOOKS, "net_create: at most 3 codebooks");
  std::vector<femasr_net::Codebook> cbs;
  if (cfg->n_codebooks <= 1 && !(cfg->n_codebooks == 1 && cfg->cb_scale[0]))
    cbs.push_back({32, cfg->n_e, cfg->e_dim});
  else
    for (int k = 0; k < cfg->n_codebooks; ++k) cbs.push_back({cfg->cb_scale[k], cfg->cb_n_e[k], cfg->cb_e_dim[k]});
  FEMASR_CHECK_ARG(cbs[0].scale == 32, "net_create: the first codebook must be at scale 32 (femasr_arch.py:255-256)");
  for (size_t k = 0; k < cbs.size(); ++k) {
    FEMASR_CHECK_ARG(cbs[k].e_dim > 0 && cbs[k].e_dim % 64 == 0 && cbs[k].e_dim <= 1024, "net_create: e_dim must be a multiple of 64");
    FEMASR_CHECK_ARG(cbs[k].n_e > 0 && cbs[k].n_e % 64 == 0, "net_create: n_e must be a multiple of 64");
    FEMASR_CHECK_ARG(k == 0 || ((cbs[k].scale == 64 || cbs[k].scale == 128) && cbs[k].scale > cbs[k - 1].scale),
                     "net_create: further codebooks must sit at increasing scales out of 64, 128");
  }
  femasr_net* n = new femasr_net();
  n->cfg = *cfg;
  n->cfg.n_e = cbs[0].n_e; n->cfg.e_dim = cbs[0].e_dim;
  n->cbs = cbs;
  for (size_t k = 0; k < cbs.size(); ++k) {
    const int lvl = cbs[k].scale == 32 ? 0 : (cbs[k].scale == 64 ? 1 : 2);
    n->level_cb[lvl] = (int)k;
    n->last_q_level = lvl;
  }
  n->depth = cfg->scale_factor == 4 ? 1 : (cfg->scale_factor == 2 ? 2 : 3);
  n->hq = cfg->scale_factor == 1;
  if (const char* ev = getenv("FEMASR_F8_CROSS")) n->f8_cross = atoi(ev) != 0;
  build_spec(n);
  *out = n;
  return FEMASR_OK;
}

extern "C" void femasr_net_destroy(femasr_net* net) { delete net; }

extern "C" int femasr_net_set_param(femasr_net* net, const char* name, const float* data, size_t numel, int on_device,
                                    void* stream) {
  FEMASR_CHECK_ARG(net && name && data, "set_param: null pointer");
  auto it = net->spec.find(name);
  if (it == net->spec.end()) return fail(FEMASR_ERR_ARG, std::string("set_param: unknown parameter ") + name);
  const ParamInfo& pi = it->second;
  if (pi.numel != numel) return fail(FEMASR_ERR_ARG, std::string("set_param: wrong size for ") + name);
  cudaStream_t st = as_stream(stream);
  DevBuf& rb = net->raw[name];
  if (!rb.p) { FEMASR_CUDA(cudaMalloc(&rb.p, numel * sizeof(float))); rb.n = numel; }
  FEMASR_CUDA(cudaMemcpyAsync(rb.p, data, numel * sizeof(float), on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  if (!on_device) FEMASR_CUDA(cudaStreamSynchronize(st));   // the host buffer may be pageable / freed by the caller
  std::string key(name);
  if (pi.kind == 1) {
    DevBuf& pb = net->packed[key];
    if (!pb.p) { FEMASR_CUDA(cudaMalloc(&pb.p, numel * sizeof(float))); pb.n = numel; }
    int s = femasr_pack_weight(rb.p, pb.p, pi.Cout, pi.Cin, pi.k, pi.k, st);
    if (s) return s;
    if (net->cfg.gemm_path == 1 && pi.k == 4 && pi.Cin == 3 && pi.Cout % 64 == 0) {
      // in_conv as a K = 48 -> 64 tensor-core GEMM over im2col rows: [Cout][64] padded matrix -> split-fp16 blob
      float* tmp = nullptr;
      FEMASR_CUDA(cudaMallocAsync(&tmp, (size_t)pi.Cout * 64 * sizeof(float), st));
      s = femasr_in_conv_pad_weight(rb.p, tmp, pi.Cout, st);
      DevBuf& tb = net->tcw[key + "#im2col"];
      const size_t bytes = femasr_tc_weight_bytes(pi.Cout, 64, 1, 1);
      if (!s && !tb.p) { if (cudaMalloc(&tb.p, bytes) != cudaSuccess) s = fail(FEMASR_ERR_CUDA, "cudaMalloc failed"); tb.n = bytes / sizeof(float); }
      if (!s) s = femasr_tc_pack_weight(tmp, tb.p, pi.Cout, 64, 1, 1, st);
      cudaFreeAsync(tmp, st);
      return s;
    }
    if (net->cfg.gemm_path == 1 && (pi.k == 1 || pi.k == 3) && pi.Cin % 64 == 0 && pi.Cout % 64 == 0) {
      DevBuf& tb = net->tcw[key];
      const size_t bytes = femasr_tc_weight_bytes(pi.Cout, pi.Cin, pi.k, pi.k);
      if (!tb.p) { FEMASR_CUDA(cudaMalloc(&tb.p, bytes)); tb.n = bytes / sizeof(float); }
      s = femasr_tc_pack_weight(rb.p, tb.p, pi.Cout, pi.Cin, pi.k, pi.k, st);
      if (s) return s;
      if (net->f8_cross && pi.k == 3) {      // a 3x3 conv may run behind the VQ: keep the F8 packing next to the fp16 one
        DevBuf& t8 = net->tcw8[key];
        if (!t8.p) { FEMASR_CUDA(cudaMalloc(&t8.p, bytes)); t8.n = bytes / sizeof(float); }
        s = femasr_tc_pack_weight_f8(rb.p, t8.p, pi.Cout, pi.Cin, pi.k, pi.k, st);
        if (s) return s;
      }
      // the five nearest-x2 -> conv3x3 sites (femasr_arch.py:172-173, 202-203) also get sub-pixel phase filters
      const std::string up1 = "multiscale_encoder.blocks." + std::to_string(net->depth + 1) + ".1.weight";
      const std::string up2 = "multiscale_encoder.blocks." + std::to_string(net->depth + 2) + ".1.weight";
      const bool is_up = pi.k == 3 && (key == up1 || key == up2 || (key.rfind("decoder_group.", 0) == 0 &&
                                        key.size() > 15 && key.compare(key.size() - 15, 15, ".block.1.weight") == 0));
      if (is_up) {
        DevBuf& ub = net->tcw_up[key];
        const size_t ubytes = femasr_tc_weight_bytes(4 * pi.Cout, pi.Cin, 2, 2);
        if (!ub.p) { FEMASR_CUDA(cudaMalloc(&ub.p, ubytes)); ub.n = ubytes / sizeof(float); }
        s = femasr_tc_pack_weight_up2(rb.p, ub.p, pi.Cout, pi.Cin, st);
        if (s || !net->f8_cross) return s;
        DevBuf& u8 = net->tcw_up8[key];
        if (!u8.p) { FEMASR_CUDA(cudaMalloc(&u8.p, ubytes)); u8.n = ubytes / sizeof(float); }
        return femasr_tc_pack_weight_up2_f8(rb.p, u8.p, pi.Cout, pi.Cin, st);
      }
      return FEMASR_OK;
    }
    return FEMASR_OK;
  }
  if (pi.kind == 2) {
    DevBuf& pb = net->packed[key];
    if (!pb.p) { FEMASR_CUDA(cudaMalloc(&pb.p, 8 * 64 * 64 * sizeof(float))); pb.n = 8 * 64 * 64; }
    DevBuf& mb = net->packed_mma[key];
    if (!mb.p) { FEMASR_CUDA(cudaMalloc(&mb.p, 8 * 64 * 64 * sizeof(float))); mb.n = 8 * 64 * 64; }
    int s = femasr_expand_rel_bias_mma(rb.p, mb.p, 8, st);
    if (s) return s;
    return femasr_expand_rel_bias(rb.p, pb.p, 8, st);
  }
  if (pi.kind == 3) {
    DevBuf& pb = net->packed[key];     // codebook^T as a GEMM operand [e_dim][n_e]
    if (!pb.p) { FEMASR_CUDA(cudaMalloc(&pb.p, numel * sizeof(float))); pb.n = numel; }
    int s = femasr_pack_weight(rb.p, pb.p, pi.Cout, pi.Cin, 1, 1, st);
    if (s) return s;
    DevBuf& eb = net->esq[key];
    if (!eb.p) { FEMASR_CUDA(cudaMalloc(&eb.p, pi.Cout * sizeof(float))); eb.n = pi.Cout; }
    s = femasr_row_sumsq(rb.p, eb.p, pi.Cout, pi.Cin, st);
    if (s) return s;
    if (net->cfg.gemm_path == 1) {     // split-fp16 planes of the [n_e, e_dim] embedding: B operand of the fused VQ
      DevBuf& tb = net->tcw[key];
      const size_t bytes = femasr_tc_weight_bytes(pi.Cout, pi.Cin, 1, 1);
      if (!tb.p) { FEMASR_CUDA(cudaMalloc(&tb.p, bytes)); tb.n = bytes / sizeof(float); }
      return femasr_tc_pack_weight(rb.p, tb.p, pi.Cout, pi.Cin, 1, 1, st);
    }
    return FEMASR_OK;
  }
  return FEMASR_OK;
}

extern "C" int femasr_net_params_complete(femasr_net* net) {
  FEMASR_CHECK_ARG(net, "params_complete: null");
  for (auto& kv : net->spec)
    if (net->raw.find(kv.first) == net->raw.end()) return fail(FEMASR_ERR_STATE, "parameter not set: " + kv.first);
  return FEMASR_OK;
}

extern "C" int femasr_net_workspace_bytes(femasr_net* net, int B, int H, int W, size_t* bytes) {
  FEMASR_CHECK_ARG(net && bytes, "workspace_bytes: null pointer");
  int s = check_geometry(net, B, H, W);
  if (s) return s;
  Ctx c; c.net = net; c.st = nullptr; c.ar.dry = true; c.ar.base = reinterpret_cast<char*>(uintptr_t(1) << 40);
  // sized for the gt_indices loss branch too (its scratch is small): one workspace serves forward and forward_gt
  c.forward(nullptr, nullptr, nullptr, nullptr, reinterpret_cast<const int64_t*>(uintptr_t(8)), B, H, W);
  *bytes = c.ar.peak + 256;
  return c.status;
}

extern "C" int femasr_net_forward(femasr_net* net, const float* x, float* y, int64_t* indices, float* cb_loss, int B,
                                  int H, int W, void* workspace, size_t workspace_bytes, void* stream) {
  return femasr_net_forward_gt(net, x, y, indices, cb_loss, nullptr, B, H, W, workspace, workspace_bytes, stream);
}

extern "C" int femasr_net_forward_gt(femasr_net* net, const float* x, float* y, int64_t* indices, float* cb_loss,
                                     const int64_t* gt_indices, int B, int H, int W, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  FEMASR_CHECK_ARG(net && x && y && workspace, "forward: null pointer");
  int s = check_geometry(net, B, H, W);
  if (s) return s;
  s = femasr_net_params_complete(net);
  if (s) return s;
  size_t need = 0;
  s = femasr_net_workspace_bytes(net, B, H, W, &need);
  if (s) return s;
  const uintptr_t mis = (256 - ((uintptr_t)workspace & 255)) & 255;
  if (workspace_bytes < need) return fail(FEMASR_ERR_STATE, "forward: workspace too small (need " + std::to_string(need) + " bytes)");
  Ctx c; c.net = net; c.st = as_stream(stream); c.ar.dry = false;
  c.ar.base = reinterpret_cast<char*>(workspace) + mis; c.ar.cap = workspace_bytes - mis;
  const long l0 = g_launches;
  c.forward(x, y, indices, cb_loss, gt_indices, B, H, W);
  net->last_launches = (int)(g_launches - l0);
  return c.status;
}

extern "C" int femasr_net_decode_workspace_bytes(femasr_net* net, int B, int h, int w, size_t* bytes) {
  FEMASR_CHECK_ARG(net && bytes && B > 0 && h > 0 && w > 0, "decode_workspace_bytes: bad argument");
  Ctx c; c.net = net; c.st = nullptr; c.ar.dry = true; c.ar.base = reinterpret_cast<char*>(uintptr_t(1) << 40);
  c.decode_indices(nullptr, nullptr, B, h, w);
  *bytes = c.ar.peak + 256;
  return c.status;
}

extern "C" int femasr_net_decode_indices(femasr_net* net, const int64_t* indices, float* y, int B, int h, int w,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  FEMASR_CHECK_ARG(net && indices && y && workspace && B > 0 && h > 0 && w > 0, "decode_indices: bad argument");
  int s = femasr_net_params_complete(net);
  if (s) return s;
  size_t need = 0;
  s = femasr_net_decode_workspace_bytes(net, B, h, w, &need);
  if (s) return s;
  if (workspace_bytes < need) return fail(FEMASR_ERR_STATE, "decode_indices: workspace too small");
  const uintptr_t mis = (256 - ((uintptr_t)workspace & 255)) & 255;
  Ctx c; c.net = net; c.st = as_stream(stream); c.ar.dry = false;
  c.ar.base = reinterpret_cast<char*>(workspace) + mis; c.ar.cap = workspace_bytes - mis;
  const long l0 = g_launches;
  c.decode_indices(indices, y, B, h, w);
  net->last_launches = (int)(g_launches - l0);
  return c.status;
}

extern "C" int femasr_net_set_tap(femasr_net* net, const char* stage, float* dst, size_t capacity) {
  FEMASR_CHECK_ARG(net && stage, "set_tap: null pointer");
  static const char* names[] = {"in_conv", "down", "swin", "up1", "up2", "z", "zq", "after_quant", "dec0", "dec1", "dec2", "z1", "z2"};
  bool known = false;
  for (const char* n : names) known = known || strcmp(n, stage) == 0;
  if (!known) return fail(FEMASR_ERR_ARG, std::string("set_tap: unknown stage ") + stage);
  if (dst) net->taps[stage] = Tap{dst, capacity};
  else net->taps.erase(stage);
  return FEMASR_OK;
}

extern "C" int femasr_net_last_launch_count(femasr_net* net) { return net ? net->last_launches : 0; }

extern "C" int femasr_net_set_profile(femasr_net* net, int enable) {
  FEMASR_CHECK_ARG(net, "set_profile: null");
  for (auto& r : net->prof) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
  net->prof.clear();
  net->profile = enable != 0;
  return FEMASR_OK;
}

// JSON {"kernel": {"launches": n, "ms": total, "flops": total}, ...} of the launches recorded since
// femasr_net_set_profile(net, 1).  Synchronises on the recorded events.
extern "C" const char* femasr_net_profile_json(femasr_net* net) {
  if (!net) return "{}";
  struct Agg { long n = 0; double ms = 0, flops = 0; };
  std::map<std::string, Agg> agg;
  for (auto& r : net->prof) {
    float ms = 0.f;
    if (cudaEventSynchronize(r.e1) != cudaSuccess || cudaEventElapsedTime(&ms, r.e0, r.e1) != cudaSuccess) continue;
    Agg& a = agg[r.name];
    a.n += 1; a.ms += ms; a.flops += r.flops;
  }
  std::string js = "{";
  bool first = true;
  for (auto& kv : agg) {
    char buf[256];
    snprintf(buf, sizeof(buf), "%s\"%s\": {\"launches\": %ld, \"ms\": %.6f, \"flops\": %.6e}", first ? "" : ", ",
             kv.first.c_str(), kv.second.n, kv.second.ms, kv.second.flops);
    js += buf;
    first = false;
  }
  js += "}";
  net->prof_json = js;
  return net->prof_json.c_str();
}

extern "C" double femasr_net_flops(femasr_net* net, int B, int H, int W) {
  if (!net) return 0.0;
  const int scale = net->cfg.scale_factor, d = net->depth;
  const double cin = chan(256 / scale);
  double f = 2.0 * 3 * 16 * cin * (H - 1) * (double)(W - 1);
  double ch = cin, hh = H, ww = W;
  for (int i = 0; i < d; ++i) {
    hh = std::floor(hh / 2); ww = std::floor(ww / 2);
    const double co = chan((256 / scale) >> (i + 1));
    f += 2.0 * 9 * ch * co * hh * ww + 4 * 2.0 * 9 * co * co * hh * ww;
    ch = co;
  }
  const double px = hh * ww;
  const double lin = 2.0 * 256 * (768 + 256 + 1024 + 1024) * px, att = 2 * 2.0 * 64 * 256 * px;
  if (!net->hq) f += 4 * (6 * (lin + att) + 2.0 * 9 * 256 * 256 * px);
  for (size_t k = 0; k < net->cbs.size(); ++k) {      // before_quant 1x1, z.E^T, after_quant 3x3 at each codebook's level
    const femasr_net::Codebook& cb = net->cbs[k];
    const double m = cb.scale / 32.0, pk = px * m * m, chk = chan(cb.scale), e = cb.e_dim;
    const double ein = k == 0 ? e : e + net->cbs[k - 1].e_dim;
    f += 2.0 * (k == 0 ? chk : 2 * chk) * e * pk + 2.0 * cb.n_e * e * pk + 2.0 * 9 * ein * chk * pk;
  }
  const double up[2][3] = {{256, 256, 2}, {256, 128, 4}};
  if (!net->hq) for (auto& u : up) f += (2.0 * 9 * u[0] * u[1] + 4 * 2.0 * 9 * u[1] * u[1]) * px * u[2] * u[2];
  const double dec[3][3] = {{256, 256, 2}, {256, 128, 4}, {128, 64, 8}};
  for (auto& u : dec) f += (2.0 * 9 * u[0] * u[1] + 4 * 2.0 * 9 * u[1] * u[1]) * px * u[2] * u[2];
  f += 2.0 * 9 * 64 * 3 * px * 64;
  return f * B;
}
