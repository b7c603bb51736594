// The skinny ends of the path and the layout / padding helpers (all HBM-bound, SIMT):
//   in_conv  4x4 p1, Cin=3   NCHW -> NHWC   (femasr_arch.py:150)
//   out_conv 3x3 p1, Cout=3  NHWC -> NCHW   (femasr_arch.py:273)
//   weight repack, NCHW<->NHWC, flip-pad (test(), :459-460), window copy (crop / tile paste)
#include <cuda_fp16.h>

#include "common.cuh"

namespace femasr {

// in_conv: 4x4, pad 1, Cin = 3.  Thread = (4 output channels) x (4 consecutive output pixels of one row): the
// 4x7x3 input patch lives in registers (loads are shared by all channel-quad threads of the pixel group through
// L1), every weight float4 is used for 16 FMAs, and the 4 stores per thread are contiguous across the warp's
// channel quads.
__global__ void __launch_bounds__(256) in_conv_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                      const float* __restrict__ bias, float* __restrict__ y,
                                                      int B, int H, int W, int Cout) {
  constexpr int KS = 4, CIN = 3, PX = 4;
  const int Ho = H - 1, Wo = W - 1;
  const int quads = Cout / 4;
  const int gpb = 256 / quads;                         // pixel groups per block
  const int q = threadIdx.x % quads;
  const int groups_x = (Wo + PX - 1) / PX;
  const long grp = (long)blockIdx.x * gpb + threadIdx.x / quads;
  const long ngrp = (long)B * Ho * groups_x;
  if (grp >= ngrp) return;
  const int gx = (int)(grp % groups_x);
  const long t = grp / groups_x;
  const int oy = (int)(t % Ho), b = (int)(t / Ho);
  const int ox0 = gx * PX;
  float patch[CIN][KS][PX + KS - 1];
#pragma unroll
  for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
    for (int r = 0; r < KS; ++r) {
      const int iy = oy + r - 1;
#pragma unroll
      for (int cidx = 0; cidx < PX + KS - 1; ++cidx) {
        const int ix = ox0 + cidx - 1;
        patch[ci][r][cidx] = (iy >= 0 && iy < H && ix >= 0 && ix < W) ? __ldg(x + (((long)b * CIN + ci) * H + iy) * W + ix) : 0.f;
      }
    }
  float4 acc[PX];
  const float4 bv = bias ? __ldg(reinterpret_cast<const float4*>(bias) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int p = 0; p < PX; ++p) acc[p] = bv;
#pragma unroll
  for (int kh = 0; kh < KS; ++kh)
#pragma unroll
    for (int kw = 0; kw < KS; ++kw)
#pragma unroll
      for (int ci = 0; ci < CIN; ++ci) {
        const float4 wv = __ldg(reinterpret_cast<const float4*>(w + ((long)(kh * KS + kw) * CIN + ci) * Cout) + q);
#pragma unroll
        for (int p = 0; p < PX; ++p) {
          const float xv = patch[ci][kh][p + kw];
          acc[p].x = fmaf(xv, wv.x, acc[p].x); acc[p].y = fmaf(xv, wv.y, acc[p].y);
          acc[p].z = fmaf(xv, wv.z, acc[p].z); acc[p].w = fmaf(xv, wv.w, acc[p].w);
        }
      }
#pragma unroll
  for (int p = 0; p < PX; ++p) {
    const int ox = ox0 + p;
    if (ox >= Wo) break;
    const long e = ((((long)b * Ho + oy) * Wo + ox) * Cout) + q * 4;
    *reinterpret_cast<float4*>(y + e) = acc[p];
  }
}

// out_conv: 3x3, Cin=64 -> 3.  The input tile (with halo) is staged in shared memory by coalesced 16-byte
// loads (NHWC rows are contiguous), pixel stride padded to 68 floats so the per-thread float4 reads are
// bank-conflict free; the 1728 weights sit in __constant__ memory (uniform across the warp -> FFMA with a
// constant operand, no load instruction).  One thread per output pixel, tile = 4 rows x 32 cols.
constexpr int OC_CIN = 64, OC_TH = 4, OC_TW = 32, OC_PS = 68;   // pixel stride in floats
__constant__ float c_outconv_w[9 * OC_CIN * 3];
__constant__ float c_outconv_b[4];

__global__ void __launch_bounds__(OC_TH * OC_TW) out_conv_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                                 int B, int H, int W) {
  extern __shared__ __align__(16) float tile[];      // [(OC_TH+2)][(OC_TW+2)][OC_PS]
  const int x0 = blockIdx.x * OC_TW, y0 = blockIdx.y * OC_TH, b = blockIdx.z;
  constexpr int TWH = OC_TW + 2, THH = OC_TH + 2;
  // cooperative halo load: (THH*TWH) pixels x 16 float4
  for (int i = threadIdx.x; i < THH * TWH * (OC_CIN / 4); i += OC_TH * OC_TW) {
    const int c4 = i % (OC_CIN / 4);
    const int pp = i / (OC_CIN / 4);
    const int px = pp % TWH, py = pp / TWH;
    const int gy = y0 + py - 1, gx = x0 + px - 1;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gy >= 0 && gy < H && gx >= 0 && gx < W)
      v = __ldg(reinterpret_cast<const float4*>(x + (((long)b * H + gy) * W + gx) * OC_CIN) + c4);
    *reinterpret_cast<float4*>(&tile[(py * TWH + px) * OC_PS + c4 * 4]) = v;
  }
  __syncthreads();
  const int lx = threadIdx.x % OC_TW, ly = threadIdx.x / OC_TW;
  const int ox = x0 + lx, oy = y0 + ly;
  float a0 = c_outconv_b[0], a1 = c_outconv_b[1], a2 = c_outconv_b[2];
#pragma unroll 1
  for (int kh = 0; kh < 3; ++kh)
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
      const float* px = &tile[((ly + kh) * TWH + lx + kw) * OC_PS];
      const float* wt = c_outconv_w + (kh * 3 + kw) * OC_CIN * 3;
#pragma unroll 4
      for (int c4 = 0; c4 < OC_CIN / 4; ++c4) {
        const float4 v = *reinterpret_cast<const float4*>(px + c4 * 4);
        const float* wk = wt + c4 * 12;
        a0 = fmaf(v.x, wk[0], a0); a1 = fmaf(v.x, wk[1], a1); a2 = fmaf(v.x, wk[2], a2);
        a0 = fmaf(v.y, wk[3], a0); a1 = fmaf(v.y, wk[4], a1); a2 = fmaf(v.y, wk[5], a2);
        a0 = fmaf(v.z, wk[6], a0); a1 = fmaf(v.z, wk[7], a1); a2 = fmaf(v.z, wk[8], a2);
        a0 = fmaf(v.w, wk[9], a0); a1 = fmaf(v.w, wk[10], a1); a2 = fmaf(v.w, wk[11], a2);
      }
    }
  if (ox < W && oy < H) {
    const long plane = (long)H * W;
    float* o = y + (long)b * 3 * plane + (long)oy * W + ox;
    o[0] = a0; o[plane] = a1; o[2 * plane] = a2;
  }
}

__global__ void pack_weight_kernel(const float* __restrict__ w, float* __restrict__ out, int Cout, int Cin, int KH, int KW) {
  const long n = (long)Cout * Cin * KH * KW;
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // i indexes the packed layout [(kh*KW+kw)*Cin + ci][co]
  const int co = (int)(i % Cout);
  long k = i / Cout;
  const int ci = (int)(k % Cin);
  const int tap = (int)(k / Cin);
  const int kh = tap / KW, kw = tap - kh * KW;
  out[i] = w[(((long)co * Cin + ci) * KH + kh) * KW + kw];
}

__global__ void nchw_to_nhwc_kernel(const float* __restrict__ x, float* __restrict__ y, int C, long HW, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;   // NHWC index
  if (i >= n) return;
  const int c = (int)(i % C);
  const long p = (i / C) % HW, b = i / C / HW;
  y[i] = x[(b * C + c) * HW + p];
}
__global__ void nhwc_to_nchw_kernel(const float* __restrict__ x, float* __restrict__ y, int C, long HW, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;   // NCHW index
  if (i >= n) return;
  const long p = i % HW;
  const int c = (int)((i / HW) % C);
  const long b = i / HW / C;
  y[i] = x[(b * HW + p) * C + c];
}

__global__ void flip_pad_kernel(const float* __restrict__ x, float* __restrict__ y, int h, int w, int hp, int wp, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int j = (int)(i % wp);
  const int r = (int)((i / wp) % hp);
  const long bc = i / wp / hp;
  const int sr = r < h ? r : 2 * h - 1 - r;          // cat([x, flip(x)])[:h+pad]
  const int sj = j < w ? j : 2 * w - 1 - j;
  y[i] = x[(bc * h + sr) * w + sj];
}

// uint8 image boundary (SURVEY 8f rank 1; inference_femasr.py:54-56,64 + basicsr/utils/img_util.py:9-35,38-94):
//   in : uint8 HWC BGR [B,h,w,3]  -> fp32 NCHW RGB /255, flip-padded to [B,3,hp,wp]  (img2tensor, /255., test() padding)
//   out: fp32 NCHW RGB [B,3,SH,SW] -> clamp to [0,1], *255, round-half-even, uint8 HWC BGR, cropped to [B,ch,cw,3]
__global__ void u8_to_input_kernel(const uint8_t* __restrict__ img, float* __restrict__ x, int h, int w, int hp, int wp, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;     // index into [B,3,hp,wp]
  if (i >= n) return;
  const int j = (int)(i % wp);
  const int r = (int)((i / wp) % hp);
  const int c = (int)((i / wp / hp) % 3);
  const long b = i / wp / hp / 3;
  const int sr = r < h ? r : 2 * h - 1 - r, sj = j < w ? j : 2 * w - 1 - j;
  x[i] = (float)img[((b * h + sr) * w + sj) * 3 + (2 - c)] / 255.0f;   // torch: float32(img) / 255.
}
__global__ void output_to_u8_kernel(const float* __restrict__ y, uint8_t* __restrict__ img, int SH, int SW, int ch, int cw, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;     // index into [B,ch,cw,3]
  if (i >= n) return;
  const int c = (int)(i % 3);
  const int j = (int)((i / 3) % cw);
  const int r = (int)((i / 3 / cw) % ch);
  const long b = i / 3 / cw / ch;
  float v = y[((b * 3 + (2 - c)) * SH + r) * SW + j];
  v = fminf(fmaxf(v, 0.0f), 1.0f);
  img[i] = (uint8_t)rintf(v * 255.0f);                              // numpy round(): half to even
}

__global__ void copy_window_kernel(const float* __restrict__ src, float* __restrict__ dst, int sh, int sw, int dh, int dw,
                                   int sy, int sx, int dy, int dx, int ch, int cw, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int j = (int)(i % cw);
  const int r = (int)((i / cw) % ch);
  const long bc = i / cw / ch;
  dst[(bc * dh + dy + r) * dw + dx + j] = src[(bc * sh + sy + r) * sw + sx + j];
}

}  // namespace femasr

using namespace femasr;

extern "C" int femasr_in_conv4x4(const float* x, const float* w, const float* bias, float* y, int B, int Cin, int H,
                                 int W, int Cout, void* stream) {
  FEMASR_CHECK_ARG(x && w && y, "in_conv: null pointer");
  FEMASR_CHECK_ARG(B > 0 && H >= 3 && W >= 3 && Cin == 3, "in_conv: needs Cin == 3 and H, W >= 3");
  FEMASR_CHECK_ARG(Cout % 4 == 0 && 256 % (Cout / 4) == 0 && Cout <= 1024, "in_conv: unsupported Cout");
  const long ngrp = (long)B * (H - 1) * cdiv(W - 1, 4);
  const int gpb = 256 / (Cout / 4);
  const unsigned grid = (unsigned)cdiv(ngrp, gpb);
  in_conv_kernel<<<grid, 256, 0, as_stream(stream)>>>(x, w, bias, y, B, H, W, Cout);
  return launch_status("in_conv_kernel");
}

// in_conv on the tensor cores: the 4x4x3 patch of every output pixel as one K = 48 (padded to 64) row of split-fp16
// operand planes, consumed by femasr_tc_igemm as a 1x1 "linear" (femasr_arch.py:150).  k = (kh * 4 + kw) * 3 + ci.
__global__ void __launch_bounds__(256) in_conv_im2col_kernel(const float* __restrict__ x, uint4* __restrict__ hi,
                                                             uint4* __restrict__ lo, int B, int H, int W, long total) {
  const long i = (long)blockIdx.x * 256 + threadIdx.x;      // (output pixel, 8-wide k chunk)
  if (i >= total) return;
  const int j = (int)(i & 7);
  const long m = i >> 3;
  const int Ho = H - 1, Wo = W - 1;
  const int ox = (int)(m % Wo);
  const long t = m / Wo;
  const int oy = (int)(t % Ho), b = (int)(t / Ho);
  __align__(16) __half h[8], l[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int k = j * 8 + e;
    float v = 0.f;
    if (k < 48) {
      const int tap = k / 3, ci = k - tap * 3;
      const int iy = oy + (tap >> 2) - 1, ix = ox + (tap & 3) - 1;
      if (iy >= 0 && iy < H && ix >= 0 && ix < W) v = __ldg(x + (((long)b * 3 + ci) * H + iy) * W + ix);
    }
    const float cl = fminf(fmaxf(v, -65504.f), 65504.f);
    h[e] = __float2half_rn(cl);
    l[e] = __float2half_rn(cl - __half2float(h[e]));
  }
  hi[i] = *reinterpret_cast<const uint4*>(h);
  lo[i] = *reinterpret_cast<const uint4*>(l);
}

// OIHW [Cout,3,4,4] -> [Cout][64] fp32 in the im2col K order, zero padded (then femasr_tc_pack_weight(.., Cout, 64, 1, 1))
__global__ void in_conv_weight_pad_kernel(const float* __restrict__ w, float* __restrict__ out, int Cout) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Cout * 64) return;
  const int co = i >> 6, k = i & 63;
  float v = 0.f;
  if (k < 48) { const int tap = k / 3, ci = k - tap * 3; v = w[((co * 3 + ci) * 4 + (tap >> 2)) * 4 + (tap & 3)]; }
  out[i] = v;
}

extern "C" int femasr_in_conv_im2col(const float* x, void* a_hi, void* a_lo, int B, int Cin, int H, int W, void* stream) {
  FEMASR_CHECK_ARG(x && a_hi && a_lo && B > 0 && H > 1 && W > 1, "in_conv_im2col: bad argument");
  FEMASR_CHECK_ARG(Cin == 3, "in_conv_im2col: Cin must be 3");
  const long total = (long)B * (H - 1) * (W - 1) * 8;
  in_conv_im2col_kernel<<<(unsigned)cdiv(total, 256), 256, 0, as_stream(stream)>>>(
      x, reinterpret_cast<uint4*>(a_hi), reinterpret_cast<uint4*>(a_lo), B, H, W, total);
  return launch_status("in_conv_im2col_kernel");
}

extern "C" int femasr_in_conv_pad_weight(const float* w_oihw, float* w_padded, int Cout, void* stream) {
  FEMASR_CHECK_ARG(w_oihw && w_padded && Cout > 0, "in_conv_pad_weight: bad argument");
  in_conv_weight_pad_kernel<<<(unsigned)cdiv((long)Cout * 64, 256), 256, 0, as_stream(stream)>>>(w_oihw, w_padded, Cout);
  return launch_status("in_conv_weight_pad_kernel");
}

extern "C" int femasr_out_conv3x3(const float* x, const float* w, const float* bias, float* y, int B, int H, int W,
                                  int Cin, void* stream) {
  FEMASR_CHECK_ARG(x && w && bias && y, "out_conv: null pointer");
  FEMASR_CHECK_ARG(B > 0 && H > 0 && W > 0, "out_conv: empty input");
  FEMASR_CHECK_ARG(Cin == OC_CIN, "out_conv: Cin must be 64 (channel_query_dict[256])");
  FEMASR_CHECK_ARG(cdiv(H, OC_TH) <= 65535 && B <= 65535, "out_conv: grid too large");
  cudaStream_t st = as_stream(stream);
  // weights travel through __constant__ memory; refreshed per call (stream-ordered) so several engines can coexist
  FEMASR_CUDA(cudaMemcpyToSymbolAsync(c_outconv_w, w, sizeof(float) * 9 * OC_CIN * 3, 0, cudaMemcpyDeviceToDevice, st));
  FEMASR_CUDA(cudaMemcpyToSymbolAsync(c_outconv_b, bias, sizeof(float) * 3, 0, cudaMemcpyDeviceToDevice, st));
  constexpr int smem = (OC_TH + 2) * (OC_TW + 2) * OC_PS * (int)sizeof(float);
  static PerDeviceFlag attr_set;
  if (!attr_set.cur()) {
    FEMASR_CUDA(cudaFuncSetAttribute(out_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_set.cur() = true;
  }
  dim3 grid((unsigned)cdiv(W, OC_TW), (unsigned)cdiv(H, OC_TH), B);
  out_conv_kernel<<<grid, OC_TH * OC_TW, smem, st>>>(x, y, B, H, W);
  return launch_status("out_conv_kernel");
}

// ------------------------------------------------------------------------------------------------
// out_conv on warp-level tensor cores (mma.sync m16n8k16, 3-term split fp16 like the big GEMMs), used by the
// tensor-core path.  The SIMT kernel above is bound by shared-memory reads (576 values per pixel for 3 outputs).
// Here the three horizontal taps are folded into the N dimension: for an output row y the warp accumulates
//     Q[x'][kw*3+co] = sum_kh sum_c X[y+kh-1][x'][c] * W[kh][kw][c][co]        (M = pixels x', N = 9 -> 16, K = 3*64)
// for the 32 halo pixels x' of its row (two m-tiles), so every activation fragment is fetched ONCE per (kh, 16
// channels) instead of once per tap, and then   out[x][co] = bias + Q[x][co] + Q[x+1][3+co] + Q[x+2][6+co]
// (a 3-term shift-add through a per-warp scratch).  Tile: 8 output rows x 30 columns per CTA (warp = row).
constexpr int OM_TH = 8, OM_TW = 30, OM_PX = 32, OM_PB = 144;     // halo pixels per row, bytes per pixel and plane (128 + pad)
constexpr int OM_PLANE = (OM_TH + 2) * OM_PX * OM_PB;             // 46080 B per fp16 plane
constexpr int OM_SMEM = 2 * OM_PLANE + OM_TH * OM_PX * 9 * (int)sizeof(float);
constexpr float OM_WSCALE = 256.0f;                               // weights * 2^8: keeps the lo plane out of fp16 subnormals
__device__ uint32_t g_outconv_bfrag[3 * 4 * 2 * 2 * 2 * 32];       // [kh][kc][nt][plane][reg][lane] B fragments (refreshed per call)

// (x, y) -> packed fp16 pairs hi = rn(v), lo = rn(v - hi), saturating at +-65504 like the big GEMMs' operand staging
__device__ __forceinline__ void oc_split2(float x, float y, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(y), "f"(x));
  const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(y - hf.y), "f"(x - hf.x));
}

// w: K-major packed [tap][c][co] fp32 (femasr_pack_weight).  One thread per (kh, kc, nt, reg, lane).
__global__ void out_conv_bfrag_kernel(const float* __restrict__ w) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 3 * 4 * 2 * 2 * 32) return;
  const int lane = idx & 31, reg = (idx >> 5) & 1, nt = (idx >> 6) & 1, kc = (idx >> 7) & 3, kh = idx >> 9;
  const int g = lane >> 2, cq = lane & 3;
  const int n = nt * 8 + g;                       // column = kw*3 + co
  float v0 = 0.f, v1 = 0.f;
  if (n < 9) {
    const int kw = n / 3, co = n - 3 * kw;
    const int ch = 16 * kc + 2 * cq + 8 * reg;    // B fragment: b0 = k 2c,2c+1; b1 = k 2c+8,2c+9
    v0 = w[(((kh * 3 + kw) * OC_CIN) + ch) * 3 + co] * OM_WSCALE;
    v1 = w[(((kh * 3 + kw) * OC_CIN) + ch + 1) * 3 + co] * OM_WSCALE;
  }
  uint32_t hi, lo;
  oc_split2(v0, v1, hi, lo);
  const int base = (((kh * 4 + kc) * 2 + nt) * 2) * 2;        // [plane][reg]
  g_outconv_bfrag[(base + 0 * 2 + reg) * 32 + lane] = hi;
  g_outconv_bfrag[(base + 1 * 2 + reg) * 32 + lane] = lo;
}

__global__ void __launch_bounds__(OM_TH * 32, 2) out_conv_mma_kernel(const float* __restrict__ x, const float* __restrict__ bias,
                                                                     float* __restrict__ y, int B, int H, int W) {
  extern __shared__ __align__(16) uint8_t om_smem[];
  uint8_t* plane_hi = om_smem;
  uint8_t* plane_lo = om_smem + OM_PLANE;
  float* qs_all = reinterpret_cast<float*>(om_smem + 2 * OM_PLANE);
  const int x0 = blockIdx.x * OM_TW - 1, y0 = blockIdx.y * OM_TH - 1, b = blockIdx.z;     // halo origin
  // stage the (TH+2) x 32 halo pixels as split fp16: 16 consecutive threads fetch one pixel's 256 bytes; the loads of
  // a batch are all issued before the first conversion (the loop is otherwise one DRAM latency per iteration)
  constexpr int NIT = (OM_TH + 2) * OM_PX * (OC_CIN / 4) / (OM_TH * 32), UB = 5;
  static_assert(NIT % UB == 0 && NIT * OM_TH * 32 == (OM_TH + 2) * OM_PX * (OC_CIN / 4), "staging loop shape");
#pragma unroll 1
  for (int it = 0; it < NIT; it += UB) {
    float4 v[UB];
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      const int i = threadIdx.x + (it + u) * (OM_TH * 32);
      const int c4 = i & 15, pp = i >> 4;
      const int gy = y0 + (pp >> 5), gx = x0 + (pp & (OM_PX - 1));
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gy >= 0 && gy < H && gx >= 0 && gx < W)
        v[u] = __ldg(reinterpret_cast<const float4*>(x + (((long)b * H + gy) * W + gx) * OC_CIN) + c4);
    }
#pragma unroll
    for (int u = 0; u < UB; ++u) {
      const int i = threadIdx.x + (it + u) * (OM_TH * 32);
      uint32_t h0, l0, h1, l1;
      oc_split2(v[u].x, v[u].y, h0, l0);
      oc_split2(v[u].z, v[u].w, h1, l1);
      const int off = (i >> 4) * OM_PB + (i & 15) * 8;
      *reinterpret_cast<uint2*>(plane_hi + off) = make_uint2(h0, h1);
      *reinterpret_cast<uint2*>(plane_lo + off) = make_uint2(l0, l1);
    }
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, cq = lane & 3;
  float acc[2][2][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = acc[mt][nt][2] = acc[mt][nt][3] = 0.f;
  // ldmatrix row address: lane -> pixel (lane & 7) + 8 * ((lane >> 3) & 1) of the m-tile, channel block 8 * (lane >> 4)
  const int lpx = (lane & 7) + 8 * ((lane >> 3) & 1), lch = 8 * (lane >> 4);
  const uint32_t hi_base = (uint32_t)__cvta_generic_to_shared(plane_hi), lo_base = (uint32_t)__cvta_generic_to_shared(plane_lo);
#pragma unroll 1
  for (int kh = 0; kh < 3; ++kh) {
    uint32_t bh[4][2][2], bl[4][2][2];            // [kc][nt][reg]
#pragma unroll
    for (int kc = 0; kc < 4; ++kc)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const int base = (((kh * 4 + kc) * 2 + nt) * 2) * 2;
          bh[kc][nt][r] = g_outconv_bfrag[(base + r) * 32 + lane];
          bl[kc][nt][r] = g_outconv_bfrag[(base + 2 + r) * 32 + lane];
        }
    const int row = warp + kh;                    // halo row feeding output row `warp` through tap row kh
#pragma unroll
    for (int kc = 0; kc < 4; ++kc)
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        const uint32_t off = (uint32_t)((row * OM_PX + mt * 16 + lpx) * OM_PB + (kc * 16 + lch) * 2);
        uint32_t ah[4], al[4];
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                     : "=r"(ah[0]), "=r"(ah[1]), "=r"(ah[2]), "=r"(ah[3]) : "r"(hi_base + off));
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                     : "=r"(al[0]), "=r"(al[1]), "=r"(al[2]), "=r"(al[3]) : "r"(lo_base + off));
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          float(&d)[4] = acc[mt][nt];
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                       : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                       : "r"(al[0]), "r"(al[1]), "r"(al[2]), "r"(al[3]), "r"(bh[kc][nt][0]), "r"(bh[kc][nt][1]));
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                       : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                       : "r"(ah[0]), "r"(ah[1]), "r"(ah[2]), "r"(ah[3]), "r"(bl[kc][nt][0]), "r"(bl[kc][nt][1]));
          asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                       : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                       : "r"(ah[0]), "r"(ah[1]), "r"(ah[2]), "r"(ah[3]), "r"(bh[kc][nt][0]), "r"(bh[kc][nt][1]));
        }
      }
  }
  // shift-add over the three horizontal taps through this warp's scratch Q[32 pixels][9]
  float* qs = qs_all + warp * OM_PX * 9;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    const int p0 = mt * 16 + g, p1 = p0 + 8;
    qs[p0 * 9 + 2 * cq] = acc[mt][0][0]; qs[p0 * 9 + 2 * cq + 1] = acc[mt][0][1];
    qs[p1 * 9 + 2 * cq] = acc[mt][0][2]; qs[p1 * 9 + 2 * cq + 1] = acc[mt][0][3];
    if (cq == 0) { qs[p0 * 9 + 8] = acc[mt][1][0]; qs[p1 * 9 + 8] = acc[mt][1][2]; }
  }
  __syncwarp();
  const int oy = blockIdx.y * OM_TH + warp, ox = blockIdx.x * OM_TW + lane;
  if (lane < OM_TW && oy < H && ox < W) {
    const long plane = (long)H * W;
    float* o = y + (long)b * 3 * plane + (long)oy * W + ox;
    const float inv = 1.0f / OM_WSCALE;
#pragma unroll
    for (int co = 0; co < 3; ++co)
      o[co * plane] = __ldg(bias + co) + ((qs[lane * 9 + co] + qs[(lane + 1) * 9 + 3 + co]) + qs[(lane + 2) * 9 + 6 + co]) * inv;
  }
}

extern "C" int femasr_out_conv3x3_mma(const float* x, const float* w, const float* bias, float* y, int B, int H, int W,
                                      int Cin, void* stream) {
  FEMASR_CHECK_ARG(x && w && bias && y, "out_conv_mma: null pointer");
  FEMASR_CHECK_ARG(B > 0 && H > 0 && W > 0, "out_conv_mma: empty input");
  FEMASR_CHECK_ARG(Cin == OC_CIN, "out_conv_mma: Cin must be 64 (channel_query_dict[256])");
  FEMASR_CHECK_ARG(cdiv(H, OM_TH) <= 65535 && B <= 65535, "out_conv_mma: grid too large");
  cudaStream_t st = as_stream(stream);
  out_conv_bfrag_kernel<<<6, 256, 0, st>>>(w);     // stream-ordered refresh of the B fragments (several engines can coexist)
  static PerDeviceFlag attr_set;
  if (!attr_set.cur()) {
    FEMASR_CUDA(cudaFuncSetAttribute(out_conv_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, OM_SMEM));
    attr_set.cur() = true;
  }
  dim3 grid((unsigned)cdiv(W, OM_TW), (unsigned)cdiv(H, OM_TH), B);
  out_conv_mma_kernel<<<grid, OM_TH * 32, OM_SMEM, st>>>(x, bias, y, B, H, W);
  return launch_status("out_conv_mma_kernel");
}

extern "C" int femasr_pack_weight(const float* w, float* out, int Cout, int Cin, int kh, int kw, void* stream) {
  FEMASR_CHECK_ARG(w && out && Cout > 0 && Cin > 0 && kh > 0 && kw > 0, "pack_weight: bad argument");
  const long n = (long)Cout * Cin * kh * kw;
  pack_weight_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(w, out, Cout, Cin, kh, kw);
  return launch_status("pack_weight_kernel");
}

extern "C" int femasr_nchw_to_nhwc(const float* x, float* y, int B, int C, int H, int W, void* stream) {
  FEMASR_CHECK_ARG(x && y && B > 0 && C > 0 && H > 0 && W > 0, "nchw_to_nhwc: bad argument");
  const long n = (long)B * C * H * W;
  nchw_to_nhwc_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(x, y, C, (long)H * W, n);
  return launch_status("nchw_to_nhwc_kernel");
}
extern "C" int femasr_nhwc_to_nchw(const float* x, float* y, int B, int C, int H, int W, void* stream) {
  FEMASR_CHECK_ARG(x && y && B > 0 && C > 0 && H > 0 && W > 0, "nhwc_to_nchw: bad argument");
  const long n = (long)B * C * H * W;
  nhwc_to_nchw_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(x, y, C, (long)H * W, n);
  return launch_status("nhwc_to_nchw_kernel");
}

extern "C" int femasr_flip_pad(const float* x, float* y, int B, int C, int h, int w, int hp, int wp, void* stream) {
  FEMASR_CHECK_ARG(x && y && B > 0 && C > 0 && h > 0 && w > 0, "flip_pad: bad argument");
  FEMASR_CHECK_ARG(hp >= h && wp >= w && hp <= 2 * h && wp <= 2 * w, "flip_pad: pad must be within one reflection");
  const long n = (long)B * C * hp * wp;
  flip_pad_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(x, y, h, w, hp, wp, n);
  return launch_status("flip_pad_kernel");
}

extern "C" int femasr_u8_to_input(const uint8_t* bgr_hwc, float* x_nchw, int B, int h, int w, int hp, int wp, void* stream) {
  FEMASR_CHECK_ARG(bgr_hwc && x_nchw && B > 0 && h > 0 && w > 0, "u8_to_input: bad argument");
  FEMASR_CHECK_ARG(hp >= h && wp >= w && hp <= 2 * h && wp <= 2 * w, "u8_to_input: pad must be within one reflection");
  const long n = (long)B * 3 * hp * wp;
  u8_to_input_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(bgr_hwc, x_nchw, h, w, hp, wp, n);
  return launch_status("u8_to_input_kernel");
}

extern "C" int femasr_output_to_u8(const float* y_nchw, uint8_t* bgr_hwc, int B, int SH, int SW, int ch, int cw, void* stream) {
  FEMASR_CHECK_ARG(y_nchw && bgr_hwc && B > 0 && ch > 0 && cw > 0 && ch <= SH && cw <= SW, "output_to_u8: bad argument");
  const long n = (long)B * ch * cw * 3;
  output_to_u8_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(y_nchw, bgr_hwc, SH, SW, ch, cw, n);
  return launch_status("output_to_u8_kernel");
}

extern "C" int femasr_copy_window(const float* src, float* dst, int B, int C, int sh, int sw, int dh, int dw, int sy,
                                  int sx, int dy, int dx, int ch, int cw, void* stream) {
  FEMASR_CHECK_ARG(src && dst && B > 0 && C > 0, "copy_window: bad argument");
  FEMASR_CHECK_ARG(ch > 0 && cw > 0 && sy >= 0 && sx >= 0 && dy >= 0 && dx >= 0 && sy + ch <= sh && sx + cw <= sw &&
                       dy + ch <= dh && dx + cw <= dw, "copy_window: window out of bounds");
  const long n = (long)B * C * ch * cw;
  copy_window_kernel<<<(unsigned)cdiv(n, 256), 256, 0, as_stream(stream)>>>(src, dst, sh, sw, dh, dw, sy, sx, dy, dx, ch, cw, n);
  return launch_status("copy_window_kernel");
}
