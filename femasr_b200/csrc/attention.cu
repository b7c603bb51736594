// Shifted-window multi-head self-attention (8x8 windows, head_dim 32), fp32 SIMT.
// One CTA per (window, head); one thread per query token.  The cyclic shift (torch.roll), the window
// partition/reverse permutes and the 0/-100 shift mask of network_swinir.py:216-279 are pure index
// arithmetic here; nothing is materialised.  0.9% of the path's FLOPs (SURVEY 8a).
#include <cuda_fp16.h>

#include "common.cuh"

namespace femasr {

constexpr int WS = 8, WT = 64, HD = 32;

__device__ __forceinline__ int shift_region(int p, int n, int shift) {
  // img_mask regions of calculate_mask(): [0,n-8) -> 0, [n-8,n-shift) -> 1, [n-shift,n) -> 2
  return p < n - WS ? 0 : (p < n - shift ? 1 : 2);
}

__global__ void __launch_bounds__(64) window_attention_kernel(const float* __restrict__ qkv,
                                                              const float* __restrict__ bias_full,
                                                              float* __restrict__ out, int H, int W, int C,
                                                              int heads, int shift) {
  __shared__ __align__(16) float ks[WT][HD];
  __shared__ __align__(16) float vs[WT][HD];
  __shared__ int region[WT];
  const int head = blockIdx.x % heads;
  const int win = blockIdx.x / heads;
  const int nwx = W / WS, nwy = H / WS;
  const int b = win / (nwx * nwy);
  const int wrem = win - b * nwx * nwy;
  const int wy = wrem / nwx, wx = wrem - wy * nwx;
  const int t = threadIdx.x;               // token within window
  const int ys = wy * WS + t / WS, xs = wx * WS + (t % WS);          // shifted-frame coordinates
  const int yo = (ys + shift) % H, xo = (xs + shift) % W;            // original coordinates (roll by -shift)
  const long tok = ((long)b * H + yo) * W + xo;
  const float* row = qkv + tok * (3 * C);
  const float scale = 0.17677669529663687f;   // head_dim ** -0.5 for head_dim 32 (network_swinir.py:84)

  float q[HD];
#pragma unroll
  for (int i = 0; i < HD / 4; ++i) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(row + head * HD) + i);
    q[4 * i] = v.x * scale; q[4 * i + 1] = v.y * scale; q[4 * i + 2] = v.z * scale; q[4 * i + 3] = v.w * scale;
  }
#pragma unroll
  for (int i = 0; i < HD / 4; ++i) {
    reinterpret_cast<float4*>(ks[t])[i] = __ldg(reinterpret_cast<const float4*>(row + C + head * HD) + i);
    reinterpret_cast<float4*>(vs[t])[i] = __ldg(reinterpret_cast<const float4*>(row + 2 * C + head * HD) + i);
  }
  region[t] = shift > 0 ? shift_region(ys, H, shift) * 3 + shift_region(xs, W, shift) : 0;
  __syncthreads();

  const float* brow = bias_full + ((long)head * WT + t) * WT;
  const int myreg = region[t];
  float s[WT];
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < WT; ++j) {
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < HD; ++k) a = fmaf(q[k], ks[j][k], a);
    a += __ldg(brow + j);
    if (shift > 0 && region[j] != myreg) a += -100.0f;
    s[j] = a;
    mx = fmaxf(mx, a);
  }
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < WT; ++j) { s[j] = expf(s[j] - mx); sum += s[j]; }
  const float inv = 1.0f / sum;
  float o[HD];
#pragma unroll
  for (int k = 0; k < HD; ++k) o[k] = 0.f;
#pragma unroll
  for (int j = 0; j < WT; ++j) {
    const float pj = s[j] * inv;
#pragma unroll
    for (int k = 0; k < HD; ++k) o[k] = fmaf(pj, vs[j][k], o[k]);
  }
  float* orow = out + tok * C + head * HD;
#pragma unroll
  for (int i = 0; i < HD / 4; ++i)
    reinterpret_cast<float4*>(orow)[i] = make_float4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
}

// ------------------------------------------------------------------------------------------------
// Tensor-core variant (warp-level mma.sync m16n8k16, fp16 operands split hi/lo, fp32 accumulate): the
// 64x32x64 per-(window, head) products are far too small for a tcgen05 tile, so the legacy warp MMA path is
// the right tool here.  One CTA of 4 warps per (window, head); warp w owns query rows [16w, 16w+16).
//   S = (q*scale) K^T  -> + rel-pos bias (+ shift mask) -> softmax (fp32, in registers) -> O = P V.
// Both products use the same 3-term split as the big GEMMs (lo*hi + hi*lo + hi*hi).
// The kernel is bound by the LSU data pipe (ncu: l1tex wavefronts 91 %), so every access is shaped to need few of them:
//   * K / V rows are fetched with 8 consecutive lanes per 128-byte row and kept ROW-MAJOR in shared memory; the
//     B fragments come from ldmatrix.x4 (K) and ldmatrix.x4.trans (V) - no transposing 2-byte stores;
//   * the head dimension of Q and K is permuted (the contraction order of an MMA is free as long as both operands
//     agree) so that a lane's 8 Q values are 32 contiguous bytes: physical dim 8c+2m+e sits at MMA k-index 8m+2c+e;
//   * the relative-position bias is pre-arranged in accumulator-fragment order (femasr_expand_rel_bias_mma): one fully
//     coalesced 16-byte load per n-tile.
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_addr(p)));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_addr(p)));
}
// (x, y) -> packed fp16 pairs hi = rn(v), lo = rn(v - hi): 2 packed converts instead of 4 scalar ones
__device__ __forceinline__ void split2(float x, float y, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(x, y);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(x - hf.x, y - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

constexpr int KV_LD = 40;   // row stride in halves (80 B): the 8 row addresses of an ldmatrix phase hit 8 distinct 16-byte slots

// 7 resident CTAs per SM (72 registers): measured 0.139 ms per layer vs 0.141 at 6 (80 registers) and 0.181 when the
// compiler is left free to use more registers
__global__ void __launch_bounds__(128, 7) window_attention_mma_kernel(const float* __restrict__ qkv,
                                                                   const float* __restrict__ bias_frag,
                                                                   float* __restrict__ out, __half* __restrict__ out_hi,
                                                                   __half* __restrict__ out_lo, int H, int W, int C,
                                                                   int heads, int shift) {
  __shared__ __align__(16) __half Kh[WT * KV_LD], Kl[WT * KV_LD];   // [key][k-index]  (k-index = permuted head dim)
  __shared__ __align__(16) __half Vh[WT * KV_LD], Vl[WT * KV_LD];   // [key][permuted dim]
  __shared__ __align__(8) int region[WT];
  __shared__ long toks[WT];
  const int head = blockIdx.x % heads;
  const int win = blockIdx.x / heads;
  const int nwx = W / WS, nwy = H / WS;
  const int b = win / (nwx * nwy);
  const int wrem = win - b * nwx * nwy;
  const int wy = wrem / nwx, wx = wrem - wy * nwx;
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, c = lane & 3;
  {
    // staging: 8 consecutive threads fetch one token's 32 K (V) values; thread = (token tid/8 + 16 i, dims [4q, 4q+4))
    const int q = tid & 7;
    const int posA = 16 * (q & 1) + 2 * (q >> 1), posB = posA + 8;    // k-index of dims 4q,4q+1 / 4q+2,4q+3
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int j = (tid >> 3) + 16 * i;
      const int ys = wy * WS + j / WS, xs = wx * WS + (j % WS);
      int yo = ys + shift, xo = xs + shift;
      if (yo >= H) yo -= H;
      if (xo >= W) xo -= W;
      const long tok = ((long)b * H + yo) * W + xo;
      if (q == 0) {
        toks[j] = tok;
        region[j] = shift > 0 ? shift_region(ys, H, shift) * 3 + shift_region(xs, W, shift) : 0;
      }
      const float* base = qkv + tok * (3 * C) + head * HD + 4 * q;
      const float4 kv = __ldg(reinterpret_cast<const float4*>(base + C));
      const float4 vv = __ldg(reinterpret_cast<const float4*>(base + 2 * C));
      uint32_t h0, l0, h1, l1;
      split2(kv.x, kv.y, h0, l0);
      split2(kv.z, kv.w, h1, l1);
      *reinterpret_cast<uint32_t*>(&Kh[j * KV_LD + posA]) = h0; *reinterpret_cast<uint32_t*>(&Kh[j * KV_LD + posB]) = h1;
      *reinterpret_cast<uint32_t*>(&Kl[j * KV_LD + posA]) = l0; *reinterpret_cast<uint32_t*>(&Kl[j * KV_LD + posB]) = l1;
      split2(vv.x, vv.y, h0, l0);
      split2(vv.z, vv.w, h1, l1);
      // V columns get the same permutation: n-tile nt, column 2c+e of the P.V accumulator is then physical dim
      // 8c+2nt+e, i.e. a lane ends up with 8 CONTIGUOUS output dims (one 16-byte store per plane and row)
      *reinterpret_cast<uint32_t*>(&Vh[j * KV_LD + posA]) = h0; *reinterpret_cast<uint32_t*>(&Vh[j * KV_LD + posB]) = h1;
      *reinterpret_cast<uint32_t*>(&Vl[j * KV_LD + posA]) = l0; *reinterpret_cast<uint32_t*>(&Vl[j * KV_LD + posB]) = l1;
    }
  }
  // this warp's bias fragments (independent of the window): issue the loads before the barrier
  float4 bf[8];
  {
    const float4* bp = reinterpret_cast<const float4*>(bias_frag) + ((long)(head * 4 + warp) * 8) * 32 + lane;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) bf[nt] = __ldg(bp + nt * 32);
  }
  __syncthreads();

  const int r0 = warp * 16 + g, r1 = r0 + 8;
  const float scale = 0.17677669529663687f;
  // Q fragments (A operand), scaled then split: a lane owns dims [8c, 8c+8) of rows r0 and r1
  uint32_t qh[2][4], ql[2][4];
  {
    const float4* q0 = reinterpret_cast<const float4*>(qkv + toks[r0] * (3 * C) + head * HD + 8 * c);
    const float4* q1 = reinterpret_cast<const float4*>(qkv + toks[r1] * (3 * C) + head * HD + 8 * c);
    const float4 a0 = __ldg(q0), a1 = __ldg(q0 + 1), b0 = __ldg(q1), b1 = __ldg(q1 + 1);
    split2(a0.x * scale, a0.y * scale, qh[0][0], ql[0][0]);   // k 2c,2c+1      <- dims 8c+0,1
    split2(b0.x * scale, b0.y * scale, qh[0][1], ql[0][1]);
    split2(a0.z * scale, a0.w * scale, qh[0][2], ql[0][2]);   // k 2c+8,2c+9    <- dims 8c+2,3
    split2(b0.z * scale, b0.w * scale, qh[0][3], ql[0][3]);
    split2(a1.x * scale, a1.y * scale, qh[1][0], ql[1][0]);   // k 16+2c,..     <- dims 8c+4,5
    split2(b1.x * scale, b1.y * scale, qh[1][1], ql[1][1]);
    split2(a1.z * scale, a1.w * scale, qh[1][2], ql[1][2]);   // k 24+2c,..     <- dims 8c+6,7
    split2(b1.z * scale, b1.w * scale, qh[1][3], ql[1][3]);
  }
  // ldmatrix lane roles: lane supplies the address of row (lane & 7) of matrix (lane >> 3)
  const int lrow = lane & 7, lmat = lane >> 3;
  float s[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
    // matrices 0..3 = k-index blocks [0,8) [8,16) [16,24) [24,32) of keys 8nt..8nt+7: (b0,b1) of kt=0, (b0,b1) of kt=1
    uint32_t kh[4], kl[4];
    const int off = (8 * nt + lrow) * KV_LD + 8 * lmat;
    ldsm_x4(kh, &Kh[off]);
    ldsm_x4(kl, &Kl[off]);
#pragma unroll
    for (int kt = 0; kt < 2; ++kt) {
      mma16816(s[nt], ql[kt], kh[2 * kt], kh[2 * kt + 1]);
      mma16816(s[nt], qh[kt], kl[2 * kt], kl[2 * kt + 1]);
      mma16816(s[nt], qh[kt], kh[2 * kt], kh[2 * kt + 1]);
    }
  }
  // bias, mask, softmax numerator (rows r0 and r1; each row is spread over the 4 lanes of a quad)
  const int reg0 = region[r0], reg1 = region[r1];
  float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int col = 8 * nt + 2 * c;
    s[nt][0] += bf[nt].x; s[nt][1] += bf[nt].y; s[nt][2] += bf[nt].z; s[nt][3] += bf[nt].w;
    if (shift > 0) {
      const int2 rc = *reinterpret_cast<const int2*>(&region[col]);
      if (rc.x != reg0) s[nt][0] += -100.0f;
      if (rc.y != reg0) s[nt][1] += -100.0f;
      if (rc.x != reg1) s[nt][2] += -100.0f;
      if (rc.y != reg1) s[nt][3] += -100.0f;
    }
    m0 = fmaxf(m0, fmaxf(s[nt][0], s[nt][1]));
    m1 = fmaxf(m1, fmaxf(s[nt][2], s[nt][3]));
  }
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
  float sum0 = 0.f, sum1 = 0.f;
  constexpr float L2E = 1.4426950408889634f;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    // exp(x - m) = 2^(x*log2e - m*log2e): one FFMA + one MUFU.EX2 per element
    s[nt][0] = ex2_approx_ftz(fmaf(s[nt][0], L2E, -m0 * L2E)); s[nt][1] = ex2_approx_ftz(fmaf(s[nt][1], L2E, -m0 * L2E));
    s[nt][2] = ex2_approx_ftz(fmaf(s[nt][2], L2E, -m1 * L2E)); s[nt][3] = ex2_approx_ftz(fmaf(s[nt][3], L2E, -m1 * L2E));
    sum0 += s[nt][0] + s[nt][1];
    sum1 += s[nt][2] + s[nt][3];
  }
  sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1); sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
  sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1); sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
  // O = P V  (P unnormalised in [0,1]; rows scaled by 1/sum at the end)
  float o[4][4];
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.f;
#pragma unroll
  for (int kt = 0; kt < 4; ++kt) {
    uint32_t ph[4], pl[4];
    split2(s[2 * kt][0], s[2 * kt][1], ph[0], pl[0]);
    split2(s[2 * kt][2], s[2 * kt][3], ph[1], pl[1]);
    split2(s[2 * kt + 1][0], s[2 * kt + 1][1], ph[2], pl[2]);
    split2(s[2 * kt + 1][2], s[2 * kt + 1][3], ph[3], pl[3]);
#pragma unroll
    for (int np = 0; np < 2; ++np) {
      // transposed 8x8 blocks of V: matrices 0,1 = keys 16kt+[0,8), +[8,16) x dims [16np, 16np+8) -> (b0,b1) of
      // n-tile 2np; matrices 2,3 the same keys x dims [16np+8, 16np+16) -> n-tile 2np+1
      uint32_t vh[4], vl[4];
      const int off = (16 * kt + 8 * (lmat & 1) + lrow) * KV_LD + 16 * np + 8 * (lmat >> 1);
      ldsm_x4_trans(vh, &Vh[off]);
      ldsm_x4_trans(vl, &Vl[off]);
#pragma unroll
      for (int h2 = 0; h2 < 2; ++h2) {
        const int nt = 2 * np + h2;
        mma16816(o[nt], pl, vh[2 * h2], vh[2 * h2 + 1]);
        mma16816(o[nt], ph, vl[2 * h2], vl[2 * h2 + 1]);
        mma16816(o[nt], ph, vh[2 * h2], vh[2 * h2 + 1]);
      }
    }
  }
  const float i0 = 1.0f / sum0, i1 = 1.0f / sum1;
  // lane c of a quad holds dims [8c, 8c+8) of rows r0 / r1 (see the V permutation above)
  const long e0 = toks[r0] * C + head * HD + 8 * c, e1 = toks[r1] * C + head * HD + 8 * c;
  if (out_hi) {              // split fp16 planes: directly the proj GEMM's A operand
    uint32_t h0[4], l0[4], h1[4], l1[4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      split2(o[nt][0] * i0, o[nt][1] * i0, h0[nt], l0[nt]);
      split2(o[nt][2] * i1, o[nt][3] * i1, h1[nt], l1[nt]);
    }
    *reinterpret_cast<uint4*>(out_hi + e0) = make_uint4(h0[0], h0[1], h0[2], h0[3]);
    *reinterpret_cast<uint4*>(out_lo + e0) = make_uint4(l0[0], l0[1], l0[2], l0[3]);
    *reinterpret_cast<uint4*>(out_hi + e1) = make_uint4(h1[0], h1[1], h1[2], h1[3]);
    *reinterpret_cast<uint4*>(out_lo + e1) = make_uint4(l1[0], l1[1], l1[2], l1[3]);
  } else {
    *reinterpret_cast<float4*>(out + e0) = make_float4(o[0][0] * i0, o[0][1] * i0, o[1][0] * i0, o[1][1] * i0);
    *reinterpret_cast<float4*>(out + e0 + 4) = make_float4(o[2][0] * i0, o[2][1] * i0, o[3][0] * i0, o[3][1] * i0);
    *reinterpret_cast<float4*>(out + e1) = make_float4(o[0][2] * i1, o[0][3] * i1, o[1][2] * i1, o[1][3] * i1);
    *reinterpret_cast<float4*>(out + e1 + 4) = make_float4(o[2][2] * i1, o[2][3] * i1, o[3][2] * i1, o[3][3] * i1);
  }
}

// bias_full[h][i][j] = table[rel_index(i,j)][h],  rel_index = (yi-yj+7)*15 + (xi-xj+7)   (network_swinir.py:91-101,127-129)
__global__ void expand_rel_bias_kernel(const float* __restrict__ table, float* __restrict__ bias_full, int heads) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= heads * WT * WT) return;
  const int j = idx % WT, i = (idx / WT) % WT, h = idx / (WT * WT);
  const int dy = i / WS - j / WS + WS - 1, dx = i % WS - j % WS + WS - 1;
  bias_full[idx] = table[(dy * (2 * WS - 1) + dx) * heads + h];
}

// The same bias in the accumulator-fragment order of window_attention_mma_kernel:
// bias_frag[h][warp][nt][lane][4] = bias[h][16 warp + g (+8)][8 nt + 2c (+1)],  g = lane / 4, c = lane % 4.
__global__ void expand_rel_bias_mma_kernel(const float* __restrict__ table, float* __restrict__ bias_frag, int heads) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= heads * WT * WT) return;
  const int e = idx & 3, lane = (idx >> 2) & 31, nt = (idx >> 7) & 7, warp = (idx >> 10) & 3, h = idx >> 12;
  const int i = 16 * warp + (lane >> 2) + 8 * (e >> 1), j = 8 * nt + 2 * (lane & 3) + (e & 1);
  const int dy = i / WS - j / WS + WS - 1, dx = i % WS - j % WS + WS - 1;
  bias_frag[idx] = table[(dy * (2 * WS - 1) + dx) * heads + h];
}

}  // namespace femasr

using namespace femasr;

extern "C" int femasr_window_attention(const float* qkv, const float* bias_full, float* out, int B, int H, int W,
                                       int C, int heads, int shift, void* stream) {
  FEMASR_CHECK_ARG(qkv && bias_full && out, "window_attention: null pointer");
  FEMASR_CHECK_ARG(B > 0 && H > 0 && W > 0, "window_attention: empty input");
  FEMASR_CHECK_ARG(H % WS == 0 && W % WS == 0, "window_attention: H and W must be multiples of the 8x8 window");
  FEMASR_CHECK_ARG(heads > 0 && C == heads * HD, "window_attention: C must equal heads*32");
  FEMASR_CHECK_ARG(shift == 0 || shift == WS / 2, "window_attention: shift must be 0 or 4");
  // note: the reference fixes shift_size from the constructor's input_resolution (32,32), not from the
  // runtime map size (network_swinir.py:190-193), so a one-window-high map is still shifted and masked.
  const long blocks = (long)B * (H / WS) * (W / WS) * heads;
  window_attention_kernel<<<(unsigned)blocks, 64, 0, as_stream(stream)>>>(qkv, bias_full, out, H, W, C, heads, shift);
  return launch_status("window_attention_kernel");
}

extern "C" int femasr_window_attention_mma(const float* qkv, const float* bias_frag, float* out, void* out_hi,
                                           void* out_lo, int B, int H, int W, int C, int heads, int shift, void* stream) {
  FEMASR_CHECK_ARG(qkv && bias_frag && (out || (out_hi && out_lo)), "window_attention_mma: null pointer");
  FEMASR_CHECK_ARG(!out_hi == !out_lo, "window_attention_mma: out_hi and out_lo go together");
  FEMASR_CHECK_ARG(B > 0 && H > 0 && W > 0, "window_attention_mma: empty input");
  FEMASR_CHECK_ARG(H % WS == 0 && W % WS == 0, "window_attention_mma: H and W must be multiples of the 8x8 window");
  FEMASR_CHECK_ARG(heads > 0 && C == heads * HD, "window_attention_mma: C must equal heads*32");
  FEMASR_CHECK_ARG(shift == 0 || shift == WS / 2, "window_attention_mma: shift must be 0 or 4");
  const long blocks = (long)B * (H / WS) * (W / WS) * heads;
  window_attention_mma_kernel<<<(unsigned)blocks, 128, 0, as_stream(stream)>>>(
      qkv, bias_frag, out, reinterpret_cast<__half*>(out_hi), reinterpret_cast<__half*>(out_lo), H, W, C, heads, shift);
  return launch_status("window_attention_mma_kernel");
}

extern "C" int femasr_expand_rel_bias_mma(const float* table, float* bias_frag, int heads, void* stream) {
  FEMASR_CHECK_ARG(table && bias_frag && heads > 0, "expand_rel_bias_mma: bad argument");
  const int n = heads * WT * WT;
  expand_rel_bias_mma_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(table, bias_frag, heads);
  return launch_status("expand_rel_bias_mma_kernel");
}

extern "C" int femasr_expand_rel_bias(const float* table, float* bias_full, int heads, void* stream) {
  FEMASR_CHECK_ARG(table && bias_full && heads > 0, "expand_rel_bias: bad argument");
  const int n = heads * WT * WT;
  expand_rel_bias_kernel<<<(n + 255) / 256, 256, 0, as_stream(stream)>>>(table, bias_full, heads);
  return launch_status("expand_rel_bias_kernel");
}
