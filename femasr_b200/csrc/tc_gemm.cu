// tcgen05 tensor-core implicit GEMM (3x3 stride-1 convolution and linear layers) for sm_100a, with
// fp32-grade accuracy from a two-term fp16 operand split:
//
//     a = a_hi + a_lo,  w*2^s = w_hi + w_lo          (fp16, 11-bit significands each)
//     D = a_hi*w_hi + a_hi*w_lo + a_lo*w_hi          (3 tcgen05.mma kind::f16 per k-step, fp32 accumulate in TMEM)
//
// i.e. ~22 significand bits per operand; the dropped a_lo*w_lo term is ~2^-22 relative (SURVEY 7.3-1:
// the path needs >=18 bits before the VQ and >=13 after it; single-pass fp16/bf16/tf32 fails parity).
//
// Structure (one persistent CTA per SM, 640 threads, warp-specialised):
//   warp 0  TMA producer: activation tile = 4-D box (64 ch x Wt x Ht x 1) of the NHWC fp16 planes at the
//           tap offset (kh-1, kw-1) - out-of-bounds rows/cols are zero-filled by TMA, which IS the conv
//           padding - and the weight tile = 2-D box (64 x BN) of the K-major fp16 planes; 128B swizzle.
//   warp 1  MMA issuer (one elected thread): 4 k-steps x 3 split products per 64-wide k-block into a
//           128 x BN fp32 accumulator in TMEM (two accumulators: the epilogue of tile i overlaps tile i+1).
//   warp 2  TMEM allocator.
//   warps 4-19 epilogue (16 warps; 8 for the 64-wide tiles): tcgen05.ld 16 columns at a time -> *2^-s + bias -> GELU -> smem transpose ->
//           + prefetched residual(s) -> coalesced fp32 NHWC (or split-fp16 plane) stores.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>

#include <algorithm>
#include <cstring>
#include <mutex>
#include <string>

#include "common.cuh"

namespace femasr {

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok;
}
// Same with a suspend-time hint: the warp may stay parked (off the issue slots) until the phase completes or `ns`
// elapse.  ncu showed 19 % of this kernel's executed instructions were poll iterations of the 16 epilogue warps, which
// compete with the epilogue's own (issue-bound) work.
__device__ __forceinline__ uint32_t mbar_try_wait_hint(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity), "r"(ns) : "memory");
  return ok;
}
// Bounded wait: a protocol bug must not hang the GPU; after 4 s the kernel traps (reported as a
// CUDA error by the next API call) instead of spinning forever.
__device__ __forceinline__ uint64_t global_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
constexpr uint32_t MBAR_HINT_NS = 20000u;
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = global_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait_hint(bar, parity, MBAR_HINT_NS)) {
    if ((++spins & 0xFFFu) == 0 && global_ns() - t0 > 4000000000ull) {   // 4 s: far beyond any legitimate wait
      printf("femasr tc_gemm: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x, bar, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
// L2 prefetch of a tensor box (no shared-memory destination, no barrier): issued a few pipeline stages ahead of the
// real load so that the load finds its lines in L2.  The activation planes stream from HBM (2.1 GB per tensor at batch
// 32), a load that misses L2 takes ~3 us under load, and the shared memory left next to resident weights holds only
// two strip stages: without the prefetch the 64 -> 64 convs were latency-bound at 48 % tensor-pipe activity (ncu).
__device__ __forceinline__ void tma_prefetch_4d(const CUtensorMap* map, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
// TMA store of a shared-memory box to a global tensor (bulk async group of the issuing thread) and its fences / waits
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }   // sources reusable
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }          // writes complete
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// One lane of a converged warp (elect.sync).  The single-thread roles (TMA producer, MMA issuer) are entered through this
// instead of `lane == 0`: with a data-dependent lane test ptxas must assume several lanes with different operands may be
// active and wraps EVERY UTCHMMA / UTMALDG in an ELECT ... BRA.U.ANY serialisation loop with R2UR moves (~10 SASS
// instructions and a branch per MMA); a 128x64x16 MMA is only 32 tensor-pipe cycles, so the issuing thread - not the
// tensor core - paced the 64-wide convs (ncu: 48 % tensor-pipe activity, no memory or epilogue limiter).
__device__ __forceinline__ bool elect_one() {
  uint32_t p;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t}"
      : "=r"(p));
  return p != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
// kind::f8f6f4 with both operands e4m3 (instruction-descriptor format fields 0 / 0, K = 32 per instruction = the same
// 32 bytes per k-step as kind::f16): the two CROSS products of the split scheme for the layers behind the VQ (F8 mode)
__device__ __forceinline__ void umma_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// the same load without the wait: the registers are valid after tmem_wait_ld()
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
// the wait names the registers as in/out operands so that no use of them can be scheduled above it
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :: "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
         "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// (x, y) -> packed fp16 hi pair and lo pair; the conversion saturates to +-65504 instead of overflowing to inf
__device__ __forceinline__ void split_pack2(float x, float y, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(y), "f"(x));     // d = {hi half: first src, lo half: second}
  const __half2 h = *reinterpret_cast<const __half2*>(&hi);
  const float2 hf = __half22float2(h);
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(y - hf.y), "f"(x - hf.x));
}

// K-major, 128B-swizzled operand tile ([rows][64 fp16], 8-row atoms of 1024 B): SBO = 1024 B, LBO unused (=1),
// descriptor version 1 (Blackwell), layout type 2 (SWIZZLE_128B).  cute::UMMA::SmemDescriptor bit layout.
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t saddr) {
  uint64_t d = (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// ------------------------------------------------------------------------------------------------ kernel
struct TcP {
  const float* bias; const float* res1; const float* res2; float* y; const float* inv_scale;
  __half* out_hi; __half* out_lo;   // when set: the result is written as split fp16 planes (next GEMM's A operand)
  float* gn_partial;                // when set: per-(image, tile, lane-quarter) GroupNorm partial sums of the OUTPUT
  int gn_rows, cpg;                 // partial rows per image; channels per group (Cout / 32)
  int B, H, W, Cin, Cout, taps, act;
  int stride;                    // 1 or 2 (3x3 stride-2: TMA traversal stride 2, tiles run over the output grid)
  int up;                        // 1: nearest-x2 upsample + 3x3 conv evaluated as 4 sub-pixel phases of 2x2 taps
  int Wt, Ht, wt_shift;          // 128-pixel tile = Ht rows x Wt cols (Wt power of two)
  int tiles_x, tiles_y, n_tiles; // per image spatial tiles, Cout / BN
  int num_tiles, cchunks;        // total tiles, Cin / 64
  int kb_begin, kb_end;          // k-block range of this launch (a K-slice; the caller sums slices through res1)
  int slice_kb;                  // >0: in-kernel K slicing - every slice_kb k-blocks the accumulator is drained into an
                                 // fp32 running sum kept in the second TMEM buffer (round-to-nearest adds by the
                                 // epilogue warps), so the truncating MMA accumulator never runs longer than a slice
  int f8;                        // F8 mode: the "lo" planes of both operands hold interleaved e4m3 bytes per 64-channel chunk
                                 // (A: [a_lo * 2^10 | a_hi * 2^-2], B: [w_hi * 2^-10 | w_lo * 2^2]); one K = 128 fp8 product per k-block
                                 // replaces the two fp16 cross products
  int tma_out;                   // 1: fp32 y, 2: split fp16 planes leave through TMA stores of the epilogue's staging tile
  int box_w, box_w_shift;        // a warp's 32 accumulator rows as a box of box_w x (32 / box_w) output pixels
  // VQ mode (template VQ): the GEMM is z . E^T and the epilogue keeps, per feature row, the four smallest distances
  // fl(fl(A + B_j) - 2 C_j) over all codes instead of storing the [N, n_e] product (femasr_arch.py:35-38, 63-66)
  const float* vq_a;             // [M]   A = sum z^2 per row
  const float* vq_esq;           // [Cout] B_j = sum e_j^2 per code
  uint2* vq_cand;                // [M][4] {distance bits, code}, ascending (distance, code)
};

constexpr int TC_BM = 128, TC_BK = 64;
// epilogue warps per TMEM lane quarter (= column split of the accumulator): 4 (16 epilogue warps) for the 128/256-wide
// tiles - measured +4 % end to end over 8 warps, the short-K layers are epilogue-issue bound - but 2 for the 64-wide
// tiles, where a warp would own a single 16-column chunk and the per-tile fixed work dominates (measured -15 %).
constexpr int nsplit_for(int BN) { return BN == 64 ? 2 : 4; }
constexpr int tc_threads_for(int BN) { return 128 + 32 * 4 * nsplit_for(BN); }
constexpr int A_PLANE_BYTES = TC_BM * TC_BK * 2;   // 16 KB

// PAIR = true: two CTAs of a cluster (one TPC) cooperate on a 256 x BN tile with tcgen05 cta_group::2 - each
// CTA stages its own 128 activation rows and only HALF of the weight tile, so the weight traffic per CTA (the
// L2->SM bottleneck of the short-K / narrow layers) is halved and one more pipeline stage fits.
// STRIP = true (3x3 stride-1 convs on maps at least 128 wide, BN <= 128): the tile is one image row of 128 pixels
// and the activation operand of the three horizontal taps (kw = 0,1,2) is ONE shared-memory strip of 130 pixels per
// (kh, 64-channel chunk): tap kw reads it through a descriptor that simply starts kw rows (kw*128 B) into the strip
// (the swizzle follows absolute address bits, see the MMA issuer).  Activation traffic from L2 drops 2.9x (3 loads
// instead of 9 per chunk) - the narrow layers are L2->SM bound (profiles/tc_igemm_traffic_r1.json).  Weights stream
// through their own ring, one tap per stage.
constexpr int STRIP_PX = 130;                         // 128 outputs + one halo pixel each side
constexpr int STRIP_PLANE_BYTES = 17 * 1024;          // 130 rows x 128 B = 16,640 B, padded to the 1024-B swizzle period

// BRES = true (strip mode, 64 -> 64 channels): the complete weight matrix (9 taps x 64 x 64, hi + lo = 144 KB) is
// loaded into shared memory ONCE per CTA and stays resident for all of its tiles; only activation strips stream.
// These layers are L2->SM bound and 60 % of their remaining L2 traffic was the weight tile re-fetched per tile.
template <int BN, bool PAIR, bool STRIP, bool BRES = false>
struct TcCfg {
  static_assert(!(PAIR && BRES), "resident-weight strips are single-CTA");
  static_assert(!BRES || (STRIP && BN == 64), "resident weights: strip mode, 64-wide tiles");
  static constexpr int B_ROWS = PAIR ? BN / 2 : BN;                 // weight-tile rows this CTA stages
  static constexpr int B_PLANE_BYTES = B_ROWS * TC_BK * 2;
  // joint A+B stages (normal / pair)
  static constexpr int STAGE_BYTES = 2 * A_PLANE_BYTES + 2 * B_PLANE_BYTES;
  static constexpr int STAGES = PAIR ? (BN == 256 ? 3 : 4) : (BN == 256 ? 2 : (BN == 128 ? 3 : 4));
  // separate rings (strip)
  // strip planes: 130 rows x 128 B; padded to 17 KB normally, packed back to back when smem is needed for weights
  // (fine: TMA and the tensor core both derive the swizzle from the absolute address, 128-B alignment suffices)
  static constexpr int SA_PLANE = BRES ? STRIP_PX * TC_BK * 2 : STRIP_PLANE_BYTES;
  static constexpr int SA_STAGES = 2, SA_BYTES = 2 * SA_PLANE;
  static constexpr int B_RES_BYTES = BRES ? 9 * 2 * B_PLANE_BYTES : 0;
  static constexpr int SB_BYTES = 2 * B_PLANE_BYTES;
  static constexpr int NSPLIT = nsplit_for(BN), EPI_WARPS = 4 * NSPLIT, THREADS = tc_threads_for(BN);
  static constexpr int BIAS_BYTES = BN * 4;     // the n-tile's bias (VQ: sum e^2) staged in shared memory for the epilogue
  static constexpr int SB_BUDGET = 232448 - 1024 - 256 - EPI_WARPS * 2048 - BIAS_BYTES - SA_STAGES * SA_BYTES;   // what is left of 227 KB
  static constexpr int SB_STAGES = BRES ? 0 : (SB_BUDGET / SB_BYTES > 6 ? 6 : SB_BUDGET / SB_BYTES);
  static constexpr int PIPE_BYTES = BRES ? B_RES_BYTES + SA_STAGES * SA_BYTES
                                         : (STRIP ? SA_STAGES * SA_BYTES + SB_STAGES * SB_BYTES : STAGES * STAGE_BYTES);
  // full/empty barriers of the rings (resident weights: one "weights landed" barrier instead of a weight ring)
  static constexpr int NBAR_PIPE = BRES ? 2 * SA_STAGES + 1 : (STRIP ? 2 * SA_STAGES + 2 * SB_STAGES : 2 * STAGES);
  static constexpr int EPI_BYTES = EPI_WARPS * 2048 /*per-warp 32x16 fp32 transpose tiles*/;
  static constexpr int SMEM_BYTES = PIPE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ + EPI_BYTES + BIAS_BYTES;
  // Multi-row strip tiles (resident weights): one work item = MR vertically adjacent image rows of 128 pixels, each its
  // own 128 x BN accumulator.  Input row s (of MR + 2) is loaded ONCE and feeds the kh = s - r tap row of every output
  // row r it touches, so a tile streams (MR + 2) / MR strips per output row instead of 3 (L2 -> SM traffic / 2 at MR = 4)
  // and every strip carries 2x the MMA work, which is what hides the strip's load latency behind only two strip stages
  // (all the shared memory the resident weights leave).
  static constexpr int MR = BRES ? 4 : 1;
  static constexpr int NACC = 2 * MR;                             // accumulator ring: two sets of MR
  // K-sliced accumulation with a THIRD buffer (tiles up to 128 wide): the MMA ping-pongs between buffers 0 / 1 while the
  // epilogue folds the finished partial into the running sum in buffer 2, so the tensor pipe no longer idles during a
  // fold (ncu on the 2-buffer protocol: 41 % of the epilogue's samples waiting for the next partial, tensor pipe 51 %).
  static constexpr bool S3 = !STRIP && BN <= 128;
  static constexpr int TMEM_COLS = S3 ? 4 * BN : (NACC * BN < 32 ? 32 : NACC * BN);   // power of two for BN in {64,128,256}
  static_assert(TMEM_COLS <= 512, "TMEM budget");
  static_assert(8 * (NBAR_PIPE + 2 * NACC) + 4 <= 256, "barrier area");
  static_assert(SMEM_BYTES <= 232448, "shared memory budget");
  static_assert(PIPE_BYTES % 1024 == 0, "the epilogue staging tiles must start on the swizzle period");
  static_assert(!STRIP || BRES || SB_STAGES >= 2, "strip weight ring too small");
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  // non-.aligned forms: the role branches leave lane 0 of the producer / MMA warps diverged from its warp
  __syncwarp();
  asm volatile("barrier.cluster.arrive.release;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
}
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma2_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma2_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void umma2_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void umma2_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
// commit of the pair's MMAs: arrives on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma2_commit_mc(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}

// RES: the layer adds a residual tile (res1) in the epilogue.  A template parameter because the prefetched residual
// chunks cost 32 registers per epilogue thread and the 640-thread CTA is capped at 96: the half of the layers
// without a residual (qkv, fc1, the first conv of every ResBlock, up / down convs) get a spill-free epilogue.
// VQ: the z . E^T product of the VectorQuantizer with the argmin fused into the epilogue (see the VQ epilogue below);
// work is ordered M-major so that one CTA sees ALL code tiles of its 128 feature rows back to back.
template <int BN, bool PAIR, bool STRIP, bool BRES, bool RES, bool VQ = false>
__global__ void __launch_bounds__(tc_threads_for(BN), 1)
tc_igemm_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_oh,
                const __grid_constant__ CUtensorMap map_ol, const TcP p) {
  using Cfg = TcCfg<BN, PAIR, STRIP, BRES>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t epi_base = smem_base + Cfg::PIPE_BYTES;           // 1024-aligned: the staging tiles are TMA-store sources
  const uint32_t bar_base = epi_base + Cfg::EPI_BYTES + Cfg::BIAS_BYTES;
  // barriers: the ring barriers (joint: full[STAGES], empty[STAGES]; strip: fullA, emptyA, fullB, emptyB),
  // then tmem_full[2], tmem_empty[2]; then the TMEM base pointer
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto fullA_bar = [&](int s) { return bar_base + 8u * s; };
  auto emptyA_bar = [&](int s) { return bar_base + 8u * (Cfg::SA_STAGES + s); };
  auto fullB_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::SA_STAGES + s); };
  auto emptyB_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::SA_STAGES + Cfg::SB_STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (Cfg::NBAR_PIPE + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (Cfg::NBAR_PIPE + Cfg::NACC + a); };
  const uint32_t tmem_slot = bar_base + 8u * (Cfg::NBAR_PIPE + 2 * Cfg::NACC);
  constexpr int MR = Cfg::MR, NACC = Cfg::NACC;

  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;     // CTA 0 of the pair issues the MMAs
  const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int nworkers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  // m-tiles of 128 pixels; a pair-tile is two consecutive m-tiles of the SAME sub-pixel phase (the two CTAs share
  // one weight tile); the second may fall off the end of the phase: dummy tile
  const int num_m = p.num_tiles / p.n_tiles;
  const int phases = p.up ? 4 : 1;
  const int m_per_phase = num_m / phases;
  const int pairs_per_phase = (m_per_phase + 1) / 2;
  const int num_work = PAIR ? phases * pairs_per_phase * p.n_tiles : p.num_tiles;
  static_assert(!VQ || (!PAIR && !STRIP && !RES), "VQ mode: plain single-CTA linear tiles");
  // it-th work item of this CTA (-1: done).  Default: items strided over the CTAs.  VQ: m-tiles strided over the
  // CTAs, and for each m-tile every n-tile (code tile) in turn.
  auto work_of = [&](int it) -> int {
    if (VQ) {
      const int mt = (it / p.n_tiles) * nworkers + worker;
      return mt < num_m ? mt * p.n_tiles + it % p.n_tiles : -1;
    }
    const int w = worker + it * nworkers;
    return w < num_work ? w : -1;
  };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::NBAR_PIPE; ++s) mbar_init(bar_base + 8u * s, 1);
    // tmem-empty: ONE arrival per epilogue warp (of both CTAs when paired), by an elected lane after __syncwarp - 512
    // per-thread arrivals per tile were 512 remote DSMEM transactions for the peer CTA of a pair
    for (int a = 0; a < NACC; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), (PAIR ? 2 : 1) * Cfg::EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (PAIR) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  const int ksz = p.taps == 9 ? 3 : 1;   // (p.up: taps == 4, offsets from the phase)

  // work item -> (n-tile, m-tile of this CTA); decodes the m-tile into (phase, image, tile row/col)
  struct TileCoord { int nt, tx, ty, b, ph; bool real; };
  auto decode = [&](int work) {
    TileCoord tc;
    tc.nt = work % p.n_tiles;
    int mt = work / p.n_tiles;
    tc.real = true;
    if (PAIR) {
      const int ph = mt / pairs_per_phase;
      const int idx = 2 * (mt - ph * pairs_per_phase) + (int)rank;
      tc.real = idx < m_per_phase;
      mt = ph * m_per_phase + (tc.real ? idx : 0);
    }
    tc.tx = mt % p.tiles_x; mt /= p.tiles_x;
    tc.ty = mt % p.tiles_y; mt /= p.tiles_y;
    tc.b = mt % p.B;
    tc.ph = mt / p.B;                                // sub-pixel phase (0 unless p.up)
    if (!tc.real) tc.b = p.B;                        // image index out of range: TMA zero-fills the dummy tile
    return tc;
  };

  if (STRIP && warp == 0 && elect_one()) {
    // ===================== TMA producer (strip mode) =====================
    // per (kh, 64-channel chunk): one 130-pixel activation strip (hi, lo), then the three taps' weight tiles
    int sa = 0, sb = 0; uint32_t pa = 0, pb = 0;
    if (BRES) {
      // the whole [64][9*64] weight matrix (hi, lo) once.  Merged layout (see the MMA issuer): per kw the hi planes of
      // kh = 2, 1, 0 back to back (3 x 8 KB), then the three lo planes - any run of consecutive kh is ONE B operand of
      // N = 64, 128 or 192 rows.
      const uint32_t bres_bar = bar_base + 8u * (2 * Cfg::SA_STAGES);
      mbar_expect_tx(bres_bar, Cfg::B_RES_BYTES);
      for (int tap = 0; tap < 9; ++tap) {
        const int kh = tap / 3, kw = tap - 3 * kh;
        const uint32_t dst_hi = smem_base + (kw * 6 + (2 - kh)) * Cfg::B_PLANE_BYTES;
        const uint32_t dst_lo = dst_hi + 3 * Cfg::B_PLANE_BYTES;
        tma_load_2d(dst_hi, &map_b_hi, bres_bar, tap * p.Cin, 0);
        tma_load_2d(dst_lo, &map_b_lo, bres_bar, tap * p.Cin, 0);
      }
    }
    // L2 prefetch cursor: runs PF_STRIPS strips ahead of the loads over the same (work, input row, chunk) sequence
    constexpr int PF_STRIPS = BRES ? 4 : 0;      // 128 -> 128 strips (streamed weights, deeper rings): measured neutral
    int pf_work = worker, pf_sr = 0, pf_cc = 0;
    auto prefetch_next = [&]() {
      if (pf_work >= num_work) return;
      const TileCoord t = decode(pf_work);
      tma_prefetch_4d(&map_a_hi, pf_cc * TC_BK, t.tx * p.Wt - 1, t.ty * MR + pf_sr - 1, t.b);
      tma_prefetch_4d(&map_a_lo, pf_cc * TC_BK, t.tx * p.Wt - 1, t.ty * MR + pf_sr - 1, t.b);
      if (++pf_cc == p.cchunks) { pf_cc = 0; if (++pf_sr == MR + 2) { pf_sr = 0; pf_work += nworkers; } }
    };
    for (int i = 0; i < PF_STRIPS; ++i) prefetch_next();
    for (int work = worker; work < num_work; work += nworkers) {
      const TileCoord tc = decode(work);
      const int x0 = tc.tx * p.Wt, y0 = tc.ty * MR, n0 = tc.nt * BN;
      // input rows y0 - 1 ... y0 + MR (MR = 1: the three kh rows of one output row)
      for (int sr = 0; sr < MR + 2; ++sr)
        for (int cc = 0; cc < p.cchunks; ++cc) {
          const int c0 = cc * TC_BK;
          if (PF_STRIPS > 0) prefetch_next();
          mbar_wait(emptyA_bar(sa), pa ^ 1u);
          const uint32_t a_dst = smem_base + Cfg::B_RES_BYTES + sa * Cfg::SA_BYTES;
          if (PAIR) {
            // CTA pair over two neighbouring row tiles: each CTA stages its own strip and HALF of every weight tile;
            // all loads complete on the LEADER's barriers, armed once for the bytes of both CTAs
            const uint32_t lead = map_to_cta(fullA_bar(sa), 0);
            if (rank == 0) mbar_expect_tx(fullA_bar(sa), 2 * (2 * STRIP_PX * TC_BK * 2));
            tma2_load_4d(a_dst, &map_a_hi, lead, c0, x0 - 1, y0 + sr - 1, tc.b);
            tma2_load_4d(a_dst + Cfg::SA_PLANE, &map_a_lo, lead, c0, x0 - 1, y0 + sr - 1, tc.b);
          } else {
            mbar_expect_tx(fullA_bar(sa), 2 * STRIP_PX * TC_BK * 2);
            tma_load_4d(a_dst, &map_a_hi, fullA_bar(sa), c0, x0 - 1, y0 + sr - 1, tc.b);
            tma_load_4d(a_dst + Cfg::SA_PLANE, &map_a_lo, fullA_bar(sa), c0, x0 - 1, y0 + sr - 1, tc.b);
          }
          if (++sa == Cfg::SA_STAGES) { sa = 0; pa ^= 1u; }
          if (BRES) continue;
          for (int kw = 0; kw < 3; ++kw) {                 // streamed weights (MR == 1: sr is kh)
            const int tap = sr * 3 + kw;
            mbar_wait(emptyB_bar(sb), pb ^ 1u);
            const uint32_t b_dst = smem_base + Cfg::SA_STAGES * Cfg::SA_BYTES + sb * Cfg::SB_BYTES;
            if (PAIR) {
              const uint32_t lead = map_to_cta(fullB_bar(sb), 0);
              const int nh = n0 + (int)rank * (BN / 2);
              if (rank == 0) mbar_expect_tx(fullB_bar(sb), 2 * Cfg::SB_BYTES);
              tma2_load_2d(b_dst, &map_b_hi, lead, tap * p.Cin + c0, nh);
              tma2_load_2d(b_dst + Cfg::B_PLANE_BYTES, &map_b_lo, lead, tap * p.Cin + c0, nh);
            } else {
              mbar_expect_tx(fullB_bar(sb), Cfg::SB_BYTES);
              tma_load_2d(b_dst, &map_b_hi, fullB_bar(sb), tap * p.Cin + c0, n0);
              tma_load_2d(b_dst + Cfg::B_PLANE_BYTES, &map_b_lo, fullB_bar(sb), tap * p.Cin + c0, n0);
            }
            if (++sb == Cfg::SB_STAGES) { sb = 0; pb ^= 1u; }
          }
        }
    }
  } else if (STRIP && warp == 1 && rank == 0 && elect_one()) {
    // ===================== MMA issuer (strip mode; leader CTA only when paired) =====================
    const uint32_t idesc = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((PAIR ? 2 * TC_BM : TC_BM) >> 4) << 24);
    int sa = 0, sb = 0; uint32_t pa = 0, pb = 0;
    int set = 0; uint32_t set_phase = 0;           // accumulator set (MR slots) of the current work item
    if (BRES) { mbar_wait(bar_base + 8u * (2 * Cfg::SA_STAGES), 0u); tc_fence_after(); }   // weights resident
    for (int work = worker; work < num_work; work += nworkers) {
      if constexpr (BRES) {
        // Multi-row strip tiles with MERGED tap rows.  ncu on these convs (profiles/ncu_r2_epilogue.json): the tensor-core
        // pipe 81 % utilised with its math sub-pipe at 42 % - a 128 x 64 x 16 MMA streams 4 KB of A and 2 KB of B out of
        // shared memory (~48 cycles at 128 B / clk) for 34 cycles of fp16 math (17 of e4m3 math): with N = 64 the operand
        // fetch, not the math, occupies the pipe.  Input strip sr feeds tap row kh = sr - r of every output row r it
        // touches WITH THE SAME A operand, and the accumulators of rows r, r + 1, ... sit side by side in TMEM, so those
        // products are ONE MMA of N = 64 x rows against the weight rows of kh = sr - r_lo, ..., sr - r_hi (contiguous in
        // the merged layout): 147 instead of 288 MMAs per 4-row work item, A fetched once per strip and k-step instead of
        // once per (row, tap).  Every accumulator still receives its contributions in (kh, kw, k, product) order, so the
        // results are bit-identical to the unmerged form.  Only the very first product into a fresh accumulator (kh = 0,
        // kw = 0, k = 0) must overwrite instead of accumulate and is issued on its own.
        auto idesc_n = [](int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24); };
        for (int sr = 0; sr < MR + 2; ++sr) {         // p.cchunks == 1 (64 input channels)
          mbar_wait(fullA_bar(sa), pa);
          tc_fence_after();
          const uint32_t a_base = smem_base + Cfg::B_RES_BYTES + sa * Cfg::SA_BYTES;
          const int r_lo = sr - 2 > 0 ? sr - 2 : 0, r_hi = sr < MR - 1 ? sr : MR - 1;
          const bool fresh = sr < MR;                  // output row r = sr (== r_hi) starts with this strip (its kh = 0 tap row)
          if (fresh) { mbar_wait(tempty_bar(set * MR + sr), set_phase ^ 1u); tc_fence_after(); }
          const int rows = r_hi - r_lo + 1;
          const uint32_t d_all = tmem_base + (uint32_t)((set * MR + r_lo) * BN);
          const uint32_t d_new = tmem_base + (uint32_t)((set * MR + r_hi) * BN);
          const uint32_t id_all = idesc_n(BN * rows), id_old = idesc_n(BN * (rows - 1)), id_one = idesc_n(BN);
          const int b_first = 2 - (sr - r_lo);         // weight plane (within the kw group) of the first merged row
          for (int kw = 0; kw < 3; ++kw) {
            const uint64_t a_hi = make_sw128_desc(a_base + kw * 128);
            const uint64_t a_lo = make_sw128_desc(a_base + Cfg::SA_PLANE + kw * 128);
            const uint32_t b_grp = smem_base + kw * 6 * Cfg::B_PLANE_BYTES;
            const uint64_t b_hi = make_sw128_desc(b_grp + b_first * Cfg::B_PLANE_BYTES);
            const uint64_t b_lo = make_sw128_desc(b_grp + (3 + b_first) * Cfg::B_PLANE_BYTES);
            // the fresh row alone: the LAST of the merged rows (kh = 0 = plane 2 of the group)
            const uint64_t b_hi_new = make_sw128_desc(b_grp + 2 * Cfg::B_PLANE_BYTES);
            const uint64_t b_lo_new = make_sw128_desc(b_grp + 5 * Cfg::B_PLANE_BYTES);
#pragma unroll
            for (int k = 0; k < TC_BK / 16; ++k) {
              const uint64_t ko = (uint64_t)((k * 32) >> 4);
              if (fresh && kw == 0 && k == 0) {
                // first product of the k-step: older rows accumulate, the fresh row overwrites
                if (p.f8) {
                  if (rows > 1) umma_f8(d_all, a_lo + ko, b_lo + ko, id_old, 1u);
                  umma_f8(d_new, a_lo + ko, b_lo_new + ko, id_one, 0u);
                } else {
                  if (rows > 1) umma_f16(d_all, a_lo + ko, b_hi + ko, id_old, 1u);
                  umma_f16(d_new, a_lo + ko, b_hi_new + ko, id_one, 0u);
                }
              } else {
                if (p.f8) umma_f8(d_all, a_lo + ko, b_lo + ko, id_all, 1u);
                else umma_f16(d_all, a_lo + ko, b_hi + ko, id_all, 1u);
              }
              if (!p.f8) umma_f16(d_all, a_hi + ko, b_lo + ko, id_all, 1u);
              umma_f16(d_all, a_hi + ko, b_hi + ko, id_all, 1u);
            }
          }
          if (sr >= 2) umma_commit(tfull_bar(set * MR + sr - 2));       // output row sr - 2 has all three tap rows
          umma_commit(emptyA_bar(sa));
          if (++sa == Cfg::SA_STAGES) { sa = 0; pa ^= 1u; }
        }
      } else
      for (int sr = 0; sr < MR + 2; ++sr)                // streamed weights: one tap's weight tile per ring stage
        for (int cc = 0; cc < p.cchunks; ++cc) {
          mbar_wait(fullA_bar(sa), pa);
          tc_fence_after();
          const uint32_t a_base = smem_base + Cfg::B_RES_BYTES + sa * Cfg::SA_BYTES;
          // input row sr is tap row kh = sr - r of output row r
          const int r_lo = sr - 2 > 0 ? sr - 2 : 0, r_hi = sr < MR - 1 ? sr : MR - 1;
          for (int r = r_lo; r <= r_hi; ++r) {
            const int kh = sr - r;
            const int slot = set * MR + r;
            const uint32_t d_tmem = tmem_base + (uint32_t)(slot * BN);
            if (kh == 0 && cc == 0) {              // first contribution to this accumulator: the epilogue must have drained it
              mbar_wait(tempty_bar(slot), set_phase ^ 1u);
              tc_fence_after();
            }
            for (int kw = 0; kw < 3; ++kw) {
              mbar_wait(fullB_bar(sb), pb);
              tc_fence_after();
              const uint32_t b_base = smem_base + Cfg::SA_STAGES * Cfg::SA_BYTES + sb * Cfg::SB_BYTES;
              // tap kw = the strip shifted by kw pixel rows.  Measured on B200: the tensor core derives the 128B-swizzle
              // XOR from the absolute shared-memory address bits (like TMA does when it writes the strip), so a start
              // address that is 128-byte but not 1024-byte aligned just works with base-offset 0; putting the row phase
              // into the descriptor's base-offset field (bits 49-51) instead produces garbage.
              const uint64_t a_hi = make_sw128_desc(a_base + kw * 128);
              const uint64_t a_lo = make_sw128_desc(a_base + Cfg::SA_PLANE + kw * 128);
              const uint64_t b_hi = make_sw128_desc(b_base), b_lo = make_sw128_desc(b_base + Cfg::B_PLANE_BYTES);
#pragma unroll
              for (int k = 0; k < TC_BK / 16; ++k) {
                const uint64_t ko = (uint64_t)((k * 32) >> 4);
                const uint32_t first = (kh | cc | kw | k) ? 1u : 0u;
                if (PAIR) {
                  if (p.f8) {
                    umma2_f8(d_tmem, a_lo + ko, b_lo + ko, idesc, first);
                  } else {
                    umma2_f16(d_tmem, a_lo + ko, b_hi + ko, idesc, first);
                    umma2_f16(d_tmem, a_hi + ko, b_lo + ko, idesc, 1u);
                  }
                  umma2_f16(d_tmem, a_hi + ko, b_hi + ko, idesc, 1u);
                } else {
                  if (p.f8) {
                    umma_f8(d_tmem, a_lo + ko, b_lo + ko, idesc, first);       // sum a_lo8 w_hi8 + sum a_hi8 w_lo8
                  } else {
                    umma_f16(d_tmem, a_lo + ko, b_hi + ko, idesc, first);
                    umma_f16(d_tmem, a_hi + ko, b_lo + ko, idesc, 1u);
                  }
                  umma_f16(d_tmem, a_hi + ko, b_hi + ko, idesc, 1u);
                }
              }
              if (PAIR) umma2_commit_mc(emptyB_bar(sb)); else umma_commit(emptyB_bar(sb));
              if (++sb == Cfg::SB_STAGES) { sb = 0; pb ^= 1u; }
            }
            if (kh == 2 && cc == p.cchunks - 1) {                                // output row r complete
              if (PAIR) umma2_commit_mc(tfull_bar(slot)); else umma_commit(tfull_bar(slot));
            }
          }
          if (PAIR) umma2_commit_mc(emptyA_bar(sa)); else umma_commit(emptyA_bar(sa));
          if (++sa == Cfg::SA_STAGES) { sa = 0; pa ^= 1u; }
        }
      if (++set == 2) { set = 0; set_phase ^= 1u; }
    }
  } else if (!STRIP && warp == 0 && elect_one()) {
    // ===================== TMA producer =====================
    int stage = 0; uint32_t phase = 0;
    // activation box of k-block kb of a tile: channel chunk and the tap's spatial offset (conv padding = TMA zero fill)
    struct ABox { int c0, x, y, b, tap; };
    auto a_box = [&](const TileCoord& tc, int kb) {
      ABox bx;
      bx.tap = kb / p.cchunks;
      bx.c0 = (kb - bx.tap * p.cchunks) * TC_BK;
      int dy = 0, dx = 0;
      if (p.up) { dy = (bx.tap >> 1) - 1 + (tc.ph >> 1); dx = (bx.tap & 1) - 1 + (tc.ph & 1); }
      else if (ksz == 3) { dy = bx.tap / 3 - 1; dx = bx.tap - (bx.tap / 3) * 3 - 1; }
      bx.x = p.stride * tc.tx * p.Wt + dx; bx.y = p.stride * tc.ty * p.Ht + dy; bx.b = tc.b;
      return bx;
    };
    // No L2 prefetch ahead of these loads (unlike the strip producer): a prefetch box costs the TMA unit as much as a
    // load, and with 2-4 joint stages of 48-96 KB these tiles are not load-latency bound - the sub-pixel up convs lost
    // 20-40 % with a prefetch 4 k-blocks ahead (profiles/microbench_r2_*).
    for (int it = 0, work; (work = work_of(it)) >= 0; ++it) {
      const TileCoord tc = decode(work);
      const int n0 = tc.ph * p.Cout + tc.nt * BN + (PAIR ? (int)rank * (BN / 2) : 0);
      for (int kb = p.kb_begin; kb < p.kb_end; ++kb) {
        const ABox bx = a_box(tc, kb);
        const int tap = bx.tap, c0 = bx.c0;
        mbar_wait(empty_bar(stage), phase ^ 1u);
        const uint32_t sa = smem_base + stage * Cfg::STAGE_BYTES;
        if (PAIR) {
          // both CTAs' loads complete on the LEADER's barrier, armed once for the bytes of both
          const uint32_t lead_full = map_to_cta(full_bar(stage), 0);
          if (rank == 0) mbar_expect_tx(full_bar(stage), 2 * Cfg::STAGE_BYTES);
          tma2_load_4d(sa, &map_a_hi, lead_full, c0, bx.x, bx.y, bx.b);
          tma2_load_4d(sa + A_PLANE_BYTES, &map_a_lo, lead_full, c0, bx.x, bx.y, bx.b);
          tma2_load_2d(sa + 2 * A_PLANE_BYTES, &map_b_hi, lead_full, tap * p.Cin + c0, n0);
          tma2_load_2d(sa + 2 * A_PLANE_BYTES + Cfg::B_PLANE_BYTES, &map_b_lo, lead_full, tap * p.Cin + c0, n0);
        } else {
          mbar_expect_tx(full_bar(stage), Cfg::STAGE_BYTES);
          tma_load_4d(sa, &map_a_hi, full_bar(stage), c0, bx.x, bx.y, bx.b);
          tma_load_4d(sa + A_PLANE_BYTES, &map_a_lo, full_bar(stage), c0, bx.x, bx.y, bx.b);
          tma_load_2d(sa + 2 * A_PLANE_BYTES, &map_b_hi, full_bar(stage), tap * p.Cin + c0, n0);
          tma_load_2d(sa + 2 * A_PLANE_BYTES + Cfg::B_PLANE_BYTES, &map_b_lo, full_bar(stage), tap * p.Cin + c0, n0);
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (!STRIP && warp == 1 && rank == 0 && elect_one()) {
    // ===================== MMA issuer (leader CTA only when paired) =====================
    // instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 (bits 4-5 = 1), A=B=f16 (0), K-major both,
    // N>>3 at bits 17-22, M>>4 at bits 24-28 (M = 256 across the CTA pair).
    const uint32_t idesc = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((PAIR ? 2 * TC_BM : TC_BM) >> 4) << 24);
    int stage = 0; uint32_t phase = 0;
    int acc = 0; uint32_t acc_phase = 0;
    const bool sliced = p.slice_kb > 0;
    const int slice_len = sliced ? p.slice_kb : (p.kb_end - p.kb_begin);
    for (int it = 0; work_of(it) >= 0; ++it) {
      for (int kb0 = p.kb_begin; kb0 < p.kb_end; kb0 += slice_len) {
        const int kb1 = min(kb0 + slice_len, p.kb_end);
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * Cfg::STAGE_BYTES;
          const uint64_t a_hi = make_sw128_desc(sa), a_lo = make_sw128_desc(sa + A_PLANE_BYTES);
          const uint64_t b_hi = make_sw128_desc(sa + 2 * A_PLANE_BYTES);
          const uint64_t b_lo = make_sw128_desc(sa + 2 * A_PLANE_BYTES + Cfg::B_PLANE_BYTES);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k) {
            const uint64_t ko = (uint64_t)((k * 32) >> 4);   // +32 bytes per k-step inside the 128B swizzle atom
            // small cross terms first, the dominant hi*hi product last
            const uint32_t first = (kb != kb0 || k != 0) ? 1u : 0u;
            if (PAIR) {
              if (p.f8) {
                umma2_f8(d_tmem, a_lo + ko, b_lo + ko, idesc, first);
              } else {
                umma2_f16(d_tmem, a_lo + ko, b_hi + ko, idesc, first);
                umma2_f16(d_tmem, a_hi + ko, b_lo + ko, idesc, 1u);
              }
              umma2_f16(d_tmem, a_hi + ko, b_hi + ko, idesc, 1u);
            } else {
              if (p.f8) {
                umma_f8(d_tmem, a_lo + ko, b_lo + ko, idesc, first);
              } else {
                umma_f16(d_tmem, a_lo + ko, b_hi + ko, idesc, first);
                umma_f16(d_tmem, a_hi + ko, b_lo + ko, idesc, 1u);
              }
              umma_f16(d_tmem, a_hi + ko, b_hi + ko, idesc, 1u);
            }
          }
          // frees the smem slot (in both CTAs of a pair) when these MMAs retire
          if (PAIR) umma2_commit_mc(empty_bar(stage)); else umma_commit(empty_bar(stage));
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        // (partial) accumulator complete -> epilogue warps (of both CTAs)
        if (PAIR) umma2_commit_mc(tfull_bar(acc)); else umma_commit(tfull_bar(acc));
        // sliced, 256-wide: one MMA target buffer (0), the other holds the running sum; else ping-pong (tiles, or the
        // partials of a sliced tile when a third buffer holds the sum)
        if (sliced && !Cfg::S3) acc_phase ^= 1u;
        else if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (8 warps) =====================
    // TMEM hands each thread one accumulator ROW; storing rows per thread would touch 32 different rows per
    // instruction.  Each warp therefore transposes 32x16 chunks through (XOR-swizzled) shared memory and
    // stores with 4 lanes per row x float4: full 64-byte row segments, 8 rows per instruction.
    // Warps 4-7 take the left half of the accumulator columns, warps 8-11 the right half (TMEM lane quarter
    // = warp_id % 4).  Residual tiles are software-prefetched one chunk ahead so their latency overlaps the
    // TMEM load / math of the current chunk (the stores may alias the residual, which otherwise pins every load
    // behind the previous store).
    const int e = warp - 4;
    const int ew = e & 3, part = e >> 2;             // TMEM lane quarter, column part
    const int row = ew * 32 + lane;
    const float inv_scale = __ldg(p.inv_scale);
    float* stage = reinterpret_cast<float*>(smem_raw + (epi_base + (uint32_t)e * 2048u - smem_u32(smem_raw)));
    // Per-column epilogue constants (bias; VQ: sum e^2) of the current n-tile live in shared memory: with the whole
    // 227 KB carved out for the pipeline there is no L1 left, and a global load per 16-column chunk was the top stall
    // of the short-K layers (16 % long-scoreboard, profiles/swin_kernels_ncu_r1.json).  Restaged only when the n-tile
    // changes; two named barriers order the rewrite against the other epilogue warps' reads.
    float* sbias = reinterpret_cast<float*>(smem_raw + (epi_base + (uint32_t)Cfg::EPI_BYTES - smem_u32(smem_raw)));
    int staged_nt = -1;
    auto stage_cols = [&](const float* src, int nt) {
      if (nt == staged_nt) return;
      const int et = (int)threadIdx.x - 128;
      const float v = et < BN ? __ldg(src + nt * BN + et) : 0.f;
      asm volatile("bar.sync 1, %0;" ::"r"(32 * Cfg::EPI_WARPS) : "memory");
      if (et < BN) sbias[et] = v;
      asm volatile("bar.sync 1, %0;" ::"r"(32 * Cfg::EPI_WARPS) : "memory");
      staged_nt = nt;
    };
    const int q = lane & 3, rsub = lane >> 2;
    constexpr int CW = BN / Cfg::NSPLIT;             // accumulator columns per warp
    constexpr int CH = 16, NCH = CW / CH;            // chunks per warp
    int acc = 0; uint32_t acc_phase = 0;
    const bool sliced = p.slice_kb > 0;
    const int nslices = sliced ? (p.kb_end - p.kb_begin + p.slice_kb - 1) / p.slice_kb : 1;
    // the MMA issuer waits on the LEADER's tmem-empty barriers; the peer's epilogue arrives there remotely
    auto release_acc = [&](int a) {          // call with the whole warp converged, after tcgen05.wait::ld + fence::before
      __syncwarp();
      if (lane == 0) { if (PAIR) mbar_arrive_cluster(map_to_cta(tempty_bar(a), 0)); else mbar_arrive(tempty_bar(a)); }
    };
    if constexpr (VQ) {
      // ===================== VQ epilogue: running top-4 of d_j = fl(fl(A + B_j) - 2 C_j) per feature row =====================
      // The thread owns one accumulator row (a feature) and CW columns (codes) of every code tile; codes arrive in
      // increasing order, so a strict '<' insertion keeps (distance, code) lexicographic order.  C_j here carries the
      // tensor core's split-fp16 / truncating-accumulator error (~1e-8 against a distance grid of ulp(A) ~ 3e-5), so
      // the FOUR best are handed to femasr_vq_finish, which recomputes the exact fp32 distance of every candidate
      // within a few ulps of the best and applies the reference's tie rule; a row whose best code is clear of the rest
      // by more than that margin needs no second look.
      constexpr int EPI_THREADS = 32 * Cfg::EPI_WARPS;
      uint2* merge = reinterpret_cast<uint2*>(smem_raw + (epi_base - smem_u32(smem_raw)));
      float td0 = INFINITY, td1 = INFINITY, td2 = INFINITY, td3 = INFINITY;
      int tj0 = 0x7fffffff, tj1 = 0x7fffffff, tj2 = 0x7fffffff, tj3 = 0x7fffffff;
      float a_row = 0.f;
      auto insert = [&](float d, int j) {          // precondition: (d, j) sorts before (td3, tj3)
        td3 = d; tj3 = j;
        if (td3 < td2 || (td3 == td2 && tj3 < tj2)) { float t = td2; td2 = td3; td3 = t; int u = tj2; tj2 = tj3; tj3 = u; }
        if (td2 < td1 || (td2 == td1 && tj2 < tj1)) { float t = td1; td1 = td2; td2 = t; int u = tj1; tj1 = tj2; tj2 = u; }
        if (td1 < td0 || (td1 == td0 && tj1 < tj0)) { float t = td0; td0 = td1; td1 = t; int u = tj0; tj0 = tj1; tj1 = u; }
      };
      for (int it = 0, work; (work = work_of(it)) >= 0; ++it) {
        const TileCoord tc = decode(work);
        const long token = (long)tc.tx * p.Wt + row;          // ksize 1: the features are one long row of tokens
        const bool valid = token < p.W;
        if (tc.nt == 0) {
          td0 = td1 = td2 = td3 = INFINITY;
          tj0 = tj1 = tj2 = tj3 = 0x7fffffff;
          a_row = valid ? __ldg(p.vq_a + token) : 0.f;
        }
        stage_cols(p.vq_esq, tc.nt);
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        const uint32_t t_row = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * BN + part * CW);
        const int colbase = tc.nt * BN + part * CW;
#pragma unroll 1
        for (int ci = 0; ci < NCH; ++ci) {
          uint32_t r[16];
          tmem_ld16(t_row + (uint32_t)(ci * CH), r);
          const float4* es4 = reinterpret_cast<const float4*>(sbias + part * CW + ci * CH);
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            const float4 es = es4[q4];
            const float ee[4] = {es.x, es.y, es.z, es.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float c = __uint_as_float(r[4 * q4 + k]) * inv_scale;                          // exact (power of two)
              const float d = __fsub_rn(__fadd_rn(a_row, ee[k]), __fmul_rn(2.0f, c));              // fl(fl(A + B_j) - 2 C_j)
              if (d < td3) insert(d, colbase + ci * CH + 4 * q4 + k);
            }
          }
        }
        tc_fence_before();
        release_acc(acc);
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        if (tc.nt == p.n_tiles - 1) {
          // the column parts of a row live in different warps: merge their lists through shared memory
          uint2* m = merge + (row * Cfg::NSPLIT + part) * 4;
          m[0] = make_uint2(__float_as_uint(td0), (uint32_t)tj0); m[1] = make_uint2(__float_as_uint(td1), (uint32_t)tj1);
          m[2] = make_uint2(__float_as_uint(td2), (uint32_t)tj2); m[3] = make_uint2(__float_as_uint(td3), (uint32_t)tj3);
          asm volatile("bar.sync 1, %0;" ::"r"(EPI_THREADS) : "memory");
          if (part == 0) {
            for (int pp = 1; pp < Cfg::NSPLIT; ++pp)
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint2 v = merge[(row * Cfg::NSPLIT + pp) * 4 + k];
                const float d = __uint_as_float(v.x);
                const int j = (int)v.y;
                if (d < td3 || (d == td3 && j < tj3)) insert(d, j);
              }
            if (valid) {
              uint4* out = reinterpret_cast<uint4*>(p.vq_cand + token * 4);
              out[0] = make_uint4(__float_as_uint(td0), (uint32_t)tj0, __float_as_uint(td1), (uint32_t)tj1);
              out[1] = make_uint4(__float_as_uint(td2), (uint32_t)tj2, __float_as_uint(td3), (uint32_t)tj3);
            }
          }
          asm volatile("bar.sync 1, %0;" ::"r"(EPI_THREADS) : "memory");
        }
      }
    } else
    for (int it = 0, work; (work = work_of(it)) >= 0; ++it)
    for (int mr = 0; mr < MR; ++mr) {          // multi-row strip tiles: one accumulator per image row, in completion order
      const TileCoord tc = decode(work);
      const int nt = tc.nt, tx = tc.tx, ty = tc.ty * MR + mr, b = tc.b, ph = tc.ph;
      const int y = ty * p.Ht + (row >> p.wt_shift), x = tx * p.Wt + (row & (p.Wt - 1));
      const bool valid = tc.real && y < p.H && x < p.W;
      const bool gn_ok = tc.real && (MR == 1 || ty < p.H);      // a multi-row tile may hang over the last image row
      const int oy = p.up ? 2 * y + (ph >> 1) : y, ox = p.up ? 2 * x + (ph & 1) : x;
      const int Ho = p.up ? 2 * p.H : p.H, Wo = p.up ? 2 * p.W : p.W;
      const int col0 = nt * BN + part * CW;
      const long myoff = valid ? (((long)b * Ho + oy) * Wo + ox) * p.Cout + col0 : -1;   // this lane's accumulator row
      long offs[4];                                  // rows it*8 + rsub of the coalesced phase, columns 4q..4q+3
#pragma unroll
      for (int it = 0; it < 4; ++it) { const long o = __shfl_sync(0xffffffffu, myoff, it * 8 + rsub); offs[it] = o < 0 ? -1 : o + 4 * q; }
      float4 cur[4], nxt[4];
      if (RES) {
#pragma unroll
        for (int it = 0; it < 4; ++it)
          cur[it] = offs[it] >= 0 ? *reinterpret_cast<const float4*>(p.res1 + offs[it]) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (p.bias) stage_cols(p.bias, nt);
      // sliced accumulation: fold all but the last partial into the running sum S (second TMEM buffer)
      const uint32_t t_sum = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)((Cfg::S3 ? 2 * BN : BN) + part * CW);
      for (int s = 0; s + 1 < nslices; ++s) {
        const int fa = Cfg::S3 ? acc : 0;              // buffer holding this partial
        mbar_wait(tfull_bar(fa), acc_phase);
        if (!Cfg::S3) acc_phase ^= 1u;
        tc_fence_after();
        const uint32_t t_part = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(fa * BN + part * CW);
#pragma unroll 1
        for (int ci = 0; ci < NCH; ++ci) {
          uint32_t pr[16];
          tmem_ld16(t_part + (uint32_t)(ci * CH), pr);
          if (s > 0) {
            uint32_t sr[16];
            tmem_ld16(t_sum + (uint32_t)(ci * CH), sr);
#pragma unroll
            for (int j = 0; j < 16; ++j) pr[j] = __float_as_uint(__uint_as_float(pr[j]) + __uint_as_float(sr[j]));
          }
          tmem_st16(t_sum + (uint32_t)(ci * CH), pr);
        }
        tmem_wait_st();
        tc_fence_before();
        release_acc(fa);
        if (Cfg::S3 && ++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * BN + part * CW);
      uint32_t rn[16];                                   // next chunk's accumulators (64-wide tiles only)
#pragma unroll 1
      for (int ci = 0; ci < NCH; ++ci) {
        const int c = ci * CH;
        if (RES && ci + 1 < NCH) {
          // next chunk's residual, requested a whole chunk ahead (DRAM latency ~ one chunk of epilogue work)
#pragma unroll
          for (int it = 0; it < 4; ++it)
            nxt[it] = offs[it] >= 0 ? *reinterpret_cast<const float4*>(p.res1 + offs[it] + c + CH) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        // this lane's 4 columns of the chunk in the coalesced phase: [c + 4q, c + 4q + 4)
        const float4 bq = p.bias ? *reinterpret_cast<const float4*>(sbias + part * CW + c + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        // 64-wide tiles (8 epilogue warps, registers to spare): the NEXT chunk's TMEM load is already in flight while this
        // chunk goes through its transpose / math / store phases (the exposed tcgen05.ld latency was 9 % of the 64 -> 64
        // conv's samples); the wide tiles sit at the 96-register cap of a 640-thread CTA and load on demand.
        constexpr bool PIPE_LD = Cfg::NSPLIT == 2;         // 8 epilogue warps: up to 168 registers per thread
        uint32_t r[16];
        if (PIPE_LD && nslices == 1) {
          if (ci == 0) tmem_ld16_async(t_row, rn);
          tmem_wait_ld(rn);
#pragma unroll
          for (int j = 0; j < 16; ++j) r[j] = rn[j];
          if (ci + 1 < NCH) tmem_ld16_async(t_row + (uint32_t)(c + CH), rn);
        } else {
          tmem_ld16(t_row + (uint32_t)c, r);
        }
        if (nslices > 1) {
          uint32_t sr[16];
          tmem_ld16(t_sum + (uint32_t)c, sr);
#pragma unroll
          for (int j = 0; j < 16; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(sr[j]));
        }
        // phase 1: the raw accumulators go straight into the (XOR-swizzled) transpose tile; scale, bias, GELU and the
        // residual adds all happen in the coalesced layout below, where a lane owns the same 4 columns in all four row
        // groups: ONE bias float4 per chunk (requested before the TMEM load), no shared-memory latency inside the math.
        if (p.tma_out) {                                   // the previous chunk's bulk store must have read the tile
          if (lane == 0) bulk_wait_read0();
          __syncwarp();
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<uint4*>(&stage[lane * 16 + 4 * (j ^ ((lane >> 1) & 3))]) = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
        __syncwarp();
        // phase 2: all four row groups are read before any is stored - distinct registers, so a store's operands are
        // never the destination of the next load (ncu: the single-register version spent 18 % of the qkv epilogue in
        // long-scoreboard stalls behind its own stores)
        float4 o4[4];
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rr = it * 8 + rsub;
          o4[it] = *reinterpret_cast<const float4*>(&stage[rr * 16 + 4 * (q ^ ((rr >> 1) & 3))]);
        }
        float sa = 0.f, ssa = 0.f, sb = 0.f, ssb = 0.f;   // GroupNorm partials of channels (x,y) and (z,w)
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          float4 o = o4[it];
          o.x = fmaf(o.x, inv_scale, bq.x); o.y = fmaf(o.y, inv_scale, bq.y);      // acc * 2^-s is exact: == (acc * inv) + bias
          o.z = fmaf(o.z, inv_scale, bq.z); o.w = fmaf(o.w, inv_scale, bq.w);
          if (p.act == FEMASR_ACT_GELU) { o.x = gelu_erf_fast_f(o.x); o.y = gelu_erf_fast_f(o.y); o.z = gelu_erf_fast_f(o.z); o.w = gelu_erf_fast_f(o.w); }
          if (RES) { o.x += cur[it].x; o.y += cur[it].y; o.z += cur[it].z; o.w += cur[it].w; }
          o4[it] = o;
        }
        if (p.res2) {
#pragma unroll
          for (int it = 0; it < 4; ++it)
            if (offs[it] >= 0) {
              const float4 rv = *reinterpret_cast<const float4*>(p.res2 + offs[it] + c);
              o4[it].x += rv.x; o4[it].y += rv.y; o4[it].z += rv.z; o4[it].w += rv.w;
            }
        }
        if (p.gn_partial) {
#pragma unroll
          for (int it = 0; it < 4; ++it)
            if (offs[it] >= 0) {
              const float4 o = o4[it];
              sa += o.x + o.y; ssa = fmaf(o.x, o.x, fmaf(o.y, o.y, ssa));
              sb += o.z + o.w; ssb = fmaf(o.z, o.z, fmaf(o.w, o.w, ssb));
            }
        }
        if (p.tma_out) {
          // The finished values go back into the staging tile and leave as ONE bulk tensor store per plane, issued by an
          // elected lane: no per-thread global addresses, no LSU wavefronts per 64-byte row segment and - the point - no
          // register held hostage by an unretired store (ncu: ~20 % of the epilogue's samples were long-scoreboard WAR
          // stalls behind STG).  Rows / columns past the tensor edge are clipped by the TMA; dummy pair tiles carry an
          // out-of-range image index and are dropped entirely.
          const int r0 = ew * 32;                          // first accumulator row of this warp
          const int bx = tx * p.Wt + (r0 & (p.Wt - 1)), by = ty * p.Ht + (r0 >> p.wt_shift);
          const uint32_t st_addr = smem_u32(stage);
          if (p.tma_out == 1) {
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              const int rr = it * 8 + rsub;
              *reinterpret_cast<float4*>(&stage[rr * 16 + 4 * (q ^ ((rr >> 1) & 3))]) = o4[it];     // in place: the cell this lane read
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) { tma_store_4d(&map_y, st_addr, col0 + c, bx, by, b); bulk_commit(); }
          } else {
            __syncwarp();                                  // every lane has read its fp32 cells before halves overwrite them
            __half* sh = reinterpret_cast<__half*>(stage);   // hi plane [32][16] halves, then the lo plane
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              const int rr = it * 8 + rsub;
              uint2 h, l;
              split_pack2(o4[it].x, o4[it].y, h.x, l.x);
              split_pack2(o4[it].z, o4[it].w, h.y, l.y);
              *reinterpret_cast<uint2*>(sh + rr * 16 + 4 * q) = h;
              *reinterpret_cast<uint2*>(sh + 512 + rr * 16 + 4 * q) = l;
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              tma_store_4d(&map_oh, st_addr, col0 + c, bx, by, b);
              tma_store_4d(&map_ol, st_addr + 1024, col0 + c, bx, by, b);
              bulk_commit();
            }
          }
        } else {
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            if (offs[it] >= 0) {
              const long off = offs[it] + c;
              const float4 o = o4[it];
              if (p.out_hi) {
                uint2 h, l;
                split_pack2(o.x, o.y, h.x, l.x);
                split_pack2(o.z, o.w, h.y, l.y);
                *reinterpret_cast<uint2*>(p.out_hi + off) = h;
                *reinterpret_cast<uint2*>(p.out_lo + off) = l;
              } else {
                *reinterpret_cast<float4*>(p.y + off) = o;
              }
            }
          }
        }
        if (p.gn_partial) {
          // fixed-order reduction over the warp's 32 rows (lanes sharing q), then one partial per group
#pragma unroll
          for (int o = 4; o <= 16; o <<= 1) {
            sa += __shfl_xor_sync(0xffffffffu, sa, o); ssa += __shfl_xor_sync(0xffffffffu, ssa, o);
            sb += __shfl_xor_sync(0xffffffffu, sb, o); ssb += __shfl_xor_sync(0xffffffffu, ssb, o);
          }
          const int tile_in_img = (ph * p.tiles_y * MR + ty) * p.tiles_x + tx;
          float* gp = p.gn_partial + (((long)b * p.gn_rows + tile_in_img * 4 + ew) * 32) * 2;
          const int ch0 = col0 + c;                      // first channel of this chunk
          if (p.cpg == 8) {
            float s1 = sa + sb, s2 = ssa + ssb;
            s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
            if (gn_ok && (lane == 0 || lane == 2)) *reinterpret_cast<float2*>(gp + (ch0 / 8 + (lane >> 1)) * 2) = make_float2(s1, s2);
          } else if (p.cpg == 4) {
            if (gn_ok && lane < 4) *reinterpret_cast<float2*>(gp + (ch0 / 4 + lane) * 2) = make_float2(sa + sb, ssa + ssb);
          } else {
            if (gn_ok && lane < 4) {
              *reinterpret_cast<float2*>(gp + (ch0 / 2 + 2 * lane) * 2) = make_float2(sa, ssa);
              *reinterpret_cast<float2*>(gp + (ch0 / 2 + 2 * lane + 1) * 2) = make_float2(sb, ssb);
            }
          }
        }
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 4; ++it) if (RES) cur[it] = nxt[it];
      }
      tc_fence_before();
      release_acc(acc);                         // one arrival per epilogue warp releases the accumulator
      if (sliced && !Cfg::S3) acc_phase ^= 1u;
      else if (++acc == NACC) { acc = 0; acc_phase ^= 1u; }
    }
  }
  if (warp >= 4 && lane == 0 && p.tma_out) bulk_wait_all();      // bulk stores read this CTA's shared memory
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------ operand preparation
__device__ __forceinline__ void split_store8(const float (&v)[8], __half* hi, __half* lo) {
  __align__(16) __half h[8], l[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float c = fminf(fmaxf(v[i], -65504.f), 65504.f);
    h[i] = __float2half_rn(c);
    l[i] = __float2half_rn(c - __half2float(h[i]));
  }
  *reinterpret_cast<uint4*>(hi) = *reinterpret_cast<const uint4*>(h);
  *reinterpret_cast<uint4*>(lo) = *reinterpret_cast<const uint4*>(l);
}

// x fp32 NHWC [B,H,W,C] -> fp16 hi/lo planes [B,H*up,W*up,C] with an optional GroupNorm+SiLU transform
// (scale/shift tables [B,C]) and optional nearest x2 replication.  8 channels per thread.
template <int MODE>
__global__ void __launch_bounds__(256) tc_prepare_kernel(const float* __restrict__ x, __half* __restrict__ hi,
                                                         __half* __restrict__ lo, const float* __restrict__ sc,
                                                         const float* __restrict__ sh, int H, int W, int C, int up,
                                                         long total8) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total8) return;
  const int c8 = C / 8;
  const int cq = (int)(i % c8);
  const long pix = i / c8;
  const int xw = (int)(pix % W);
  const long t = pix / W;
  const int yh = (int)(t % H);
  const int b = (int)(t / H);
  const float4* src = reinterpret_cast<const float4*>(x + pix * C + cq * 8);
  const float4 a = __ldg(src), bq = __ldg(src + 1);
  float v[8] = {a.x, a.y, a.z, a.w, bq.x, bq.y, bq.z, bq.w};
  if (MODE == FEMASR_PRO_GN_SILU) {
    const float4* ps = reinterpret_cast<const float4*>(sc + (long)b * C + cq * 8);
    const float4* pt = reinterpret_cast<const float4*>(sh + (long)b * C + cq * 8);
    const float4 s0 = __ldg(ps), s1 = __ldg(ps + 1), t0 = __ldg(pt), t1 = __ldg(pt + 1);
    const float s[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
    const float tt[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = silu_f(fmaf(v[k], s[k], tt[k]));
  }
  if (!up) {
    split_store8(v, hi + pix * C + cq * 8, lo + pix * C + cq * 8);
  } else {
    const int W2 = 2 * W;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const long op = (((long)b * 2 * H + 2 * yh + dy) * W2 + 2 * xw + dx) * C + cq * 8;
        split_store8(v, hi + op, lo + op);
      }
  }
}

// Same transform without replication, organised for bandwidth: the image is a flat array of float4 (4 channels), a warp
// reads 512 contiguous bytes per request and every thread keeps PREP_U independent requests in flight; blockIdx.y = b.
constexpr int PREP_U = 4;
template <int MODE>
__global__ void __launch_bounds__(256) tc_prepare_flat_kernel(const float4* __restrict__ x, uint2* __restrict__ hi,
                                                              uint2* __restrict__ lo, const float* __restrict__ sc,
                                                              const float* __restrict__ sh, int C, int per_image4) {
  const int b = blockIdx.y;
  const long base = (long)b * per_image4;
  const int i0 = blockIdx.x * (256 * PREP_U) + threadIdx.x;
  const int c4 = C >> 2;
  float4 v[PREP_U];
#pragma unroll
  for (int u = 0; u < PREP_U; ++u) {
    const int i = i0 + u * 256;
    if (i < per_image4) v[u] = __ldg(x + base + i);
  }
#pragma unroll
  for (int u = 0; u < PREP_U; ++u) {
    const int i = i0 + u * 256;
    // `continue`, not `break` (same result: i grows with u): with `break` the optimiser sinks each load above next to its
    // use, and the fast-SiLU variant kept one request in flight instead of PREP_U (27 instead of 40 registers)
    if (i >= per_image4) continue;
    float w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
    if (MODE == FEMASR_PRO_GN_SILU || MODE == FEMASR_PRO_GN_SILU_FAST) {
      const int c = (i % c4) * 4;
      const float4 s = __ldg(reinterpret_cast<const float4*>(sc + (long)b * C + c));
      const float4 t = __ldg(reinterpret_cast<const float4*>(sh + (long)b * C + c));
      const float ss[4] = {s.x, s.y, s.z, s.w}, tt[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float n = fmaf(w[k], ss[k], tt[k]);
        // fast form: 2 MUFU + 3 FP32 ops instead of ~25 instructions (this pass is issue-bound with the exact one)
        w[k] = MODE == FEMASR_PRO_GN_SILU_FAST ? __fdividef(n, 1.0f + __expf(-n)) : silu_f(n);
      }
    }
    __align__(8) __half h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float cl = fminf(fmaxf(w[k], -65504.f), 65504.f);
      h[k] = __float2half_rn(cl);
      l[k] = __float2half_rn(cl - __half2float(h[k]));
    }
    hi[base + i] = *reinterpret_cast<const uint2*>(h);
    lo[base + i] = *reinterpret_cast<const uint2*>(l);
  }
}

// F8 staging (layers behind the VQ): the hi plane as above; the second plane holds, per pixel and 64-channel chunk, 128
// bytes = [e4m3((v - hi) * 2^10) x 64 | e4m3(v * 2^-2) x 64] - the A operand of the single K = 128 fp8 MMA group that
// replaces the two fp16 cross products (the weights carry [e4m3(w_hi * 2^-10) | e4m3(w_lo * 2^2)] at the matching offsets,
// so both power-of-two scales cancel inside the dot product).
// Error budget: scripts/exp_fp8_cross.py, 1.2e-4 output max-abs for the whole post-VQ scope (bar 1e-3).
// The scales place the operands in e4m3's normal range (4 significant bits down to 2^-6, fewer below, nothing under 2^-10).
// The first recipe, (2^12, 2^0), was tuned on the kaiming-uniform random-init weights, whose magnitudes all lie within a
// factor 2 of the per-tensor maximum; a TRAINED conv is bell-shaped with typical |w| ~ max / 10 ... max / 50, for which
// e4m3(w_hi * 2^-12) <= 0.25 * |w| / max is already subnormal.  scripts/exp_fp8_scales.py (weights of the layers behind the
// VQ redrawn from a normal / a Student-t(3) distribution of the same standard deviation; output max-abs uniform / normal /
// t(3)): (12, 0) 1.2e-4 / 1.1e-4 / 5.8e-4, (10, 2) 1.3e-4 / 1.4e-4 / 1.8e-4 - the minimax choice over a 10-recipe sweep.
// Activations keep full e4m3 precision for |a| in [2^-4, 1792] (a_lo * 2^10 ~ a / 4 likewise).
constexpr float F8_LO_SCALE = 1024.0f;       // a_lo * 2^10 against w_hi * 2^-10
constexpr float F8_VAL_SCALE = 0.25f;        // a * 2^-2 against w_lo * 2^2
__device__ __forceinline__ uint32_t pack_e4m3x4(float a, float b, float c, float d) {
  const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E4M3);
  const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, __NV_E4M3);
  return lo | (hi << 16);
}
template <int MODE>
__global__ void __launch_bounds__(256) tc_prepare_flat_f8_kernel(const float4* __restrict__ x, uint4* __restrict__ hi,
                                                                 uint2* __restrict__ x8, const float* __restrict__ sc,
                                                                 const float* __restrict__ sh, int C, int per_image8) {
  // one thread = 8 consecutive channels of a pixel: 32 bytes in, 16 (hi) + 8 (lo8) + 8 (value8) bytes out
  constexpr int U = 2;
  const int b = blockIdx.y;
  const long base = (long)b * per_image8;
  const int i0 = blockIdx.x * (256 * U) + threadIdx.x;
  const int c8 = C >> 3;
  float4 v[U][2];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int i = i0 + u * 256;
    if (i < per_image8) { v[u][0] = __ldg(x + 2 * (base + i)); v[u][1] = __ldg(x + 2 * (base + i) + 1); }
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int i = i0 + u * 256;
    if (i >= per_image8) break;
    float w[8] = {v[u][0].x, v[u][0].y, v[u][0].z, v[u][0].w, v[u][1].x, v[u][1].y, v[u][1].z, v[u][1].w};
    const int c = (i % c8) * 8;
    if (MODE == FEMASR_PRO_GN_SILU || MODE == FEMASR_PRO_GN_SILU_FAST) {
      const float4* ps = reinterpret_cast<const float4*>(sc + (long)b * C + c);
      const float4* pt = reinterpret_cast<const float4*>(sh + (long)b * C + c);
      const float4 s0 = __ldg(ps), s1 = __ldg(ps + 1), t0 = __ldg(pt), t1 = __ldg(pt + 1);
      const float ss[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
      const float tt[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float n = fmaf(w[k], ss[k], tt[k]);
        w[k] = MODE == FEMASR_PRO_GN_SILU_FAST ? __fdividef(n, 1.0f + __expf(-n)) : silu_f(n);
      }
    }
    float l[8];
    uint32_t hp[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      uint32_t lo_unused;
      const float a = fminf(fmaxf(w[2 * k], -65504.f), 65504.f), bq = fminf(fmaxf(w[2 * k + 1], -65504.f), 65504.f);
      asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hp[k]) : "f"(bq), "f"(a));
      const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hp[k]));
      l[2 * k] = (a - hf.x) * F8_LO_SCALE; l[2 * k + 1] = (bq - hf.y) * F8_LO_SCALE;
      w[2 * k] = a; w[2 * k + 1] = bq;
      (void)lo_unused;
    }
    hi[base + i] = make_uint4(hp[0], hp[1], hp[2], hp[3]);
    // byte layout of the pixel's x8 row: chunk (c / 64) * 128 + (c % 64) for the lo part, + 64 for the value part
    const long pix = (base + i) / c8;
    const long q = pix * (C >> 2) + (c >> 6) * 16 + ((c & 63) >> 3);          // index in 8-byte units
    x8[q] = make_uint2(pack_e4m3x4(l[0], l[1], l[2], l[3]), pack_e4m3x4(l[4], l[5], l[6], l[7]));
    x8[q + 8] = make_uint2(pack_e4m3x4(w[0] * F8_VAL_SCALE, w[1] * F8_VAL_SCALE, w[2] * F8_VAL_SCALE, w[3] * F8_VAL_SCALE),
                           pack_e4m3x4(w[4] * F8_VAL_SCALE, w[5] * F8_VAL_SCALE, w[6] * F8_VAL_SCALE, w[7] * F8_VAL_SCALE));
  }
}

// LayerNorm (C = 256, eps) fused with the split: one warp per token row.
__global__ void __launch_bounds__(256) tc_prepare_ln_kernel(const float* __restrict__ x, __half* __restrict__ hi,
                                                            __half* __restrict__ lo, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, long M, float eps) {
  // two rows per warp, all four 512-byte requests of the warp in flight before the first reduction (the one-row version
  // ran at 5.2 TB/s against 6.5-6.9 of the flat staging kernels)
  constexpr int LN_ROWS = 2;
  const long row0 = ((long)blockIdx.x * 8 + (threadIdx.x >> 5)) * LN_ROWS;
  if (row0 >= M) return;
  const int lane = threadIdx.x & 31;
  // lane owns columns [4 lane, 4 lane + 4) and [128 + 4 lane, ...): two fully coalesced 512-byte requests per row
  float4 a[LN_ROWS], b[LN_ROWS];
#pragma unroll
  for (int rr = 0; rr < LN_ROWS; ++rr) {
    if (row0 + rr < M) {
      const float4* r = reinterpret_cast<const float4*>(x + (row0 + rr) * 256) + lane;
      a[rr] = __ldg(r); b[rr] = __ldg(r + 32);
    }
  }
  const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma) + lane), g1 = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32);
  const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta) + lane), b1 = __ldg(reinterpret_cast<const float4*>(beta) + lane + 32);
  const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
  const float be[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
  for (int rr = 0; rr < LN_ROWS; ++rr) {
    const long row = row0 + rr;
    if (row >= M) break;
    float v[8] = {a[rr].x, a[rr].y, a[rr].z, a[rr].w, b[rr].x, b[rr].y, b[rr].z, b[rr].w};
    float s = ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
    s = warp_sum(s);
    const float mu = s * (1.0f / 256.0f);
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) { const float d = v[k] - mu; q = fmaf(d, d, q); }
    q = warp_sum(q) * (1.0f / 256.0f);
    const float rs = 1.0f / sqrtf(q + eps);
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = (v[k] - mu) * rs * g[k] + be[k];
    uint2 h0, l0, h1, l1;
    split_pack2(v[0], v[1], h0.x, l0.x); split_pack2(v[2], v[3], h0.y, l0.y);
    split_pack2(v[4], v[5], h1.x, l1.x); split_pack2(v[6], v[7], h1.y, l1.y);
    uint2* ph = reinterpret_cast<uint2*>(hi + row * 256) + lane;
    uint2* pl = reinterpret_cast<uint2*>(lo + row * 256) + lane;
    ph[0] = h0; ph[32] = h1;
    pl[0] = l0; pl[32] = l1;
  }
}

// weights: OIHW fp32 -> [Cout][taps*Cin] fp16 hi/lo planes of w * 2^s, s chosen so max|w|*2^s is in [512,1024)
__global__ void absmax_kernel(const float* __restrict__ w, unsigned int* __restrict__ out, long n) {
  float m = 0.f;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(w[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));   // non-negative floats order like uints
}
__global__ void tc_pack_weight_kernel(const float* __restrict__ w, __half* __restrict__ hi, __half* __restrict__ lo,
                                      const unsigned int* __restrict__ absmax, float* __restrict__ inv_scale, int Cout,
                                      int Cin, int KH, int KW) {
  const float mx = __uint_as_float(*absmax);
  int ex = 0;
  if (mx > 0.f) frexpf(mx, &ex);          // mx = f * 2^ex, f in [0.5,1)
  const int s = mx > 0.f ? 10 - ex : 0;   // mx * 2^s in [512, 1024)
  const float scale = ldexpf(1.0f, s);
  const long n = (long)Cout * Cin * KH * KW;
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *inv_scale = ldexpf(1.0f, -s);
  if (i >= n) return;
  // i indexes the packed layout [co][(kh*KW+kw)*Cin + ci]
  const long K = (long)Cin * KH * KW;
  const int co = (int)(i / K);
  const long k = i - (long)co * K;
  const int tap = (int)(k / Cin), ci = (int)(k - (long)tap * Cin);
  const int kh = tap / KW, kw = tap - kh * KW;
  const float v = w[(((long)co * Cin + ci) * KH + kh) * KW + kw] * scale;   // exact (power of two)
  const __half h = __float2half_rn(v);
  hi[i] = h;
  lo[i] = __float2half_rn(v - __half2float(h));
}

// F8 variant of the packed weights: hi plane as above; the second plane holds per (row, 64-wide k chunk) 128 bytes =
// [e4m3(w_hi * 2^-10) x 64 | e4m3(w_lo * 2^2) x 64] (see tc_prepare_flat_f8_kernel)
__global__ void tc_pack_weight_f8_kernel(const float* __restrict__ w, __half* __restrict__ hi, uint8_t* __restrict__ x8,
                                         const unsigned int* __restrict__ absmax, float* __restrict__ inv_scale, int Cout,
                                         int Cin, int KH, int KW) {
  const float mx = __uint_as_float(*absmax);
  int ex = 0;
  if (mx > 0.f) frexpf(mx, &ex);
  const int s = mx > 0.f ? 10 - ex : 0;
  const float scale = ldexpf(1.0f, s);
  const long n = (long)Cout * Cin * KH * KW;
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) *inv_scale = ldexpf(1.0f, -s);
  if (i >= n) return;
  const long K = (long)Cin * KH * KW;
  const int co = (int)(i / K);
  const long k = i - (long)co * K;
  const int tap = (int)(k / Cin), ci = (int)(k - (long)tap * Cin);
  const int kh = tap / KW, kw = tap - kh * KW;
  const float v = w[(((long)co * Cin + ci) * KH + kh) * KW + kw] * scale;
  const __half h = __float2half_rn(v);
  hi[i] = h;
  const float hf = __half2float(h);
  uint8_t* row = x8 + (long)co * K * 2 + (k >> 6) * 128 + (k & 63);
  row[0] = (uint8_t)__nv_cvt_float_to_fp8(hf * (1.0f / F8_LO_SCALE), __NV_SATFINITE, __NV_E4M3);
  row[64] = (uint8_t)__nv_cvt_float_to_fp8((v - hf) * (1.0f / F8_VAL_SCALE), __NV_SATFINITE, __NV_E4M3);
}

// nearest-x2 upsample followed by a 3x3 conv == four 2x2 convs on the low-res grid (one per output phase
// (py,px)), whose weights are sums of the 3x3 taps that land on the same source pixel:
//   rows: py=0 -> {kh=0 | kh=1,2},  py=1 -> {kh=0,1 | kh=2};  same for columns.  2.25x fewer MACs.
// out: fp32 [4*Cout][Cin][2][2] (OIHW of the stacked phase filters), summed in a fixed order.
__global__ void subpixel_weights_kernel(const float* __restrict__ w, float* __restrict__ out, int Cout, int Cin) {
  const long n = (long)4 * Cout * Cin * 4;
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int bq = (int)(i & 1), a = (int)((i >> 1) & 1);
  long r = i >> 2;
  const int ci = (int)(r % Cin); r /= Cin;
  const int co = (int)(r % Cout);
  const int ph = (int)(r / Cout);
  const int py = ph >> 1, px = ph & 1;
  const int kh0 = py == 0 ? (a == 0 ? 0 : 1) : (a == 0 ? 0 : 2), kh1 = py == 0 ? (a == 0 ? 0 : 2) : (a == 0 ? 1 : 2);
  const int kw0 = px == 0 ? (bq == 0 ? 0 : 1) : (bq == 0 ? 0 : 2), kw1 = px == 0 ? (bq == 0 ? 0 : 2) : (bq == 0 ? 1 : 2);
  const float* wp = w + ((long)co * Cin + ci) * 9;
  float sum = 0.f;
  for (int kh = kh0; kh <= kh1; ++kh)
    for (int kw = kw0; kw <= kw1; ++kw) sum += wp[kh * 3 + kw];
  out[i] = sum;
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

static int make_map(CUtensorMap* m, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                    const cuuint32_t* box, int spatial_stride = 1, CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_FLOAT16,
                    CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(FEMASR_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint32_t estr[4] = {1, (cuuint32_t)spatial_stride, (cuuint32_t)spatial_stride, 1};
  if (rank == 2) estr[1] = 1;
  CUresult r = enc(m, dtype, (cuuint32_t)rank, const_cast<void*>(ptr), dims, strides_bytes, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(FEMASR_ERR_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
  return FEMASR_OK;
}

// Launch in clusters of cluster_x CTAs along x (2: the CTA pairs of the cta_group::2 kernels; 1: a plain launch).
template <class... KArgs, class... Args>
static cudaError_t launch_clustered(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                   int cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = cluster_x; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cfg.attrs = &attr; cfg.numAttrs = cluster_x > 1 ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// output maps of the TMA-store epilogue (valid when p.tma_out != 0; otherwise copies of an input map, never dereferenced)
struct OutMaps { CUtensorMap y, oh, ol; };

template <int BN, bool PAIR, bool STRIP, bool BRES, bool RES>
static int launch_tc_v(const CUtensorMap& ah, const CUtensorMap& al, const CUtensorMap& bh, const CUtensorMap& bl,
                       const OutMaps& om, const TcP& p, cudaStream_t st) {
  using Cfg = TcCfg<BN, PAIR, STRIP, BRES>;
  static PerDeviceFlag attr_set;      // per template instantiation AND per device
  if (!attr_set.cur()) {
    FEMASR_CUDA(cudaFuncSetAttribute(tc_igemm_kernel<BN, PAIR, STRIP, BRES, RES>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set.cur() = true;
  }
  if constexpr (!PAIR) {
    const int grid = p.num_tiles < sm_count() ? p.num_tiles : sm_count();
    FEMASR_CUDA(launch_clustered(tc_igemm_kernel<BN, false, STRIP, BRES, RES>, dim3(grid), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, st, 1,
                           ah, al, bh, bl, om.y, om.oh, om.ol, p));
    return launch_status("tc_igemm_kernel");
  } else {
    const int num_m = p.num_tiles / p.n_tiles;
    const int phases = p.up ? 4 : 1;
    const int work = phases * ((num_m / phases + 1) / 2) * p.n_tiles;
    const int pairs = work < sm_count() / 2 ? work : sm_count() / 2;
    FEMASR_CUDA(launch_clustered(tc_igemm_kernel<BN, true, STRIP, false, RES>, dim3(2 * pairs), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, st, 2,
                           ah, al, bh, bl, om.y, om.oh, om.ol, p));
    return launch_status("tc_igemm_kernel(pair)");
  }
}

template <int BN, bool PAIR, bool STRIP, bool BRES = false>
static int launch_tc(const CUtensorMap& ah, const CUtensorMap& al, const CUtensorMap& bh, const CUtensorMap& bl,
                     const OutMaps& om, const TcP& p, cudaStream_t st) {
  return p.res1 ? launch_tc_v<BN, PAIR, STRIP, BRES, true>(ah, al, bh, bl, om, p, st)
                : launch_tc_v<BN, PAIR, STRIP, BRES, false>(ah, al, bh, bl, om, p, st);
}

template <int BN>
static int launch_vq(const CUtensorMap& ah, const CUtensorMap& al, const CUtensorMap& bh, const CUtensorMap& bl,
                     const TcP& p, cudaStream_t st) {
  using Cfg = TcCfg<BN, false, false, false>;
  static PerDeviceFlag attr_set;
  if (!attr_set.cur()) {
    FEMASR_CUDA(cudaFuncSetAttribute(tc_igemm_kernel<BN, false, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set.cur() = true;
  }
  const int num_m = p.num_tiles / p.n_tiles;
  const int grid = num_m < sm_count() ? num_m : sm_count();
  FEMASR_CUDA(launch_clustered(tc_igemm_kernel<BN, false, false, false, false, true>, dim3(grid), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, st, 1,
                         ah, al, bh, bl, ah, ah, ah, p));
  return launch_status("tc_igemm_kernel(vq)");
}

}  // namespace femasr

using namespace femasr;

static void tc_tile_shape(int H, int W, int* Wt, int* Ht) {
  int best_wt = 8; long best_cost = -1;
  for (int wt = 128; wt >= 8; wt >>= 1) {
    const int ht = 128 / wt;
    const long cost = cdiv(W, wt) * wt * cdiv(H, ht) * ht;
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_wt = wt; }
  }
  *Wt = best_wt; *Ht = 128 / best_wt;
}

// Tiling decisions shared by femasr_tc_igemm and femasr_tc_gn_partial_rows.  (H, W) = the grid the tiles run over.
struct TilePlan { int Wt, Ht, wt_shift, tiles_x, tiles_y, BN; bool pair, strip; };
static TilePlan plan_tiles(const femasr_tc_args* a, int H, int W) {
  TilePlan t;
  const int stride = a->stride == 2 ? 2 : 1;
  const int taps = a->upsample ? 4 : a->ksize * a->ksize;
  t.BN = a->Cout % 256 == 0 ? 256 : (a->Cout % 128 == 0 ? 128 : 64);
  // CTA pairs (tcgen05 cta_group::2): a->pair 1 = on, 0 = off, -1 = automatic.
  // Measured (profiles/microbench_*): pairing pays when the weight tile is wide and the K loop long enough to
  // amortise the pair's coupling - BN = 256 and K >= 1024 (+10..22 %); narrow / short-K layers are faster unpaired.
  // Round-2 sweep with the cheap (elect.sync) MMA issue (profiles/sweep_bn_pair_r2.txt): the plain fp32-output linears with
  // three or more column tiles (qkv) also gain 5 % paired; fc1 (GELU + split epilogue, issue-bound) and proj do not.
  const bool wide_plain_linear = a->ksize == 1 && a->act == FEMASR_ACT_NONE && a->y && a->Cout >= 768;
  t.pair = a->pair >= 0 ? a->pair != 0 : (t.BN == 256 && ((long)taps * a->Cin >= 1024 || wide_plain_linear));
  // K-sliced layers (in front of the VQ): 128-wide tiles - the accumulator drain of a slice is half as long, twice as
  // many tiles overlap it (fc2 0.210 -> 0.197 ms),
  // and with 128-wide tiles the three-buffer protocol applies (the MMA no longer waits for the fold): fc2 0.213 -> 0.181,
  // 256 -> 256 @64² sliced conv 0.367 -> 0.319 ms paired (profiles/sweep_bn_pair_r2.txt)
  if (a->slice_kb > 0 && t.BN == 256 && a->pair < 0) {
    t.BN = 128;
    t.pair = a->ksize == 3 && (long)taps * a->Cin >= 1024;
  }
  // strip mode (one activation strip shared by the three horizontal taps) wherever the layer allows it; a->strip 0 turns
  // it off, like a->pair
  const bool strip_ok = a->ksize == 3 && stride == 1 && !a->upsample && t.BN <= 128 && W >= 128 && a->kb_begin == 0 &&
                        a->kb_count == 0 && a->slice_kb == 0;
  t.strip = strip_ok && a->strip != 0;
  if (t.strip) {
    // strips over a CTA pair (two neighbouring row tiles share every weight tile, each CTA stages half of it): 128-wide
    // tiles with streamed weights only, unless a->pair = 0 asks for single-CTA strips.  The 128 -> 128 @256² convs
    // re-stream the whole 590 KB weight matrix per row tile and are L2-bound in F8 mode; same-box: 1.156 -> 1.056 ms
    // (F8), 1.490 -> 1.412 ms (three fp16 products), bit-identical results
    t.pair = t.BN == 128 && a->pair != 0;
    t.Wt = 128; t.Ht = 1;
  } else {
    tc_tile_shape(H, W, &t.Wt, &t.Ht);   // the widest power-of-two Wt <= 128 that wastes the fewest padded pixels
  }
  t.wt_shift = 0; while ((1 << t.wt_shift) < t.Wt) ++t.wt_shift;
  t.tiles_x = (int)cdiv(W, t.Wt); t.tiles_y = (int)cdiv(H, t.Ht);
  return t;
}

// rows of GroupNorm partials femasr_tc_igemm will write per image for this conv (same decision logic as the launch)
extern "C" int femasr_tc_gn_partial_rows(const femasr_tc_args* a) {
  if (!a) return 0;
  int H = a->H, W = a->W;
  if (a->stride == 2) { H = (H - 1) / 2 + 1; W = (W - 1) / 2 + 1; }
  const TilePlan t = plan_tiles(a, H, W);
  return (a->upsample ? 4 : 1) * t.tiles_x * t.tiles_y * 4;
}

extern "C" size_t femasr_tc_weight_bytes(int Cout, int Cin, int kh, int kw) {
  return (size_t)2 * Cout * Cin * kh * kw * sizeof(__half) + 256;   // hi plane, lo plane, then {absmax, inv_scale}
}

// Layout of the packed tensor-core weight blob: [hi plane][lo plane | F8: interleaved e4m3 plane][uint absmax][float inv_scale].
static int tc_pack_weight_impl(const float* w_oihw, void* blob, int Cout, int Cin, int kh, int kw, bool f8, void* stream) {
  FEMASR_CHECK_ARG(w_oihw && blob && Cout > 0 && Cin > 0 && kh > 0 && kw > 0, "tc_pack_weight: bad argument");
  FEMASR_CHECK_ARG(!f8 || Cin % 64 == 0, "tc_pack_weight_f8: Cin must be a multiple of 64");
  const long n = (long)Cout * Cin * kh * kw;
  __half* hi = reinterpret_cast<__half*>(blob);
  __half* lo = hi + n;
  unsigned int* amax = reinterpret_cast<unsigned int*>(lo + n);
  float* inv = reinterpret_cast<float*>(amax + 1);
  cudaStream_t st = as_stream(stream);
  FEMASR_CUDA(cudaMemsetAsync(amax, 0, 8, st));
  absmax_kernel<<<(unsigned)std::min<long>(cdiv(n, 256), 1024), 256, 0, st>>>(w_oihw, amax, n);
  int s = launch_status("absmax_kernel");
  if (s) return s;
  if (f8) {
    tc_pack_weight_f8_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(w_oihw, hi, reinterpret_cast<uint8_t*>(lo), amax, inv, Cout, Cin, kh, kw);
    return launch_status("tc_pack_weight_f8_kernel");
  }
  tc_pack_weight_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(w_oihw, hi, lo, amax, inv, Cout, Cin, kh, kw);
  return launch_status("tc_pack_weight_kernel");
}
extern "C" int femasr_tc_pack_weight(const float* w_oihw, void* blob, int Cout, int Cin, int kh, int kw, void* stream) {
  return tc_pack_weight_impl(w_oihw, blob, Cout, Cin, kh, kw, false, stream);
}
extern "C" int femasr_tc_pack_weight_f8(const float* w_oihw, void* blob, int Cout, int Cin, int kh, int kw, void* stream) {
  return tc_pack_weight_impl(w_oihw, blob, Cout, Cin, kh, kw, true, stream);
}

// Packed phase filters for the fused upsample+conv: a blob like femasr_tc_pack_weight's for the stacked
// [4*Cout][Cin][2][2] filter bank (femasr_tc_weight_bytes(4*Cout, Cin, 2, 2) bytes).
static int tc_pack_weight_up2_impl(const float* w_oihw, void* blob, int Cout, int Cin, bool f8, void* stream) {
  FEMASR_CHECK_ARG(w_oihw && blob && Cout > 0 && Cin > 0, "tc_pack_weight_up2: bad argument");
  cudaStream_t st = as_stream(stream);
  float* tmp = nullptr;
  const long n = (long)16 * Cout * Cin;
  FEMASR_CUDA(cudaMallocAsync(&tmp, n * sizeof(float), st));
  subpixel_weights_kernel<<<(unsigned)cdiv(n, 256), 256, 0, st>>>(w_oihw, tmp, Cout, Cin);
  int s = launch_status("subpixel_weights_kernel");
  if (!s) s = tc_pack_weight_impl(tmp, blob, 4 * Cout, Cin, 2, 2, f8, stream);
  cudaFreeAsync(tmp, st);
  return s;
}
extern "C" int femasr_tc_pack_weight_up2(const float* w_oihw, void* blob, int Cout, int Cin, void* stream) {
  return tc_pack_weight_up2_impl(w_oihw, blob, Cout, Cin, false, stream);
}
extern "C" int femasr_tc_pack_weight_up2_f8(const float* w_oihw, void* blob, int Cout, int Cin, void* stream) {
  return tc_pack_weight_up2_impl(w_oihw, blob, Cout, Cin, true, stream);
}

// F8 operand staging (see tc_prepare_flat_f8_kernel): modes NONE / GN_SILU / GN_SILU_FAST, no replication
extern "C" int femasr_tc_prepare_f8(const float* x, void* a_hi, void* a_x8, int mode, const float* pro_a, const float* pro_b,
                                    int B, int H, int W, int C, void* stream) {
  FEMASR_CHECK_ARG(x && a_hi && a_x8 && B > 0 && H > 0 && W > 0, "tc_prepare_f8: bad argument");
  FEMASR_CHECK_ARG(C % 64 == 0, "tc_prepare_f8: C must be a multiple of 64");
  FEMASR_CHECK_ARG((long)H * W * (C / 4) < (1l << 30) && B <= 65535, "tc_prepare_f8: tensor too large for the flat kernel");
  cudaStream_t st = as_stream(stream);
  const int per8 = H * W * (C / 8);
  const dim3 grid((unsigned)cdiv(per8, 256 * 2), (unsigned)B);
  const float4* x4 = reinterpret_cast<const float4*>(x);
  uint4* hi = reinterpret_cast<uint4*>(a_hi);
  uint2* x8 = reinterpret_cast<uint2*>(a_x8);
  if (mode == FEMASR_PRO_GN_SILU || mode == FEMASR_PRO_GN_SILU_FAST) {
    FEMASR_CHECK_ARG(pro_a && pro_b, "tc_prepare_f8: GN mode needs the scale/shift tables");
    if (mode == FEMASR_PRO_GN_SILU) tc_prepare_flat_f8_kernel<FEMASR_PRO_GN_SILU><<<grid, 256, 0, st>>>(x4, hi, x8, pro_a, pro_b, C, per8);
    else tc_prepare_flat_f8_kernel<FEMASR_PRO_GN_SILU_FAST><<<grid, 256, 0, st>>>(x4, hi, x8, pro_a, pro_b, C, per8);
  } else if (mode == FEMASR_PRO_NONE) {
    tc_prepare_flat_f8_kernel<FEMASR_PRO_NONE><<<grid, 256, 0, st>>>(x4, hi, x8, nullptr, nullptr, C, per8);
  } else {
    return fail(FEMASR_ERR_ARG, "tc_prepare_f8: bad mode");
  }
  return launch_status("tc_prepare_flat_f8_kernel");
}

extern "C" int femasr_tc_prepare(const float* x, void* a_hi, void* a_lo, int mode, const float* pro_a, const float* pro_b,
                                 const float* gamma, const float* beta, int B, int H, int W, int C, int upsample,
                                 float eps, void* stream) {
  FEMASR_CHECK_ARG(x && a_hi && a_lo && B > 0 && H > 0 && W > 0, "tc_prepare: bad argument");
  FEMASR_CHECK_ARG(C % 8 == 0, "tc_prepare: C must be a multiple of 8");
  cudaStream_t st = as_stream(stream);
  __half* hi = reinterpret_cast<__half*>(a_hi);
  __half* lo = reinterpret_cast<__half*>(a_lo);
  if (mode == FEMASR_PRO_LN) {
    FEMASR_CHECK_ARG(C == 256 && gamma && beta && !upsample, "tc_prepare: LN mode needs C=256, gamma/beta, no upsample");
    const long M = (long)B * H * W;
    tc_prepare_ln_kernel<<<(unsigned)cdiv(M, 16), 256, 0, st>>>(x, hi, lo, gamma, beta, M, eps);
    return launch_status("tc_prepare_ln_kernel");
  }
  if (!upsample && (long)H * W * (C / 4) < (1l << 30) && B <= 65535 &&
      (mode == FEMASR_PRO_GN_SILU || mode == FEMASR_PRO_GN_SILU_FAST || mode == FEMASR_PRO_NONE)) {
    const int per4 = H * W * (C / 4);
    const dim3 grid((unsigned)cdiv(per4, 256 * PREP_U), (unsigned)B);
    const float4* x4 = reinterpret_cast<const float4*>(x);
    uint2* hi2 = reinterpret_cast<uint2*>(hi);
    uint2* lo2 = reinterpret_cast<uint2*>(lo);
    if (mode == FEMASR_PRO_GN_SILU) {
      FEMASR_CHECK_ARG(pro_a && pro_b, "tc_prepare: GN mode needs the scale/shift tables");
      tc_prepare_flat_kernel<FEMASR_PRO_GN_SILU><<<grid, 256, 0, st>>>(x4, hi2, lo2, pro_a, pro_b, C, per4);
    } else if (mode == FEMASR_PRO_GN_SILU_FAST) {
      FEMASR_CHECK_ARG(pro_a && pro_b, "tc_prepare: GN mode needs the scale/shift tables");
      tc_prepare_flat_kernel<FEMASR_PRO_GN_SILU_FAST><<<grid, 256, 0, st>>>(x4, hi2, lo2, pro_a, pro_b, C, per4);
    } else {
      tc_prepare_flat_kernel<FEMASR_PRO_NONE><<<grid, 256, 0, st>>>(x4, hi2, lo2, nullptr, nullptr, C, per4);
    }
    return launch_status("tc_prepare_flat_kernel");
  }
  const long total8 = (long)B * H * W * (C / 8);
  const unsigned grid = (unsigned)cdiv(total8, 256);
  if (mode == FEMASR_PRO_GN_SILU_FAST) mode = FEMASR_PRO_GN_SILU;     // replicating variant: exact SiLU only
  if (mode == FEMASR_PRO_GN_SILU) {
    FEMASR_CHECK_ARG(pro_a && pro_b, "tc_prepare: GN mode needs the scale/shift tables");
    tc_prepare_kernel<FEMASR_PRO_GN_SILU><<<grid, 256, 0, st>>>(x, hi, lo, pro_a, pro_b, H, W, C, upsample, total8);
  } else if (mode == FEMASR_PRO_NONE) {
    tc_prepare_kernel<FEMASR_PRO_NONE><<<grid, 256, 0, st>>>(x, hi, lo, nullptr, nullptr, H, W, C, upsample, total8);
  } else {
    return fail(FEMASR_ERR_ARG, "tc_prepare: bad mode");
  }
  return launch_status("tc_prepare_kernel");
}

// VectorQuantizer distance stage on the tensor cores (femasr_arch.py:35-38, 63-66): for every feature row the four
// smallest d_j = fl(fl(A + B_j) - 2 z.e_j) with their codes, ascending in (d, j); the [N, n_e] product never leaves the SM.
extern "C" int femasr_vq_match_tc(const void* z_hi, const void* z_lo, const void* cb_blob, const float* a, const float* esq,
                                  void* cand, int N, int n_e, int e_dim, void* stream) {
  FEMASR_CHECK_ARG(z_hi && z_lo && cb_blob && a && esq && cand, "vq_match_tc: null pointer");
  FEMASR_CHECK_ARG(N > 0 && n_e > 0 && e_dim > 0 && n_e % 64 == 0 && e_dim % 64 == 0, "vq_match_tc: n_e and e_dim must be positive multiples of 64");
  const long nw = (long)n_e * e_dim;
  const __half* w_hi = reinterpret_cast<const __half*>(cb_blob);
  const __half* w_lo = w_hi + nw;
  TcP p;
  memset(&p, 0, sizeof(p));
  p.inv_scale = reinterpret_cast<const float*>(reinterpret_cast<const unsigned int*>(w_lo + nw) + 1);
  p.vq_a = a; p.vq_esq = esq; p.vq_cand = reinterpret_cast<uint2*>(cand);
  p.B = 1; p.H = 1; p.W = N; p.Cin = e_dim; p.Cout = n_e; p.taps = 1; p.stride = 1;
  p.Wt = 128; p.Ht = 1; p.wt_shift = 7; p.tiles_x = (int)cdiv(N, 128); p.tiles_y = 1;
  const int BN = n_e % 256 == 0 ? 256 : (n_e % 128 == 0 ? 128 : 64);
  p.n_tiles = n_e / BN;
  p.num_tiles = p.tiles_x * p.n_tiles; p.cchunks = e_dim / 64;
  p.kb_begin = 0; p.kb_end = p.cchunks; p.cpg = 1;
  CUtensorMap mah, mal, mbh, mbl;
  {
    const cuuint64_t dims[4] = {(cuuint64_t)e_dim, (cuuint64_t)N, 1, 1};
    const cuuint64_t str[3] = {(cuuint64_t)e_dim * 2, (cuuint64_t)N * e_dim * 2, (cuuint64_t)N * e_dim * 2};
    const cuuint32_t box[4] = {64, 128, 1, 1};
    int s = make_map(&mah, z_hi, 4, dims, str, box);
    if (s) return s;
    s = make_map(&mal, z_lo, 4, dims, str, box);
    if (s) return s;
  }
  {
    const cuuint64_t dims[2] = {(cuuint64_t)e_dim, (cuuint64_t)n_e};
    const cuuint64_t str[1] = {(cuuint64_t)e_dim * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)BN};
    int s = make_map(&mbh, w_hi, 2, dims, str, box);
    if (s) return s;
    s = make_map(&mbl, w_lo, 2, dims, str, box);
    if (s) return s;
  }
  cudaStream_t st = as_stream(stream);
  if (BN == 256) return launch_vq<256>(mah, mal, mbh, mbl, p, st);
  if (BN == 128) return launch_vq<128>(mah, mal, mbh, mbl, p, st);
  return launch_vq<64>(mah, mal, mbh, mbl, p, st);
}

// y = act(conv(a) + bias) + res1 + res2 with a given as fp16 hi/lo planes at the conv-input resolution.
extern "C" int femasr_tc_igemm(const femasr_tc_args* a, void* stream) {
  FEMASR_CHECK_ARG(a && a->a_hi && a->a_lo && a->w_blob, "tc_igemm: null pointer");
  FEMASR_CHECK_ARG(a->y || (a->out_hi && a->out_lo), "tc_igemm: need y or the out_hi/out_lo planes");
  FEMASR_CHECK_ARG(!a->out_hi == !a->out_lo, "tc_igemm: out_hi and out_lo go together");
  FEMASR_CHECK_ARG(a->B > 0 && a->H > 0 && a->W > 0, "tc_igemm: empty input");
  FEMASR_CHECK_ARG(a->ksize == 1 || a->ksize == 3, "tc_igemm: ksize must be 1 or 3");
  FEMASR_CHECK_ARG(!a->upsample || a->ksize == 3, "tc_igemm: upsample fusion needs ksize 3 (and an up2 weight blob)");
  FEMASR_CHECK_ARG(a->Cin % 64 == 0 && a->Cout % 64 == 0, "tc_igemm: Cin and Cout must be multiples of 64");
  int B = a->B, H = a->H, W = a->W;
  const int stride = a->stride == 2 ? 2 : 1;
  FEMASR_CHECK_ARG(a->stride >= 0 && a->stride <= 2, "tc_igemm: stride must be 1 or 2");
  FEMASR_CHECK_ARG(stride == 1 || (a->ksize == 3 && !a->upsample), "tc_igemm: stride 2 needs a plain 3x3 conv");
  if (a->ksize == 1) { W = B * H * W; H = 1; B = 1; }     // pointwise: one long row of tokens
  const int Hin = H, Win = W;                             // activation-plane dims
  if (stride == 2) { H = (H - 1) / 2 + 1; W = (W - 1) / 2 + 1; }   // tiles run over the output grid
  FEMASR_CHECK_ARG((long)W < (1l << 31), "tc_igemm: too many rows");
  const int taps = a->upsample ? 4 : a->ksize * a->ksize;
  const int phases = a->upsample ? 4 : 1;
  const long Ktot = (long)taps * a->Cin;
  const long nw = (long)phases * a->Cout * Ktot;
  const __half* w_hi = reinterpret_cast<const __half*>(a->w_blob);
  const __half* w_lo = w_hi + nw;
  const float* inv_scale = reinterpret_cast<const float*>(reinterpret_cast<const unsigned int*>(w_lo + nw) + 1);

  TcP p;
  memset(&p, 0, sizeof(p));
  p.bias = a->bias; p.res1 = a->res1; p.res2 = a->res2; p.y = a->y; p.inv_scale = inv_scale;
  p.out_hi = reinterpret_cast<__half*>(a->out_hi); p.out_lo = reinterpret_cast<__half*>(a->out_lo);
  p.gn_partial = a->gn_partial; p.cpg = a->Cout / 32; p.gn_rows = 0;
  FEMASR_CHECK_ARG(!a->gn_partial || (a->ksize == 3 && (a->Cout == 64 || a->Cout == 128 || a->Cout == 256)),
                   "tc_igemm: gn_partial needs a 3x3 conv with Cout in {64,128,256}");
  p.B = B; p.H = H; p.W = W; p.Cin = a->Cin; p.Cout = a->Cout; p.taps = taps; p.act = a->act;
  p.up = a->upsample ? 1 : 0; p.stride = stride;
  p.f8 = a->f8 ? 1 : 0;
  FEMASR_CHECK_ARG(!a->f8 || a->slice_kb == 0, "tc_igemm: the F8 cross-term mode is for the layers behind the VQ (no K slicing)");
  const TilePlan plan = plan_tiles(a, H, W);
  p.Wt = plan.Wt; p.Ht = plan.Ht; p.wt_shift = plan.wt_shift; p.tiles_x = plan.tiles_x; p.tiles_y = plan.tiles_y;
  const int BN = plan.BN;
  p.n_tiles = a->Cout / BN;
  const bool pair = plan.pair, strip = plan.strip;
  FEMASR_CHECK_ARG(!(a->strip == 1 && !strip), "tc_igemm: strip mode needs a plain 3x3 stride-1 conv, Cout tile <= 128, W >= 128, no K slicing");
  p.gn_rows = phases * p.tiles_x * p.tiles_y * 4;           // one partial row per (128-pixel tile, lane quarter)
  // 64 -> 64 channels: weights resident in shared memory, work items of 4 image rows
  const bool bres = strip && a->Cin == 64 && a->Cout == 64;
  if (bres) p.tiles_y = (int)cdiv(H, TcCfg<64, false, true, true>::MR);
  const long ntile = (long)phases * B * p.tiles_x * p.tiles_y * p.n_tiles;
  FEMASR_CHECK_ARG(ntile < (1l << 31), "tc_igemm: too many tiles");
  p.num_tiles = (int)ntile; p.cchunks = a->Cin / 64;
  const int nkb_total = taps * p.cchunks;
  p.kb_begin = a->kb_begin; p.kb_end = a->kb_count > 0 ? a->kb_begin + a->kb_count : nkb_total;
  FEMASR_CHECK_ARG(p.kb_begin >= 0 && p.kb_begin < p.kb_end && p.kb_end <= nkb_total, "tc_igemm: bad k-block slice");
  FEMASR_CHECK_ARG(a->slice_kb >= 0, "tc_igemm: slice_kb must be >= 0");
  p.slice_kb = (a->slice_kb > 0 && a->slice_kb < p.kb_end - p.kb_begin) ? a->slice_kb : 0;

  CUtensorMap mah, mal, mbh, mbl;
  {
    const cuuint64_t dims[4] = {(cuuint64_t)a->Cin, (cuuint64_t)Win, (cuuint64_t)Hin, (cuuint64_t)B};
    const cuuint64_t str[3] = {(cuuint64_t)a->Cin * 2, (cuuint64_t)Win * a->Cin * 2, (cuuint64_t)Hin * Win * a->Cin * 2};
    // with a traversal stride s the box spans s*Wt x s*Ht source pixels and lands Wt x Ht of them in smem
    const cuuint32_t box[4] = {64, (cuuint32_t)(strip ? STRIP_PX : p.Wt * stride), (cuuint32_t)(p.Ht * stride), 1};
    int s = make_map(&mah, a->a_hi, 4, dims, str, box, stride);
    if (s) return s;
    s = make_map(&mal, a->a_lo, 4, dims, str, box, stride);
    if (s) return s;
  }
  {
    const cuuint64_t dims[2] = {(cuuint64_t)Ktot, (cuuint64_t)phases * a->Cout};
    const cuuint64_t str[1] = {(cuuint64_t)Ktot * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)(pair ? BN / 2 : BN)};
    int s = make_map(&mbh, w_hi, 2, dims, str, box);
    if (s) return s;
    s = make_map(&mbl, w_lo, 2, dims, str, box);
    if (s) return s;
  }
  // TMA-store epilogue: the output is a plain [B, H, W, Cout] tensor (no sub-pixel phases) -> the staging tile of each
  // epilogue warp (32 accumulator rows x 16 columns) leaves as one bulk tensor store; edge tiles are clipped by the TMA
  OutMaps om;
  om.y = mah; om.oh = mah; om.ol = mah;
  p.tma_out = 0;
  p.box_w = p.Wt < 32 ? p.Wt : 32;
  p.box_w_shift = 0; while ((1 << p.box_w_shift) < p.box_w) ++p.box_w_shift;
  // Measured same-box A/B (profiles/microbench_r2_tma_store_ab.txt): linears +3..6 %, 64-wide strip convs -5..9 % (8
  // epilogue warps: the extra staging write and the read-wait of the bulk store cost more than the stores they replace),
  // other convs neutral -> enabled for ksize 1 only.
  if (a->ksize == 1 && !a->upsample) {
    const cuuint64_t dims[4] = {(cuuint64_t)a->Cout, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    const cuuint32_t box[4] = {16, (cuuint32_t)p.box_w, (cuuint32_t)(32 / p.box_w), 1};
    if (a->y) {
      const cuuint64_t str[3] = {(cuuint64_t)a->Cout * 4, (cuuint64_t)W * a->Cout * 4, (cuuint64_t)H * W * a->Cout * 4};
      int s = make_map(&om.y, a->y, 4, dims, str, box, 1, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, CU_TENSOR_MAP_SWIZZLE_64B);
      if (s) return s;
      p.tma_out = 1;
    } else {
      const cuuint64_t str[3] = {(cuuint64_t)a->Cout * 2, (cuuint64_t)W * a->Cout * 2, (cuuint64_t)H * W * a->Cout * 2};
      int s = make_map(&om.oh, a->out_hi, 4, dims, str, box, 1, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, CU_TENSOR_MAP_SWIZZLE_NONE);
      if (s) return s;
      s = make_map(&om.ol, a->out_lo, 4, dims, str, box, 1, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, CU_TENSOR_MAP_SWIZZLE_NONE);
      if (s) return s;
      p.tma_out = 2;
    }
  }
  cudaStream_t st = as_stream(stream);
  if (strip) {
    if (BN == 128 && pair) return launch_tc<128, true, true>(mah, mal, mbh, mbl, om, p, st);
    if (BN == 128) return launch_tc<128, false, true>(mah, mal, mbh, mbl, om, p, st);
    if (bres) return launch_tc<64, false, true, true>(mah, mal, mbh, mbl, om, p, st);
    return launch_tc<64, false, true>(mah, mal, mbh, mbl, om, p, st);
  }
  if (pair) {
    if (BN == 256) return launch_tc<256, true, false>(mah, mal, mbh, mbl, om, p, st);
    if (BN == 128) return launch_tc<128, true, false>(mah, mal, mbh, mbl, om, p, st);
    return launch_tc<64, true, false>(mah, mal, mbh, mbl, om, p, st);
  }
  if (BN == 256) return launch_tc<256, false, false>(mah, mal, mbh, mbl, om, p, st);
  if (BN == 128) return launch_tc<128, false, false>(mah, mal, mbh, mbl, om, p, st);
  return launch_tc<64, false, false>(mah, mal, mbh, mbl, om, p, st);
}
