/* femasr_b200.h - C ABI of the B200-native FeMaSR inference hot path.
 *
 * This shared library (libfemasr_b200.so, sm_100a only) is the drop-in boundary underneath the
 * reference's Python operator surface `basicsr.archs.femasr_arch.FeMaSRNet`
 * (/root/reference/basicsr/archs/femasr_arch.py:214-479).  Signatures use plain pointers and
 * sizes only: device pointers are raw CUDA addresses, `stream` is a cudaStream_t passed as void*.
 * Every entry point returns 0 on success or a negative femasr_status; femasr_last_error() gives
 * the message (thread-local).  Nothing here owns caller memory; nothing falls back to the CPU.
 *
 * Data layout: activations between kernels are NHWC fp32 ([B,H,W,C]; Swin tokens [B,HW,C] are the
 * same bytes).  Images at the public boundary are NCHW fp32 like the reference's tensors.
 */
#ifndef FEMASR_B200_H
#define FEMASR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  FEMASR_OK = 0,
  FEMASR_ERR_ARG = -1,       /* bad shape / null pointer / unsupported configuration */
  FEMASR_ERR_CUDA = -2,      /* a CUDA runtime/driver call failed */
  FEMASR_ERR_STATE = -3,     /* missing parameter, workspace too small, ... */
  FEMASR_ERR_NO_DEVICE = -4  /* no sm_100 device: there is no CPU fallback */
} femasr_status;

const char* femasr_last_error(void);
int femasr_abi_version(void);
/* compute capability major*10+minor of the current device, or negative status */
int femasr_device_cc(void);

/* ------------------------------------------------------------------------------------------------
 * Network-level API: replaces FeMaSRNet.encode_and_decode / test / decode_indices
 * (femasr_arch.py:311-374, 449-468, 376-385) for norm 'gn', act 'silu'; LQ_stage=True with scale_factor 2 or 4,
 * or the HQ autoencoder (LQ_stage=False) as scale_factor 1; one codebook at scale 32, or the multi-scale
 * variant (femasr_arch.py:280-299) with further codebooks at 64 / 128.
 * ---------------------------------------------------------------------------------------------- */
typedef struct femasr_net femasr_net;
#define FEMASR_MAX_CODEBOOKS 3

typedef struct {
  int scale_factor;   /* 2 or 4            (femasr_arch.py:225) */
  int n_e;            /* codebook entries  (codebook_params[0][1]) */
  int e_dim;          /* codebook dim      (codebook_params[0][2]), multiple of 64 */
  int in_channel;     /* 3 */
  int use_quantize;   /* femasr_arch.py:224,349-350: 0 => z_quant = feat_to_quant (VQ still runs) */
  int use_residual;   /* femasr_arch.py:226,361-362 */
  int gemm_path;      /* 0 = fp32 SIMT implicit GEMM, 1 = tcgen05 split-fp16 tensor-core GEMM */
  /* multi-scale codebooks (femasr_arch.py:231-235, 280-299): rows of codebook_params.  n_codebooks 0 or 1 = the single
   * codebook (32, n_e, e_dim) above; else cb_scale[0] must be 32 (it fixes the depth, :255-256), the others an
   * increasing subset of {64, 128}; n_e / e_dim above are ignored. */
  int n_codebooks;
  int cb_scale[FEMASR_MAX_CODEBOOKS];
  int cb_n_e[FEMASR_MAX_CODEBOOKS];     /* multiples of 64 */
  int cb_e_dim[FEMASR_MAX_CODEBOOKS];   /* multiples of 64 */
} femasr_net_config;

int femasr_net_create(const femasr_net_config* cfg, femasr_net** out);
void femasr_net_destroy(femasr_net* net);

/* Upload one state_dict tensor by its reference name (SURVEY.md 8b), fp32, contiguous, from HOST
 * or DEVICE memory (`on_device` says which).  The engine keeps its own repacked device copy.
 * int64 buffers (relative_position_index, attn_mask) are derived, not uploaded. */
int femasr_net_set_param(femasr_net* net, const char* name, const float* data, size_t numel,
                         int on_device, void* stream);
/* 0 if every parameter has been set, else FEMASR_ERR_STATE (message names the first missing). */
int femasr_net_params_complete(femasr_net* net);

/* Bytes of device workspace femasr_net_forward needs for a [B,3,H,W] input. */
int femasr_net_workspace_bytes(femasr_net* net, int B, int H, int W, size_t* bytes);

/* encode_and_decode (femasr_arch.py:311-374).
 *   x_nchw    [B,3,H,W] fp32 device.  H,W such that the Swin stage (H/2 for x4, H/4 for x2) is a
 *             multiple of 8, else FEMASR_ERR_ARG (the reference raises from window_partition).
 *   y_nchw    [B,3,s*H,s*W] fp32 device, unclamped.
 *   indices   [B,1,h,w] int64 device (may be NULL).  Multi-scale nets: the maps of all codebooks back to back in
 *             codebook order ([B,1,h,w], then [B,1,2h,2w] for a codebook at 64, [B,1,4h,4w] at 128).
 *   cb_loss   1 float device: codebook_loss = sum over codebooks of 1.25*mean((z_q-z)^2)
 *             (femasr_arch.py:84-92, 371); may be NULL.
 */
int femasr_net_forward(femasr_net* net, const float* x_nchw, float* y_nchw, int64_t* indices,
                       float* cb_loss, int B, int H, int W, void* workspace, size_t workspace_bytes,
                       void* stream);
/* forward(input, gt_indices) (femasr_arch.py:470-474): gt_indices = the HQ stage's codes laid out like `indices`
 * (all codebooks back to back).  They change only cb_loss, and only in the LQ stage (scale_factor 2 | 4):
 * per codebook 0.25*mean((E[gt]-z)^2) + mean((G(z)-G(E[gt]))^2), G = per-image Gram matrix z^T z / hw
 * (femasr_arch.py:40-48, 70-78, 87-90).  gt_indices == NULL is femasr_net_forward. */
int femasr_net_forward_gt(femasr_net* net, const float* x_nchw, float* y_nchw, int64_t* indices,
                          float* cb_loss, const int64_t* gt_indices, int B, int H, int W, void* workspace,
                          size_t workspace_bytes, void* stream);

/* decode_indices (femasr_arch.py:376-385): indices [B,1,h,w] int64 -> y [B,3,8h,8w]. */
int femasr_net_decode_indices(femasr_net* net, const int64_t* indices, float* y_nchw, int B, int h,
                              int w, void* workspace, size_t workspace_bytes, void* stream);
int femasr_net_decode_workspace_bytes(femasr_net* net, int B, int h, int w, size_t* bytes);

/* Stage taps for parity tests: when `dst` is set for a stage name, the next forward copies that
 * stage's NHWC fp32 tensor there (device, `capacity` floats).  Names: in_conv, down, swin, up1, up2,
 * z, zq, after_quant, dec0, dec1, dec2 (z / zq / after_quant: first codebook), z1, z2 (features in front of the
 * second / third codebook).  dst == NULL removes the tap. */
int femasr_net_set_tap(femasr_net* net, const char* stage, float* dst, size_t capacity);
/* Number of kernels the last femasr_net_forward launched (bench.py's gpu_launches). */
int femasr_net_last_launch_count(femasr_net* net);
/* Per-kernel timing for bench.py's roofline: while enabled, every launch of femasr_net_forward is
 * bracketed by CUDA events on the launching stream; femasr_net_profile_json returns
 * {"kernel": {"launches": n, "ms": total, "flops": algorithmic total}, ...} (valid until the next call). */
int femasr_net_set_profile(femasr_net* net, int enable);
const char* femasr_net_profile_json(femasr_net* net);
/* Algorithmic FLOPs (2*MAC, conv+linear+QK/PV+VQ distance) of one forward on [B,3,H,W]. */
double femasr_net_flops(femasr_net* net, int B, int H, int W);

/* test() padding (femasr_arch.py:455-460): flip-pad [B,3,h,w] -> [B,3,hp,wp]. */
int femasr_flip_pad(const float* x, float* y, int B, int C, int h, int w, int hp, int wp, void* stream);
/* crop / paste used by test() (:465) and test_tile() (:444-446): copies the window
 * src[:, :, sy:sy+ch, sx:sx+cw] to dst[:, :, dy:dy+ch, dx:dx+cw]. */
int femasr_copy_window(const float* src, float* dst, int B, int C, int sh, int sw, int dh, int dw,
                       int sy, int sx, int dy, int dx, int ch, int cw, void* stream);

/* uint8 image boundary fused on the device (inference_femasr.py:54-56,64; utils/img_util.py:9-35,38-94):
 *   femasr_u8_to_input:  uint8 HWC BGR [B,h,w,3] -> fp32 NCHW RGB in [0,1], flip-padded to [B,3,hp,wp]
 *                        (= img2tensor, /255., and test()'s padding in one pass)
 *   femasr_output_to_u8: fp32 NCHW RGB [B,3,SH,SW] -> uint8 HWC BGR [B,ch,cw,3] of the top-left ch x cw crop
 *                        (= test()'s crop and tensor2img: clamp to [0,1], *255, round half to even) */
int femasr_u8_to_input(const uint8_t* bgr_hwc, float* x_nchw, int B, int h, int w, int hp, int wp, void* stream);
int femasr_output_to_u8(const float* y_nchw, uint8_t* bgr_hwc, int B, int SH, int SW, int ch, int cw, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Operator-level API (what the network is built from; exported so each kernel has its own parity
 * test).  All tensors device fp32 unless stated.
 * ---------------------------------------------------------------------------------------------- */

/* Repack a conv weight OIHW [Cout,Cin,kh,kw] -> K-major GEMM operand [kh*kw*Cin][Cout]
 * (linear weights [N,K] are the kh=kw=1 case). */
int femasr_pack_weight(const float* w_oihw, float* w_packed, int Cout, int Cin, int kh, int kw, void* stream);

enum { FEMASR_PRO_NONE = 0, FEMASR_PRO_GN_SILU = 1, FEMASR_PRO_LN = 2,
       /* femasr_tc_prepare only: GN + SiLU with ex2.approx / rcp.approx (relative error <= 4e-7 instead of 1.2e-7);
          the engine uses it behind the VQ, where the bar is 1e-3 on the output, never in front of the index decision */
       FEMASR_PRO_GN_SILU_FAST = 3 };
enum { FEMASR_ACT_NONE = 0, FEMASR_ACT_GELU = 1 };

/* Implicit-GEMM convolution / linear:  y = act(conv(pro(x)) + bias) + res1 + res2.
 *   ksize 3 (pad 1) or 1 (pad 0); stride 1|2; upsample=1 applies nearest x2 to pro(x) first
 *   (nn.Upsample, femasr_arch.py:172,202).  Linear layers are ksize=1 with Hin*Win = tokens.
 *   prologue GN_SILU: x' = silu(x*pro_scale[b,c] + pro_shift[b,c])   (tables from femasr_gn_stats)
 *   prologue LN:      x' = (x - row_mean[m])*row_rstd[m]*gamma[c] + beta[c]
 * Replaces nn.Conv2d / nn.Linear call sites femasr_arch.py:150-203,273,298; fema_utils.py:75-90;
 * network_swinir.py:19-21,105-107,465. */
typedef struct {
  const float* x;          /* NHWC [B,Hin,Win,Cin] */
  const float* w;          /* packed [ksize*ksize*Cin][Cout] */
  const float* bias;       /* [Cout] or NULL */
  const float* res1;       /* NHWC like y, or NULL; may alias y */
  const float* res2;       /* NHWC like y, or NULL */
  float* y;                /* NHWC [B,Ho,Wo,Cout] */
  const float* pro_a;      /* GN: scale [B,Cin];  LN: row_mean [M] */
  const float* pro_b;      /* GN: shift [B,Cin];  LN: row_rstd [M] */
  const float* gamma;      /* LN only: [Cin] */
  const float* beta;       /* LN only: [Cin] */
  int B, Hin, Win, Cin, Cout;
  int ksize, stride, upsample;
  int prologue;            /* FEMASR_PRO_* */
  int act;                 /* FEMASR_ACT_* */
} femasr_igemm_args;
int femasr_igemm_simt(const femasr_igemm_args* a, void* stream);

/* ---- tcgen05 tensor-core implicit GEMM (gemm_path 1): same contract as femasr_igemm_simt for ksize 1|3,
 * stride 1, Cin%64==0, Cout%64==0, computed as a 3-product split-fp16 GEMM (a_hi*w_hi + a_hi*w_lo + a_lo*w_hi,
 * fp32 accumulate in TMEM).  The activation operand is staged once per layer as two fp16 NHWC planes by
 * femasr_tc_prepare (which also applies the GN+SiLU / LayerNorm prologue and the nearest x2 upsample);
 * weights are packed once by femasr_tc_pack_weight into a blob of femasr_tc_weight_bytes bytes. */
typedef struct {
  const void* a_hi;        /* fp16 NHWC [B,H,W,Cin] at the conv-input resolution (after any upsample) */
  const void* a_lo;
  const void* w_blob;      /* from femasr_tc_pack_weight */
  const float* bias;       /* [Cout] or NULL */
  const float* res1;       /* fp32 NHWC like y, or NULL; may alias y */
  const float* res2;
  float* y;                /* fp32 NHWC [B,H,W,Cout] */
  int B, H, W, Cin, Cout;
  int ksize;               /* 1 or 3 (pad 1) */
  int act;                 /* FEMASR_ACT_* */
  void* out_hi;            /* optional: write the result as split fp16 NHWC planes (the next GEMM's operand) */
  void* out_lo;            /*           instead of fp32 y (y may then be NULL) */
  int stride;              /* 0|1: stride 1.  2: 3x3 stride-2 conv (pad 1); H,W are the INPUT dims, y is
                              [B,(H-1)/2+1,(W-1)/2+1,Cout] (TMA traversal stride 2 on the activation planes) */
  int kb_begin, kb_count;  /* K-slice in 64-wide k-blocks (k = tap*Cin + c); kb_count 0 = everything.  Slices are summed
                              by the caller in fp32 (round-to-nearest) by chaining launches with res1 = y, which bounds
                              the tensor-core accumulator's truncation error to one slice */
  int slice_kb;            /* >0: the same slicing inside ONE launch - every slice_kb k-blocks the MMA accumulator is
                              drained into an fp32 running sum held in the second TMEM buffer (tcgen05.ld/st, RN adds) */
  int pair;                /* 1: CTA pairs (tcgen05 cta_group::2, 256-row tiles, each CTA stages half the weight tile);
                              0: single-CTA tiles; -1: library default */
  int strip;               /* 1: row-strip tiles (one image row of 128 pixels; the three horizontal taps share one
                              130-pixel activation strip in shared memory): plain 3x3 stride-1 convs, Cout tile <= 128,
                              W >= 128, no K slicing.  0: off; -1: automatic */
  float* gn_partial;       /* optional: GroupNorm(32) partial sums of the OUTPUT, [B][rows][32][2] fp32 with
                              rows = femasr_tc_gn_partial_rows(args); finished by femasr_gn_finalize_rows */
  int upsample;            /* 1: y [B,2H,2W,Cout] = conv3x3(nearest_x2(a)), evaluated as 4 sub-pixel 2x2 convs on the
                              low-res grid; a_* are at the LOW resolution and w_blob comes from femasr_tc_pack_weight_up2 */
  int f8;                  /* 1: F8 cross-term mode (layers behind the VQ, error budget 1e-3 on the output): a_lo and the
                              blob's second plane hold interleaved e4m3 bytes (femasr_tc_prepare_f8 /
                              femasr_tc_pack_weight_f8) and the two cross products a_lo*w_hi + a_hi*w_lo run as ONE
                              kind::f8f6f4 product at twice the fp16 rate: 2.0 instead of 3.0 MMA units per k-step */
} femasr_tc_args;
size_t femasr_tc_weight_bytes(int Cout, int Cin, int kh, int kw);
int femasr_tc_pack_weight(const float* w_oihw, void* blob, int Cout, int Cin, int kh, int kw, void* stream);
/* blob of femasr_tc_weight_bytes(4*Cout, Cin, 2, 2) bytes for the upsample-fused form (femasr_tc_args.upsample) */
int femasr_tc_pack_weight_up2(const float* w_oihw_3x3, void* blob, int Cout, int Cin, void* stream);
/* mode FEMASR_PRO_NONE | GN_SILU (pro_a/pro_b = scale/shift tables) | LN (gamma/beta, C=256, stats computed
 * in-kernel).  x fp32 NHWC [B,H,W,C] -> a_hi/a_lo fp16 NHWC [B,H*u,W*u,C], u = upsample ? 2 : 1. */
int femasr_tc_prepare(const float* x, void* a_hi, void* a_lo, int mode, const float* pro_a, const float* pro_b,
                      const float* gamma, const float* beta, int B, int H, int W, int C, int upsample,
                      float eps, void* stream);
/* F8 cross-term mode (femasr_tc_args.f8): per 64-channel chunk the second operand plane holds 128 bytes
 * [e4m3(lo * 2^10) x 64 | e4m3(value * 2^-2) x 64] (activations) resp. [e4m3(w_hi * 2^-10) x 64 | e4m3(w_lo * 2^2) x 64]
 * (weights); the scales cancel in the product and are an implementation detail of the prepare / pack pair. */
int femasr_tc_prepare_f8(const float* x, void* a_hi, void* a_x8, int mode, const float* pro_a, const float* pro_b,
                         int B, int H, int W, int C, void* stream);
int femasr_tc_pack_weight_f8(const float* w_oihw, void* blob, int Cout, int Cin, int kh, int kw, void* stream);
int femasr_tc_pack_weight_up2_f8(const float* w_oihw_3x3, void* blob, int Cout, int Cin, void* stream);
int femasr_tc_igemm(const femasr_tc_args* a, void* stream);
/* number of GroupNorm partial rows per image femasr_tc_igemm will write for these arguments (the tiling is
 * chosen from the shape / flags; pointers in `a` are not read) */
int femasr_tc_gn_partial_rows(const femasr_tc_args* a);
/* scale/shift tables (as femasr_gn_stats) from the partial rows a femasr_tc_igemm epilogue produced;
 * HW = pixels per image of the tensor the partials describe. */
int femasr_gn_finalize_rows(const float* partial, const float* gamma, const float* beta, float* scale, float* shift,
                            int B, int rows, int HW, int C, float eps, void* stream);

/* GroupNorm(32 groups, eps) statistics of NHWC x[B,HW,C] folded with the affine parameters into
 * per-(sample,channel) scale/shift: scale = rstd*gamma, shift = beta - mean*rstd*gamma
 * (nn.GroupNorm, fema_utils.py:21-22).  `scratch` >= femasr_gn_scratch_floats(B,HW,C) floats. */
size_t femasr_gn_scratch_floats(int B, int HW, int C);
int femasr_gn_stats(const float* x, const float* gamma, const float* beta, float* scale, float* shift,
                    float* scratch, int B, int HW, int C, float eps, void* stream);

/* LayerNorm statistics per token row of x[M,C] (C == 256): mean[M], rstd[M] (network_swinir.py:199,207). */
int femasr_ln_stats(const float* x, float* mean, float* rstd, int M, int C, float eps, void* stream);

/* Shifted-window multi-head attention (network_swinir.py:114-145, 239-279 minus the linears):
 * qkv [B*H*W, 3*C] in token order -> out [B*H*W, C] in token order; 8x8 windows, C = heads*32,
 * cyclic shift `shift` (0 or 4) and its 0/-100 mask are applied by index arithmetic.
 * bias_full [heads][64][64] = relative_position_bias_table[relative_position_index] (:127-129). */
int femasr_window_attention(const float* qkv, const float* bias_full, float* out, int B, int H, int W,
                            int C, int heads, int shift, void* stream);
/* Same contract on warp-level tensor cores (mma.sync m16n8k16, 3-term split-fp16, fp32 softmax); heads*32 == C.
 * bias_frag: the same [heads][64][64] bias values in the kernel's accumulator-fragment order, made by
 * femasr_expand_rel_bias_mma (one coalesced 16-byte load per lane and n-tile instead of 16 strided 8-byte ones).
 * out_hi/out_lo non-NULL: the result is written as split fp16 planes [B*H*W, C] instead of fp32 `out`. */
int femasr_window_attention_mma(const float* qkv, const float* bias_frag, float* out, void* out_hi, void* out_lo,
                                int B, int H, int W, int C, int heads, int shift, void* stream);
int femasr_expand_rel_bias(const float* table /*[225,heads]*/, float* bias_full, int heads, void* stream);
int femasr_expand_rel_bias_mma(const float* table /*[225,heads]*/, float* bias_frag /*heads*4096*/, int heads, void* stream);

/* VectorQuantizer.forward (femasr_arch.py:50-100) given zc = z @ codebook^T:
 *   d_j = fl(fl(sum z^2 + esq_j) - 2*zc_j), idx = argmin (lowest index on ties), zq = z + (e_idx - z),
 *   loss_rows[i] = sum_k (e_idx - z)^2.  esq from femasr_row_sumsq(codebook). */
int femasr_row_sumsq(const float* x, float* out, int rows, int cols, void* stream);
int femasr_vq_select(const float* z, const float* zc, const float* codebook, const float* esq,
                     int64_t* idx, float* zq, float* loss_rows, int N, int n_e, int e_dim,
                     int write_zq_passthrough, void* stream);
/* Fused VQ feature matching on the tensor cores (femasr_arch.py:35-38, 50-100) - the [N, n_e] distance matrix and the
 * one-hot of the reference never exist:
 *   femasr_vq_match_tc  z (split fp16 planes [N, e_dim]) x codebook (femasr_tc_pack_weight blob of the [n_e, e_dim]
 *                       embedding) on tcgen05; the epilogue evaluates d_j = fl(fl(A + B_j) - 2 C_j) and keeps per row the
 *                       four smallest (d, j) in cand[N][4] = {float bits, int32} pairs, ascending.  a = row_sumsq(z),
 *                       esq = row_sumsq(codebook).
 *   femasr_vq_finish    exact fp32 re-evaluation of the candidates that lie within rounding distance of the best
 *                       (whole-codebook rescan if all four do), lowest-index tie rule, then idx / zq = z + (e - z) /
 *                       loss_rows like femasr_vq_select.  stats (3 x uint32, may be NULL) counts refined rows, rescanned
 *                       rows and rows whose code changed.  Bit-identical indices to femasr_vq_select on exact z.E^T. */
int femasr_vq_match_tc(const void* z_hi, const void* z_lo, const void* cb_blob, const float* a, const float* esq,
                       void* cand, int N, int n_e, int e_dim, void* stream);
int femasr_vq_finish(const float* z, const float* a, const void* cand, const float* codebook, const float* esq,
                     int64_t* idx, float* zq, float* loss_rows, unsigned int* stats, int N, int n_e, int e_dim,
                     void* stream);
/* Compact wire format of codebook-index maps (extension; the reference moves int64 maps, femasr_arch.py:100,376-385):
 * ceil(log2 n_e) bits per code, little-endian bit stream.  femasr_packed_code_bytes gives the stream length;
 * *status (device int) becomes 1 if a code lies outside [0, n_e). */
size_t femasr_packed_code_bytes(size_t numel, int n_e);
int femasr_pack_codes(const int64_t* indices, void* packed, size_t numel, int n_e, int* status, void* stream);
int femasr_unpack_codes(const void* packed, int64_t* indices, size_t numel, int n_e, void* stream);
/* out[0] = scale * sum(x[0..n)) accumulated in double in a fixed order. */
int femasr_sum_scaled(const float* x, float* out, size_t n, double scale, void* stream);
/* out[0] += scale * sum(x[0..n)) (the running sum over codebooks, femasr_arch.py:371). */
int femasr_sum_scaled_add(const float* x, float* out, size_t n, double scale, void* stream);
/* torch.cat((a, nearest(b -> H x W)), dim=channels) on NHWC fp32: the before_quant input of the later codebooks
 * (femasr_arch.py:332-335, Hb=H, Wb=W) and CombineQuantBlock (fema_utils.py:92-99, F.interpolate default mode). */
int femasr_concat_channels(const float* a, int Ca, const float* b, int Hb, int Wb, int Cb, float* out, int B, int H,
                           int W, void* stream);
/* gt_indices loss branch (femasr_arch.py:70-78, 87-88): zq_gt[N,e] = codebook[gt], rows[i] = sum_k (zq_gt - z)^2. */
int femasr_vq_gt_rows(const float* z, const float* codebook, const int64_t* gt, float* zq_gt, float* rows, int N,
                      int n_e, int e_dim, void* stream);
/* gram_loss (femasr_arch.py:40-48) on x, y [B,HW,C] (C multiple of 32): partial[B * femasr_gram_diff_tiles(C)] holds
 * the per-tile sums of (x^T x / HW - y^T y / HW)^2; the loss is their sum / (B*C*C). */
int femasr_gram_diff_tiles(int C);
int femasr_gram_diff(const float* x, const float* y, float* partial, int B, int HW, int C, void* stream);
/* get_codebook_entry (femasr_arch.py:102-112): zq[N,e] = codebook[idx]. */
int femasr_codebook_gather(const int64_t* idx, const float* codebook, float* zq, int N, int n_e,
                           int e_dim, void* stream);

/* MultiScaleEncoder.in_conv (femasr_arch.py:150): 4x4, pad 1, NCHW [B,Cin,H,W] -> NHWC [B,H-1,W-1,Cout].
 * w packed [16*Cin][Cout]. */
int femasr_in_conv4x4(const float* x_nchw, const float* w, const float* bias, float* y_nhwc, int B,
                      int Cin, int H, int W, int Cout, void* stream);
/* in_conv on the tensor cores (femasr_arch.py:150): femasr_in_conv_im2col writes, per output pixel of the 4x4 p1 conv,
 * its 48 input values (k = (kh*4+kw)*3+ci, zero padded to 64) as split fp16 planes [B*(H-1)*(W-1)][64]; the conv is then
 * femasr_tc_igemm with ksize 1, Cin 64 on a weight blob packed from femasr_in_conv_pad_weight's [Cout][64] matrix. */
int femasr_in_conv_im2col(const float* x_nchw, void* a_hi, void* a_lo, int B, int Cin, int H, int W, void* stream);
int femasr_in_conv_pad_weight(const float* w_oihw, float* w_padded, int Cout, void* stream);
/* out_conv (femasr_arch.py:273): 3x3 pad 1, NHWC [B,H,W,Cin] -> NCHW [B,3,H,W].  w packed [9*Cin][3]. */
int femasr_out_conv3x3(const float* x_nhwc, const float* w, const float* bias, float* y_nchw, int B,
                       int H, int W, int Cin, void* stream);
/* Same contract on warp-level tensor cores (mma.sync, 3-term split fp16; the three horizontal taps folded into N):
 * fp32-grade accuracy (not ATen-identical rounding), used by gemm_path 1.
 * Both out_conv entry points stage the 1728 weights in library-global device memory (`__constant__` / fragment
 * buffer) that is refreshed by every call in stream order: calls issued on DIFFERENT streams must not overlap
 * (one engine handle = one host thread = one stream at a time, see the threading note in INTEGRATION.md). */
int femasr_out_conv3x3_mma(const float* x_nhwc, const float* w, const float* bias, float* y_nchw, int B,
                           int H, int W, int Cin, void* stream);

/* layout helpers for tests */
int femasr_nchw_to_nhwc(const float* x, float* y, int B, int C, int H, int W, void* stream);
int femasr_nhwc_to_nchw(const float* x, float* y, int B, int C, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FEMASR_B200_H */
