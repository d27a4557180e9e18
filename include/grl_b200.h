/* grl_b200.h -- C ABI of libgrl_b200.so: the B200 (sm_100a) implementation of GRL's forward hot path.
 *
 * The reference (ofsoundof/GRL-Image-Restoration) is pure Python/ATen: it has no FFI, plugin or
 * operator registry for this path.  Its boundary is the nn.Module contract (SURVEY.md section 8b);
 * every entry point below therefore cites the reference *Python interface* it replaces
 * (paths relative to the reference root) and INTEGRATION.md shows the ctypes binding a maintainer
 * adds.  Conventions for every function:
 *   - plain pointers + sizes only; all data pointers are DEVICE pointers unless the name ends in
 *     _host; `stream` is a cudaStream_t passed as void*;
 *   - no allocation, no synchronisation; re-entrant per stream.  Process-wide state is limited to: the
 *     per-thread error string, an atomic launch counter (grl_launch_count), the attention-kernel
 *     selector (grl_tc_attn_variant) and the environment switches read once (GRL_ATTN_SPLIT,
 *     GRL_GEMM_PERSISTENT, GRL_ATTN2_*), the per-device "shared-memory attribute set" flags, and the
 *     watchdog record of grl_tc_attn2_debug.  None of it depends on the data of a call;
 *   - returns 0 on success, a negative GrlStatus otherwise; grl_last_error() gives the message
 *     (the Python wrappers raise RuntimeError -- same behaviour as a failing ATen call).
 * Activations are channels-last: a (B, L, C) token tensor is the same memory as (B, H, W, C).
 */
#ifndef GRL_B200_H_
#define GRL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GRL_B200_ABI_VERSION 3

typedef enum {
  GRL_OK = 0,
  GRL_ERR_INVALID = -1,   /* bad argument / unsupported shape */
  GRL_ERR_CUDA = -2,      /* a CUDA runtime/driver call failed */
  GRL_ERR_WORKSPACE = -3, /* workspace too small */
  GRL_ERR_ARCH = -4       /* device is not sm_100 */
} GrlStatus;

typedef enum { GRL_ACT_NONE = 0, GRL_ACT_GELU = 1, GRL_ACT_LEAKY = 2 } GrlAct;

/* One attention "level": a (H x W) token grid cut into (wh x ww) windows/stripes after a cyclic
 * roll by (-sh, -sw)  [torch.roll + window_partition: mixed_attn_block_efficient.py:139-147,
 * :234-247; models/common/ops.py:36-54]. */
typedef struct {
  int32_t H, W;   /* grid size (tokens, or anchors = tokens / df) */
  int32_t wh, ww; /* window / stripe size on this grid */
  int32_t sh, sw; /* cyclic shift on this grid (0 = none) */
} GrlGrid;

const char* grl_last_error(void);
int grl_abi_version(void);
/* number of kernels this library has launched since it was loaded (bench.py's gpu_launches) */
uint64_t grl_launch_count(void);
/* 1 if the current device is compute capability 10.x */
int grl_device_ok(void);

/* ---- geometry, host side (bit-exact restatement of models/common/ops.py; used by tests and by the
 * Python surface to honour the reference's table/index/mask arguments) ------------------------- */
/* get_relative_position_index_simple (ops.py:352-375): out is (n1, n2) int64, row-major.
 * window_to_anchor != 0: n1 = wh*ww, n2 = (wh/df)*(ww/df); else transposed roles. */
int grl_rel_index_host(int wh, int ww, int df, int window_to_anchor, int64_t* out);
/* calculate_mask / calculate_mask_all (ops.py:112-157): out is (nW, n1, n2) fp32 of 0 / -100. */
int grl_shift_mask_host(int H, int W, int wh, int ww, int sh, int sw, int df, int window_to_anchor, float* out);
/* get_relative_coords_table_all (ops.py:225-271), pretrained size 0: out is ((wh+awh-1)*(ww+aww-1), 2) fp32 */
int grl_coords_table_host(int wh, int ww, int df, float* out);
/* torch.roll(-shift) + window_partition (ops.py:36-53, efficient.py:141-143,:236-241) as a gather map: out is
 * (nW, wh*ww) int32, the flat index y*W + x (un-rolled image) of token n of window w -- the addressing every attention
 * kernel folds into its loads and stores. */
int grl_token_map_host(GrlGrid g, int32_t* out);
/* Tokens per TMA box of the persistent attention kernel for this grid (csrc/attn2.cu): runs of that many
 * tokens starting at multiples of it are contiguous in memory for every window.  0 = no box form (gather kernel). */
int grl_tc_attn_box_tokens(GrlGrid g);

/* ---- fp32 operators (exact-parity path; every one is a hand-written sm_100a kernel) ---------- */

/* AffineTransform bias: out[h, r] = 16*sigmoid(CPB_MLP(table[r]))  for r < rows
 * (mixed_attn_block_efficient.py:41-47 with the gather commuted out; mixed_attn_block.py:24-31).
 * table (rows,2); w1 (hidden,2); b1 (hidden); w2 (heads,hidden); out (heads, rows). */
int grl_bias_table_f32(const float* table, int rows, const float* w1, const float* b1, const float* w2,
                       int hidden, int heads, float* out, void* stream);

/* AffineTransform.forward on a materialised map (mixed_attn_block_efficient.py:36-58):
 * attn (B_, heads, n1, n2) in place: attn*exp(min(logit_scale,ln100)) + bias[h, index[i,j]] + mask[b_%nW,i,j].
 * bias = output of grl_bias_table_f32; index (n1,n2) int64; mask (nW,n1,n2) or NULL. */
int grl_affine_f32(float* attn, int64_t B_, int heads, int n1, int n2, const float* logit_scale,
                   const float* bias, int rows, const int64_t* index, const float* mask, int nW, void* stream);

/* y[m, n] = act(sum_k x[m*ldx + k] * w[n*K + k] + b[n]) (+ res[m*ldr + n]);  nn.Linear / QKVProjection /
 * AnchorLinear.reduction / Mlp.fc1,fc2 / MixedAttention.proj (mixed_attn_block.py:661-676,:714-736;
 * swin_v1_block.py:37-43; mixed_attn_block_efficient.py:379). b, res may be NULL. */
int grl_linear_f32(const float* x, int64_t ldx, const float* w, const float* b, const float* res, int64_t ldr,
                   float* y, int64_t ldy, int64_t M, int N, int K, int act, float slope, void* stream);

/* 3x3 / stride 1 / pad 1 convolution on channels-last data (nn.Conv2d in CAB mixed_attn_block.py:973-977,
 * TransformerStage.conv grl.py:136,:168, conv_first / conv_after_body / upsampler heads grl.py:293,:348-379).
 * x (B,H,W,Cin); w packed (Cout, 9*Cin) with k = (ky*3+kx)*Cin + c; y (B,H,W,Cout); res optional (B,H,W,Cout). */
int grl_conv3x3_f32(const float* x, const float* w, const float* b, const float* res, float* y, int B, int H, int W,
                    int Cin, int Cout, int act, float slope, void* stream);

/* AvgPool2d(df, df) on channels-last data (AnchorLinear.pooling, mixed_attn_block.py:725,:733). */
int grl_avgpool_f32(const float* x, float* y, int B, int H, int W, int C, int df, void* stream);

/* out = (x ? x : 0) + res_scale * LayerNorm(u; gamma, beta, eps) (+ cab_y * cab_gate[b, c])
 * (post-norm residual, mixed_attn_block_efficient.py:543-554; norm_start/norm_end grl.py:494,:501 with x = NULL).
 * Rows M = B*L; cab_y (M,C) and cab_gate (B,C) optional (both or none). */
int grl_ln_residual_f32(const float* x, const float* u, const float* gamma, const float* beta, float eps,
                        float res_scale, const float* cab_y, const float* cab_gate, int64_t L, float* out,
                        int64_t M, int C, void* stream);

/* ChannelAttention gate (mixed_attn_block.py:948-967): gate[b,c] = sigmoid(W2 relu(W1 mean_L(y[b]) + b1) + b2).
 * y (B,L,C); w1 (R,C); w2 (C,R); workspace >= grl_channel_gate_workspace(B,L,C) bytes. */
size_t grl_channel_gate_workspace(int B, int64_t L, int C);
int grl_channel_gate_f32(const float* y, int B, int64_t L, int C, const float* w1, const float* b1, const float* w2,
                         const float* b2, int R, float* gate, void* workspace, size_t workspace_bytes, void* stream);

/* WindowAttention.forward (mixed_attn_block_efficient.py:128-165) fused: roll + partition + cosine attention
 * + learned scale + relative-position bias + shift mask + softmax + AV + merge + reverse roll.
 * qkv: token rows of `ld_qkv` floats; the window half starts at qkv and is laid out (3, heads, d).
 * out: token rows of `ld_out` floats, channel = head*d + e.  bias (heads, rows) from grl_bias_table_f32 with
 * rows = (2wh-1)(2ww-1).  use_mask: apply the region-id shift mask (mask argument not None in the reference). */
int grl_window_attn_f32(const float* qkv, int64_t ld_qkv, float* out, int64_t ld_out, int B, GrlGrid grid, int heads,
                        int d, const float* logit_scale, const float* bias, int use_mask, void* stream);

/* AnchorStripeAttention.forward (mixed_attn_block_efficient.py:215-270) fused: two chained attentions
 * X1 = softmax(a k^T) v (anchors attend to the stripe), Y = softmax(q a^T) X1.
 * qkv: stripe half (3, heads, d) per token; anchor (B, H/df, W/df, heads*d) rows of `ld_anchor` floats;
 * tok = stripe grid on tokens, anc = the same stripes on the anchor grid; bias1/scale1 = attn_transform1
 * (a2w index), bias2/scale2 = attn_transform2 (w2a index).  workspace >= grl_stripe_attn_workspace bytes. */
size_t grl_stripe_attn_workspace(int B, GrlGrid tok, GrlGrid anc, int heads, int d);
int grl_stripe_attn_f32(const float* qkv, int64_t ld_qkv, const float* anchor, int64_t ld_anchor, float* out,
                        int64_t ld_out, int B, GrlGrid tok, GrlGrid anc, int heads, int d, const float* logit_scale1,
                        const float* bias1, const float* logit_scale2, const float* bias2, int use_mask,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- bf16 tensor-core operators (throughput path: tcgen05.mma + TMEM + TMA, sm_100a only) ----------------
 * Activations are bf16 with channel pitches padded to a multiple of 64; attention heads live in 32-wide "slots"
 * (head_dim zero-padded to 32).  The residual stream, LayerNorm, softmax statistics and all accumulators stay fp32. */

/* grl_bias_table_f32 scaled by `mul` (log2(e) for the exp2-domain softmax of grl_tc_attn) and written as FOUR
 * copies, copy c shifted right by c entries: out[(h*4 + c)*rows_pad + r + c] = bias[h][r].  `out` (heads, 4, rows_pad)
 * must be zero-initialised; rows_pad % 4 == 0, rows_pad >= rows + 4.  The attention kernel reads runs of four
 * consecutive table entries as one aligned 16-byte load from the copy that matches the run's alignment. */
int grl_tc_bias_table4(const float* table, int rows, const float* w1, const float* b1, const float* w2, int hidden,
                       int heads, float mul, int rows_pad, float* out, void* stream);

/* `fmt` selects the 16-bit operand format everywhere below: 0 = fp16 (default: 11-bit mantissa, saturating
 * converts; needed for the 0.01 dB PSNR gate), 1 = bf16.  Both run kind::f16 tcgen05.mma at the same rate. */

/* fp32 (M, C) rows of pitch ldx -> 16-bit (M, Cpad) zero-padded; and back (16-bit rows of pitch ldx, column offset). */
int grl_tc_pack16(const float* x, int64_t ldx, void* y16, int64_t M, int C, int Cpad, int fmt, void* stream);
int grl_tc_unpack16(const void* x16, int64_t ldx, int x_off, float* y, int64_t ldy, int64_t M, int C, int fmt, void* stream);
/* Network input in one pass: check_image_size (reflect pad on the bottom / right up to (Hp, Wp); zero pad when the pad
 * exceeds the image, as grl.py:485-488 falls back) + (x - mean) * img_range (grl.py:510-511) + bchw -> channels-last +
 * 16-bit pack.  x (B, Cin <= 4, H, W) fp32 -> y16 (B, Hp, Wp, Cpad), zero in [Cin, Cpad); y32 (may be NULL): the fp32
 * channels-last copy (B, Hp, Wp, Cin) the no-upsampler heads add back (grl.py:540-547).  mean4: 4 HOST floats. */
int grl_tc_head_pack(const float* x, int B, int Cin, int H, int W, int Hp, int Wp, const float* mean4, float range, void* y16,
                     int Cpad, float* y32, int fmt, void* stream);
/* AvgPool2d(df) on 16-bit channels-last data (AnchorLinear.pooling, mixed_attn_block.py:725). */
int grl_tc_avgpool16(const void* x16, void* y16, int B, int H, int W, int Cpad, int df, int fmt, void* stream);
/* Per-slot multipliers of the packed qkv layout [win q|k|v][stripe q|k|v] x heads: exp(min(logit_scale, ln100))*log2(e)
 * on window q, stripe q (attn_transform2) and stripe k (attn_transform1); 1 on the other q/k slots; 0 on v slots
 * (mixed_attn_block_efficient.py:39). out: (3*hw + 3*hs) floats. */
int grl_tc_slot_scale(const float* ls_window, const float* ls_stripe1, const float* ls_stripe2, int heads_w, int heads_s,
                      float* out, void* stream);
/* ChannelAttention gate from bf16 CAB features y (B, L, ld) (mixed_attn_block.py:948-967). */
size_t grl_tc_channel_gate_workspace(int B, int64_t L, int C);
int grl_tc_channel_gate(const void* y16, int64_t ld, int fmt, int B, int64_t L, int C, const float* w1, const float* b1,
                        const float* w2, const float* b2, int R, float* gate, void* workspace, size_t workspace_bytes,
                        void* stream);

/* Tensor-core GEMM / implicit-GEMM 3x3 conv with a fused epilogue.  x: bf16 (M, kpad) or (B, H, W, kpad) when taps == 9;
 * w: bf16 (npad, taps*kpad) K-major (conv: k = tap*kpad + c, tap = ky*3+kx); bias: (npad) fp32, zero in the pad.
 *   epi 0  y = act(acc + b) (+ res_f32)           -> out_bf16 (n_store cols) and/or out_f32 (n_real cols)
 *          nn.Linear / nn.Conv2d of Mlp.fc1, CAB, TransformerStage.conv, conv_first/after_body/upsampler heads
 *   epi 1  per 32-wide slot: (acc + b) * slot_scale / max(||.||2, 1e-12) (slot_scale <= 0: untouched) -> out_bf16
 *          QKVProjection / AnchorLinear.reduction fused with F.normalize + logit scale (efficient.py:39,:85)
 *   epi 2  out = res_f32 + res_scale * LayerNorm(acc + b) (+ cab_y * cab_gate[token / L]) -> out_f32 + out_bf16
 *          MixedAttention.proj + norm1 + CAB add, Mlp.fc2 + norm2 (efficient.py:543-554); needs npad <= 256. */
typedef struct {
  int32_t fmt; /* 0 = fp16, 1 = bf16 */
  const void* x;
  const void* w;
  const float* bias;
  int64_t M;
  int32_t B, H, W;
  int32_t kpad, npad, taps, epi;
  int32_t n_store, n_real;
  void* out_bf16;
  int64_t ldo_bf16;
  float* out_f32;
  int64_t ldo_f32;
  const float* res_f32;
  int64_t ldr;
  int32_t act;
  float slope;
  const float* slot_scale;
  int32_t C;
  const float* gamma;
  const float* beta;
  float eps, res_scale;
  const void* cab_y;
  int64_t ld_caby;
  const float* cab_gate;
  int64_t L;
  /* head / tail fusion (taps == 9 only; zero = off).
   * ps_r > 0: PixelShuffle(ps_r) folded into the 16-bit store (models/common/upsample.py:6-30): w rows must be packed so
   *   that output column n' = q * (n_store / r^2) + c holds torch channel c * r^2 + q; out_bf16 is (B, H r, W r, ldo_bf16).
   * out_nchw: final image planes (B, n_real / nchw_r^2, Hc, Wc) fp32 = value * post_scale + post_shift[c]: x / img_range +
   *   mean, the crop to (Hc, Wc) and bhwc -> bchw (grl.py:549-551) folded into the store; nchw_r > 1 additionally folds
   *   UpsampleOneStep's PixelShuffle (upsample.py:33-50, torch channel order). */
  int32_t ps_r;
  float* out_nchw;
  int32_t nchw_r, Hc, Wc;
  float post_scale;
  float post_shift[4];
} GrlTcGemm;
int grl_tc_gemm(const GrlTcGemm* p, void* stream);

/* Transformer MLP of one block fused with norm2 and the residual (Mlp.forward, swin_v1_block.py:37-43, then
 * norm2 + residual, efficient.py:554):
 *   out = res_f32 + res_scale * LayerNorm(fc2(GELU(fc1(x) + b1)) + b2; gamma, beta, eps) -> out_f32 (C cols) + out_bf16
 * in one persistent launch; the hidden activation never leaves the SM.  Same arithmetic as grl_tc_gemm epi 0 (GELU, 16-bit
 * out_bf16 of the hidden) followed by grl_tc_gemm epi 2 on that hidden.  x: 16-bit (M, cpad); w1: (hpad, cpad) and
 * w2: (n_ln, hpad), both K-major and zero in the pads; b1 (hpad) and b2 (n_ln) fp32, zero in the pads.
 * cpad % 64 == 0, cpad <= n_ln, n_ln in {64, 128, 192}, hpad % 64 == 0, C % 4 == 0, C <= min(cpad, 188); out_bf16 is written
 * up to ldo_bf16 columns (zero beyond C); ldo_f32 and ldr % 4 == 0, ldo_bf16 % 8 == 0. */
typedef struct {
  int32_t fmt; /* 0 = fp16, 1 = bf16 */
  const void* x;
  const void* w1;
  const float* b1;
  const void* w2;
  const float* b2;
  int64_t M;
  int32_t C, cpad, hpad, n_ln;
  const float* gamma;
  const float* beta;
  float eps, res_scale;
  const float* res_f32;
  int64_t ldr;
  float* out_f32;
  int64_t ldo_f32;
  void* out_bf16;
  int64_t ldo_bf16;
} GrlTcMlp;
int grl_tc_mlp(const GrlTcMlp* p, void* stream);

/* Fused cosine attention over packed bf16 head slots: out = softmax2(q k^T + bias + mask) v, one call per
 * WindowAttention.forward and two per AnchorStripeAttention.forward (efficient.py:128-165,:215-270).
 * q/k/v: bf16 token rows (pitch ld*, element offset *_off of head 0's slot); v_dense/o_dense: the (B_, heads, N, 32)
 * intermediate X1 of the stripe attention; bias: (heads, 4, rows_pad) fp32 from grl_tc_bias_table4(.., log2 e, ..). */
typedef struct {
  int32_t fmt; /* 0 = fp16, 1 = bf16 */
  GrlGrid gq, gk;
  const void* q;
  int64_t ldq;
  int32_t q_off;
  const void* k;
  int64_t ldk;
  int32_t k_off;
  const void* v;
  int64_t ldv;
  int32_t v_off;
  int32_t v_dense;
  void* out;
  int64_t ldo;
  int32_t o_off;
  int32_t o_dense;
  int32_t B, heads;
  const float* bias; /* (heads, 4, rows_pad) from grl_tc_bias_table4 */
  int32_t rows;
  int32_t rows_pad;
  int32_t use_mask;
  int32_t ones_col; /* 1: column 31 of every V row is 1.0 (head_dim < 32) -> the row sum comes out of the P V MMA */
} GrlTcAttn;
int grl_tc_attn(const GrlTcAttn* p, void* stream);

/* Kernel behind grl_tc_attn: 5 (default) = the persistent warp-specialised kernel of csrc/attn2.cu -- Q / K / V tiles by TMA
 * boxes of the (B, H, W, C) tensors, S and P in TMEM (P V reads its A operand from TMEM), O accumulated in TMEM with a lazy
 * rescale, several query tiles sharing every K / V tile -- for every geometry whose rolled window rows split into runs of
 * >= 8 contiguous tokens (grl_tc_attn_box_tokens > 0); other geometries, and 0, run the gather kernel of csrc/attn_tc.cu
 * (one CTA per 128-query tile, cp.async row gathers).  Initial value: environment variable GRL_ATTN_SPLIT (unset = 5).
 * Returns the previous value; anything but 0 / 5 only queries.  Both kernels compute the same function. */
int grl_tc_attn_variant(int variant);
/* Diagnosis of the persistent attention kernel's pipeline: out8 = {1 if an mbarrier wait timed out (~0.5 s) since the last
 * call, wait site id (csrc/attn2.cu), block, warp, parity, barrier shared-memory offset, 0, 0}; reading clears it.  A timed-out
 * launch finishes with undefined results instead of hanging the GPU. */
int grl_tc_attn2_debug(int* out8);

/* ---- validation metric (SURVEY.md 8f row 3) -------------------------------------------------- */
/* Per-image PSNR of the reference's validation step in one fused pass: tensor_round (utils/utils_image.py:30-33) of
 * both images, `border` pixels shaved on every side (engines/base.py:265-267, utils_image.py:8-11), mean squared error
 * over (C, H, W) and -10 log10 (utils/metrics/psnr.py:44-48).  restored / target: (B, C, H, W) fp32, C <= 4.
 * psnr_y (may be NULL): the same on the luma of MATLAB's rgb2ycbcr rounded to 8 bit (utils_image.py:43-80) when C == 3,
 * else a copy of psnr_rgb.  The error is accumulated exactly (integers), so the result does not depend on the launch
 * geometry.  workspace: 16 * B bytes of device memory (zeroed by the call). */
int grl_psnr_f32(const float* restored, const float* target, int B, int C, int H, int W, int border, void* workspace,
                 size_t workspace_bytes, float* psnr_rgb, float* psnr_y, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GRL_B200_H_ */
