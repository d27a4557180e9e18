// ops_tc.h -- launcher declarations of the bf16 tensor-core path (gemm_tc.cu, attn_tc.cu, misc_tc.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/grl_b200.h"

namespace grl {
namespace tc {

enum { EPI_BIAS_ACT = 0, EPI_QKV = 1, EPI_LN = 2 };

struct GemmTcArgs {
  int fmt;  // operand / 16-bit activation format: 0 = fp16, 1 = bf16
  // filled by launch_gemm_tc
  long long M;
  int nk, taps, n_tiles, total_tiles;
  int H, W, tiles_x, tiles_y;
  int epi_mode;  // 0 = 16-bit staging, 1 = fp32 staging, 2 = direct
  // epilogue
  int N;      // columns computed/stored as bf16 (zero beyond the real outputs)
  int N_f32;  // real outputs (fp32 store / residual width)
  const float* bias;  // (npad), zero in the pad
  void* out_bf16;  // 16-bit output (fp16 or bf16 per fmt)
  long long ldo_bf16;
  float* out_f32;
  long long ldo_f32;
  const float* res_f32;
  long long ldr;
  int act;
  float slope;
  // EPI_QKV
  const float* slot_scale;  // per 32-wide slot: > 0 normalise and multiply, <= 0 leave as is
  // EPI_LN
  int C;
  const float* gamma;
  const float* beta;
  float eps, res_scale;
  const void* cab_y;  // 16-bit
  long long ld_caby;
  const float* cab_gate;
  long long L;
  // head / tail fusion (conv only)
  int ps_r;         // > 0: PixelShuffle(ps_r) folded into the 16-bit store: column n' = q * (N / r^2) + c goes to pixel
                    // (y r + q / r, x r + q % r), channel c of a (B, H r, W r, ldo) tensor (weights packed in that order)
  float* out_nchw;  // direct epilogue: final image planes (B, N_f32 / nchw_r^2, Hc, Wc) = value * post_scale + post_shift[c],
  int nchw_r;       // PixelShuffle(nchw_r) (torch channel order c r^2 + dy r + dx) and the crop to (Hc, Wc) folded into the store
  int Hc, Wc;
  float post_scale, post_shift[4];
};

struct GemmTcProblem {
  const void* x;  // bf16 activations
  const void* w;  // bf16 weights (npad, taps*kpad)
  long long M;    // linear: rows
  int B, H, W;    // conv: image
  int kpad, npad, taps, epi;
};

int launch_gemm_tc(const GemmTcProblem& p, GemmTcArgs a, cudaStream_t st);

// Fused transformer MLP (gemm_tc.cu, mlp_tcp_kernel): out = res + rs * LayerNorm(fc2(GELU(fc1(x)))).  The LayerNorm
// epilogue takes its arguments from a GemmTcArgs as an EPI_LN grl_tc_gemm would (bias = fc2 bias, C, gamma, beta, eps,
// res_scale, res_f32, out_f32, out_bf16).
struct MlpTcProblem {
  const void* x;   // 16-bit (M, cpad)
  const void* w1;  // 16-bit (hpad, cpad), K-major
  const float* b1; // (hpad), zero in the pad
  const void* w2;  // 16-bit (n_ln, hpad), K-major
  long long M;
  int cpad, hpad, n_ln;
};
struct MlpTcArgs {
  GemmTcArgs ep;
  const float* bias1;
  int nk1, nj;  // cpad / 64, hpad / 64
};
int launch_mlp_tc(const MlpTcProblem& p, GemmTcArgs a, cudaStream_t st);

// Fused attention on packed bf16 head slots (32 wide).  See attn_tc.cu.
struct AttnTcArgs {
  int fmt;  // 0 = fp16, 1 = bf16 (all 16-bit operands and outputs)
  GrlGrid gq, gk;
  const __nv_bfloat16* q;
  long long ldq;  // elements per token row
  int q_off;      // element offset of head 0's slot
  const __nv_bfloat16* k;
  long long ldk;
  int k_off;
  const __nv_bfloat16* v;
  long long ldv;
  int v_off;
  int v_dense;  // V is the dense (B_, heads, Nk, 32) X1 buffer
  __nv_bfloat16* out;
  long long ldo;
  int o_off;
  int o_dense;
  int B, heads;
  const float* bias;  // (heads, 4, rows_pad) fp32, log2 domain: copy c holds the table shifted right by c entries
  int rows, rows_pad;
  int use_mask;
  int ones_col;  // V[:, 31] == 1 for every key: take the softmax denominator from O[:, 31]
};
int launch_attn_tc(const AttnTcArgs& a, cudaStream_t st);
// 5 = attn2.cu where the geometry allows it (default), 0 = always this file's gather kernel; -1 (or anything else): query only
int attn_variant(int set);
// persistent warp-specialised kernel (attn2.cu): P and O in TMEM, NWG query tiles share each K / V tile; returns +1 when the
// geometry has no TMA box form
int launch_attn2(const AttnTcArgs& a, cudaStream_t st);
int attn_tma_box_tokens(const GrlGrid& g);  // tokens per TMA box of attn2.cu for this grid, 0 = no box form
int attn2_debug(int* out8);  // {timed_out, wait site, block, warp, parity, barrier smem offset, 0, 0} of the first timed-out wait; clears it

}  // namespace tc
}  // namespace grl

namespace grl {
namespace tc {
// reflect-pad (or zero-pad when the pad exceeds the image, as grl.py:485-488 falls back) + (x - mean) * range + NCHW -> NHWC +
// 16-bit pack of the network input: x (B, Cin, H, W) fp32 -> y16 (B, Hp, Wp, Cpad) and, optionally, y32 (B, Hp, Wp, Cin)
int launch_head_pack(const float* x, int B, int Cin, int H, int W, int Hp, int Wp, const float* mean4, float range, void* y16,
                     int Cpad, float* y32, int fmt, cudaStream_t st);
int launch_pack_bf16(const float* x, long long ldx, void* y, long long M, int C, int Cpad, int fmt, cudaStream_t st);
int launch_unpack_bf16(const void* x, long long ldx, int x_off, float* y, long long ldy, long long M, int C, int fmt,
                       cudaStream_t st);
int launch_avgpool_bf16(const void* x, void* y, int B, int H, int W, int Cpad, int df, int fmt, cudaStream_t st);
size_t channel_partial_bf16_ws(int B, long long L, int C);
int launch_channel_partial_bf16(const void* y, int B, long long L, long long ld, int C, int fmt, float* partial,
                                int* chunks_out, cudaStream_t st);
int launch_slot_scale(const float* ls_w, const float* ls_s1, const float* ls_s2, int hw, int hs, float* out,
                      cudaStream_t st);
}  // namespace tc
}  // namespace grl
