// capi.cu -- the extern "C" surface declared in include/grl_b200.h.
#include <math.h>
#include <string.h>

#include "grl_common.cuh"
#include "ops_f32.h"
#include "ops_tc.h"

namespace grl {
char* error_buffer() {
  static thread_local char buf[512] = {0};
  return buf;
}
unsigned long long& launch_counter() {
  static unsigned long long n = 0;
  return n;
}
}  // namespace grl

using namespace grl;

extern "C" {

const char* grl_last_error(void) { return error_buffer(); }
int grl_abi_version(void) { return GRL_B200_ABI_VERSION; }
uint64_t grl_launch_count(void) { return launch_counter(); }

int grl_device_ok(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10;
}

// ---------------------------------------------------------------- geometry (host)
int grl_rel_index_host(int wh, int ww, int df, int window_to_anchor, int64_t* out) {
  GRL_REQUIRE(wh > 0 && ww > 0 && df > 0 && out, "rel_index: bad arguments");
  const int awh = wh / df, aww = ww / df;
  const int n1 = window_to_anchor ? wh * ww : awh * aww;
  const int n2 = window_to_anchor ? awh * aww : wh * ww;
  const int qww = window_to_anchor ? ww : aww;
  const int kwh = window_to_anchor ? awh : wh, kww = window_to_anchor ? aww : ww;
  for (int i = 0; i < n1; ++i)
    for (int j = 0; j < n2; ++j)
      out[(size_t)i * n2 + j] = rel_index(i / qww, i % qww, j / kww, j % kww, qww, kwh, kww);
  return GRL_OK;
}

int grl_token_map_host(GrlGrid g, int32_t* out) {
  GRL_REQUIRE(out != nullptr, "token_map: null output");
  int rc;
  if ((rc = check_grid(g, "token_map")) != GRL_OK) return rc;
  const int nwh = g.H / g.wh, nww = g.W / g.ww, n = g.wh * g.ww;
  for (int wr = 0; wr < nwh; ++wr)
    for (int wc = 0; wc < nww; ++wc)
      for (int i = 0; i < n; ++i) {
        const Tok t = locate(g, wr, wc, i);
        out[((size_t)wr * nww + wc) * n + i] = t.y * g.W + t.x;
      }
  return GRL_OK;
}

int grl_tc_attn_box_tokens(GrlGrid g) {
  if (check_grid(g, "attn_box_tokens") != GRL_OK) return 0;
  return tc::attn_tma_box_tokens(g);
}

int grl_shift_mask_host(int H, int W, int wh, int ww, int sh, int sw, int df, int window_to_anchor, float* out) {
  GRL_REQUIRE(df > 0 && out, "shift_mask: bad arguments");
  GrlGrid gt = {H, W, wh, ww, sh, sw};
  GrlGrid ga = {H / df, W / df, wh / df, ww / df, sh / df, sw / df};
  int rc;
  if ((rc = check_grid(gt, "shift_mask(tokens)")) != GRL_OK) return rc;
  if ((rc = check_grid(ga, "shift_mask(anchors)")) != GRL_OK) return rc;
  const GrlGrid& gq = window_to_anchor ? gt : ga;
  const GrlGrid& gk = window_to_anchor ? ga : gt;
  const int n1 = gq.wh * gq.ww, n2 = gk.wh * gk.ww;
  const int nwh = gq.H / gq.wh, nww = gq.W / gq.ww;
  for (int wr = 0; wr < nwh; ++wr)
    for (int wc = 0; wc < nww; ++wc) {
      float* o = out + (size_t)(wr * nww + wc) * n1 * n2;
      for (int i = 0; i < n1; ++i) {
        Tok tq = locate(gq, wr, wc, i);
        const int rq = region_id(gq, tq.r, tq.c);
        for (int j = 0; j < n2; ++j) {
          Tok tk = locate(gk, wr, wc, j);
          o[(size_t)i * n2 + j] = (rq != region_id(gk, tk.r, tk.c)) ? -100.0f : 0.0f;
        }
      }
    }
  return GRL_OK;
}

int grl_coords_table_host(int wh, int ww, int df, float* out) {
  GRL_REQUIRE(wh > 0 && ww > 0 && df > 0 && out, "coords_table: bad arguments");
  const int ws[2] = {wh, ww}, aws[2] = {wh / df, ww / df};
  int hi[2], lo[2];
  for (int a = 0; a < 2; ++a) {
    hi[a] = ws[a] - 1 - (ws[a] - aws[a]) / 2;
    lo[a] = -(aws[a] - 1) - (ws[a] - aws[a]) / 2;
  }
  const int nh = hi[0] - lo[0] + 1, nw = hi[1] - lo[1] + 1;
  // same operation order as ops.py:257-269: v / hi (fp32), * 8 (fp32), sign * log2(|v| + 1) (fp32), then a
  // division by the float64 scalar np.log2(8) == 3.0 carried out in fp32 (torch keeps the tensor dtype).
  for (int i = 0; i < nh; ++i)
    for (int j = 0; j < nw; ++j) {
      const int c[2] = {lo[0] + i, lo[1] + j};
      for (int a = 0; a < 2; ++a) {
        float v = (float)c[a] / (float)hi[a];
        v = v * 8.0f;
        float s = (v > 0.f) ? 1.f : (v < 0.f ? -1.f : 0.f);
        out[((size_t)i * nw + j) * 2 + a] = s * log2f(fabsf(v) + 1.0f) / 3.0f;
      }
    }
  return GRL_OK;
}

// ---------------------------------------------------------------- fp32 operators
int grl_bias_table_f32(const float* table, int rows, const float* w1, const float* b1, const float* w2, int hidden,
                       int heads, float* out, void* stream) {
  return launch_bias_table(table, rows, w1, b1, w2, hidden, heads, 1.0f, 1, rows, out, (cudaStream_t)stream);
}

int grl_tc_bias_table4(const float* table, int rows, const float* w1, const float* b1, const float* w2, int hidden,
                       int heads, float mul, int rows_pad, float* out, void* stream) {
  GRL_REQUIRE(rows_pad % 4 == 0 && rows_pad >= rows + 4, "tc_bias_table4: rows_pad must be a multiple of 4 and >= rows + 4");
  return launch_bias_table(table, rows, w1, b1, w2, hidden, heads, mul, 4, rows_pad, out, (cudaStream_t)stream);
}

int grl_affine_f32(float* attn, int64_t B_, int heads, int n1, int n2, const float* logit_scale, const float* bias,
                   int rows, const int64_t* index, const float* mask, int nW, void* stream) {
  return launch_affine(attn, B_, heads, n1, n2, logit_scale, bias, rows, (const long long*)index, mask, nW,
                       (cudaStream_t)stream);
}

int grl_linear_f32(const float* x, int64_t ldx, const float* w, const float* b, const float* res, int64_t ldr,
                   float* y, int64_t ldy, int64_t M, int N, int K, int act, float slope, void* stream) {
  GRL_REQUIRE(M >= 0 && N >= 0 && K > 0 && ldx >= K && ldy >= N, "linear: bad shape M=%lld N=%d K=%d", (long long)M, N,
              K);
  GemmArgs a = {x, ldx, w, b, res, ldr, y, ldy, M, N, K, act, slope, 0, 0, 0};
  return launch_gemm(a, false, (cudaStream_t)stream);
}

int grl_conv3x3_f32(const float* x, const float* w, const float* b, const float* res, float* y, int B, int H, int W,
                    int Cin, int Cout, int act, float slope, void* stream) {
  GRL_REQUIRE(B >= 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0, "conv3x3: bad shape");
  GemmArgs a = {x, 0, w, b, res, Cout, y, Cout, (long long)B * H * W, Cout, 9 * Cin, act, slope, H, W, Cin};
  return launch_gemm(a, true, (cudaStream_t)stream);
}

int grl_avgpool_f32(const float* x, float* y, int B, int H, int W, int C, int df, void* stream) {
  return launch_avgpool(x, y, B, H, W, C, df, (cudaStream_t)stream);
}

int grl_ln_residual_f32(const float* x, const float* u, const float* gamma, const float* beta, float eps,
                        float res_scale, const float* cab_y, const float* cab_gate, int64_t L, float* out, int64_t M,
                        int C, void* stream) {
  return launch_ln_residual(x, u, gamma, beta, eps, res_scale, cab_y, cab_gate, L, out, M, C, (cudaStream_t)stream);
}

size_t grl_channel_gate_workspace(int B, int64_t L, int C) { return channel_gate_ws(B, L, C); }

int grl_channel_gate_f32(const float* y, int B, int64_t L, int C, const float* w1, const float* b1, const float* w2,
                         const float* b2, int R, float* gate, void* workspace, size_t workspace_bytes, void* stream) {
  return launch_channel_gate(y, B, L, C, w1, b1, w2, b2, R, gate, workspace, workspace_bytes, (cudaStream_t)stream);
}

int grl_window_attn_f32(const float* qkv, int64_t ld_qkv, float* out, int64_t ld_out, int B, GrlGrid grid, int heads,
                        int d, const float* logit_scale, const float* bias, int use_mask, void* stream) {
  AttnArgs a;
  memset(&a, 0, sizeof(a));
  const int c = heads * d;
  a.gq = grid;
  a.gk = grid;
  a.q = qkv, a.ldq = ld_qkv, a.q_off = 0;
  a.k = qkv, a.ldk = ld_qkv, a.k_off = c;
  a.v = qkv, a.ldv = ld_qkv, a.v_off = 2 * c;
  a.out = out, a.ldo = ld_out, a.o_off = 0;
  a.B = B, a.heads = heads, a.d = d;
  a.logit_scale = logit_scale;
  a.bias = bias;
  a.rows = (2 * grid.wh - 1) * (2 * grid.ww - 1);
  a.use_mask = use_mask;
  return launch_attn(a, (cudaStream_t)stream);
}

size_t grl_stripe_attn_workspace(int B, GrlGrid tok, GrlGrid anc, int heads, int d) {
  (void)tok;
  return sizeof(float) * (size_t)B * anc.H * anc.W * heads * d;
}

int grl_stripe_attn_f32(const float* qkv, int64_t ld_qkv, const float* anchor, int64_t ld_anchor, float* out,
                        int64_t ld_out, int B, GrlGrid tok, GrlGrid anc, int heads, int d, const float* logit_scale1,
                        const float* bias1, const float* logit_scale2, const float* bias2, int use_mask,
                        void* workspace, size_t workspace_bytes, void* stream) {
  const size_t need = grl_stripe_attn_workspace(B, tok, anc, heads, d);
  if (workspace_bytes < need) return fail(GRL_ERR_WORKSPACE, "stripe_attn: workspace %zu < %zu", workspace_bytes, need);
  const int c = heads * d;
  const int rows = (tok.wh + anc.wh - 1) * (tok.ww + anc.ww - 1);
  float* x1 = (float*)workspace;
  AttnArgs a;
  memset(&a, 0, sizeof(a));
  // pass 1: anchors attend to the stripe's tokens (a2w)   efficient.py:256-258
  a.gq = anc, a.gk = tok;
  a.q = anchor, a.ldq = ld_anchor, a.q_off = 0;
  a.k = qkv, a.ldk = ld_qkv, a.k_off = c;
  a.v = qkv, a.ldv = ld_qkv, a.v_off = 2 * c;
  a.out = x1, a.o_dense = 1;
  a.B = B, a.heads = heads, a.d = d;
  a.logit_scale = logit_scale1, a.bias = bias1, a.rows = rows, a.use_mask = use_mask;
  int rc = launch_attn(a, (cudaStream_t)stream);
  if (rc != GRL_OK) return rc;
  // pass 2: tokens attend to the anchors, values = X1 (w2a)   efficient.py:259
  memset(&a, 0, sizeof(a));
  a.gq = tok, a.gk = anc;
  a.q = qkv, a.ldq = ld_qkv, a.q_off = 0;
  a.k = anchor, a.ldk = ld_anchor, a.k_off = 0;
  a.v = x1, a.v_dense = 1;
  a.out = out, a.ldo = ld_out, a.o_off = 0;
  a.B = B, a.heads = heads, a.d = d;
  a.logit_scale = logit_scale2, a.bias = bias2, a.rows = rows, a.use_mask = use_mask;
  return launch_attn(a, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- bf16 tensor-core operators
static int check_fmt(int fmt) {
  GRL_REQUIRE(fmt == 0 || fmt == 1, "tc: operand format must be 0 (fp16) or 1 (bf16), got %d", fmt);
  return GRL_OK;
}
int grl_tc_pack16(const float* x, int64_t ldx, void* y, int64_t M, int C, int Cpad, int fmt, void* stream) {
  if (check_fmt(fmt)) return GRL_ERR_INVALID;
  return tc::launch_pack_bf16(x, ldx, y, M, C, Cpad, fmt, (cudaStream_t)stream);
}
int grl_tc_unpack16(const void* x, int64_t ldx, int x_off, float* y, int64_t ldy, int64_t M, int C, int fmt,
                    void* stream) {
  if (check_fmt(fmt)) return GRL_ERR_INVALID;
  return tc::launch_unpack_bf16(x, ldx, x_off, y, ldy, M, C, fmt, (cudaStream_t)stream);
}
int grl_tc_head_pack(const float* x, int B, int Cin, int H, int W, int Hp, int Wp, const float* mean4, float range, void* y16,
                     int Cpad, float* y32, int fmt, void* stream) {
  if (check_fmt(fmt)) return GRL_ERR_INVALID;
  GRL_REQUIRE(x && y16, "head_pack: null argument");
  return tc::launch_head_pack(x, B, Cin, H, W, Hp, Wp, mean4, range, y16, Cpad, y32, fmt, (cudaStream_t)stream);
}
int grl_tc_avgpool16(const void* x, void* y, int B, int H, int W, int Cpad, int df, int fmt, void* stream) {
  if (check_fmt(fmt)) return GRL_ERR_INVALID;
  return tc::launch_avgpool_bf16(x, y, B, H, W, Cpad, df, fmt, (cudaStream_t)stream);
}
int grl_tc_slot_scale(const float* ls_w, const float* ls_s1, const float* ls_s2, int hw, int hs, float* out,
                      void* stream) {
  GRL_REQUIRE(hw >= 1 && hs >= 1 && hw <= 8 && hs <= 8, "slot_scale: bad head counts");
  return tc::launch_slot_scale(ls_w, ls_s1, ls_s2, hw, hs, out, (cudaStream_t)stream);
}
size_t grl_tc_channel_gate_workspace(int B, int64_t L, int C) { return tc::channel_partial_bf16_ws(B, L, C); }
int grl_tc_channel_gate(const void* y, int64_t ld, int fmt, int B, int64_t L, int C, const float* w1, const float* b1,
                        const float* w2, const float* b2, int R, float* gate, void* ws, size_t ws_bytes, void* stream) {
  if (check_fmt(fmt)) return GRL_ERR_INVALID;
  if (ws_bytes < tc::channel_partial_bf16_ws(B, L, C)) return fail(GRL_ERR_WORKSPACE, "tc_channel_gate: workspace too small");
  int chunks = 0;
  int rc = tc::launch_channel_partial_bf16(y, B, L, ld, C, fmt, (float*)ws, &chunks, (cudaStream_t)stream);
  if (rc != GRL_OK) return rc;
  return launch_channel_gate_from_partial((const float*)ws, chunks, B, L, C, w1, b1, w2, b2, R, gate, (cudaStream_t)stream);
}

int grl_tc_gemm(const GrlTcGemm* p, void* stream) {
  GRL_REQUIRE(p != nullptr, "tc_gemm: null problem");
  if (!grl_device_ok()) return fail(GRL_ERR_ARCH, "tc_gemm: tcgen05 kernels need an sm_100 device");
  tc::GemmTcProblem q = {p->x, p->w, p->M, p->B, p->H, p->W, p->kpad, p->npad, p->taps, p->epi};
  tc::GemmTcArgs a;
  memset(&a, 0, sizeof(a));
  if (check_fmt(p->fmt)) return GRL_ERR_INVALID;
  a.fmt = p->fmt;
  a.N = p->n_store, a.N_f32 = p->n_real;
  a.bias = p->bias;
  a.out_bf16 = p->out_bf16, a.ldo_bf16 = p->ldo_bf16;
  a.out_f32 = p->out_f32, a.ldo_f32 = p->ldo_f32;
  a.res_f32 = p->res_f32, a.ldr = p->ldr;
  a.act = p->act, a.slope = p->slope;
  a.slot_scale = p->slot_scale;
  a.C = p->C, a.gamma = p->gamma, a.beta = p->beta, a.eps = p->eps, a.res_scale = p->res_scale;
  a.cab_y = p->cab_y, a.ld_caby = p->ld_caby, a.cab_gate = p->cab_gate, a.L = p->L;
  a.ps_r = p->ps_r, a.out_nchw = p->out_nchw, a.nchw_r = p->nchw_r > 0 ? p->nchw_r : 1, a.Hc = p->Hc, a.Wc = p->Wc;
  a.post_scale = p->post_scale;
  for (int c = 0; c < 4; ++c) a.post_shift[c] = p->post_shift[c];
  GRL_REQUIRE(p->bias != nullptr, "tc_gemm: bias is required (pass zeros)");
  GRL_REQUIRE(p->n_store <= p->npad && p->n_real <= p->npad, "tc_gemm: n_store/n_real exceed npad");
  if (p->epi == tc::EPI_QKV) GRL_REQUIRE(p->slot_scale && p->out_bf16 && p->ldo_bf16 >= p->npad, "tc_gemm: QKV epilogue arguments");
  if (p->epi == tc::EPI_LN)
    GRL_REQUIRE(p->gamma && p->beta && p->res_f32 && p->out_f32 && p->out_bf16 && p->C > 0 && p->C <= p->npad &&
                    p->L > 0 && (p->ldo_f32 % 4) == 0 && (p->ldo_bf16 % 8) == 0,
                "tc_gemm: LN epilogue arguments");
  if (p->out_bf16) GRL_REQUIRE((p->ldo_bf16 % 8) == 0, "tc_gemm: bf16 output pitch must be a multiple of 8");
  return tc::launch_gemm_tc(q, a, (cudaStream_t)stream);
}

int grl_tc_mlp(const GrlTcMlp* p, void* stream) {
  GRL_REQUIRE(p != nullptr, "tc_mlp: null problem");
  if (!grl_device_ok()) return fail(GRL_ERR_ARCH, "tc_mlp: tcgen05 kernels need an sm_100 device");
  if (check_fmt(p->fmt)) return GRL_ERR_INVALID;
  GRL_REQUIRE(p->x && p->w1 && p->b1 && p->w2 && p->b2 && p->gamma && p->beta && p->res_f32 && p->out_f32 && p->out_bf16,
              "tc_mlp: null argument");
  GRL_REQUIRE(p->ldr >= p->C && p->ldo_f32 >= p->C && p->ldo_bf16 >= p->C && (p->ldr % 4) == 0 && (p->ldo_f32 % 4) == 0 &&
                  (p->ldo_bf16 % 8) == 0,
              "tc_mlp: pitches must hold C columns, fp32 pitches a multiple of 4 and the 16-bit pitch a multiple of 8");
  tc::MlpTcProblem q = {p->x, p->w1, p->b1, p->w2, p->M, p->cpad, p->hpad, p->n_ln};
  tc::GemmTcArgs a;
  memset(&a, 0, sizeof(a));
  a.fmt = p->fmt;
  a.bias = p->b2;
  a.C = p->C, a.gamma = p->gamma, a.beta = p->beta, a.eps = p->eps, a.res_scale = p->res_scale;
  a.res_f32 = p->res_f32, a.ldr = p->ldr;
  a.out_f32 = p->out_f32, a.ldo_f32 = p->ldo_f32;
  a.out_bf16 = p->out_bf16, a.ldo_bf16 = p->ldo_bf16;
  a.L = 1;
  return tc::launch_mlp_tc(q, a, (cudaStream_t)stream);
}

int grl_tc_attn(const GrlTcAttn* p, void* stream) {
  GRL_REQUIRE(p != nullptr, "tc_attn: null problem");
  if (!grl_device_ok()) return fail(GRL_ERR_ARCH, "tc_attn: tcgen05 kernels need an sm_100 device");
  tc::AttnTcArgs a;
  memset(&a, 0, sizeof(a));
  if (check_fmt(p->fmt)) return GRL_ERR_INVALID;
  a.fmt = p->fmt;
  a.gq = p->gq, a.gk = p->gk;
  a.q = (const __nv_bfloat16*)p->q, a.ldq = p->ldq, a.q_off = p->q_off;
  a.k = (const __nv_bfloat16*)p->k, a.ldk = p->ldk, a.k_off = p->k_off;
  a.v = (const __nv_bfloat16*)p->v, a.ldv = p->ldv, a.v_off = p->v_off, a.v_dense = p->v_dense;
  a.out = (__nv_bfloat16*)p->out, a.ldo = p->ldo, a.o_off = p->o_off, a.o_dense = p->o_dense;
  a.B = p->B, a.heads = p->heads, a.bias = p->bias, a.rows = p->rows, a.rows_pad = p->rows_pad, a.use_mask = p->use_mask;
  a.ones_col = p->ones_col;
  GRL_REQUIRE((p->ldq % 8) == 0 && (p->ldk % 8) == 0 && (p->v_dense || (p->ldv % 8) == 0) &&
                  (p->o_dense || (p->ldo % 8) == 0) && (p->q_off % 8) == 0 && (p->k_off % 8) == 0 &&
                  (p->v_off % 8) == 0 && (p->o_off % 8) == 0,
              "tc_attn: pitches and offsets must be multiples of 8 elements (16 bytes)");
  GRL_REQUIRE(p->rows == (p->gq.wh + p->gk.wh - 1) * (p->gq.ww + p->gk.ww - 1), "tc_attn: bias table has %d rows, expected %d",
              p->rows, (p->gq.wh + p->gk.wh - 1) * (p->gq.ww + p->gk.ww - 1));
  return tc::launch_attn_tc(a, (cudaStream_t)stream);
}

int grl_tc_attn_variant(int variant) { return tc::attn_variant(variant); }
int grl_tc_attn2_debug(int* out8) { return tc::attn2_debug(out8); }

int grl_psnr_f32(const float* restored, const float* target, int B, int C, int H, int W, int border, void* workspace,
                 size_t workspace_bytes, float* psnr_rgb, float* psnr_y, void* stream) {
  GRL_REQUIRE(restored && target && psnr_rgb, "psnr: null argument");
  GRL_REQUIRE(workspace && workspace_bytes >= sizeof(unsigned long long) * 2 * (size_t)(B > 0 ? B : 0),
              "psnr: workspace %zu bytes < %zu", workspace_bytes, sizeof(unsigned long long) * 2 * (size_t)(B > 0 ? B : 0));
  return launch_psnr(restored, target, B, C, H, W, border, (unsigned long long*)workspace, psnr_rgb, psnr_y,
                     (cudaStream_t)stream);
}

}  // extern "C"
