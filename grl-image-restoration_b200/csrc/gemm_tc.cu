// gemm_tc.cu -- bf16 tcgen05 GEMM / implicit-GEMM 3x3 convolution with fused epilogues (the non-attention half
// of a GRL block on the throughput path).
//
//   D[128 x BN] (fp32, TMEM) = A[128 x K] (bf16, TMA -> smem, SWIZZLE_128B) * W[BN x K]^T (bf16, TMA -> smem)
//
// A is either a row-major (tokens x Kpad) activation matrix (nn.Linear: QKVProjection, AnchorLinear, proj, Mlp) or
// the channels-last image itself read through a 4-D tensor map: one CTA owns an 8x16 pixel patch and each of the
// 9 taps is the same TMA box shifted by (dy, dx) -- the zero padding of the convolution is TMA's out-of-bounds
// fill, no im2col buffer exists (CAB convs mixed_attn_block.py:973-977, TransformerStage.conv grl.py:164-170).
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + single-thread MMA issuer,
// warps 2-5 = epilogue (one accumulator row per thread, read with tcgen05.ld 32x32b).
// Two CTAs are co-resident per SM (<= 100 KB smem, <= 256 TMEM columns each) so one CTA's epilogue overlaps the
// other's loads and MMAs; these GEMMs are short-K and HBM/epilogue bound, not tensor bound (DESIGN.md).
//
// Epilogues:
//   EPI_BIAS_ACT : y = act(acc + b) (+ res)                       -> bf16 and/or fp32     (fc1, CAB, convs, heads)
//   EPI_QKV      : per 32-wide head slot  y = (acc + b) * scale / max(||.||, 1e-12)  -> bf16 (q^, k^, a^; v untouched)
//                  (F.normalize + logit scale of Attention.attn / AffineTransform, efficient.py:39,:85)
//   EPI_LN       : x' = x + rs * LayerNorm(acc + b) (+ cab_y * gate) -> fp32 residual stream + bf16 operand copy
//                  (efficient.py:543-554)
// mlp_tcp_kernel fuses the transformer MLP (fc1 -> GELU -> fc2 -> EPI_LN) into one persistent launch (see there).
#include <algorithm>
#include <stdlib.h>

#include "grl_common.cuh"
#include "tc_common.cuh"
#include "ops_tc.h"

namespace grl {
namespace tc {

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// erf-form GELU for the tensor-core epilogues: Abramowitz-Stegun 7.1.26 (|erf error| <= 1.5e-7 plus ~1e-6 from the
// approximate reciprocal / exp2; far below the 16-bit rounding that follows): 2 MUFU + 11 FMA-class instructions
// instead of erff's ~30.  The fp32 parity path keeps erff.
__device__ __forceinline__ float gelu_as(float x) {
  const float z = fabsf(x) * 0.70710678118654752440f;
  float t, e;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-z * z * 1.4426950408889634f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float erf_abs = fmaf(-p * t, e, 1.0f);  // erf(|x| / sqrt 2)
  const float half_x = 0.5f * x;
  return fmaf(half_x, copysignf(erf_abs, x), half_x);  // 0.5 x (1 + erf(x / sqrt 2))
}
__device__ __forceinline__ float tc_act(float v, int act, float slope) {
  if (act == GRL_ACT_GELU) return gelu_as(v);
  if (act == GRL_ACT_LEAKY) return v > 0.f ? v : v * slope;
  return v;
}

// ---- differential-timing builds (tools/kernel_diag.py): each GRL_GEMM_DIAG_* define removes ONE stream of the
// epilogue so that its cost shows up as a time difference.  Results of such builds are wrong by construction; the
// default build is bit-for-bit the production kernel.
#ifdef GRL_GEMM_DIAG_NORES  // fp32 residual tile never fetched
#define GRL_GDIAG_RES(x) false
#else
#define GRL_GDIAG_RES(x) (x)
#endif
#ifdef GRL_GEMM_DIAG_NOCAB  // CAB features / gate never fetched
#define GRL_GDIAG_CAB(x) false
#else
#define GRL_GDIAG_CAB(x) (x)
#endif
#ifdef GRL_GEMM_DIAG_NOST32  // fp32 residual stream never written
#define GRL_GDIAG_ST32(x) false
#else
#define GRL_GDIAG_ST32(x) (x)
#endif
#ifdef GRL_GEMM_DIAG_NOST16  // 16-bit operand copy never written
#define GRL_GDIAG_ST16(x) false
#else
#define GRL_GDIAG_ST16(x) (x)
#endif

constexpr int kStages = 2;
constexpr int kBM = 128, kBK = 64;
constexpr int kTH = 8, kTW = 16;  // conv patch (kTH * kTW == kBM)

// Epilogue staging: the accumulator tile is first written to shared memory by its row owners (phase A, thread = row,
// straight from TMEM), then streamed to global memory row-major by all epilogue threads with 16-byte accesses
// (phase B) -- fully coalesced residual reads and stores with many independent requests in flight.  The staging
// tile aliases the TMA pipeline buffers (the main loop is over when the epilogue starts).
//   fp32 staging (LayerNorm / fp32 outputs): [128][pitch32] floats, pitch32 % 8 == 4  -> conflict-free 16 B rows
//   16-bit staging (fp16/bf16-only outputs): [128][BN + 8] halves
__host__ __device__ constexpr int stage_pitch32(int c) { return (c % 8 == 4) ? c : ((c + 3) / 4 * 4 % 8 == 4 ? (c + 3) / 4 * 4 : (c + 3) / 4 * 4 + 4); }

template <int BN>
struct GemmSmem {
  static constexpr int A_BYTES = kBM * kBK * 2;
  static constexpr int B_BYTES = BN * kBK * 2;
  static constexpr int STAGE = A_BYTES + B_BYTES;
  static constexpr int PIPE = kStages * STAGE;
  static constexpr int STG32 = (BN == 96) ? 0 : kBM * stage_pitch32(BN <= 192 ? (BN == 192 ? 188 : BN) : 4) * 4;  // C <= 188 at BN = 192
  static constexpr int STG16 = kBM * (BN + 8) * 2;
  static constexpr int STG = (STG32 > STG16 ? STG32 : STG16);
  static constexpr int OFF_TOK = ((PIPE > STG ? PIPE : STG) + 15) / 16 * 16;  // long long tok[128]
  static constexpr int OFF_PAR = OFF_TOK + 128 * 8 + 128 * 4;  // (+ int img[128]) float bias[BN], gamma[BN], beta[BN]
  static constexpr int OFF_BAR = OFF_PAR + 3 * BN * 4;
  static constexpr int TOTAL = OFF_BAR + 128 + 1024 /*align slack*/;
};

__device__ __forceinline__ uint32_t tmem_cols_for(int bn) { return bn <= 32 ? 32 : bn <= 64 ? 64 : bn <= 128 ? 128 : 256; }

__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

template <int BN, int EPI, bool CONV>
__global__ void __launch_bounds__(192, (BN <= 96 ? 3 : 2))
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  using S = GemmSmem<BN>;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* empty = full + kStages;
  uint64_t* tmem_full = empty + kStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
  long long* s_tok = reinterpret_cast<long long*>(smem + S::OFF_TOK);
  int* s_img = reinterpret_cast<int*>(smem + S::OFF_TOK + 128 * 8);  // image (batch) index of every row (CAB gate)
  float* s_bias = reinterpret_cast<float*>(smem + S::OFF_PAR);      // this tile's columns [n0, n0 + BN)
  float* s_gamma = s_bias + BN;
  float* s_beta = s_gamma + BN;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // 1-D grid, N tile fastest: the CTAs that share an A tile (same rows, different output columns) are scheduled
  // together, so the tile is read from DRAM once and from L2 afterwards (QKV: 3 column tiles, fc1: 2).
  const int n_tiles = a.n_tiles;
  const int m_idx = blockIdx.x / n_tiles;
  const int n0 = (blockIdx.x - m_idx * n_tiles) * BN;
  const int nk_total = a.taps * a.nk;

  // tile coordinates
  int m0 = 0, tb = 0, ty0 = 0, tx0 = 0;
  if (CONV) {
    int t = m_idx;
    const int tx = t % a.tiles_x;
    t /= a.tiles_x;
    const int ty = t % a.tiles_y;
    tb = t / a.tiles_y;
    ty0 = ty * kTH;
    tx0 = tx * kTW;
  } else {
    m0 = m_idx * kBM;
  }

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    mbar_init_fence();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) tmem_alloc(tmem_slot, tmem_cols_for(BN));
  // per-column constants once per CTA (every row-owner thread needs all of them: smem broadcast instead of a global
  // load per accumulator element)
  for (int c = threadIdx.x; c < BN; c += blockDim.x) {
    const int n = n0 + c;
    s_bias[c] = (n < a.N) ? a.bias[n] : 0.f;
    if (EPI == EPI_LN) {
      s_gamma[c] = (c < a.C) ? a.gamma[c] : 0.f;
      s_beta[c] = (c < a.C) ? a.beta[c] : 0.f;
    }
  }
  if (warp >= 2) {  // token (global row) of every accumulator row, -1 = outside the problem
    const int r = (warp & 3) * 32 + lane;
    long long tok;
    if (CONV) {
      const int y = ty0 + r / kTW, x = tx0 + r % kTW;
      tok = (y < a.H && x < a.W) ? ((long long)tb * a.H + y) * a.W + x : -1;
    } else {
      tok = (long long)m0 + r;
      if (tok >= a.M) tok = -1;
    }
    s_tok[r] = tok;
    s_img[r] = (EPI == EPI_LN && tok >= 0) ? (int)(tok / a.L) : 0;  // one 64-bit division per row, not per access
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int kc = 0; kc < nk_total; ++kc) {
        const int s = kc % kStages;
        const uint32_t ph = (kc / kStages) & 1;
        mbar_wait(&empty[s], ph ^ 1);
        uint8_t* sa = smem + s * S::STAGE;
        uint8_t* sb = sa + S::A_BYTES;
        mbar_expect_tx(&full[s], S::STAGE);
        if (CONV) {
          const int tap = kc / a.nk, c0 = (kc - tap * a.nk) * kBK;
          tma_load_4d(sa, &tmA, &full[s], c0, tx0 + (tap % 3) - 1, ty0 + (tap / 3) - 1, tb);
        } else {
          tma_load_2d(sa, &tmA, &full[s], kc * kBK, m0);
        }
        tma_load_2d(sb, &tmB, &full[s], kc * kBK, n0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc(kBM, BN, a.fmt, 0, 0);
      for (int kc = 0; kc < nk_total; ++kc) {
        const int s = kc % kStages;
        const uint32_t ph = (kc / kStages) & 1;
        mbar_wait(&full[s], ph);
        tcgen05_fence_after();
        const uint32_t sa = smem_u32(smem + s * S::STAGE);
        const uint32_t sb = sa + S::A_BYTES;
#pragma unroll
        for (int k = 0; k < kBK / 16; ++k) {
          const uint64_t ad = umma_desc(sa + k * 32, 16, 1024, SWZ_128B);
          const uint64_t bd = umma_desc(sb + k * 32, 16, 1024, SWZ_128B);
          umma_ss(tmem, ad, bd, idesc, (kc | k) != 0);
        }
        umma_commit(&empty[s]);
      }
      umma_commit(tmem_full);
    }
  } else {
    // ================================================================== epilogue (4 warps, 128 threads)
    const int q = warp & 3;       // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;  // accumulator row owned in phase A
    const int et = threadIdx.x - 64;  // 0..127
    const int fmt = a.fmt;
    uint16_t* out16 = reinterpret_cast<uint16_t*>(a.out_bf16);
    mbar_wait(tmem_full, 0);  // all MMAs done -> accumulators valid AND the pipeline smem is free for staging
    tcgen05_fence_after();
    const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);
    uint32_t v[32];

    // epi_mode (chosen on the host): 1 = fp32 staging (LayerNorm / fp32 result / residual, whole row in this tile),
    // 0 = 16-bit staging, 2 = direct per-row stores (odd widths such as the 3-channel image head)
    if (EPI == EPI_BIAS_ACT && a.epi_mode == 2) {
      const long long tok = s_tok[row];
      for (int c0 = 0; c0 < BN; c0 += 32) {
        if (n0 + c0 >= a.N) break;
        tmem_ld32(trow + c0, v);
        tmem_ld_wait();
        if (tok < 0) continue;
        float o[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int n = n0 + c0 + j;
          float val = tc_act(__uint_as_float(v[j]) + s_bias[c0 + j], a.act, a.slope);
          if (a.res_f32 && n < a.N_f32) val += __ldg(a.res_f32 + tok * a.ldr + n);
          o[j] = (n < a.N) ? val : 0.f;
          if (a.out_f32 && n < a.N_f32) a.out_f32[tok * a.ldo_f32 + n] = o[j];
          if (CONV && a.out_nchw && n < a.N_f32) {
            // tail fusion: x / img_range + mean (grl.py:549), the crop (:551), channels-last -> bchw and, for the one-step
            // head, PixelShuffle (upsample.py:33-50; torch order n = c r^2 + dy r + dx) folded into the store
            const int r = a.nchw_r, rr = r * r;
            const int c = n / rr, q = n - c * rr;
            const int yy = (ty0 + row / kTW) * r + q / r, xx = (tx0 + row % kTW) * r + q % r;
            if (yy < a.Hc && xx < a.Wc)
              a.out_nchw[(((long long)tb * (a.N_f32 / rr) + c) * a.Hc + yy) * a.Wc + xx] = fmaf(o[j], a.post_scale, a.post_shift[c & 3]);
          }
        }
        if (out16) {
#pragma unroll
          for (int j = 0; j < 32; j += 8)
            if (n0 + c0 + j < a.ldo_bf16)
              *reinterpret_cast<uint4*>(out16 + tok * a.ldo_bf16 + n0 + c0 + j) =
                  make_uint4(pack16(o[j], o[j + 1], fmt), pack16(o[j + 2], o[j + 3], fmt), pack16(o[j + 4], o[j + 5], fmt),
                             pack16(o[j + 6], o[j + 7], fmt));
        }
      }
    } else if (a.epi_mode == 1) {
      const int Cw = (EPI == EPI_LN) ? a.C : a.N_f32;  // real fp32 columns of this tile row (n0 == 0 when wide)
      const int pitch = stage_pitch32(Cw);
      float* stg = reinterpret_cast<float*>(smem);
      // ---------------- residual tile -> staging, asynchronously (cp.async, 16 B per request, the whole 128 x C
      // tile in flight at once); it lands while the row moments are computed from TMEM.  Phase A then adds its
      // result in place, so phase B has no fp32 loads left.
      const bool res_in_stage = GRL_GDIAG_RES(a.res_f32 != nullptr);
      if (res_in_stage) {
        const int C4r = Cw >> 2, ewr = et >> 5;
        for (int r = ewr; r < kBM; r += 4) {
          const long long rtok = s_tok[r];
          for (int c4 = lane; c4 < C4r; c4 += 32)
            cp_async_16(stg + r * pitch + c4 * 4, a.res_f32 + (rtok >= 0 ? rtok : 0) * a.ldr + c4 * 4, rtok >= 0);
        }
        cp_async_commit();
      }
      // ---------------- phase A
      if (EPI == EPI_LN) {
        // one pass over TMEM for both moments, shifted by the row's first element (no catastrophic cancellation):
        //   mean = x0 + S1/C,  var = S2/C - (S1/C)^2   with S1 = sum(x - x0), S2 = sum((x - x0)^2)
        float s1 = 0.f, s2 = 0.f, x0 = 0.f;
        for (int c0 = 0; c0 < Cw; c0 += 32) {
          tmem_ld32(trow + c0, v);
          tmem_ld_wait();
          if (c0 == 0) x0 = __uint_as_float(v[0]) + s_bias[0];
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (c0 + j < Cw) {
              const float d = __uint_as_float(v[j]) + s_bias[c0 + j] - x0;
              s1 += d;
              s2 = fmaf(d, d, s2);
            }
        }
        const float m1 = s1 / (float)Cw;
        const float mean = x0 + m1;
        const float var = fmaxf(s2 / (float)Cw - m1 * m1, 0.f) * (float)Cw;  // (kept as a sum for the line below)
        const float rstd = rsqrtf(var / (float)Cw + a.eps);
        if (res_in_stage) {  // every thread's share of the residual tile has landed and is visible to the row owners
          cp_async_wait<0>();
          epi_barrier();
        }
        for (int c0 = 0; c0 < Cw; c0 += 32) {
          tmem_ld32(trow + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (c0 + j < Cw) {  // Cw % 4 == 0
              float4* sp = reinterpret_cast<float4*>(stg + row * pitch + c0 + j);
              float4 acc4 = res_in_stage ? *sp : make_float4(0.f, 0.f, 0.f, 0.f);
              float o4[4] = {acc4.x, acc4.y, acc4.z, acc4.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int c = c0 + j + e;
                o4[e] += ((__uint_as_float(v[j + e]) + s_bias[c] - mean) * rstd * s_gamma[c] + s_beta[c]) * a.res_scale;
              }
              *sp = make_float4(o4[0], o4[1], o4[2], o4[3]);
            }
          }
        }
      } else {
        if (res_in_stage) {
          cp_async_wait<0>();
          epi_barrier();
        }
        for (int c0 = 0; c0 < Cw; c0 += 32) {
          tmem_ld32(trow + c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (c0 + j < Cw) {
              float4* sp = reinterpret_cast<float4*>(stg + row * pitch + c0 + j);
              float4 acc4 = res_in_stage ? *sp : make_float4(0.f, 0.f, 0.f, 0.f);
              float o4[4] = {acc4.x, acc4.y, acc4.z, acc4.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) o4[e] += tc_act(__uint_as_float(v[j + e]) + s_bias[c0 + j + e], a.act, a.slope);
              *sp = make_float4(o4[0], o4[1], o4[2], o4[3]);
            }
          }
        }
      }
      tcgen05_fence_before();
      epi_barrier();
      // ---------------- phase B: row-major streaming, 4 columns per thread, warp = row group.
      // All global loads of a batch of RB rows are issued before any store (the compiler cannot prove the output
      // and residual pointers distinct, so interleaving would serialise every row on a DRAM round trip).
      const int C4 = Cw >> 2;                              // float4 items with real data
      const int P4 = out16 ? (int)(a.ldo_bf16 >> 2) : C4;  // the 16-bit copy is written up to its (zero) pad
      const int ew = et >> 5;
      const bool has_cab = GRL_GDIAG_CAB((EPI == EPI_LN) && a.cab_y != nullptr);
      const uint16_t* caby = reinterpret_cast<const uint16_t*>(a.cab_y);
      constexpr int RB = 8;
      for (int cbase = 0; cbase < P4; cbase += 32) {
        const int c4 = cbase + lane;
        const bool col_real = c4 < C4, col_any = c4 < P4;
        for (int rb = 0; rb < 32; rb += RB) {  // this warp's rows: ew, ew + 4, ...
          long long tok[RB];
          float4 gg[RB];
          uint2 cy[RB];
#pragma unroll
          for (int i = 0; i < RB; ++i) {
            tok[i] = s_tok[ew + 4 * (rb + i)];
            gg[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            cy[i] = make_uint2(0u, 0u);
            if (tok[i] >= 0 && col_real) {
              if (has_cab) {
                cy[i] = __ldg(reinterpret_cast<const uint2*>(caby + tok[i] * a.ld_caby + c4 * 4));
                gg[i] = __ldg(reinterpret_cast<const float4*>(a.cab_gate + (long long)s_img[ew + 4 * (rb + i)] * Cw + c4 * 4));
              }
            }
          }
#pragma unroll
          for (int i = 0; i < RB; ++i) {
            if (tok[i] < 0 || !col_any) continue;
            float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
            if (col_real) {
              val = *reinterpret_cast<const float4*>(stg + (ew + 4 * (rb + i)) * pitch + c4 * 4);
              if (has_cab) {
                const float2 c01 = unpack16(cy[i].x, fmt), c23 = unpack16(cy[i].y, fmt);
                val.x = fmaf(c01.x, gg[i].x, val.x), val.y = fmaf(c01.y, gg[i].y, val.y);
                val.z = fmaf(c23.x, gg[i].z, val.z), val.w = fmaf(c23.y, gg[i].w, val.w);
              }
              if (GRL_GDIAG_ST32(a.out_f32)) *reinterpret_cast<float4*>(a.out_f32 + tok[i] * a.ldo_f32 + c4 * 4) = val;
            }
            if (GRL_GDIAG_ST16(out16))
              *reinterpret_cast<uint2*>(out16 + tok[i] * a.ldo_bf16 + c4 * 4) =
                  make_uint2(pack16(val.x, val.y, fmt), pack16(val.z, val.w, fmt));
          }
        }
      }
    } else {
      // ---------------- 16-bit outputs only: phase A packs into a [128][BN + 8] tile
      constexpr int P16 = BN + 8;
      uint16_t* stg = reinterpret_cast<uint16_t*>(smem);
      const int ncols = min(BN, a.N - n0);  // columns of this tile that exist (multiple of 32)
      for (int c0 = 0; c0 < ncols; c0 += 32) {
        tmem_ld32(trow + c0, v);
        tmem_ld_wait();
        float o[32];
        if (EPI == EPI_QKV) {
          const int slot = (n0 + c0) >> 5;
          float ss = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            o[j] = __uint_as_float(v[j]) + s_bias[c0 + j];
            ss = fmaf(o[j], o[j], ss);
          }
          const float sc = __ldg(a.slot_scale + slot);
          // x / max(||x||, 1e-12) == x * rsqrt(max(||x||^2, 1e-24));  scale <= 0 marks a value slot
          const float mul = sc > 0.f ? sc * rsqrtf(fmaxf(ss, 1e-24f)) : 1.0f;
#pragma unroll
          for (int j = 0; j < 32; ++j) o[j] *= mul;
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) o[j] = tc_act(__uint_as_float(v[j]) + s_bias[c0 + j], a.act, a.slope);
        }
#pragma unroll
        for (int j = 0; j < 32; j += 8)
          *reinterpret_cast<uint4*>(stg + row * P16 + c0 + j) =
              make_uint4(pack16(o[j], o[j + 1], fmt), pack16(o[j + 2], o[j + 3], fmt), pack16(o[j + 4], o[j + 5], fmt),
                         pack16(o[j + 6], o[j + 7], fmt));
      }
      tcgen05_fence_before();
      epi_barrier();
      const int nvec = min((long long)ncols, a.ldo_bf16 - n0) >> 3;  // 16-byte vectors per row
      const int ew = et >> 5;
      if (CONV && a.ps_r > 0) {
        // PixelShuffle folded into the store (upsample.py:6-30): the weights are packed so that column n' = q * Cq + c
        // holds torch's channel c r^2 + q, i.e. Cq consecutive columns are ONE output pixel's channels
        const int ps = a.ps_r, Cq = a.N / (ps * ps);
        const int nv = min(BN, a.N - n0) >> 3;
#pragma unroll 4
        for (int r = ew; r < kBM; r += 4) {
          if (s_tok[r] < 0) continue;
          const int y = ty0 + r / kTW, x = tx0 + r % kTW;
          for (int vv = lane; vv < nv; vv += 32) {
            const int n = n0 + vv * 8;
            const int q = n / Cq, c = n - q * Cq;
            const long long dtok = ((long long)tb * a.H * ps + y * ps + q / ps) * ((long long)a.W * ps) + x * ps + q % ps;
            *reinterpret_cast<uint4*>(out16 + dtok * a.ldo_bf16 + c) = *reinterpret_cast<const uint4*>(stg + r * P16 + vv * 8);
          }
        }
      } else {
#pragma unroll 4
        for (int r = ew; r < kBM; r += 4) {
          const long long tok = s_tok[r];
          if (tok < 0) continue;
          for (int vv = lane; vv < nvec; vv += 32)
            if (GRL_GDIAG_ST16(true))
              *reinterpret_cast<uint4*>(out16 + tok * a.ldo_bf16 + n0 + vv * 8) = *reinterpret_cast<const uint4*>(stg + r * P16 + vv * 8);
        }
      }
    }
  }
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem, tmem_cols_for(BN));
  }
}

// -------------------------------------------------------------------------------------
// Persistent variant (GRL_GEMM_PERSISTENT=1): grid = min(#SMs, tiles), every CTA walks tiles blockIdx.x, blockIdx.x +
// gridDim.x, ... (N tile fastest).  Three decoupled pipelines: the TMA producer fills a 3-stage operand ring that is
// continuous across tiles, the MMA thread accumulates into the other half of TMEM (two accumulator buffers), and EIGHT
// epilogue warps -- two threads per accumulator row, the row's 32-column chunks split between them, LayerNorm moments
// merged through shared memory -- drain the current tile through a staging tile of its own.  One CTA per SM; the first
// version of this kernel (4 epilogue warps) lost to the 2-CTA kernel above because these GEMMs are epilogue-bound.
// -------------------------------------------------------------------------------------
constexpr int kStagesP = 3;
constexpr int kPersistentDefault = 15;  // measured: 412.9 -> 394.4 ms per 16-tile GRL-Base x4 forward with all four classes on
constexpr int kEpiWarpsP = 8, kEpiThreadsP = kEpiWarpsP * 32, kThreadsP = 64 + kEpiThreadsP;

template <int BN>
struct GemmSmemP {
  static constexpr int A_BYTES = kBM * kBK * 2;
  static constexpr int B_BYTES = BN * kBK * 2;
  static constexpr int STAGE = A_BYTES + B_BYTES;
  static constexpr int PIPE = kStagesP * STAGE;
  static constexpr int STG = GemmSmem<BN>::STG;
  static constexpr int OFF_STG = (PIPE + 1023) / 1024 * 1024;
  static constexpr int OFF_TOK = (OFF_STG + STG + 15) / 16 * 16;  // long long tok[128]
  static constexpr int OFF_PAR = OFF_TOK + 128 * 8 + 128 * 4;      // (+ int img[128]) float bias[BN], gamma[BN], beta[BN]
  static constexpr int OFF_MOM = OFF_PAR + 3 * BN * 4;             // float mom[2][128][3]
  static constexpr int OFF_BAR = OFF_MOM + 2 * 128 * 3 * 4;
  static constexpr int TOTAL = OFF_BAR + 128 + 1024 /*align slack*/;
  static_assert(TOTAL <= 232448, "shared memory budget");
};

__device__ __forceinline__ void epi_barrier_p() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// fp32-staged epilogue of the persistent kernels (epi_mode 1): residual prefetch into the staging tile, phase A from TMEM
// (LayerNorm moments and normalise, or bias / activation), phase B row-major streaming stores.  Called by the 256 threads of
// the eight epilogue warps (named barrier 1) of gemm_tcp_kernel and mlp_tcp_kernel; trow = this row's TMEM lane quarter in
// the accumulator buffer, row / half = the accumulator row and the column half (32-column chunks) this thread owns.
template <int EPI>
__device__ __forceinline__ void epilogue_f32_p(const GemmTcArgs& a, uint32_t trow, float* stg, const long long* s_tok,
                                               const int* s_img, const float* s_bias, const float* s_gamma,
                                               const float* s_beta, float* s_mom, int row, int half, int et, int lane) {
  const int fmt = a.fmt;
  uint16_t* out16 = reinterpret_cast<uint16_t*>(a.out_bf16);
  uint32_t v[32];
  const int Cw = (EPI == EPI_LN) ? a.C : a.N_f32;  // real fp32 columns of this tile row (n0 == 0 when wide)
  const int pitch = stage_pitch32(Cw);
  // ---------------- residual tile -> staging, asynchronously (cp.async, 16 B per request, the whole 128 x C
  // tile in flight at once); it lands while the row moments are computed from TMEM.  Phase A then adds its
  // result in place, so phase B has no fp32 loads left.
  const bool res_in_stage = GRL_GDIAG_RES(a.res_f32 != nullptr);
  if (res_in_stage) {
    const int C4r = Cw >> 2, ewr = et >> 5;
    for (int r = ewr; r < kBM; r += kEpiWarpsP) {
      const long long rtok = s_tok[r];
      for (int c4 = lane; c4 < C4r; c4 += 32)
        cp_async_16(stg + r * pitch + c4 * 4, a.res_f32 + (rtok >= 0 ? rtok : 0) * a.ldr + c4 * 4, rtok >= 0);
    }
    cp_async_commit();
  }
  // ---------------- phase A
  if (EPI == EPI_LN) {
    // One pass over TMEM for the moments of THIS THREAD'S HALF of the row (its 32-column chunks), shifted by the half's
    // first element (no catastrophic cancellation): mean_h = x0 + S1/n, M2_h = S2 - S1^2/n with S1 = sum(x - x0),
    // S2 = sum((x - x0)^2).  The two halves are merged with the pairwise update (Chan et al.):
    //   mean = mean_0 + d n_1 / n,  M2 = M2_0 + M2_1 + d^2 n_0 n_1 / n,  d = mean_1 - mean_0.
    float s1 = 0.f, s2 = 0.f, x0 = 0.f;
    int nh = 0;
    for (int c0 = 32 * half; c0 < Cw; c0 += 64) {
      tmem_ld32(trow + c0, v);
      tmem_ld_wait();
      if (c0 == 32 * half) x0 = __uint_as_float(v[0]) + s_bias[c0];
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (c0 + j < Cw) {
          const float d = __uint_as_float(v[j]) + s_bias[c0 + j] - x0;
          s1 += d;
          s2 = fmaf(d, d, s2);
          ++nh;
        }
    }
    {
      const float fn = (float)nh;
      const float m1 = nh > 0 ? s1 / fn : 0.f;
      s_mom[(half * kBM + row) * 3 + 0] = x0 + m1;
      s_mom[(half * kBM + row) * 3 + 1] = nh > 0 ? fmaxf(s2 - s1 * m1, 0.f) : 0.f;
      s_mom[(half * kBM + row) * 3 + 2] = fn;
    }
    if (res_in_stage) cp_async_wait<0>();  // this thread's share of the residual tile has landed ...
    epi_barrier_p();                         // ... and is visible to the row owners; so are both halves' moments
    float mean, rstd;
    {
      const float m0 = s_mom[row * 3 + 0], q0 = s_mom[row * 3 + 1], c0n = s_mom[row * 3 + 2];
      const float m1 = s_mom[(kBM + row) * 3 + 0], q1 = s_mom[(kBM + row) * 3 + 1], c1n = s_mom[(kBM + row) * 3 + 2];
      const float n = c0n + c1n, d = (c1n > 0.f) ? m1 - m0 : 0.f;
      mean = m0 + d * (c1n / n);
      const float M2 = q0 + q1 + d * d * (c0n * c1n / n);
      rstd = rsqrtf(M2 / n + a.eps);
    }
    for (int c0 = 32 * half; c0 < Cw; c0 += 64) {
      tmem_ld32(trow + c0, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        if (c0 + j < Cw) {  // Cw % 4 == 0
          float4* sp = reinterpret_cast<float4*>(stg + row * pitch + c0 + j);
          float4 acc4 = res_in_stage ? *sp : make_float4(0.f, 0.f, 0.f, 0.f);
          float o4[4] = {acc4.x, acc4.y, acc4.z, acc4.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int c = c0 + j + e;
            o4[e] += ((__uint_as_float(v[j + e]) + s_bias[c] - mean) * rstd * s_gamma[c] + s_beta[c]) * a.res_scale;
          }
          *sp = make_float4(o4[0], o4[1], o4[2], o4[3]);
        }
      }
    }
  } else {
    if (res_in_stage) {
      cp_async_wait<0>();
      epi_barrier_p();
    }
    for (int c0 = 32 * half; c0 < Cw; c0 += 64) {
      tmem_ld32(trow + c0, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        if (c0 + j < Cw) {
          float4* sp = reinterpret_cast<float4*>(stg + row * pitch + c0 + j);
          float4 acc4 = res_in_stage ? *sp : make_float4(0.f, 0.f, 0.f, 0.f);
          float o4[4] = {acc4.x, acc4.y, acc4.z, acc4.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) o4[e] += tc_act(__uint_as_float(v[j + e]) + s_bias[c0 + j + e], a.act, a.slope);
          *sp = make_float4(o4[0], o4[1], o4[2], o4[3]);
        }
      }
    }
  }
  tcgen05_fence_before();
  epi_barrier_p();
  // ---------------- phase B: row-major streaming, 4 columns per thread, warp = row group.
  // All global loads of a batch of RB rows are issued before any store (the compiler cannot prove the output
  // and residual pointers distinct, so interleaving would serialise every row on a DRAM round trip).
  const int C4 = Cw >> 2;                              // float4 items with real data
  const int P4 = out16 ? (int)(a.ldo_bf16 >> 2) : C4;  // the 16-bit copy is written up to its (zero) pad
  const int ew = et >> 5;
  const bool has_cab = GRL_GDIAG_CAB((EPI == EPI_LN) && a.cab_y != nullptr);
  const uint16_t* caby = reinterpret_cast<const uint16_t*>(a.cab_y);
  constexpr int RB = 8;
  for (int cbase = 0; cbase < P4; cbase += 32) {
    const int c4 = cbase + lane;
    const bool col_real = c4 < C4, col_any = c4 < P4;
    for (int rb = 0; rb < kBM / kEpiWarpsP; rb += RB) {  // this warp's rows: ew, ew + 8, ...
      long long tok[RB];
      float4 gg[RB];
      uint2 cy[RB];
#pragma unroll
      for (int i = 0; i < RB; ++i) {
        tok[i] = s_tok[ew + kEpiWarpsP * (rb + i)];
        gg[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        cy[i] = make_uint2(0u, 0u);
        if (tok[i] >= 0 && col_real) {
          if (has_cab) {
            cy[i] = __ldg(reinterpret_cast<const uint2*>(caby + tok[i] * a.ld_caby + c4 * 4));
            gg[i] = __ldg(reinterpret_cast<const float4*>(a.cab_gate + (long long)s_img[ew + kEpiWarpsP * (rb + i)] * Cw + c4 * 4));
          }
        }
      }
#pragma unroll
      for (int i = 0; i < RB; ++i) {
        if (tok[i] < 0 || !col_any) continue;
        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
        if (col_real) {
          val = *reinterpret_cast<const float4*>(stg + (ew + kEpiWarpsP * (rb + i)) * pitch + c4 * 4);
          if (has_cab) {
            const float2 c01 = unpack16(cy[i].x, fmt), c23 = unpack16(cy[i].y, fmt);
            val.x = fmaf(c01.x, gg[i].x, val.x), val.y = fmaf(c01.y, gg[i].y, val.y);
            val.z = fmaf(c23.x, gg[i].z, val.z), val.w = fmaf(c23.y, gg[i].w, val.w);
          }
          if (GRL_GDIAG_ST32(a.out_f32)) *reinterpret_cast<float4*>(a.out_f32 + tok[i] * a.ldo_f32 + c4 * 4) = val;
        }
        if (GRL_GDIAG_ST16(out16))
          *reinterpret_cast<uint2*>(out16 + tok[i] * a.ldo_bf16 + c4 * 4) =
              make_uint2(pack16(val.x, val.y, fmt), pack16(val.z, val.w, fmt));
      }
    }
  }
}

template <int BN, int EPI, bool CONV>
__global__ void __launch_bounds__(kThreadsP, 1)
gemm_tcp_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  using S = GemmSmemP<BN>;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* empty = full + kStagesP;
  uint64_t* tmem_full = empty + kStagesP;   // [2] accumulator buffer b complete            (tcgen05.commit)
  uint64_t* tmem_empty = tmem_full + 2;    // [2] accumulator buffer b drained by the epilogue (1 arrival)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  long long* s_tok = reinterpret_cast<long long*>(smem + S::OFF_TOK);
  int* s_img = reinterpret_cast<int*>(smem + S::OFF_TOK + 128 * 8);  // image (batch) index of every row (CAB gate)
  float* s_bias = reinterpret_cast<float*>(smem + S::OFF_PAR);      // this tile's columns [n0, n0 + BN)
  float* s_gamma = s_bias + BN;
  float* s_beta = s_gamma + BN;
  float* s_mom = reinterpret_cast<float*>(smem + S::OFF_MOM);  // [2][128][3]: (mean, M2, n) of each column half of a row

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = a.n_tiles;
  const int total_tiles = a.total_tiles;
  const int nk_total = a.taps * a.nk;
  const uint32_t TC = tmem_cols_for(BN);  // columns per accumulator buffer

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStagesP; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], 1);
    }
    mbar_init_fence();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) tmem_alloc(tmem_slot, 2 * TC);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;

  // tile -> coordinates (N tile fastest: the CTAs that share an A tile run together, so it is read from DRAM once)
  auto coords = [&](int tile, int& n0, int& m0, int& tb, int& ty0, int& tx0) {
    const int m_idx = tile / n_tiles;
    n0 = (tile - m_idx * n_tiles) * BN;
    m0 = 0, tb = 0, ty0 = 0, tx0 = 0;
    if (CONV) {
      int t = m_idx;
      const int tx = t % a.tiles_x;
      t /= a.tiles_x;
      const int ty = t % a.tiles_y;
      tb = t / a.tiles_y;
      ty0 = ty * kTH;
      tx0 = tx * kTW;
    } else {
      m0 = m_idx * kBM;
    }
  };

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        int n0, m0, tb, ty0, tx0;
        coords(tile, n0, m0, tb, ty0, tx0);
        for (int kc = 0; kc < nk_total; ++kc, ++it) {
          const int s = it % kStagesP;
          mbar_wait(&empty[s], ((it / kStagesP) & 1) ^ 1);
          uint8_t* sa = smem + s * S::STAGE;
          uint8_t* sb = sa + S::A_BYTES;
          mbar_expect_tx(&full[s], S::STAGE);
          if (CONV) {
            const int tap = kc / a.nk, c0 = (kc - tap * a.nk) * kBK;
            tma_load_4d(sa, &tmA, &full[s], c0, tx0 + (tap % 3) - 1, ty0 + (tap / 3) - 1, tb);
          } else {
            tma_load_2d(sa, &tmA, &full[s], kc * kBK, m0);
          }
          tma_load_2d(sb, &tmB, &full[s], kc * kBK, n0);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc(kBM, BN, a.fmt, 0, 0);
      uint32_t it = 0, lt = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
        const uint32_t b = lt & 1;
        mbar_wait(&tmem_empty[b], ((lt >> 1) & 1) ^ 1);  // the epilogue has drained this accumulator buffer
        tcgen05_fence_after();
        for (int kc = 0; kc < nk_total; ++kc, ++it) {
          const int s = it % kStagesP;
          mbar_wait(&full[s], (it / kStagesP) & 1);
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(smem + s * S::STAGE);
          const uint32_t sb = sa + S::A_BYTES;
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k) {
            const uint64_t ad = umma_desc(sa + k * 32, 16, 1024, SWZ_128B);
            const uint64_t bd = umma_desc(sb + k * 32, 16, 1024, SWZ_128B);
            umma_ss(tmem + b * TC, ad, bd, idesc, (kc | k) != 0);
          }
          umma_commit(&empty[s]);
        }
        umma_commit(&tmem_full[b]);
      }
    }
  } else {
    // ================================================================== epilogue (8 warps, 256 threads): TWO threads per
    // accumulator row -- warps w and w + 4 share a TMEM lane quarter and split the row's 32-column chunks (even / odd)
    const int q = warp & 3;       // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;  // accumulator row owned in phase A
    const int et = threadIdx.x - 64;  // 0..255
    const int half = et >> 7;         // which chunks of the row: c0 = 32 * half, + 64, ...
    const int fmt = a.fmt;
    uint16_t* out16 = reinterpret_cast<uint16_t*>(a.out_bf16);
    uint32_t v[32];
    uint32_t lt = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
      int n0, m0, tb, ty0, tx0;
      coords(tile, n0, m0, tb, ty0, tx0);
      // per-tile tables: token (global row) of every accumulator row (-1 = outside the problem), its image, and the
      // per-column constants of this N tile (every row-owner thread needs all of them: smem broadcast)
      {
        long long tok;
        if (CONV) {
          const int y = ty0 + row / kTW, x = tx0 + row % kTW;
          tok = (y < a.H && x < a.W) ? ((long long)tb * a.H + y) * a.W + x : -1;
        } else {
          tok = (long long)m0 + row;
          if (tok >= a.M) tok = -1;
        }
        if (half == 0) {
          s_tok[row] = tok;
          s_img[row] = (EPI == EPI_LN && tok >= 0) ? (int)(tok / a.L) : 0;  // one 64-bit division per row, not per access
        }
        for (int c = et; c < BN; c += kEpiThreadsP) {
          const int n = n0 + c;
          s_bias[c] = (n < a.N) ? a.bias[n] : 0.f;
          if (EPI == EPI_LN) {
            s_gamma[c] = (c < a.C) ? a.gamma[c] : 0.f;
            s_beta[c] = (c < a.C) ? a.beta[c] : 0.f;
          }
        }
      }
      epi_barrier_p();
      const uint32_t b = lt & 1;
      mbar_wait(&tmem_full[b], (lt >> 1) & 1);  // all MMAs of this tile done -> accumulators valid
      tcgen05_fence_after();
      const uint32_t trow = tmem + b * TC + ((uint32_t)(q * 32) << 16);


      // epi_mode (chosen on the host): 1 = fp32 staging (LayerNorm / fp32 result / residual, whole row in this tile),
      // 0 = 16-bit staging, 2 = direct per-row stores (odd widths such as the 3-channel image head)
      if (EPI == EPI_BIAS_ACT && a.epi_mode == 2) {
        const long long tok = s_tok[row];
        for (int c0 = 32 * half; c0 < BN; c0 += 64) {
          if (n0 + c0 >= a.N) break;
          tmem_ld32(trow + c0, v);
          tmem_ld_wait();
          if (tok < 0) continue;
          float o[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int n = n0 + c0 + j;
            float val = tc_act(__uint_as_float(v[j]) + s_bias[c0 + j], a.act, a.slope);
            if (a.res_f32 && n < a.N_f32) val += __ldg(a.res_f32 + tok * a.ldr + n);
            o[j] = (n < a.N) ? val : 0.f;
            if (a.out_f32 && n < a.N_f32) a.out_f32[tok * a.ldo_f32 + n] = o[j];
            if (CONV && a.out_nchw && n < a.N_f32) {
              // tail fusion: x / img_range + mean (grl.py:549), the crop (:551), channels-last -> bchw and, for the one-step
              // head, PixelShuffle (upsample.py:33-50; torch order n = c r^2 + dy r + dx) folded into the store
              const int r = a.nchw_r, rr = r * r;
              const int c = n / rr, q = n - c * rr;
              const int yy = (ty0 + row / kTW) * r + q / r, xx = (tx0 + row % kTW) * r + q % r;
              if (yy < a.Hc && xx < a.Wc)
                a.out_nchw[(((long long)tb * (a.N_f32 / rr) + c) * a.Hc + yy) * a.Wc + xx] = fmaf(o[j], a.post_scale, a.post_shift[c & 3]);
            }
          }
          if (out16) {
#pragma unroll
            for (int j = 0; j < 32; j += 8)
              if (n0 + c0 + j < a.ldo_bf16)
                *reinterpret_cast<uint4*>(out16 + tok * a.ldo_bf16 + n0 + c0 + j) =
                    make_uint4(pack16(o[j], o[j + 1], fmt), pack16(o[j + 2], o[j + 3], fmt), pack16(o[j + 4], o[j + 5], fmt),
                               pack16(o[j + 6], o[j + 7], fmt));
          }
        }
      } else if (a.epi_mode == 1) {
        epilogue_f32_p<EPI>(a, trow, reinterpret_cast<float*>(smem + S::OFF_STG), s_tok, s_img, s_bias, s_gamma, s_beta, s_mom,
                            row, half, et, lane);
      } else {
        // ---------------- 16-bit outputs only: phase A packs into a [128][BN + 8] tile
        constexpr int P16 = BN + 8;
        uint16_t* stg = reinterpret_cast<uint16_t*>(smem + S::OFF_STG);
        const int ncols = min(BN, a.N - n0);  // columns of this tile that exist (multiple of 32)
        for (int c0 = 32 * half; c0 < ncols; c0 += 64) {
          tmem_ld32(trow + c0, v);
          tmem_ld_wait();
          float o[32];
          if (EPI == EPI_QKV) {
            const int slot = (n0 + c0) >> 5;
            float ss = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              o[j] = __uint_as_float(v[j]) + s_bias[c0 + j];
              ss = fmaf(o[j], o[j], ss);
            }
            const float sc = __ldg(a.slot_scale + slot);
            // x / max(||x||, 1e-12) == x * rsqrt(max(||x||^2, 1e-24));  scale <= 0 marks a value slot
            const float mul = sc > 0.f ? sc * rsqrtf(fmaxf(ss, 1e-24f)) : 1.0f;
#pragma unroll
            for (int j = 0; j < 32; ++j) o[j] *= mul;
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) o[j] = tc_act(__uint_as_float(v[j]) + s_bias[c0 + j], a.act, a.slope);
          }
#pragma unroll
          for (int j = 0; j < 32; j += 8)
            *reinterpret_cast<uint4*>(stg + row * P16 + c0 + j) =
                make_uint4(pack16(o[j], o[j + 1], fmt), pack16(o[j + 2], o[j + 3], fmt), pack16(o[j + 4], o[j + 5], fmt),
                           pack16(o[j + 6], o[j + 7], fmt));
        }
        tcgen05_fence_before();
        epi_barrier_p();
        const int nvec = min((long long)ncols, a.ldo_bf16 - n0) >> 3;  // 16-byte vectors per row
        const int ew = et >> 5;
        if (CONV && a.ps_r > 0) {
          // PixelShuffle folded into the store (upsample.py:6-30): the weights are packed so that column n' = q * Cq + c
          // holds torch's channel c r^2 + q, i.e. Cq consecutive columns are ONE output pixel's channels
          const int ps = a.ps_r, Cq = a.N / (ps * ps);
          const int nv = min(BN, a.N - n0) >> 3;
#pragma unroll 4
          for (int r = ew; r < kBM; r += kEpiWarpsP) {
            if (s_tok[r] < 0) continue;
            const int y = ty0 + r / kTW, x = tx0 + r % kTW;
            for (int vv = lane; vv < nv; vv += 32) {
              const int n = n0 + vv * 8;
              const int q = n / Cq, c = n - q * Cq;
              const long long dtok = ((long long)tb * a.H * ps + y * ps + q / ps) * ((long long)a.W * ps) + x * ps + q % ps;
              *reinterpret_cast<uint4*>(out16 + dtok * a.ldo_bf16 + c) = *reinterpret_cast<const uint4*>(stg + r * P16 + vv * 8);
            }
          }
        } else {
#pragma unroll 4
          for (int r = ew; r < kBM; r += kEpiWarpsP) {
            const long long tok = s_tok[r];
            if (tok < 0) continue;
            for (int vv = lane; vv < nvec; vv += 32)
              if (GRL_GDIAG_ST16(true))
                *reinterpret_cast<uint4*>(out16 + tok * a.ldo_bf16 + n0 + vv * 8) = *reinterpret_cast<const uint4*>(stg + r * P16 + vv * 8);
          }
        }
      }

      // end of tile: every TMEM read of this buffer and every read of the staging tile / tables is done
      tcgen05_fence_before();
      epi_barrier_p();
      if (et == 0) mbar_arrive(&tmem_empty[b]);
    }
  }
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem, 2 * TC);
  }
}

// -------------------------------------------------------------------------------------
// Fused transformer MLP (grl_tc_mlp):  z = x + rs * LayerNorm2(fc2(GELU(fc1(y))))  -> z32 (fp32) + z16 (16-bit, zero pad).
// Persistent, one CTA per SM, 128-row tiles walked with stride gridDim.x.  The hidden activation never leaves the SM: each
// 64-wide hidden chunk j is accumulated in TMEM (H[j & 1] = A W1_j^T), turned into GELU'd 16-bit pairs in place by the
// GELU warps (tcgen05.ld -> gelu_as -> pack16 -> tcgen05.st), and read back by the fc2 MMA as its TMEM A operand
// (O[t & 1] += H16 W2_j^T).  The arithmetic is that of the two-launch route fc1 (EPI_BIAS_ACT, GELU) + fc2 (EPI_LN): the
// same gelu_as, the same 16-bit rounding of the hidden, the same K order of every fp32 accumulation, and the same
// LayerNorm epilogue function.
//   warp 0       TMA producer: the A tile (128 x cpad, resident while the tile runs fc1) and a ring of weight chunks,
//                W1 rows [64j, 64j + 64) or W2 columns [64j, 64j + 64), in the order the MMAs consume them
//   warp 1       TMEM allocator + single-thread MMA issuer: fc1(j + 1) is issued before fc2(j), so GELU(j) overlaps the
//                next fc1 chunk; fc1(j + 2) reuses H[j & 1] only after fc2(j) was issued, and the tensor pipe runs one
//                thread's MMAs in issue order
//   warps 2-5    GELU, one thread per hidden row (TMEM lane quarter warp & 3)
//   warps 6-13   LayerNorm epilogue of the persistent GEMM (epilogue_f32_p<EPI_LN>) on O[t & 1]
// TMEM: O[2] (n_ln columns each) + H[2] (64 columns each) = 512 columns at n_ln = 192.
// -------------------------------------------------------------------------------------
constexpr int kStagesM = 3;
constexpr int kGeluWarpsM = 4;
constexpr int kThreadsM = 64 + 32 * kGeluWarpsM + kEpiThreadsP;  // 448

template <int NLN>
struct MlpSmem {
  // cpad <= NLN: the A tile is NLN / 64 boxes of 128 x 64, a W1 chunk NLN / 64 boxes of 64 x 64, a W2 chunk NLN x 64
  static constexpr int A_BOX = kBM * kBK * 2;
  static constexpr int W1_BOX = 64 * kBK * 2;
  static constexpr int STAGE = NLN * kBK * 2;  // == (NLN / 64) * W1_BOX
  static constexpr int OFF_RING = (NLN / 64) * A_BOX;
  static constexpr int OFF_STG = OFF_RING + kStagesM * STAGE;
  static constexpr int STG = kBM * stage_pitch32(NLN == 192 ? 188 : NLN) * 4;  // fp32 LayerNorm staging, C <= 188
  static constexpr int OFF_TOK = OFF_STG + STG;                // long long tok[128], int img[128]
  static constexpr int OFF_PAR = OFF_TOK + 128 * 8 + 128 * 4;  // float bias2[NLN], gamma[NLN], beta[NLN]
  static constexpr int OFF_MOM = OFF_PAR + 3 * NLN * 4;        // float mom[2][128][3]
  static constexpr int OFF_BAR = OFF_MOM + 2 * 128 * 3 * 4;
  static constexpr int TOTAL = OFF_BAR + 256 + 1024 /*align slack*/;
  static_assert(STAGE == (NLN / 64) * W1_BOX, "ring stage holds a W1 or a W2 chunk");
  static_assert(OFF_TOK % 16 == 0, "alignment");
  static_assert(TOTAL <= 232448, "shared memory budget");
};

template <int NLN>
__global__ void __launch_bounds__(kThreadsM, 1)
mlp_tcp_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW1,
               const __grid_constant__ CUtensorMap tmW2, const MlpTcArgs m) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  using S = MlpSmem<NLN>;
  const GemmTcArgs& a = m.ep;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* empty = full + kStagesM;
  uint64_t* a_full = empty + kStagesM;  // A tile loaded                                  (TMA bytes)
  uint64_t* a_empty = a_full + 1;       // last fc1 MMA of the tile done: A may be replaced (tcgen05.commit)
  uint64_t* h_full = a_empty + 1;       // [2] fc1 chunk accumulated in H[b]                (tcgen05.commit)
  uint64_t* h_ready = h_full + 2;       // [2] H[b] holds the GELU'd 16-bit chunk           (one arrival per GELU warp)
  uint64_t* tmem_full = h_ready + 2;    // [2] O[b] complete                                (tcgen05.commit)
  uint64_t* tmem_empty = tmem_full + 2; // [2] O[b] drained by the LayerNorm epilogue       (1 arrival)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  long long* s_tok = reinterpret_cast<long long*>(smem + S::OFF_TOK);
  int* s_img = reinterpret_cast<int*>(smem + S::OFF_TOK + 128 * 8);
  float* s_bias = reinterpret_cast<float*>(smem + S::OFF_PAR);
  float* s_gamma = s_bias + NLN;
  float* s_beta = s_gamma + NLN;
  float* s_mom = reinterpret_cast<float*>(smem + S::OFF_MOM);

  constexpr uint32_t kColH = 2 * NLN;  // H[0], H[1] follow O[0], O[1]
  constexpr uint32_t kTmemCols = 2 * NLN + 128 <= 256 ? 256 : 512;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_tiles = a.total_tiles, nk1 = m.nk1, nj = m.nj;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStagesM; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&h_full[b], 1);
      mbar_init(&h_ready[b], kGeluWarpsM);
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], 1);
    }
    mbar_init_fence();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW1);
    tma_prefetch_desc(&tmW2);
  }
  if (warp == 1) tmem_alloc(tmem_slot, kTmemCols);
  for (int c = threadIdx.x; c < NLN; c += blockDim.x) {  // the weights are the same for every tile: one table per CTA
    s_bias[c] = a.bias[c];
    s_gamma[c] = (c < a.C) ? a.gamma[c] : 0.f;
    s_beta[c] = (c < a.C) ? a.beta[c] : 0.f;
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t it = 0, lt = 0;
      auto load_w = [&](bool w2, int j) {
        const int s = it % kStagesM;
        mbar_wait(&empty[s], ((it / kStagesM) & 1) ^ 1);
        uint8_t* sw = smem + S::OFF_RING + s * S::STAGE;
        if (w2) {
          mbar_expect_tx(&full[s], S::STAGE);
          tma_load_2d(sw, &tmW2, &full[s], j * kBK, 0);
        } else {
          mbar_expect_tx(&full[s], nk1 * S::W1_BOX);
          for (int kc = 0; kc < nk1; ++kc) tma_load_2d(sw + kc * S::W1_BOX, &tmW1, &full[s], kc * kBK, j * 64);
        }
        ++it;
      };
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
        mbar_wait(a_empty, (lt & 1) ^ 1);
        mbar_expect_tx(a_full, nk1 * S::A_BOX);
        for (int kc = 0; kc < nk1; ++kc) tma_load_2d(smem + kc * S::A_BOX, &tmA, a_full, kc * kBK, tile * kBM);
        load_w(false, 0);  // consumption order: W1_0, then (W1_{j+1}, W2_j) for every j
        for (int j = 0; j < nj; ++j) {
          if (j + 1 < nj) load_w(false, j + 1);
          load_w(true, j);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc1 = umma_idesc(kBM, 64, a.fmt, 0, 0);
      const uint32_t idesc2 = umma_idesc(kBM, NLN, a.fmt, 0, 0);
      const uint32_t sa = smem_u32(smem);
      uint32_t it = 0, lt = 0, g = 0;  // g: hidden chunks issued so far over all tiles; chunk g lives in H[g & 1]
      auto fc1 = [&](uint32_t hb) {
        const int s = it % kStagesM;
        mbar_wait(&full[s], (it / kStagesM) & 1);
        tcgen05_fence_after();
        const uint32_t sw = smem_u32(smem + S::OFF_RING + s * S::STAGE);
        for (int kc = 0; kc < nk1; ++kc)
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k)
            umma_ss(tmem + kColH + hb * 64, umma_desc(sa + kc * S::A_BOX + k * 32, 16, 1024, SWZ_128B),
                    umma_desc(sw + kc * S::W1_BOX + k * 32, 16, 1024, SWZ_128B), idesc1, (kc | k) != 0);
        umma_commit(&empty[s]);
        umma_commit(&h_full[hb]);
        ++it;
      };
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
        const uint32_t b = lt & 1;
        mbar_wait(&tmem_empty[b], ((lt >> 1) & 1) ^ 1);  // the LayerNorm epilogue has drained O[b]
        mbar_wait(a_full, lt & 1);
        tcgen05_fence_after();
        fc1(g & 1);
        if (nj == 1) umma_commit(a_empty);
        for (int j = 0; j < nj; ++j, ++g) {
          if (j + 1 < nj) {
            fc1((g + 1) & 1);  // H[(g + 1) & 1]: its previous chunk's fc2 was issued in the last iteration
            if (j + 2 == nj) umma_commit(a_empty);
          }
          mbar_wait(&h_ready[g & 1], (g >> 1) & 1);
          tcgen05_fence_after();
          const int s = it % kStagesM;
          mbar_wait(&full[s], (it / kStagesM) & 1);
          tcgen05_fence_after();
          const uint32_t sw = smem_u32(smem + S::OFF_RING + s * S::STAGE);
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k)
            umma_ts(tmem + b * NLN, tmem + kColH + (g & 1) * 64 + k * 8, umma_desc(sw + k * 32, 16, 1024, SWZ_128B), idesc2,
                    (j | k) != 0);
          umma_commit(&empty[s]);
          ++it;
        }
        umma_commit(&tmem_full[b]);
      }
    }
  } else if (warp < 2 + kGeluWarpsM) {
    // ================================================================== GELU: thread = hidden row of its lane quarter
    const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
    const int fmt = a.fmt;
    uint32_t g = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      for (int j = 0; j < nj; ++j, ++g) {
        const uint32_t th = tmem + kColH + (g & 1) * 64 + lane_off;
        const float4* b1 = reinterpret_cast<const float4*>(m.bias1 + j * 64);
        mbar_wait(&h_full[g & 1], (g >> 1) & 1);
        tcgen05_fence_after();
        uint32_t pk[32];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t v[32];
          tmem_ld32(th + h * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const float4 bb = __ldg(b1 + h * 8 + c);
            pk[h * 16 + 2 * c] = pack16(gelu_as(__uint_as_float(v[4 * c]) + bb.x), gelu_as(__uint_as_float(v[4 * c + 1]) + bb.y), fmt);
            pk[h * 16 + 2 * c + 1] =
                pack16(gelu_as(__uint_as_float(v[4 * c + 2]) + bb.z), gelu_as(__uint_as_float(v[4 * c + 3]) + bb.w), fmt);
          }
        }
        tmem_st32(th, pk);  // 64 hidden values -> 32 columns of 16-bit pairs, the fc2 MMA's A operand
        tmem_st_wait();
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&h_ready[g & 1]);
      }
    }
  } else {
    // ================================================================== LayerNorm epilogue (8 warps, 256 threads)
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int et = threadIdx.x - (64 + 32 * kGeluWarpsM);  // 0..255
    const int half = et >> 7;
    float* stg = reinterpret_cast<float*>(smem + S::OFF_STG);
    uint32_t lt = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
      if (half == 0) {
        const long long tok = (long long)tile * kBM + row;
        s_tok[row] = tok < a.M ? tok : -1;
        s_img[row] = 0;
      }
      epi_barrier_p();
      const uint32_t b = lt & 1;
      mbar_wait(&tmem_full[b], (lt >> 1) & 1);
      tcgen05_fence_after();
      epilogue_f32_p<EPI_LN>(a, tmem + b * NLN + ((uint32_t)(q * 32) << 16), stg, s_tok, s_img, s_bias, s_gamma, s_beta,
                             s_mom, row, half, et, lane);
      // end of tile: every TMEM read of O[b] and every read of the staging tile / row table is done
      tcgen05_fence_before();
      epi_barrier_p();
      if (et == 0) mbar_arrive(&tmem_empty[b]);
    }
  }
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem, kTmemCols);
  }
}

// -------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------
static int make_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                    const cuuint32_t* box, int fmt) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return fail(GRL_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint32_t ones[5] = {1, 1, 1, 1, 1};
  CUresult rc = fn(m, fmt == FMT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_bytes,
                   box, ones, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) return fail(GRL_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)rc);
  return GRL_OK;
}

template <int BN, int EPI, bool CONV>
static int launch_one(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmTcArgs& a, dim3 grid, cudaStream_t st) {
  auto kern = gemm_tc_kernel<BN, EPI, CONV>;
  // the attribute is per device: a process that drives several GPUs configures each one once
  static bool configured[kMaxDevices] = {false};
  int dev = 0;
  GRL_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices || !configured[dev]) {
    GRL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmSmem<BN>::TOTAL));
    if (dev >= 0 && dev < kMaxDevices) configured[dev] = true;
  }
  kern<<<grid, 192, GemmSmem<BN>::TOTAL, st>>>(tmA, tmB, a);
  GRL_LAUNCH_CHECK("gemm_tc_kernel");
  return GRL_OK;
}

template <int BN, int EPI, bool CONV>
static int launch_one_p(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmTcArgs& a, cudaStream_t st) {
  auto kern = gemm_tcp_kernel<BN, EPI, CONV>;
  static bool configured[kMaxDevices] = {false};
  int dev = 0;
  GRL_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices || !configured[dev]) {
    GRL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmSmemP<BN>::TOTAL));
    if (dev >= 0 && dev < kMaxDevices) configured[dev] = true;
  }
  const unsigned grid = (unsigned)std::min(sm_count(), a.total_tiles);  // one CTA per SM walks the tiles
  kern<<<grid, kThreadsP, GemmSmemP<BN>::TOTAL, st>>>(tmA, tmB, a);
  GRL_LAUNCH_CHECK("gemm_tcp_kernel");
  return GRL_OK;
}

template <int EPI, bool CONV>
static int dispatch_bn(int bn, const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmTcArgs& a, dim3 grid,
                       cudaStream_t st, bool persistent) {
  if (persistent) {
    switch (bn) {
      case 64: return launch_one_p<64, EPI, CONV>(tmA, tmB, a, st);
      case 128: return launch_one_p<128, EPI, CONV>(tmA, tmB, a, st);
      case 192: return launch_one_p<192, EPI, CONV>(tmA, tmB, a, st);
      case 256: return launch_one_p<256, EPI, CONV>(tmA, tmB, a, st);
    }
  }
  switch (bn) {
    case 64: return launch_one<64, EPI, CONV>(tmA, tmB, a, grid, st);
    case 96: return launch_one<96, EPI, CONV>(tmA, tmB, a, grid, st);
    case 128: return launch_one<128, EPI, CONV>(tmA, tmB, a, grid, st);
    case 192: return launch_one<192, EPI, CONV>(tmA, tmB, a, grid, st);
    case 256: return launch_one<256, EPI, CONV>(tmA, tmB, a, grid, st);
  }
  return fail(GRL_ERR_INVALID, "gemm_tc: unsupported tile width %d", bn);
}

int pick_bn(int npad) {
  if (npad <= 64) return 64;
  if (npad <= 128) return 128;
  if (npad % 192 == 0 || npad <= 192) return 192;
  if (npad % 256 == 0) return 256;
  return npad % 128 == 0 ? 128 : 192;
}

// x: bf16 (M, Kpad) row-major or (B, H, W, Kpad) channels-last; w: bf16 (Npad, taps*Kpad) K-major.
int launch_gemm_tc(const GemmTcProblem& p, GemmTcArgs a, cudaStream_t st) {
  GRL_REQUIRE(p.kpad % kBK == 0 && p.kpad > 0, "gemm_tc: K pad %d must be a multiple of 64", p.kpad);
  GRL_REQUIRE(p.npad % 32 == 0 && p.npad > 0, "gemm_tc: N pad %d must be a multiple of 32", p.npad);
  int bn = (p.epi == EPI_LN) ? (p.npad <= 64 ? 64 : p.npad <= 128 ? 128 : p.npad <= 192 ? 192 : 256) : pick_bn(p.npad);
  // 16-bit-only epilogues (QKV, fc1, CAB conv2): 96-wide tiles need 58 KB smem / 128 TMEM columns -> 3 CTAs per SM
  static int narrow = -1;
  if (narrow < 0) {
    const char* e = getenv("GRL_GEMM_BN96");
    narrow = (e && e[0] == '1') ? 1 : 0;  // opt-in: measured no gain on B200 (profiles/r1_tc_path_final.md)
  }
  if (narrow && p.epi != EPI_LN && !a.out_f32 && !a.res_f32 && p.npad % 96 == 0 && p.npad >= 192) bn = 96;
  GRL_REQUIRE(p.epi != EPI_LN || p.npad <= 256, "gemm_tc: LayerNorm epilogue needs the whole row in one tile (N=%d)",
              p.npad);
  // Which GEMM classes run the persistent 8-epilogue-warp kernel: GRL_GEMM_PERSISTENT = bit mask (1 LayerNorm epilogue,
  // 2 QKV epilogue, 4 bias / activation linear, 8 3x3 conv; default kPersistentDefault; 0 = the 2-CTA kernel everywhere).
  static int persistent_mask = -1;
  if (persistent_mask < 0) {
    const char* e = getenv("GRL_GEMM_PERSISTENT");
    persistent_mask = e ? atoi(e) & 15 : kPersistentDefault;
  }
  const int cls = p.taps == 9 ? 8 : p.epi == EPI_LN ? 1 : p.epi == EPI_QKV ? 2 : 4;
  bool persistent = (persistent_mask & cls) != 0 && bn != 96;
  const bool conv = p.taps == 9;
  if (a.ps_r > 0)
    GRL_REQUIRE(conv && p.epi == EPI_BIAS_ACT && !a.out_f32 && !a.res_f32 && a.out_bf16 && a.N % (a.ps_r * a.ps_r) == 0 &&
                    (a.N / (a.ps_r * a.ps_r)) % 8 == 0 && a.ldo_bf16 >= a.N / (a.ps_r * a.ps_r),
                "gemm_tc: pixel-shuffle store needs a 16-bit-only conv epilogue with N %% r^2 == 0 and N / r^2 %% 8 == 0");
  if (a.out_nchw)
    GRL_REQUIRE(conv && p.epi == EPI_BIAS_ACT && a.nchw_r >= 1 && a.N_f32 % (a.nchw_r * a.nchw_r) == 0 &&
                    a.N_f32 / (a.nchw_r * a.nchw_r) <= 4 && a.Hc > 0 && a.Wc > 0,
                "gemm_tc: NCHW tail store needs a conv with <= 4 output channels");
  GRL_REQUIRE(p.taps == 1 || p.taps == 9, "gemm_tc: taps must be 1 or 9");
  // Epilogue mode.  fp32 staging (LayerNorm, fp32 output, residual) needs the whole output row in one tile, 16-byte
  // aligned fp32 rows and a tile that fits the staging area; anything else with an fp32 side takes the direct path.
  a.epi_mode = 0;
  if (p.epi == EPI_LN || (p.epi == EPI_BIAS_ACT && (a.out_f32 || a.res_f32))) {
    const int cw = p.epi == EPI_LN ? a.C : a.N_f32;
    const int cap = bn == 64 ? GemmSmem<64>::OFF_TOK : bn == 128 ? GemmSmem<128>::OFF_TOK : bn == 192 ? GemmSmem<192>::OFF_TOK
                                                                                                     : GemmSmem<256>::OFF_TOK;
    const int cap_p = bn == 64 ? GemmSmem<64>::STG : bn == 128 ? GemmSmem<128>::STG : bn == 192 ? GemmSmem<192>::STG : GemmSmem<256>::STG;
    if (persistent && kBM * stage_pitch32(cw > 0 ? cw : 4) * 4 > cap_p) persistent = false;  // its staging tile is smaller
    const bool ok = bn != 96 && p.npad <= bn && cw > 0 && cw % 4 == 0 && kBM * stage_pitch32(cw) * 4 <= cap &&
                    (!a.out_f32 || a.ldo_f32 % 4 == 0) && (!a.res_f32 || a.ldr % 4 == 0) &&
                    (!a.out_bf16 || a.ldo_bf16 % 4 == 0);
    GRL_REQUIRE(ok || p.epi != EPI_LN, "gemm_tc: LayerNorm epilogue needs C %% 4 == 0 and C <= 188 (got %d)", cw);
    a.epi_mode = ok ? 1 : 2;
  }
  if (a.out_nchw) a.epi_mode = 2;
  CUtensorMap tmA, tmB;
  int rc;
  dim3 grid;
  a.nk = p.kpad / kBK;
  a.taps = p.taps;
  if (conv) {
    cuuint64_t dims[4] = {(cuuint64_t)p.kpad, (cuuint64_t)p.W, (cuuint64_t)p.H, (cuuint64_t)p.B};
    cuuint64_t str[3] = {(cuuint64_t)p.kpad * 2, (cuuint64_t)p.W * p.kpad * 2, (cuuint64_t)p.H * p.W * p.kpad * 2};
    cuuint32_t box[4] = {(cuuint32_t)kBK, (cuuint32_t)kTW, (cuuint32_t)kTH, 1};
    if ((rc = make_map(&tmA, p.x, 4, dims, str, box, a.fmt)) != GRL_OK) return rc;
    a.H = p.H, a.W = p.W;
    a.tiles_x = ceil_div(p.W, kTW), a.tiles_y = ceil_div(p.H, kTH);
    a.M = (long long)p.B * p.H * p.W;
    a.n_tiles = ceil_div(p.npad, bn);
    GRL_REQUIRE((long long)a.tiles_x * a.tiles_y * p.B * a.n_tiles < (1ll << 31), "gemm_tc: grid too large");
    grid = dim3((unsigned)(a.tiles_x * a.tiles_y * p.B * a.n_tiles));
    a.total_tiles = (int)grid.x;
  } else {
    cuuint64_t dims[2] = {(cuuint64_t)p.kpad, (cuuint64_t)p.M};
    cuuint64_t str[1] = {(cuuint64_t)p.kpad * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)kBM};
    if ((rc = make_map(&tmA, p.x, 2, dims, str, box, a.fmt)) != GRL_OK) return rc;
    a.M = p.M;
    a.n_tiles = ceil_div(p.npad, bn);
    GRL_REQUIRE((long long)ceil_div(p.M, kBM) * a.n_tiles < (1ll << 31), "gemm_tc: grid too large");
    grid = dim3((unsigned)(ceil_div(p.M, kBM) * a.n_tiles));
    a.total_tiles = (int)grid.x;
  }
  if (a.M == 0) return GRL_OK;
  {
    cuuint64_t dims[2] = {(cuuint64_t)p.kpad * p.taps, (cuuint64_t)p.npad};
    cuuint64_t str[1] = {(cuuint64_t)p.kpad * p.taps * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)bn};
    if ((rc = make_map(&tmB, p.w, 2, dims, str, box, a.fmt)) != GRL_OK) return rc;
  }
  switch (p.epi) {
    case EPI_BIAS_ACT:
      return conv ? dispatch_bn<EPI_BIAS_ACT, true>(bn, tmA, tmB, a, grid, st, persistent)
                  : dispatch_bn<EPI_BIAS_ACT, false>(bn, tmA, tmB, a, grid, st, persistent);
    case EPI_QKV:
      GRL_REQUIRE(!conv, "gemm_tc: QKV epilogue is linear-only");
      return dispatch_bn<EPI_QKV, false>(bn, tmA, tmB, a, grid, st, persistent);
    case EPI_LN:
      GRL_REQUIRE(!conv, "gemm_tc: LN epilogue is linear-only");
      return dispatch_bn<EPI_LN, false>(bn, tmA, tmB, a, grid, st, persistent);
  }
  return fail(GRL_ERR_INVALID, "gemm_tc: unknown epilogue %d", p.epi);
}

template <int NLN>
static int launch_mlp_one(const CUtensorMap& tmA, const CUtensorMap& tmW1, const CUtensorMap& tmW2, const MlpTcArgs& m,
                          cudaStream_t st) {
  auto kern = mlp_tcp_kernel<NLN>;
  static bool configured[kMaxDevices] = {false};
  int dev = 0;
  GRL_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices || !configured[dev]) {
    GRL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, MlpSmem<NLN>::TOTAL));
    if (dev >= 0 && dev < kMaxDevices) configured[dev] = true;
  }
  const unsigned grid = (unsigned)std::min(sm_count(), m.ep.total_tiles);
  kern<<<grid, kThreadsM, MlpSmem<NLN>::TOTAL, st>>>(tmA, tmW1, tmW2, m);
  GRL_LAUNCH_CHECK("mlp_tcp_kernel");
  return GRL_OK;
}

// x: 16-bit (M, cpad); w1: (hpad, cpad); w2: (n_ln, hpad), both K-major (the BlockPlan packing of fc1 / fc2).
int launch_mlp_tc(const MlpTcProblem& p, GemmTcArgs a, cudaStream_t st) {
  GRL_REQUIRE(p.n_ln == 64 || p.n_ln == 128 || p.n_ln == 192, "tc_mlp: n_ln must be 64, 128 or 192 (got %d)", p.n_ln);
  GRL_REQUIRE(p.cpad % kBK == 0 && p.cpad > 0 && p.cpad <= p.n_ln, "tc_mlp: cpad %d must be a multiple of 64 and <= n_ln %d",
              p.cpad, p.n_ln);
  GRL_REQUIRE(p.hpad % 64 == 0 && p.hpad > 0, "tc_mlp: hidden pad %d must be a positive multiple of 64", p.hpad);
  const int stg = p.n_ln == 64 ? MlpSmem<64>::STG : p.n_ln == 128 ? MlpSmem<128>::STG : MlpSmem<192>::STG;
  GRL_REQUIRE(a.C > 0 && a.C % 4 == 0 && a.C <= p.cpad && kBM * stage_pitch32(a.C) * 4 <= stg,
              "tc_mlp: LayerNorm epilogue needs C %% 4 == 0 and C <= 188, C <= cpad (got C=%d, cpad=%d)", a.C, p.cpad);
  GRL_REQUIRE(p.M >= 0 && (p.M + kBM - 1) / kBM < (1ll << 31), "tc_mlp: bad row count %lld", p.M);
  a.M = p.M;
  a.total_tiles = (int)((p.M + kBM - 1) / kBM);
  if (a.M == 0) return GRL_OK;
  CUtensorMap tmA, tmW1, tmW2;
  int rc;
  {
    cuuint64_t dims[2] = {(cuuint64_t)p.cpad, (cuuint64_t)p.M};
    cuuint64_t str[1] = {(cuuint64_t)p.cpad * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)kBM};
    if ((rc = make_map(&tmA, p.x, 2, dims, str, box, a.fmt)) != GRL_OK) return rc;
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)p.cpad, (cuuint64_t)p.hpad};
    cuuint64_t str[1] = {(cuuint64_t)p.cpad * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBK, 64};
    if ((rc = make_map(&tmW1, p.w1, 2, dims, str, box, a.fmt)) != GRL_OK) return rc;
  }
  {
    cuuint64_t dims[2] = {(cuuint64_t)p.hpad, (cuuint64_t)p.n_ln};
    cuuint64_t str[1] = {(cuuint64_t)p.hpad * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)p.n_ln};
    if ((rc = make_map(&tmW2, p.w2, 2, dims, str, box, a.fmt)) != GRL_OK) return rc;
  }
  MlpTcArgs m;
  m.ep = a;
  m.bias1 = p.b1;
  m.nk1 = p.cpad / kBK;
  m.nj = p.hpad / 64;
  switch (p.n_ln) {
    case 64: return launch_mlp_one<64>(tmA, tmW1, tmW2, m, st);
    case 128: return launch_mlp_one<128>(tmA, tmW1, tmW2, m, st);
    default: return launch_mlp_one<192>(tmA, tmW1, tmW2, m, st);
  }
}

}  // namespace tc
}  // namespace grl
