// attn2.cu -- persistent, warp-specialised fused cosine attention for sm_100a (WindowAttention and both passes of
// AnchorStripeAttention; mixed_attn_block_efficient.py:77-94,:128-165,:215-270).  Same math and operands as attn_tc.cu
// (packed 16-bit head slots, q^ / k^ pre-normalised and pre-scaled, log2-domain bias table); different machine mapping:
//
//   * one CTA per SM, persistent over work items (window|stripe, head, group of NWG query tiles of 128 rows);
//   * NWG softmax warpgroups share every K / V tile: K_t / V_t travel global -> shared ONCE per NWG*128 queries, as TMA
//     boxes of the (B, H, W, C) tensors (a run of gcd(window width, shift) tokens stays contiguous under torch.roll);
//   * S = Q K^T lands in TMEM; the softmax thread (one query row = one TMEM lane) turns it into P IN PLACE
//     (tcgen05.ld -> exp2 -> tcgen05.st): P never touches shared memory and P V reads its A operand from TMEM;
//   * O accumulates in TMEM across key tiles (tcgen05.mma accumulate); the running-max rescale is LAZY: O is touched
//     by the softmax warps only when a row's maximum grew by more than 2^8 since its reference was fixed, which is
//     rare after the first tile -- the 32-register output accumulator and its per-tile fold are gone;
//   * the softmax is ONE pass per tile with speculative exponentials (the lazy rescale makes the reference known before the
//     row maximum of the tile is): tcgen05.ld / bias LDS / packed FADD2 / FMNMX3 / MUFU.EX2 / pack as straight-line code;
//   * measured (DESIGN.md 5.3): at head_dim 32 neither the tensor pipe (11 % active) nor the exp2 unit (47 %) binds, the
//     SM's LSU / TMEM data path does -- 80 KB per 128 x 64 score tile for S out of TMEM, P back and the bias from shared memory.
//
// Roles (threads = NWG * 128 + 64): warpgroups 0..NWG-1 softmax; warp 4 NWG = TMA producer; warp 4 NWG + 1 = the MMA issuer (one
// elected thread issues every tcgen05.mma; GRL_A2_MULTI_ISSUER builds one issuer warp per warpgroup instead: no faster).
// (No setmaxnreg: the register pool of a CTA is what its own warps release.)
//
// TMEM columns per warpgroup g (base 160 g): [0, 64) = S buffer 0, [64, 128) = S buffer 1, [128, 160) = O_g.  S_g(t) lands
// in buffer t & 1 and is overwritten in place by P_g(t) (16-bit pairs in the first 32 columns of the buffer).  Q K^T runs
// TWO tiles ahead of the softmax: the issuer sends  P V_g(t) ; Q K^T_g(t+2)  back to back -- both touch buffer t & 1, and
// the tensor pipe executes one thread's MMAs in issue order, so the second overwrites what the first has read -- which
// means S_g(t+1) is already complete when the softmax warps finish tile t: they never wait for the MMA round trip.
#include <type_traits>
#include <stdlib.h>

#include <algorithm>

#include "attn_tc.cuh"
#include "grl_common.cuh"
#include "ops_f32.h"
#include "ops_tc.h"
#include "tc_common.cuh"

namespace grl {
namespace tc {

namespace {

// ---- differential-timing builds (tools/attn2_diag.py): each GRL_A2_DIAG_* define removes ONE ingredient so that its cost
// shows up as a time difference.  Results of such builds are WRONG by construction; the default build defines none.
#ifdef GRL_A2_DIAG_NOBIAS
#define A2_BIAS(expr) make_float4(0.f, 0.f, 0.f, 0.f)
#else
#define A2_BIAS(expr) (expr)
#endif
#ifdef GRL_A2_DIAG_NOEXP
#define A2_EX2(x) (x)
#else
#define A2_EX2(x) ex2(x)
#endif
#ifdef GRL_A2_DIAG_NOLDTM
#define A2_LDTM(stmt)
#else
#define A2_LDTM(stmt) stmt
#endif
#ifdef GRL_A2_DIAG_NOSTTM
#define A2_STTM(stmt)
#else
#define A2_STTM(stmt) stmt
#endif
#ifdef GRL_A2_DIAG_NOPV
#define A2_PV(stmt)
#else
#define A2_PV(stmt) stmt
#endif
#ifdef GRL_A2_DIAG_NOQK
#define A2_QK(stmt)
#else
#define A2_QK(stmt) stmt
#endif
#ifdef GRL_A2_DIAG_NOKVCOMMIT
#define A2_KVCOMMIT(bar) mbar_arrive(bar)
#else
#define A2_KVCOMMIT(bar) umma_commit(bar)
#endif
#ifdef GRL_A2_DIAG_ONEBOX  // the producer issues ONE box per Q / K / V tile (garbage data): what does TMA issue cost?
#define A2_BOXCNT(cnt, bw) min((cnt), (bw))
#else
#define A2_BOXCNT(cnt, bw) (cnt)
#endif
#ifdef GRL_A2_DIAG_NOMAX
#define A2_MAX(expr) 0.f
#else
#define A2_MAX(expr) (expr)
#endif

constexpr int kKT2 = 64;       // keys per tile
constexpr float kTau = 8.0f;   // lazy-rescale threshold (log2 units): P <= 2^8 stays far inside fp16 / bf16 range
constexpr int kColsPerWg = 160;  // TMEM columns per warpgroup: S buffer 0 | S buffer 1 | O

constexpr int kMaxStages2 = 16;

// Shared memory (bytes): [Q tiles NWG x 8 KB][barriers 1 KB][koff / rid 8 KB][K ring NS x 4 KB][V ring NS x 4 KB][bias table].
// The ring depth NS is chosen at launch from what is left of the 227 KB: tiles t .. t+2 are live in the MMA pipeline, the
// rest is prefetch distance -- a K / V tile comes from HBM / L2 through TMA in ~1.6 us, so a shallow ring bounds the
// whole kernel by that latency (measured: 5 stages -> every variant of the kernel, even one without any math, took ~1 ms).
template <int NWG>
struct A2Smem {
  static constexpr int Q_BYTES = kQT * 64;
  static constexpr int KV_BYTES = kKT2 * 64;
  static constexpr int OFF_BAR = NWG * Q_BYTES;
  static constexpr int OFF_META = OFF_BAR + 1024;                            // int koff[16][KT], krid[16][KT]
  static constexpr int OFF_K = OFF_META + kMaxStages2 * 2 * kKT2 * 4;
  static constexpr int FIXED = OFF_K + 1024;                                 // + alignment slack
  __host__ __device__ static constexpr int off_v(int ns) { return OFF_K + ns * KV_BYTES; }
  __host__ __device__ static constexpr int off_bias(int ns) { return OFF_K + 2 * ns * KV_BYTES; }
  __host__ __device__ static constexpr int total(int ns, int bias_bytes) { return FIXED + 2 * ns * KV_BYTES + bias_bytes; }
};

struct A2Geom {
  int bw_q, bw_k;   // tokens per TMA box
  int n_qg;         // query groups (NWG * 128 rows) per window
  int per_head;     // B * windows * n_qg work items per head; CTA b works on head b / (gridDim / heads)
  int stages;       // K / V ring depth
  int ntiles;       // key tiles per window: ceil(Nk / 64) (host-computed: one constant load instead of a divide chain per tile)
};

// Lean mbarrier wait: mbarrier.try_wait suspends the thread in hardware until the phase completes or a system time limit
// passes, so the retry loop is two instructions.  A wall-clock bound (checked every 4096 retries) turns a protocol bug into
// a recorded diagnosis instead of a hung GPU: the first waiter that times out writes (site, block, warp, parity) to
// g_a2_dbg and raises an abort flag; every wait then falls through, the kernel finishes with garbage and the host can
// read the record (grl_tc_attn2_debug).
__device__ int g_a2_dbg[8];
__device__ __forceinline__ void mbar_wait2_sa(uint32_t bar_sa, uint32_t parity, int site = 0) {  // bar_sa: shared-window address
  uint32_t ok;
  int spins = 0;
  long long t0 = 0;
  for (;;) {
#ifdef GRL_A2_SPIN  // A/B: non-blocking test_wait in a spin loop instead of the hardware-suspended try_wait
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar_sa), "r"(parity)
        : "memory");
#else
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar_sa), "r"(parity)
        : "memory");
#endif
    if (ok) return;
    if ((++spins & 4095) == 0) {
      if (*reinterpret_cast<volatile int*>(&g_a2_dbg[0]) != 0) return;  // somebody timed out: drain
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 1000000000ll) {
        if (atomicCAS(&g_a2_dbg[0], 0, 1) == 0) {
          g_a2_dbg[1] = site, g_a2_dbg[2] = blockIdx.x, g_a2_dbg[3] = threadIdx.x >> 5, g_a2_dbg[4] = (int)parity;
          g_a2_dbg[5] = (int)(bar_sa & 0xffff);
          __threadfence();
        }
        return;
      }
    }
  }
}

__device__ __forceinline__ void mbar_wait2(uint64_t* bar, uint32_t parity, int site = 0) { mbar_wait2_sa(smem_u32(bar), parity, site); }
__device__ __forceinline__ void mbar_arrive_sa(uint32_t bar_sa) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_sa) : "memory");
}

// Warp-collective wait (call sites are warp-uniform).
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity, int site = 0) {
#ifdef GRL_A2_ONE_LANE_POLL  // measured slightly slower than letting every lane poll (the warp instruction is one request)
  if ((threadIdx.x & 31) == 0) mbar_wait2(bar, parity, site);
  __syncwarp();
#else
  mbar_wait2(bar, parity, site);
#endif
}

// Waits of the producer / issuer warps: they are off the softmax warps' critical path (deep K / V ring, S two tiles ahead),
// so they may sleep in hardware (try_wait with a suspend-time hint) instead of polling next to the warps doing the math.
__device__ __forceinline__ void mbar_wait_bg(uint64_t* bar, uint32_t parity, int site = 0) {
#ifdef GRL_A2_BG_SLEEP
  mbar_wait(bar, parity);
#else
  mbar_wait2(bar, parity, site);
#endif
}

// shared-memory loads by 32-bit shared address (the tile base is aligned through integer arithmetic, after which the
// compiler only sees a generic pointer and would emit generic LD instead of LDS)
__device__ __forceinline__ float4 lds128(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}
__device__ __forceinline__ float lds32f(uint32_t saddr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(saddr));
  return v;
}
__device__ __forceinline__ int lds32i(uint32_t saddr) {
  int v;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(saddr));
  return v;
}

// packed fp32 pairs (sm_100 FADD2: two adds per issued instruction; the softmax warps are issue / latency bound)
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
  return d;
}
__device__ __forceinline__ float lo2(uint64_t v) { return __uint_as_float((uint32_t)v); }
__device__ __forceinline__ float hi2(uint64_t v) { return __uint_as_float((uint32_t)(v >> 32)); }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// MMA issuer warps per CTA: one for every warpgroup (GRL_A2_MULTI_ISSUER, A/B build) or a single one (default)
template <int NWG>
__host__ __device__ constexpr int kIssuers2() {
#ifdef GRL_A2_MULTI_ISSUER
  return NWG;
#else
  return 1;
#endif
}

struct Item {
  int qg, h, bw, b, wr, wc, nact;
};

// position in the K / V ring: stage and the parity of the fill that is current for it
struct Ring {
  int st;
  uint32_t ph;
  __device__ __forceinline__ void adv(int ns) {
    if (++st == ns) st = 0, ph ^= 1u;
  }
  __device__ __forceinline__ void skip(int n, int ns) {  // n tiles at once (a warpgroup sitting an item out)
    const int tot = st + n;
    ph ^= (uint32_t)(tot / ns) & 1u;
    st = tot % ns;
  }
};

template <int NWG, int KW, int VAR, bool BS>
__global__ void __launch_bounds__(NWG * 128 + 32 + kIssuers2<NWG>() * 32, 1)
attn2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
             const __grid_constant__ CUtensorMap tmV, const AttnTcArgs a, const A2Geom tg) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  using S = A2Smem<NWG>;
  constexpr int KT = kKT2;
  const int NS = tg.stages;
  uint8_t* Qs = smem;
  uint8_t* Ks = smem + S::OFF_K;
  uint8_t* Vs = smem + S::off_v(NS);
  int* koff_s = reinterpret_cast<int*>(smem + S::OFF_META);  // [16][KT]
  int* krid_s = koff_s + kMaxStages2 * KT;                    // [16][KT]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* q_full = bars;                  // [NWG]  Q tile of warpgroup g landed            (TMA tx)
  uint64_t* q_empty = q_full + 4;           // [NWG]  every Q K^T of the item that reads it is done  (tcgen05.commit)
  uint64_t* bar_s = q_empty + 4;            // [NWG][2]  buffer t & 1: S_g(t) ready / P V_g(t-2) done; every tile commits once
  uint64_t* p_full = bar_s + 8;             // [NWG][2]  P_g(t) written to TMEM, buffer t & 1    (4 warp arrivals)
  uint64_t* item_done = p_full + 8;         // [NWG]  warpgroup g has consumed the item's closing completions (4 warp arrivals)
  uint64_t* kv_full = item_done + 4;           // [NS]  K_t, V_t landed                       (TMA tx)
  uint64_t* kv_empty = kv_full + kMaxStages2;  // [NS]  every MMA that reads the stage is done (tcgen05.commit)
  uint64_t* meta_full = kv_empty + kMaxStages2;  // [NS]  koff / rid of the stage written      (32 arrivals)
  uint64_t* bias_full = meta_full + kMaxStages2;      // the head's bias table landed in shared memory (BS)   (bulk-copy tx)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bias_full + 1);
  float* bias_s = reinterpret_cast<float*>(smem + S::off_bias(NS));

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wg = warp >> 2;
  const int Nq = a.gq.wh * a.gq.ww, Nk = a.gk.wh * a.gk.ww;
  const int nww = a.gq.W / a.gq.ww, nwh = a.gq.H / a.gq.wh;
  const int nW = nwh * nww;
  const int Wt = a.gq.ww + a.gk.ww - 1;
  const int ntiles = tg.ntiles;
  static_assert(NWG * kColsPerWg <= 512, "two S buffers + O per warpgroup: at most 3 warpgroups fit the 512 TMEM columns");
  constexpr uint32_t TMEM_COLS = (NWG * kColsPerWg <= 128) ? 128 : (NWG * kColsPerWg <= 256) ? 256 : 512;
  constexpr int fmt = (VAR & 1) ? FMT_BF16 : FMT_F16;
  constexpr bool ones = (VAR & 2) != 0;

  if (tid == 0) {
    for (int g = 0; g < NWG; ++g) {
      mbar_init(&q_full[g], 1);
      mbar_init(&q_empty[g], 1);
      mbar_init(&bar_s[2 * g], 1);
      mbar_init(&bar_s[2 * g + 1], 1);
      mbar_init(&p_full[2 * g], 4);
      mbar_init(&p_full[2 * g + 1], 4);
      mbar_init(&item_done[g], 4);
    }
    for (int s = 0; s < NS; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], kIssuers2<NWG>());
      mbar_init(&meta_full[s], 1);
    }
    mbar_init(bias_full, 1);
    mbar_init_fence();
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
  }
  if (warp == 4 * NWG + 1) tmem_alloc(tmem_slot, TMEM_COLS);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;

  // Static head partition: CTA b serves head b / cph only (cph = CTAs per head), so a CTA needs ONE bias table for its
  // whole life -- it can live in shared memory (BS), and without BS the table stays hot in this SM's L1.
  const int cph = gridDim.x / a.heads;
  const int my_h = blockIdx.x / cph, my_c = blockIdx.x - my_h * cph;
  auto decode = [&](int idx) {
    Item it;
    it.qg = idx % tg.n_qg;
    it.bw = idx / tg.n_qg;
    it.h = my_h;
    it.b = it.bw / nW;
    const int w = it.bw - it.b * nW;
    it.wr = w / nww;
    it.wc = w - it.wr * nww;
    const int left = Nq - it.qg * NWG * kQT;
    it.nact = min(NWG, (left + kQT - 1) / kQT);
    return it;
  };

  if (warp >= 4 * NWG) {
    if (warp == 4 * NWG) {
      // =============================================================== TMA producer
      // A run of `bw` consecutive tokens of one window row is contiguous in the (B, H, W, C) tensor even after the
      // roll (bw divides gcd(window width, shift)), so it is ONE 4-D box (32 channels x bw x 1 x 1) that lands as bw
      // rows of 64 bytes, 64-byte swizzled by the copy engine -- the layout the UMMA descriptors below expect.
      // ONE lane issues every box, with running (row, column) coordinates: per-lane coordinates would make the compiler
      // serialise the warp into an elect / broadcast loop around each UTMALDG, and this warp -- not the tensor or the MUFU
      // pipe -- was what bounded an earlier version of the kernel (~2000 cycles per key tile).
      struct Cur {
        int ih, iw;
      };
      auto tma_run = [&](const CUtensorMap* m1, int c1, uint8_t* d1, const CUtensorMap* m2, int c2, uint8_t* d2,
                         const GrlGrid& g, const Item& it, Cur& cur, int cnt, int bw, uint64_t* bar) {  // lane 0
        const int yb = it.wr * g.wh + g.sh, xb = it.wc * g.ww + g.sw;
        for (int n = 0; n < A2_BOXCNT(cnt, bw); n += bw) {
          int y = yb + cur.ih, x = xb + cur.iw;
          if (y >= g.H) y -= g.H;
          if (x >= g.W) x -= g.W;
          tma_load_4d(d1 + n * 64, m1, bar, c1, x, y, it.b);
          if (m2) tma_load_4d(d2 + n * 64, m2, bar, c2, x, y, it.b);
          cur.iw += bw;
          if (cur.iw >= g.ww) cur.iw = 0, ++cur.ih;
        }
      };
      const bool mask_fast_p = (KW > 0) && (a.gk.sw == 0 || ((a.gk.ww - a.gk.sw) & 3) == 0);
      uint32_t kv_it = 0, q_cnt[NWG];
      Ring rp = {0, 0};
#pragma unroll
      for (int g = 0; g < NWG; ++g) q_cnt[g] = 0;
      if (BS && elect_one()) {  // the head's table: 4 shifted copies, contiguous in global memory, one bulk copy
        const uint32_t bytes = 16u * (uint32_t)a.rows_pad;
        mbar_expect_tx(bias_full, bytes);
        bulk_load_1d(bias_s, a.bias + (size_t)my_h * 4 * a.rows_pad, bytes, bias_full);
      }
      for (int item = my_c; item < tg.per_head; item += cph) {
        const Item it = decode(item);
        const bool need_mask = a.use_mask && (it.wr == nwh - 1 || it.wc == nww - 1);
#pragma unroll
        for (int g = 0; g < NWG; ++g) {
          if (g < it.nact) {
            mbar_wait_bg(&q_empty[g], (q_cnt[g] & 1) ^ 1, 1);
            ++q_cnt[g];
            const int q0 = (it.qg * NWG + g) * kQT;
            const int cnt = min(kQT, Nq - q0);
            if (elect_one()) {
              mbar_expect_tx(&q_full[g], (uint32_t)A2_BOXCNT(cnt, tg.bw_q) * 64u);
              Cur cq = {q0 / a.gq.ww, q0 % a.gq.ww};
              tma_run(&tmQ, a.q_off + it.h * kDP, Qs + g * S::Q_BYTES, nullptr, 0, nullptr, a.gq, it, cq, cnt, tg.bw_q, &q_full[g]);
            }
            __syncwarp();
          }
        }
        Cur ck = {0, 0};  // in-window (row, column) of the first key of the next tile
        for (int t = 0; t < ntiles; ++t, ++kv_it, rp.adv(NS)) {
          const int st = rp.st;
          mbar_wait_bg(&kv_empty[st], rp.ph ^ 1, 2);
          const int k0 = t * KT, cnt = min(KT, Nk - k0);
          uint8_t* kd = Ks + st * S::KV_BYTES;
          uint8_t* vd = Vs + st * S::KV_BYTES;
          if (cnt < KT && !a.v_dense) {  // ragged tile: V rows past Nk meet P == 0 and must be finite
            for (int i = lane; i < (KT - cnt) * 4; i += 32) *reinterpret_cast<uint4*>(vd + cnt * 64 + i * 16) = make_uint4(0, 0, 0, 0);
            fence_proxy_async_smem();
          }
          // koff / rid of the keys: read by the generic bias path (ragged tile, KW == 0) and by the shift mask
          if ((need_mask && !mask_fast_p) || KW == 0 || cnt < KT) {
            for (int r = lane; r < KT; r += 32) {
              const int kj = k0 + r;
              const Tok tk = locate(a.gk, it.wr, it.wc, kj < Nk ? kj : 0);
              koff_s[st * KT + r] = tk.ih * Wt + tk.iw;
              krid_s[st * KT + r] = region_id(a.gk, tk.r, tk.c);
            }
          }
          __syncwarp();  // every lane's koff / rid stores are ordered before lane 0's release
          if (elect_one()) mbar_arrive(&meta_full[st]);
          if (elect_one()) {
            mbar_expect_tx(&kv_full[st], (uint32_t)(A2_BOXCNT(cnt, tg.bw_k) + (a.v_dense ? KT : A2_BOXCNT(cnt, tg.bw_k))) * 64u);
            if (a.v_dense) {  // V = (B_, heads, Nk, 32) rows: one 2-D box (rows past this head's Nk: next head / zero fill, P == 0)
              tma_run(&tmK, a.k_off + it.h * kDP, kd, nullptr, 0, nullptr, a.gk, it, ck, cnt, tg.bw_k, &kv_full[st]);
              tma_load_2d(vd, &tmV, &kv_full[st], 0, (int)(((long long)it.bw * a.heads + it.h) * Nk + k0));
            } else {  // K and V rows of a token sit in the same tensor: same coordinates, two channel offsets
              tma_run(&tmK, a.k_off + it.h * kDP, kd, &tmV, a.v_off + it.h * kDP, vd, a.gk, it, ck, cnt, tg.bw_k, &kv_full[st]);
            }
          }
          __syncwarp();
        }
      }
#ifdef GRL_A2_MULTI_ISSUER
    } else if (warp <= 4 * NWG + NWG) {
      // =============================================================== MMA issuers: one warp (one thread) per warpgroup.
      // Each issuer owns the MMAs of ONE warpgroup (the ordering the S / P aliasing needs is within a warpgroup); all of
      // them release the K / V stages (kv_empty counts NWG).  After EVERY tile t the issuer commits to bar_s[t & 1]:
      // that completion means "P V(t) done and, if it exists, S(t+2) ready".  The softmax warps consume these completions
      // strictly in order per buffer, so every parity wait is exact; the two completions past the last tile are the
      // "O final" signal.  Nothing on the softmax warps' critical path waits for an MMA that was issued in the same tile.
      const int g = warp - (4 * NWG + 1);
      const uint32_t idesc_qk = umma_idesc(kQT, KT, fmt, 0, 0);
      const uint32_t idesc_pv = umma_idesc(kQT, kDP, fmt, 0, 1);
      // descriptors: only the 14-bit start-address field (16-byte units) changes between uses
      const uint64_t q_desc = umma_desc(smem_u32(Qs + g * S::Q_BYTES), 16, 512, SWZ_64B);
      const uint64_t k_desc0 = umma_desc(smem_u32(Ks), 16, 512, SWZ_64B);
      const uint64_t v_desc0 = umma_desc(smem_u32(Vs), 16, 512, SWZ_64B);
      const uint32_t wg_ta = tmem + g * kColsPerWg;
      uint32_t kv_it = 0, q_cnt = 0, p_par = 0, d_cnt = 0;  // p_par: bit b = parity to wait for on p_full[2 g + b]
      Ring r0 = {0, 0}, r2 = {0, 0}, rl = {0, 0};  // tile t, tile t + 2, last tile handled
      r2.adv(NS);
      r2.adv(NS);
      auto issue_qk = [&](int st, int buf, bool last) {  // lane 0
        const uint64_t kd = k_desc0 + (uint64_t)(st * (S::KV_BYTES >> 4));
        A2_QK(umma_ss(wg_ta + buf * 64, q_desc, kd, idesc_qk, false));
        A2_QK(umma_ss(wg_ta + buf * 64, q_desc + 2, kd + 2, idesc_qk, true));
        if (last) umma_commit(&q_empty[g]);
      };
      for (int item = my_c; item < tg.per_head; item += cph) {
        const Item it = decode(item);
        const bool active = g < it.nact;
        if (active) {
          mbar_wait_bg(&q_full[g], q_cnt & 1, 3);
          ++q_cnt;
        }
        // prologue: S_g(0) and S_g(1)
        Ring rq = r0;  // ring position of tile t0
        for (int t0 = 0; t0 < 2 && t0 < ntiles; ++t0, rq.adv(NS)) {
          const int st = rq.st;
          mbar_wait_bg(&kv_full[st], rq.ph, 4);
          if (active && elect_one()) {
            tcgen05_fence_after();
            issue_qk(st, t0, t0 + 1 == ntiles);
            umma_commit(&bar_s[2 * g + t0]);
          }
          __syncwarp();
        }
        if (ntiles == 1 && active && elect_one()) umma_commit(&bar_s[2 * g + 1]);  // keep both buffers' counts in step
        __syncwarp();
        for (int t = 0; t < ntiles; ++t, ++kv_it, rl = r0, r0.adv(NS), r2.adv(NS)) {
          const int st = r0.st, st2 = r2.st;
          if (t + 2 < ntiles) mbar_wait_bg(&kv_full[st2], r2.ph, 5);
          if (active) {
            // (per S buffer: the softmax warps run up to two tiles ahead of this thread, and an mbarrier that completes
            // twice before its waiter has looked is indistinguishable from one that has not completed)
            mbar_wait_bg(&p_full[2 * g + (t & 1)], (p_par >> (t & 1)) & 1u, 6);
            p_par ^= 1u << (t & 1);
            if (elect_one()) {
              tcgen05_fence_after();
              const uint64_t vd = v_desc0 + (uint64_t)(st * (S::KV_BYTES >> 4));
              const uint32_t p_ta = wg_ta + (t & 1) * 64;
#pragma unroll
              for (int k = 0; k < KT / 16; ++k) A2_PV(umma_ts(wg_ta + 128, p_ta + k * 8, vd + (uint64_t)(k * 64), idesc_pv, (t | k) != 0));
              if (t + 2 < ntiles) issue_qk(st2, t & 1, t + 3 == ntiles);
              umma_commit(&bar_s[2 * g + (t & 1)]);  // P V(t) done (+ S(t+2) ready)
              A2_KVCOMMIT(&kv_empty[st]);            // every MMA of this warpgroup that reads stage st has been issued
            }
          } else if (elect_one()) {
            mbar_arrive(&kv_empty[st]);  // sitting this item out: release the stage (after its fill: kv_full(st2) / prologue waits)
          }
          __syncwarp();
        }
        if (active) {  // the warpgroup has consumed this item's closing completions of bar_s (see its epilogue)
          mbar_wait_bg(&item_done[g], d_cnt & 1, 7);
          ++d_cnt;
        }
      }
      // every commit has arrived before the CTA's shared memory goes away (kv_empty needs all NWG issuers)
      if (kv_it > 0) mbar_wait_bg(&kv_empty[rl.st], rl.ph, 8);
    }
#else
    } else if (warp == 4 * NWG + 1) {
      // =============================================================== MMA issuer: ONE warp (one thread) serves every
      // warpgroup in turn (measured ~10 % faster end to end than one issuer warp per warpgroup: fewer warps polling next
      // to the softmax warps).  After EVERY tile t of warpgroup g it commits to bar_s[g][t & 1] ("P V(t) done and, if it
      // exists, S(t+2) ready"); the softmax warps consume these completions strictly in order per buffer, so every parity
      // wait is exact; the two completions past the last tile are the "O final" signal.
      const uint32_t idesc_qk = umma_idesc(kQT, KT, fmt, 0, 0);
      const uint32_t idesc_pv = umma_idesc(kQT, kDP, fmt, 0, 1);
      // descriptors: only the 14-bit start-address field (16-byte units) changes between uses
      const uint64_t q_desc0 = umma_desc(smem_u32(Qs), 16, 512, SWZ_64B);
      const uint64_t k_desc0 = umma_desc(smem_u32(Ks), 16, 512, SWZ_64B);
      const uint64_t v_desc0 = umma_desc(smem_u32(Vs), 16, 512, SWZ_64B);
      // parities to wait for, one bit per barrier (arrays indexed by t & 1 would live in local memory)
      uint32_t kv_it = 0, q_par = 0, p_par = 0, d_par = 0;
      Ring r0 = {0, 0}, r2 = {0, 0}, rl = {0, 0};  // tile t, tile t + 2, last tile handled
      r2.adv(NS);
      r2.adv(NS);
      auto issue_qk = [&](int g, int st, int buf, bool last) {  // lane 0
        const uint64_t qd = q_desc0 + (uint64_t)(g * (S::Q_BYTES >> 4));
        const uint64_t kd = k_desc0 + (uint64_t)(st * (S::KV_BYTES >> 4));
        A2_QK(umma_ss(tmem + g * kColsPerWg + buf * 64, qd, kd, idesc_qk, false));
        A2_QK(umma_ss(tmem + g * kColsPerWg + buf * 64, qd + 2, kd + 2, idesc_qk, true));
        if (last) umma_commit(&q_empty[g]);
      };
      for (int item = my_c; item < tg.per_head; item += cph) {
        const Item it = decode(item);
        // prologue: S_g(0) and S_g(1)
        Ring rq = r0;  // ring position of tile t0
        for (int t0 = 0; t0 < 2 && t0 < ntiles; ++t0, rq.adv(NS)) {
          const int st = rq.st;
          mbar_wait_bg(&kv_full[st], rq.ph, 4);
#pragma unroll
          for (int g = 0; g < NWG; ++g) {
            if (g < it.nact) {
              if (t0 == 0) {
                mbar_wait_bg(&q_full[g], (q_par >> g) & 1u, 3);
                q_par ^= 1u << g;
              }
              if (elect_one()) {
                tcgen05_fence_after();
                issue_qk(g, st, t0, t0 + 1 == ntiles);
                umma_commit(&bar_s[2 * g + t0]);
                if (ntiles == 1) umma_commit(&bar_s[2 * g + 1]);  // keep both buffers' counts in step
              }
              __syncwarp();
            }
          }
        }
        for (int t = 0; t < ntiles; ++t, ++kv_it, rl = r0, r0.adv(NS), r2.adv(NS)) {
          const int st = r0.st, st2 = r2.st;
          if (t + 2 < ntiles) mbar_wait_bg(&kv_full[st2], r2.ph, 5);
#ifndef GRL_A2_ILV  // default: one warpgroup after the other, each as soon as its P is there (the warpgroups need not run in step)
#pragma unroll
          for (int g = 0; g < NWG; ++g) {
            if (g < it.nact) {
              mbar_wait_bg(&p_full[2 * g + (t & 1)], (p_par >> (2 * g + (t & 1))) & 1u, 6);
              p_par ^= 1u << (2 * g + (t & 1));
              if (elect_one()) {
                tcgen05_fence_after();
                const uint64_t vd = v_desc0 + (uint64_t)(st * (S::KV_BYTES >> 4));
                const uint32_t wg_ta = tmem + g * kColsPerWg;
                const uint32_t p_ta = wg_ta + (t & 1) * 64;
#pragma unroll
                for (int k = 0; k < KT / 16; ++k) A2_PV(umma_ts(wg_ta + 128, p_ta + k * 8, vd + (uint64_t)(k * 64), idesc_pv, (t | k) != 0));
                if (t + 2 < ntiles) issue_qk(g, st2, t & 1, t + 3 == ntiles);
                umma_commit(&bar_s[2 * g + (t & 1)]);  // P V(t) done (+ S(t+2) ready)
              }
              __syncwarp();
            }
          }
#else
          // (per S buffer: the softmax warps run up to two tiles ahead of this thread, and an mbarrier that completes
          // twice before its waiter has looked is indistinguishable from one that has not completed)
#pragma unroll
          for (int g = 0; g < NWG; ++g) {
            if (g < it.nact) {
              mbar_wait_bg(&p_full[2 * g + (t & 1)], (p_par >> (2 * g + (t & 1))) & 1u, 6);
              p_par ^= 1u << (2 * g + (t & 1));
            }
          }
          if (elect_one()) {
            // A/B build (GRL_A2_ILV): the MMAs of the three warpgroups interleaved k-step by k-step, so that consecutive
            // MMAs are independent.  Measured: no gain (1.71 vs 1.66 ms) -- the tensor pipe is not what the hand-off waits for.
            tcgen05_fence_after();
            const uint64_t vd = v_desc0 + (uint64_t)(st * (S::KV_BYTES >> 4));
            const uint64_t kd2 = k_desc0 + (uint64_t)(st2 * (S::KV_BYTES >> 4));
            const uint32_t bo = (uint32_t)(t & 1) * 64u;
#pragma unroll
            for (int k = 0; k < KT / 16; ++k) {
#pragma unroll
              for (int g = 0; g < NWG; ++g)
                if (g < it.nact) A2_PV(umma_ts(tmem + g * kColsPerWg + 128, tmem + g * kColsPerWg + bo + k * 8, vd + (uint64_t)(k * 64), idesc_pv, (t | k) != 0));
            }
            if (t + 2 < ntiles) {
#pragma unroll
              for (int k = 0; k < 2; ++k) {
#pragma unroll
                for (int g = 0; g < NWG; ++g)
                  if (g < it.nact) A2_QK(umma_ss(tmem + g * kColsPerWg + bo, q_desc0 + (uint64_t)(g * (S::Q_BYTES >> 4)) + 2 * k, kd2 + 2 * k, idesc_qk, k != 0));
              }
              if (t + 3 == ntiles) {
#pragma unroll
                for (int g = 0; g < NWG; ++g)
                  if (g < it.nact) umma_commit(&q_empty[g]);
              }
            }
#pragma unroll
            for (int g = 0; g < NWG; ++g)
              if (g < it.nact) umma_commit(&bar_s[2 * g + (t & 1)]);  // P V(t) done (+ S(t+2) ready)
          }
          __syncwarp();
#endif
          if (elect_one()) A2_KVCOMMIT(&kv_empty[st]);  // every MMA that reads stage st has been issued
          __syncwarp();
        }
#pragma unroll
        for (int g = 0; g < NWG; ++g) {
          if (g < it.nact) {  // the warpgroup has consumed this item's closing completions of bar_s (see its epilogue)
            mbar_wait_bg(&item_done[g], (d_par >> g) & 1u, 7);
            d_par ^= 1u << g;
          }
        }
      }
      // every commit has arrived before the CTA's shared memory goes away
      if (kv_it > 0) mbar_wait_bg(&kv_empty[rl.st], rl.ph, 8);
    }
#endif
  } else {
    // =============================================================== softmax warpgroups: thread = query row
    const int row = tid & 127;
#ifdef GRL_A2_SKEW  // A/B: start warpgroup g  g * GRL_A2_SKEW  cycles late, so that the warpgroups' MUFU / LSU phases do not coincide
    if (wg > 0) {
      const long long t_start = clock64();
      while (clock64() - t_start < (long long)wg * GRL_A2_SKEW) {
      }
    }
#endif
    uint32_t ts0 = tmem + ((uint32_t)((warp & 3) * 32) << 16) + wg * kColsPerWg;  // S / P buffer 0 of this row
    asm volatile("" : "+r"(ts0));  // opaque: kept in a register instead of being rebuilt from %tid (S2R + shifts) every tile
    const uint32_t to = ts0 + 128;                                                        // O columns
    bool bias_ready = false;
    const uint32_t bias_sa = smem_u32(bias_s), koff_sa = smem_u32(koff_s), krid_sa = smem_u32(krid_s);
    // shared-window addresses of this warpgroup's barriers, computed once (a generic pointer costs a window-base computation
    // per use: S2UR CgaCtaId / ULEA / ... on the per-tile critical path)
    const uint32_t bar_s_sa = smem_u32(&bar_s[2 * wg]), p_full_sa = smem_u32(&p_full[2 * wg]);
    uint32_t s_par = 0;  // bit b: parity of the next completion of bar_s[2 wg + b] (every tile consumes exactly one)
    Ring rs = {0, 0};
    for (int item = my_c; item < tg.per_head; item += cph) {
      const Item it = decode(item);
      if (wg >= it.nact) {
        rs.skip(ntiles, NS);
        continue;
      }
      const int qi = (it.qg * NWG + wg) * kQT + row;
      const bool q_ok = qi < Nq;
      const Tok tq = locate(a.gq, it.wr, it.wc, q_ok ? qi : it.qg * NWG * kQT);
      const float* bias_h = a.bias + (size_t)it.h * 4 * a.rows_pad;
      if (BS && !bias_ready) {
        mbar_wait_warp(bias_full, 0, 9);
        bias_ready = true;
      }
      const int base_i = (tq.ih + a.gk.wh - 1) * Wt + tq.iw + a.gk.ww - 1;
      const int q_rid = region_id(a.gq, tq.r, tq.c);
      // shift mask (ops.py:112-157): only windows of the last row / column carry one.  Region id of key (kh, kw) of this
      // window = 3 (a1 + [a1 & kh >= wh - sh]) + (b1 + [b1 & kw >= ww - sw])  (grl_geometry.h region_id in window coordinates)
      const bool a1 = it.wr == nwh - 1, b1 = it.wc == nww - 1;
      const bool need_mask = a.use_mask && (a1 || b1);
      const int kh_th = (a1 && a.gk.sh > 0) ? a.gk.wh - a.gk.sh : 0x7fffffff;  // first key row of the wrapped region
      const int kw_th = (b1 && a.gk.sw > 0) ? a.gk.ww - a.gk.sw : 0x7fffffff;  // first key column of the wrapped region
      // closed-form masks need every aligned group of 4 keys to lie on one side of kw_th
      const bool mask_fast = (KW > 0) && (a.gk.sw == 0 || ((a.gk.ww - a.gk.sw) & 3) == 0);
      float m_ref = 0.f, l_run = 0.f;

      for (int t = 0; t < ntiles; ++t, rs.adv(NS)) {
        const int k0 = t * KT, st = rs.st, buf = t & 1;
        const uint32_t ts = ts0 + buf * 64;
        const bool full_tile = (KW > 0) && (k0 + KT <= Nk);
        // Tiles whose bias row is a closed-form run (full tile of a rectangular window, mask absent or closed-form) of a table
        // that lives in SHARED memory take the single-pass path below; ragged tiles / metadata masks keep the two-phase path
        // after it, and so do tables read through L1 (BS == false: the 64 x 128 stripes of the denoising models, 290 KB):
        // the two-phase path has all 16 LDG.128 of a tile in flight before S is waited for, the chunked single pass would
        // expose the L1 / L2 latency four times per tile (measured: cfg3 290 -> 322 ms per step).
        const bool fastp = BS && full_tile && (!need_mask || mask_fast);
        uint32_t pk[32];
        if (fastp) {
          // ---- S_t
          mbar_wait2_sa(bar_s_sa + 8u * (uint32_t)buf, (s_par >> buf) & 1u, 10);
          s_par ^= 1u << buf;
          tcgen05_fence_after();
          // One pass over the tile in two 32-key chunks: x = S + bias (+ mask), running row maximum and -- SPECULATIVELY, with
          // the reference the row already has -- P = exp2(x - m_ref) packed to 16 bits.  The lazy rescale makes the speculation
          // pay: the reference moves on ~7 % of the tiles only, so the exponentials do not have to wait for the maximum and
          // the MUFU stream of one chunk overlaps the adds / maxima of the other (the two-phase version serialised
          // LDS -> FADD -> LDTM -> FADD -> FMNMX -> MUFU per warp; the warps, not the MUFU pipe, bounded the kernel).  When a
          // row does outgrow the reference the tile is simply recomputed from TMEM (S is still there: P overwrites it last).
          float ps = 0.f;
          auto pass = [&](const float mref, auto DO_EXP, auto MASKED) -> float {  // compile-time flags: straight-line code
            constexpr bool do_exp = decltype(DO_EXP)::value, masked = decltype(MASKED)::value;
            constexpr int KWS = KW > 0 ? KW : 32;
            float mxa = -INFINITY, mxb = -INFINITY, psa = 0.f, psb = 0.f;
            const uint64_t negm = pack2(-mref, -mref);
#pragma unroll
            for (int c0 = 0; c0 < KT; c0 += 16) {  // 16 consecutive keys of one key row (registers: P 32 + S 16 + bias 16)
              uint32_t v[16];
#ifdef GRL_A2_DIAG_NOLDTM
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = 0;
#else
              tmem_ld16(ts + c0, v);  // in flight while the bias run is fetched
#endif
              const int kj = k0 + c0;  // first key of the run (CTA-uniform, multiple of 16)
              const int kh = kj / KWS, kw0 = kj % KWS;
              const int s0 = base_i - (kh * Wt + kw0) - 3;  // table index of key kj + 3
              const int cpy = (-s0) & 3;
              const float4* bp = reinterpret_cast<const float4*>(bias_h + (size_t)cpy * a.rows_pad + (s0 + cpy));
              const uint32_t bps = bias_sa + (uint32_t)(cpy * a.rows_pad + (s0 + cpy)) * 4u;  // BS: LDS.128
              float bsv[16];
#pragma unroll
              for (int qd = 0; qd < 4; ++qd) {
                const float4 bb = A2_BIAS(BS ? lds128(bps - 16u * qd) : __ldg(bp - qd));
                bsv[4 * qd + 0] = bb.w, bsv[4 * qd + 1] = bb.z, bsv[4 * qd + 2] = bb.y, bsv[4 * qd + 3] = bb.x;
              }
              if (masked) {
                const int rid_lo = 3 * ((int)a1 + (int)(kh >= kh_th)) + (int)b1;
                const float off_lo = (rid_lo != q_rid) ? kMaskLog2 : 0.f;
                const float off_hi = (rid_lo + 1 != q_rid) ? kMaskLog2 : 0.f;
#pragma unroll
                for (int qd = 0; qd < 4; ++qd) {
                  const float off = (kw0 + 4 * qd >= kw_th) ? off_hi : off_lo;
#pragma unroll
                  for (int e = 0; e < 4; ++e) bsv[4 * qd + e] += off;
                }
              }
#ifndef GRL_A2_DIAG_NOLDTM
              tmem_ld_wait();
#endif
              uint64_t x2[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) x2[j] = add2(pack2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), pack2(bsv[2 * j], bsv[2 * j + 1]));
#pragma unroll
              for (int j = 0; j < 8; j += 2) {
                mxa = fmax3(mxa, lo2(x2[j]), hi2(x2[j]));
                mxb = fmax3(mxb, lo2(x2[j + 1]), hi2(x2[j + 1]));
              }
              if (do_exp) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const uint64_t y = add2(x2[j], negm);
                  const float p0 = A2_EX2(lo2(y)), p1 = A2_EX2(hi2(y));
                  if (!ones) psa += p0, psb += p1;
                  pk[c0 / 2 + j] = (fmt == FMT_BF16) ? pack_bf16(p0, p1) : pack_f16(p0, p1);
                }
              }
            }
            ps = psa + psb;
            return A2_MAX(fmaxf(mxa, mxb));
          };
          const bool first = (t == 0);
          auto tile = [&](auto MASKED) {
            using T = std::true_type;
            using F = std::false_type;
            // (no reference yet on the first tile of an item: maximum only)
            const float mx = first ? pass(m_ref, F{}, MASKED) : pass(m_ref, T{}, MASKED);
            if (__any_sync(0xffffffffu, first || mx - m_ref > kTau)) {
              float delta = first ? mx : fmaxf(mx - m_ref, 0.f);
              if (!(fabsf(delta) < 1e30f)) delta = 0.f;  // rows of a partial query tile hold garbage
              m_ref += delta;
              if (!first) {
                // O_g must hold P V of every tile < t: peek at the next completion of the other buffer's barrier (see below)
                mbar_wait2_sa(bar_s_sa + 8u * (uint32_t)(buf ^ 1), (s_par >> (buf ^ 1)) & 1u, 12);
                tcgen05_fence_after();
                const float sc = ex2(-delta);
                uint32_t v[32];
                tmem_ld32(to, v);
                tmem_ld_wait();
#pragma unroll
                for (int e = 0; e < kDP; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * sc);
                tmem_st32(to, v);
                l_run *= sc;
              }
              (void)pass(m_ref, T{}, MASKED);  // P against the new reference
            }
          };
          if (need_mask) tile(std::true_type{});  // (item-uniform)
          else tile(std::false_type{});
          if (!ones) l_run += ps;
        } else {
          // ---- x = bias (+ mask) - m_ref first: these loads and adds do not depend on S and run while Q K^T is in flight.
          // Nothing here may touch the per-stage metadata: a warpgroup that sat out the previous item is a whole item
          // ahead of the producer, and an mbarrier parity wait only orders phases that are at most one apart.
          float x[KT];
          if (full_tile) {
            constexpr int KWS = KW > 0 ? KW : 4;
            constexpr int RW = (KWS >= 32) ? 32 : KWS;  // consecutive keys of one key row
#pragma unroll
            for (int r0 = 0; r0 < KT; r0 += RW) {
              const int kj = k0 + r0;  // first key of the run (CTA-uniform, multiple of 4)
              const int kh = kj / KWS, kw0 = kj % KWS;
              const int s0 = base_i - (kh * Wt + kw0) - 3;  // table index of key kj + 3
              const int cpy = (-s0) & 3;
              const float4* bp = reinterpret_cast<const float4*>(bias_h + (size_t)cpy * a.rows_pad + (s0 + cpy));
              const uint32_t bps = bias_sa + (uint32_t)(cpy * a.rows_pad + (s0 + cpy)) * 4u;  // BS: LDS.128
              if (need_mask && mask_fast) {  // (item-uniform branch: windows without a mask skip the per-group selects)
                const int rid_lo = 3 * ((int)a1 + (int)(kh >= kh_th)) + (int)b1;
                const float off_lo = (rid_lo != q_rid) ? m_ref - kMaskLog2 : m_ref;
                const float off_hi = (rid_lo + 1 != q_rid) ? m_ref - kMaskLog2 : m_ref;
#pragma unroll
                for (int qd = 0; qd < RW / 4; ++qd) {
                  const float4 bb = A2_BIAS(BS ? lds128(bps - 16u * qd) : __ldg(bp - qd));
                  const int j = r0 + 4 * qd;
                  const float off = (kw0 + 4 * qd >= kw_th) ? off_hi : off_lo;
                  x[j + 0] = bb.w - off, x[j + 1] = bb.z - off, x[j + 2] = bb.y - off, x[j + 3] = bb.x - off;
                }
              } else {
#pragma unroll
                for (int qd = 0; qd < RW / 4; ++qd) {
                  const float4 bb = A2_BIAS(BS ? lds128(bps - 16u * qd) : __ldg(bp - qd));
                  const int j = r0 + 4 * qd;
                  x[j + 0] = bb.w - m_ref, x[j + 1] = bb.z - m_ref, x[j + 2] = bb.y - m_ref, x[j + 3] = bb.x - m_ref;
                }
              }
            }
          }
          // ---- S_t
          mbar_wait2_sa(bar_s_sa + 8u * (uint32_t)buf, (s_par >> buf) & 1u, 10);
          s_par ^= 1u << buf;
          tcgen05_fence_after();
          const bool meta_mask = need_mask && !(full_tile && mask_fast);
          if (!full_tile || meta_mask) mbar_wait_warp(&meta_full[st], rs.ph, 11);  // S_t ready => this fill is the current one
          if (!full_tile) {
#pragma unroll
            for (int j = 0; j < KT; ++j) x[j] = (BS ? lds32f(bias_sa + 4u * (uint32_t)(base_i - lds32i(koff_sa + 4u * (st * KT + j))))
                         : __ldg(bias_h + base_i - lds32i(koff_sa + 4u * (st * KT + j)))) - m_ref;
          }
#pragma unroll
          for (int c0 = 0; c0 < KT; c0 += 32) {
            A2_LDTM({
              uint32_t v[32];
              tmem_ld32(ts + c0, v);
              tmem_ld_wait();
              _Pragma("unroll") for (int j = 0; j < 32; ++j) x[c0 + j] += __uint_as_float(v[j]);
            })
          }
          if (meta_mask) {
#pragma unroll
            for (int j = 0; j < KT; ++j)
              if (lds32i(krid_sa + 4u * (st * KT + j)) != q_rid) x[j] += kMaskLog2;
          }
          if (k0 + KT > Nk) {  // after the add: K rows past Nk are stale shared memory, S there may be anything
#pragma unroll
            for (int j = 0; j < KT; ++j)
              if (k0 + j >= Nk) x[j] = -INFINITY;
          }
          float mx0 = fmax3(x[0], x[1], x[2]), mx1 = fmax3(x[3], x[4], x[5]);
#pragma unroll
          for (int j = 6; j + 3 < KT; j += 4) {
            mx0 = fmax3(mx0, x[j], x[j + 1]);
            mx1 = fmax3(mx1, x[j + 2], x[j + 3]);
          }
          const float mx = A2_MAX(fmax3(mx0, mx1, fmaxf(x[KT - 2], x[KT - 1])));
          // ---- lazy rescale: move the reference only when a row outgrew it by 2^kTau (always on the first tile)
          const bool first = (t == 0);
          if (__any_sync(0xffffffffu, first || mx > kTau)) {
            float delta = first ? mx : fmaxf(mx, 0.f);
            if (!(fabsf(delta) < 1e30f)) delta = 0.f;  // rows of a partial query tile hold garbage
            m_ref += delta;
#pragma unroll
            for (int j = 0; j < KT; ++j) x[j] -= delta;
            if (!first) {
              // O_g must hold P V of every tile < t.  The NEXT completion of the other buffer's barrier (S(t+1) ready, or the
              // closing completion when t is the last tile) is committed right after P V(t-1): peek at it (the wait at tile
              // t+1 / in the epilogue consumes it), which keeps the wait exact and off the common path.
              mbar_wait2_sa(bar_s_sa + 8u * (uint32_t)(buf ^ 1), (s_par >> (buf ^ 1)) & 1u, 12);
              tcgen05_fence_after();
              const float sc = ex2(-delta);
              uint32_t v[32];
              tmem_ld32(to, v);
              tmem_ld_wait();
#pragma unroll
              for (int e = 0; e < kDP; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * sc);
              tmem_st32(to, v);
              l_run *= sc;
            }
          }
          // ---- P_t = exp2(x) -> 16-bit pairs -> TMEM (over S_t)
          float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
          for (int c = 0; c < KT / 2; ++c) {
            const float p0 = A2_EX2(x[2 * c]), p1 = A2_EX2(x[2 * c + 1]);
            if (!ones) ps0 += p0, ps1 += p1;
            pk[c] = (fmt == FMT_BF16) ? pack_bf16(p0, p1) : pack_f16(p0, p1);
          }
          if (!ones) l_run += ps0 + ps1;
        }
        A2_STTM(tmem_st32(ts, pk));
        tmem_st_wait();
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_sa(p_full_sa + 8u * (uint32_t)buf);
      }
      // ---- epilogue: O_g final
      // closing completions: buffer ntiles & 1 (P V(ntiles-2) done), then buffer (ntiles+1) & 1 (P V(ntiles-1) done = O final)
      mbar_wait_warp(&bar_s[2 * wg + (ntiles & 1)], (s_par >> (ntiles & 1)) & 1u, 13);
      s_par ^= 1u << (ntiles & 1);
      mbar_wait_warp(&bar_s[2 * wg + ((ntiles + 1) & 1)], (s_par >> ((ntiles + 1) & 1)) & 1u, 14);
      s_par ^= 1u << ((ntiles + 1) & 1);
      // "item consumed": the issuer may now commit the next item's S(0) / S(1) to these barriers (an mbarrier must not
      // complete twice before its waiter has looked: a parity wait cannot tell phases two apart)
      __syncwarp();
      if (lane == 0) mbar_arrive(&item_done[wg]);
      tcgen05_fence_after();
      {
        uint32_t v[32];
        tmem_ld32(to, v);
        tmem_ld_wait();
        if (q_ok) {
          const float inv = 1.0f / (ones ? __uint_as_float(v[kDP - 1]) : l_run);
          const long long q_tok = (long long)(it.b * a.gq.H + tq.y) * a.gq.W + tq.x;
          __nv_bfloat16* dst = a.o_dense ? a.out + (((long long)it.bw * a.heads + it.h) * Nq + qi) * kDP
                                         : a.out + q_tok * a.ldo + a.o_off + it.h * kDP;
#pragma unroll
          for (int e = 0; e < kDP; e += 8) {
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = __uint_as_float(v[e + i]) * inv;
            *reinterpret_cast<uint4*>(dst + e) = make_uint4(pack16(o[0], o[1], fmt), pack16(o[2], o[3], fmt),
                                                            pack16(o[4], o[5], fmt), pack16(o[6], o[7], fmt));
          }
        }
      }
      tcgen05_fence_before();
    }
  }
  __syncthreads();
  if (warp == 4 * NWG + 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
// Tokens per box for a window of width ww rolled by sw: the largest power of two <= 64 dividing gcd(ww, sw) (ww if the
// grid is not rolled horizontally).  0 = no usable box (runs shorter than 8 tokens = 512 bytes, the 64-byte-swizzle repeat).
int box_tokens2(const GrlGrid& g) {
  int d = g.ww;
  if (g.sw > 0) {
    int x = g.ww, y = g.sw;
    while (y) {
      const int t = x % y;
      x = y, y = t;
    }
    d = x;
  }
  int bw = 64;
  while (bw > 1 && d % bw) bw >>= 1;
  return bw >= 8 ? bw : 0;
}

int make_token_map2(CUtensorMap* m, const void* base, long long ld, const GrlGrid& g, int B, int bw) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return fail(GRL_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  const cuuint64_t dims[4] = {(cuuint64_t)ld, (cuuint64_t)g.W, (cuuint64_t)g.H, (cuuint64_t)B};
  const cuuint64_t str[3] = {(cuuint64_t)ld * 2, (cuuint64_t)g.W * ld * 2, (cuuint64_t)g.H * g.W * ld * 2};
  const cuuint32_t box[4] = {(cuuint32_t)kDP, (cuuint32_t)bw, 1, 1};
  const cuuint32_t ones[4] = {1, 1, 1, 1};
  const CUresult rc = fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<void*>(base), dims, str, box, ones,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) return fail(GRL_ERR_CUDA, "cuTensorMapEncodeTiled (attention tokens) failed with CUresult %d", (int)rc);
  return GRL_OK;
}

int make_dense_map2(CUtensorMap* m, const void* base, long long rows, int box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return fail(GRL_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  const cuuint64_t dims[2] = {(cuuint64_t)kDP, (cuuint64_t)rows};
  const cuuint64_t str[1] = {(cuuint64_t)kDP * 2};
  const cuuint32_t box[2] = {(cuuint32_t)kDP, (cuuint32_t)box_rows};
  const cuuint32_t ones[2] = {1, 1};
  const CUresult rc = fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, const_cast<void*>(base), dims, str, box, ones,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) return fail(GRL_ERR_CUDA, "cuTensorMapEncodeTiled (dense V) failed with CUresult %d", (int)rc);
  return GRL_OK;
}

constexpr int kMaxSmem = 232448;  // 227 KB: the per-CTA shared-memory limit of sm_100

template <int NWG, int KW, int VAR, bool BS>
int launch2_var(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const AttnTcArgs& a, A2Geom tg,
                cudaStream_t st) {
  auto kern = attn2_kernel<NWG, KW, VAR, BS>;
  static bool configured[kMaxDevices] = {false};
  int dev = 0;
  GRL_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices || !configured[dev]) {
    GRL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    if (dev >= 0 && dev < kMaxDevices) configured[dev] = true;
  }
  const int Nq = a.gq.wh * a.gq.ww;
  tg.n_qg = ceil_div(Nq, NWG * kQT);
  tg.ntiles = ceil_div(a.gk.wh * a.gk.ww, kKT2);
  const long long per_head = (long long)a.B * (a.gq.H / a.gq.wh) * (a.gq.W / a.gq.ww) * tg.n_qg;
  GRL_REQUIRE(per_head * a.heads < (1ll << 31), "attn2: too many work items");
  tg.per_head = (int)per_head;
  const long long cph = std::max(1ll, std::min((long long)(sm_count() / a.heads), per_head));  // CTAs per head
  const unsigned grid = (unsigned)(cph * a.heads);
  const int bias_bytes = BS ? 16 * a.rows_pad : 0;
  tg.stages = std::min(kMaxStages2, (kMaxSmem - A2Smem<NWG>::FIXED - bias_bytes) / (2 * A2Smem<NWG>::KV_BYTES));
  GRL_REQUIRE(tg.stages >= 4, "attn2: no room for the K / V ring");
  const int smem = A2Smem<NWG>::total(tg.stages, bias_bytes);
  kern<<<grid, NWG * 128 + 32 + kIssuers2<NWG>() * 32, smem, st>>>(tq, tk, tv, a, tg);
  GRL_LAUNCH_CHECK("attn2_kernel");
  return GRL_OK;
}

template <int NWG, int KW, int VAR>
int launch2_bs(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const AttnTcArgs& a, const A2Geom& tg,
               cudaStream_t st) {
  // the 4-copy table in shared memory when it fits next to the tiles: LDS.128 costs 4 wavefronts where the L1 path pays
  // ~7.5 tag lookups (the 128-byte runs of the four copies are not line aligned) -- the L1 data pipe was the busiest unit
  static const bool off = [] { const char* e = getenv("GRL_ATTN2_NO_SMEM_BIAS"); return e && e[0] == '1'; }();
  // ... as long as the table leaves room for a ring deep enough to cover the TMA latency (>= min_ring stages)
  static const int min_ring = [] { const char* e = getenv("GRL_ATTN2_MIN_RING"); return e ? atoi(e) : 6; }();
  if (KW > 0 && !off && A2Smem<NWG>::total(min_ring, 16 * a.rows_pad) <= kMaxSmem)
    return launch2_var<NWG, KW, VAR, (KW > 0)>(tq, tk, tv, a, tg, st);
  return launch2_var<NWG, KW, VAR, false>(tq, tk, tv, a, tg, st);
}

template <int NWG, int KW>
int launch2_kw(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const AttnTcArgs& a, const A2Geom& tg,
               cudaStream_t st) {
  switch ((a.fmt == FMT_BF16 ? 1 : 0) | (a.ones_col ? 2 : 0)) {
    case 0: return launch2_bs<NWG, KW, 0>(tq, tk, tv, a, tg, st);
    case 1: return launch2_bs<NWG, KW, 1>(tq, tk, tv, a, tg, st);
    case 2: return launch2_bs<NWG, KW, 2>(tq, tk, tv, a, tg, st);
    default: return launch2_bs<NWG, KW, 3>(tq, tk, tv, a, tg, st);
  }
}

template <int NWG>
int launch2_nwg(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const AttnTcArgs& a, const A2Geom& tg,
                cudaStream_t st) {
  switch (a.gk.ww) {
    case 16: return launch2_kw<NWG, 16>(tq, tk, tv, a, tg, st);
    case 32: return launch2_kw<NWG, 32>(tq, tk, tv, a, tg, st);
    case 64: return launch2_kw<NWG, 64>(tq, tk, tv, a, tg, st);
    case 128: return launch2_kw<NWG, 128>(tq, tk, tv, a, tg, st);
    default: return launch2_kw<NWG, 0>(tq, tk, tv, a, tg, st);
  }
}

int attn2_debug_read(int* out8) {
  int tmp[8] = {0};
  if (cudaMemcpyFromSymbol(tmp, g_a2_dbg, sizeof(tmp)) != cudaSuccess) return -1;
  for (int i = 0; i < 8; ++i) out8[i] = tmp[i];
  int zero[8] = {0};
  cudaMemcpyToSymbol(g_a2_dbg, zero, sizeof(zero));
  return 0;
}

}  // namespace

int attn2_debug(int* out8) { return attn2_debug_read(out8); }
int attn_tma_box_tokens(const GrlGrid& g) { return box_tokens2(g); }

// Returns GRL_OK after launching, a negative error, or +1 when this geometry cannot be expressed as TMA boxes (the
// caller then launches the gather kernel of attn_tc.cu).  Arguments already validated by launch_attn_tc.
int launch_attn2(const AttnTcArgs& a, cudaStream_t st) {
  A2Geom tg;
  tg.bw_q = box_tokens2(a.gq);
  tg.bw_k = box_tokens2(a.gk);
  tg.n_qg = tg.per_head = 0;
  if (tg.bw_q == 0 || tg.bw_k == 0) return 1;
  if (a.gq.W < tg.bw_q || a.gk.W < tg.bw_k) return 1;
  if ((reinterpret_cast<uintptr_t>(a.q) | reinterpret_cast<uintptr_t>(a.k) | reinterpret_cast<uintptr_t>(a.v)) & 15) return 1;
  CUtensorMap tq, tk, tv;
  int rc;
  if ((rc = make_token_map2(&tq, a.q, a.ldq, a.gq, a.B, tg.bw_q)) != GRL_OK) return rc;
  if ((rc = make_token_map2(&tk, a.k, a.ldk, a.gk, a.B, tg.bw_k)) != GRL_OK) return rc;
  if (a.v_dense) {
    const long long rows = (long long)a.B * (a.gk.H / a.gk.wh) * (a.gk.W / a.gk.ww) * a.heads * a.gk.wh * a.gk.ww;
    if (rows < kKT2) return 1;  // the dense-V box is 64 rows: keep it inside the tensor
    if ((rc = make_dense_map2(&tv, a.v, rows, kKT2)) != GRL_OK) return rc;
  } else {
    if ((rc = make_token_map2(&tv, a.v, a.ldv, a.gk, a.B, tg.bw_k)) != GRL_OK) return rc;
  }
#ifndef GRL_A2_NWG  // A/B builds: 1 or 2 softmax warpgroups per CTA (how the time per tile depends on the co-resident warpgroups)
#define GRL_A2_NWG 3
#endif
  return launch2_nwg<GRL_A2_NWG>(tq, tk, tv, a, tg, st);
}

}  // namespace tc
}  // namespace grl
