// tc_common.cuh -- sm_100a primitives used by the tensor-core path: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (TMEM alloc / mma / commit / ld / st), UMMA shared-memory + instruction descriptors, cp.async.
// Inline PTX only; bit layouts follow the PTX ISA "tcgen05 matrix descriptor" / "instruction descriptor"
// tables (the same fields CUTLASS's cute/arch/mma_sm100_desc.hpp encodes).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace grl {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  // suspend-time hint: the thread sleeps in hardware until the phase completes (or ~1 ms passes) instead of
  // spinning -- waiting warps must not eat the issue slots of the warps doing the softmax / epilogue math.
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(1000000u)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (-> CUDA error reported through the C ABI) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  int spins = 0;
  long long t0 = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 63) == 0) {  // wall-clock bound (~2 s), checked rarely so that waiting costs no issue slots
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ll) __trap();
    }
  }
}

// ------------------------------------------------------------------ proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(smem)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// ------------------------------------------------------------------ cp.async (LDGSTS) for gathered rows
__device__ __forceinline__ void cp_async_16(void* smem, const void* gmem, bool valid) {
  const int sz = valid ? 16 : 0;  // src-size 0 -> zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem)), "l"(gmem), "r"(sz) : "memory");
}
// 1-D bulk copy global -> shared (TMA engine, no tensor map): bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_load_1d(void* smem, const void* gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem)),
               "l"(gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------ TMEM
// Called by ONE full warp.  ncols: power of two in [32, 512].
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// 32 lanes x 32 columns of 32-bit: thread t of the warp gets TMEM lane (lane_base + t), columns [col, col+32).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 16 columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 lanes x 32 columns of 32-bit, the inverse of tmem_ld32.
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------ UMMA descriptors
enum : uint32_t { SWZ_NONE = 0, SWZ_128B = 2, SWZ_64B = 4, SWZ_32B = 6 };

// Shared-memory matrix descriptor (64-bit): start address, leading / stride byte offsets (16-byte units),
// descriptor version 1 (Blackwell), swizzle mode in bits [61,64).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t swz) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)swz << 61;
  return d;
}

// Instruction descriptor for kind::f16: D fp32, A/B both `fmt` (0 = fp16, 1 = bf16), majors 0 = K-major, 1 = MN-major.
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N, int fmt, int a_mn_major, int b_mn_major) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)a_mn_major << 15) |
         ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]; issued by ONE thread.  A: 128 lanes x K 16-bit values packed in pairs (K / 2 columns).
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
// One lane of a converged warp (elect.sync).  Code under `if (elect_one())` is "one-lane uniform" to ptxas: operands of the
// UTCHMMA / UTMALDG / UTCBAR instructions in it move to uniform registers with plain R2UR, where code under
// `if (lane == 0)` gets an ELECT / R2UR.BROADCAST / BRA.U.ANY loop (about 13 instructions) around each of them.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// All previously issued MMAs of this thread arrive on `bar` when they complete (implies fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
// Operand formats of the tensor-core path: FMT_F16 (default: 11-bit mantissa, saturating converts) or FMT_BF16.
enum : int { FMT_F16 = 0, FMT_BF16 = 1 };
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ uint32_t pack16(float lo, float hi, int fmt) {
  return fmt == FMT_BF16 ? pack_bf16(lo, hi) : pack_f16(lo, hi);
}
__device__ __forceinline__ float2 unpack16(uint32_t v, int fmt) {
  if (fmt == FMT_BF16) return make_float2(__uint_as_float(v << 16), __uint_as_float(v & 0xFFFF0000u));
  return __half22float2(*reinterpret_cast<const __half2*>(&v));
}
__device__ __forceinline__ float unpack16_one(uint16_t v, int fmt) {
  if (fmt == FMT_BF16) return __uint_as_float((uint32_t)v << 16);
  return __half2float(*reinterpret_cast<const __half*>(&v));
}

// ------------------------------------------------------------------ host: tensor maps without linking libcuda
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn();  // gemm_tc.cu

}  // namespace tc
}  // namespace grl
