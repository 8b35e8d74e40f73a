// Thin inline-PTX layer for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM
// alloc / ld / st / commit / fences) and the UMMA shared-memory / instruction descriptors.
// Hand-written for this repository; bit layouts follow the PTX ISA "tcgen05" chapter (the same
// layouts CUTLASS documents in cute/arch/mma_sm100_desc.hpp).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace mfa {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ uint32_t lane_id() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(r));
  return r;
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "elect.sync _|P, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier -------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred P;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n"
      "selp.u32 %0, 1, 0, P;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// Bounded wait: a protocol bug must surface as a trapped kernel (an error the host reports), never
// as a hung GPU.  ~4 s at 2 GHz; the check costs nothing on the fast path.
#ifndef MFA_MBAR_TIMEOUT_CYCLES
#define MFA_MBAR_TIMEOUT_CYCLES (8000000000ll)
#endif
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long start = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ffu) == 0 && clock64() - start > MFA_MBAR_TIMEOUT_CYCLES) {
      printf("mfa_b200: mbarrier timeout block (%d,%d) thread %d bar@%u parity %u\n", blockIdx.x, blockIdx.y,
             threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
  }
}

// ---------------------------------------------------------------- streaming global loads -----
// Read-once data (O and dO rows for D = rowsum(dO * O)): no L1 line is allocated for the miss.  The kernels run with up
// to 225 KB of shared memory, which leaves ~30 KB of L1; a 128-row tile's 48 KB in flight through allocating loads
// serialised on L1 lines (measured: -5 % on the persistent dQ kernel at N >= 4096 when its shared memory grew by 48 KB).
__device__ __forceinline__ float4 ldg_stream_f32x4(const float *p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}
__device__ __forceinline__ uint2 ldg_stream_u32x2(const void *p) {
  uint2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}

// ---------------------------------------------------------------- TMA ------------------------
__device__ __forceinline__ void prefetch_tensormap(const void *map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
// 3-D tiled load global -> shared, completion counted in bytes on `bar`
__device__ __forceinline__ void tma_load_3d(void *smem_dst, const void *map, uint64_t *bar, int32_t c0, int32_t c1,
                                            int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// 3-D tiled store shared -> global (bulk async-group completion).  The issuing THREAD owns the group: the same thread
// commits and later waits.  Generic-proxy writes to the source tile need fence.proxy.async before the store is issued.
__device__ __forceinline__ void tma_store_3d(const void *map, uint32_t smem_src, int32_t c0, int32_t c1, int32_t c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// every committed group of this thread has finished READING shared memory (the source tile may be rewritten)
__device__ __forceinline__ void tma_store_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... has completed (the global writes are done)
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// 1-D bulk copy global -> shared (no tensor map): `bytes` a multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_load_1d(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gmem_src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---------------------------------------------------------------- tcgen05: TMEM management ----
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_result, uint32_t columns) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
               "r"(columns)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t columns) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(columns) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// all tcgen05.mma issued so far by this thread -> one arrival on `bar` when they complete
// (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---------------------------------------------------------------- tcgen05: descriptors --------
// Shared-memory matrix descriptor, 128-byte swizzle (what TMA SWIZZLE_128B writes):
//   [0,14) start address >> 4   [16,30) leading byte offset >> 4   [32,46) stride byte offset >> 4
//   [46,48) version = 1 (sm_100)   [49,52) base offset = 0   [61,64) layout type: 2 = SWIZZLE_128B
// K-major operand  (rows = M or N index, 64 16-bit K elements = one 128 B swizzle row):
//   SBO = distance between 8-row groups (1024 B); LBO unused.
// MN-major operand (rows = K index, 64 16-bit MN elements per 128 B row):
//   SBO = distance between 8-row (K) groups (1024 B); LBO = distance between 64-element MN blocks.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t desc = 0;
  desc |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  desc |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  desc |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  desc |= static_cast<uint64_t>(1) << 46;
  desc |= static_cast<uint64_t>(2) << 61;
  return desc;
}

// Instruction descriptor for kind::f16 (FP16/BF16 inputs, FP32 accumulate):
//   [4,6) D format: 1 = F32   [7,10) A format, [10,13) B format: 0 = F16, 1 = BF16
//   [15] A major, [16] B major: 0 = K-major, 1 = MN-major   [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_f16_mixed(uint32_t M, uint32_t N, uint32_t a_format,
                                                            uint32_t b_format, uint32_t a_mn_major,
                                                            uint32_t b_mn_major) {
  return (1u << 4) | (a_format << 7) | (b_format << 10) | (a_mn_major << 15) | (b_mn_major << 16) |
         ((N >> 3) << 17) | ((M >> 4) << 24);
}
__host__ __device__ constexpr uint32_t make_idesc_f16(uint32_t M, uint32_t N, uint32_t ab_format, uint32_t a_mn_major,
                                                      uint32_t b_mn_major) {
  return make_idesc_f16_mixed(M, N, ab_format, ab_format, a_mn_major, b_mn_major);
}

// D[tmem] (+)= A[smem] * B[smem]
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]   (A: 128 lanes x K/2 32-bit columns, two 16-bit K elements per column)
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ---------------------------------------------------------------- tcgen05: TMEM <-> registers --
// 32x32b shape: thread i of the warp owns TMEM lane (lane base + i); .xN moves N consecutive columns.
#define MFA_R4(v, o) "%" #o ", %" #v
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
#undef MFA_R4
// 64 consecutive columns in one instruction (the wait is the caller's: several loads may be put in flight first)
__device__ __forceinline__ void tmem_ld64(uint32_t taddr, uint32_t (&r)[64]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%32], "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31};" ::"r"(r[0]),
      "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
      "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]),
      "r"(r[29]), "r"(r[30]), "r"(r[31]), "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%16], "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15};" ::"r"(r[0]),
      "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(taddr)
      : "memory");
}

// ---------------------------------------------------------------- shared memory, explicit state space ----
// Pointers derived from the manually aligned dynamic shared-memory base are generic to the compiler (LD.E / ST.E in
// SASS); the staging tiles of the epilogues go through these instead so that they compile to LDS / STS.
__device__ __forceinline__ void sts_f32x4(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds_f32x4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

// ---------------------------------------------------------------- math helpers ----------------
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// ---- packed FP32x2 arithmetic (Blackwell FFMA2 / FADD2: two FP32 lanes per issue slot) ----
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(d)
      : "l"(*reinterpret_cast<const uint64_t *>(&a)), "l"(*reinterpret_cast<const uint64_t *>(&b)),
        "l"(*reinterpret_cast<const uint64_t *>(&c)));
  return *reinterpret_cast<float2 *>(&d);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;"
      : "=l"(d)
      : "l"(*reinterpret_cast<const uint64_t *>(&a)), "l"(*reinterpret_cast<const uint64_t *>(&b)));
  return *reinterpret_cast<float2 *>(&d);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;"
      : "=l"(d)
      : "l"(*reinterpret_cast<const uint64_t *>(&a)), "l"(*reinterpret_cast<const uint64_t *>(&b)));
  return *reinterpret_cast<float2 *>(&d);
}
__device__ __forceinline__ float max_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float min_nan(float a, float b) {
  float r;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
// exp2 of two values on the FMA / ALU pipes (no MUFU): Cody-Waite split x = n + f, n = round(x), f in [-0.5, 0.5],
// 2^f by a degree-3 minimax polynomial (max relative error 7.6e-5, below the 16-bit rounding P gets anyway), then
// n is added to the exponent field.
// kClampUpper = false is for callers whose inputs cannot be large (the backward pass: x = s - L <= ~0 because L is the
// row's log-sum-exp): it saves two of the ~12 instructions per pair.
template <bool kClampUpper = true>
__device__ __forceinline__ float2 exp2_poly2(float2 x) {
  const float kMagic = 12582912.0f;  // 1.5 * 2^23: adding it leaves round(x) in the low mantissa bits
  // clamp to the finite exponent range: -inf / very negative inputs give ~0, and an input far above the running max
  // (stale or unset m) gives a huge finite value, which is what the caller's overflow check looks for
  // (max.NaN / min.NaN: a NaN score stays NaN -- it reaches the sum, the caller's overflow check and the output, as
  // it does through ex2.approx -- where fmaxf would quietly turn it into 2^-126)
  x.x = max_nan(x.x, -126.0f);
  x.y = max_nan(x.y, -126.0f);
  if (kClampUpper) {
    x.x = min_nan(x.x, 127.0f);
    x.y = min_nan(x.y, 127.0f);
  }
  const float2 t = fadd2(x, make_float2(kMagic, kMagic));
  const float2 n = fadd2(t, make_float2(-kMagic, -kMagic));
  const float2 f = fadd2(x, make_float2(-n.x, -n.y));
  float2 p = ffma2(make_float2(0.055168044f, 0.055168044f), f, make_float2(0.24260214f, 0.24260214f));
  p = ffma2(p, f, make_float2(0.69326079f, 0.69326079f));
  p = ffma2(p, f, make_float2(0.99992865f, 0.99992865f));
  float2 r;
  r.x = __uint_as_float(__float_as_uint(p.x) + (__float_as_uint(t.x) << 23));
  r.y = __uint_as_float(__float_as_uint(p.y) + (__float_as_uint(t.y) << 23));
  return r;
}

// pack two FP32 into one 32-bit register of 16-bit values: low half = lo, high half = hi
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// the two 16-bit halves of a packed register, widened back to FP32 (exact)
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t w) {
  return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xFFFF0000u));
}
__device__ __forceinline__ float2 unpack_f16x2(uint32_t w) {
  float2 r;
  asm("{\n"
      ".reg .b16 lo, hi;\n"
      "mov.b32 {lo, hi}, %2;\n"
      "cvt.f32.f16 %0, lo;\n"
      "cvt.f32.f16 %1, hi;\n"
      "}\n"
      : "=f"(r.x), "=f"(r.y)
      : "r"(w));
  return r;
}

// ---------------------------------------------------------------- online-softmax inner loop ---

// One half-row (64 scores, FP32 bits in v) -> P = exp2(s * scale_log2 - m) rounded to 16 bits in `packed`; returns the
// half-row sum.  v is consumed in place.  kPolyPairs of every 4 element pairs take exp2 on the FMA pipe (exp2_poly2)
// instead of the MUFU pipe.
template <bool kBF16, uint32_t kPolyPairs>
__device__ __forceinline__ float softmax_exp_half(uint32_t (&v)[64], uint32_t (&packed)[32], float scale_log2, float m) {
  // Pairs by which "sum and pack" trails "exp2".  A warp issues in order: with the consumer of an ex2 right behind it
  // (what a plain loop compiles to) every pair exposes the MUFU latency -- measured 26 cycles per pair against the
  // pipe's 16 (two ex2 at 4 lanes / clk / sub-partition).
  constexpr uint32_t kSkew = 4;
  const float2 scale2 = make_float2(scale_log2, scale_log2), negm2 = make_float2(-m, -m);
  float2 acc0 = make_float2(0.f, 0.f), acc1 = make_float2(0.f, 0.f);
#pragma unroll
  for (uint32_t i = 0; i < 32 + kSkew; ++i) {
    if (i < 32) {
      float2 x = ffma2(make_float2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1])), scale2, negm2);
      if (kPolyPairs > 0 && (i & 3) < kPolyPairs) {
        x = exp2_poly2(x);
      } else {
        x.x = ex2_approx(x.x);
        x.y = ex2_approx(x.y);
      }
      v[2 * i] = __float_as_uint(x.x);
      v[2 * i + 1] = __float_as_uint(x.y);
    }
    if (i >= kSkew) {
      const uint32_t k = i - kSkew;
      float2 e = make_float2(__uint_as_float(v[2 * k]), __uint_as_float(v[2 * k + 1]));
      packed[k] = kBF16 ? pack_bf16x2(e.x, e.y) : pack_f16x2(e.x, e.y);
      if (k & 1)
        acc1 = fadd2(acc1, e);
      else
        acc0 = fadd2(acc0, e);
    }
  }
  const float2 acc = fadd2(acc0, acc1);
  return acc.x + acc.y;
}

// ---------------------------------------------------------------- register reallocation ------
template <uint32_t RegCount>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(RegCount));
}
template <uint32_t RegCount>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(RegCount));
}

}  // namespace ptx
}  // namespace mfa
