// tcgen05 / mbarrier / bulk-copy PTX wrappers shared by the tensor-core kernels (sm_100a).
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

namespace umma {

// ---- PTX wrappers -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t a, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t a) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t a, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint32_t a, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
               "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(a), "r"(parity) : "memory");
  return ok != 0;
}
// non-blocking poll (test_wait never suspends the thread, unlike try_wait)
__device__ __forceinline__ bool mbar_poll(uint32_t a, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
               "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(a), "r"(parity) : "memory");
  return ok != 0;
}
// bounded wait: a stuck pipeline raises the abort flag instead of hanging the GPU
__device__ __forceinline__ bool mbar_wait(uint32_t a, uint32_t parity, volatile int* abort_flag, int code = 0, long long limit = 1000000000LL) {
  if (mbar_test(a, parity)) return true;
  const long long t0 = clock64();
  while (true) {
    if (mbar_test(a, parity)) return true;
    if (*abort_flag) return false;
    if (clock64() - t0 > limit) {
      if (atomicCAS((int*)abort_flag, 0, 1) == 0) ((int*)abort_flag)[1] = code;   // first failing wait wins
      return false;
    }
  }
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void group_sync(int m) { asm volatile("bar.sync %0, %1;" ::"r"(1 + m), "r"(128) : "memory"); }
// group barrier that also ANDs a predicate over the 128 threads of the tile group
__device__ __forceinline__ bool group_sync_and(int m, bool pred) {
  uint32_t r;
  asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %3, 0;\n\tbarrier.cta.red.and.pred q, %1, %2, p;\n\t"
               "selp.u32 %0, 1, 0, q;\n\t}" : "=r"(r) : "r"(1 + m), "r"(128), "r"((uint32_t)pred) : "memory");
  return r != 0;
}
// ACC: 0 = overwrite the accumulator, 1 = accumulate
template <int ACC>
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "n"(ACC) : "memory");
}
__device__ __forceinline__ void tc_mma_dyn(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               ::"r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
               "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
               "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                 "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                 "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
               : "r"(taddr));
}
// A operand from tensor memory (row = lane, two 16-bit K elements per 32-bit column: K = 16 is 8 columns)
template <int ACC>
__device__ __forceinline__ void tc_mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b, uint32_t idesc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
               ::"r"(d_tmem), "r"(a_tmem), "l"(b), "r"(idesc), "n"(ACC) : "memory");
}
__device__ __forceinline__ void tc_mma_ts_dyn(uint32_t d_tmem, uint32_t a_tmem, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
               ::"r"(d_tmem), "r"(a_tmem), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tc_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
               "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                 "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, no-swizzle canonical layout: 8-row x 16-byte core matrices; rows 16 B apart,
// 8-row groups SBO (=128 B) apart, 16-byte K chunks LBO apart (cute::UMMA::SmemDescriptor, version 1).
// `lo` = (shared address >> 4) | ((LBO >> 4) << 16); the high word is the same for every operand here.
__device__ __forceinline__ uint64_t desc_from_lo(uint32_t lo) { return ((uint64_t)0x4008u << 32) | lo; }
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}
// cute::UMMA::InstrDescriptor: c=F32 (bit 4), a/b format (bits 7,10: F16=0, BF16=1), K-major, N>>3 @17, M>>4 @24
__host__ __device__ constexpr uint32_t make_idesc(int fmt, int M, int N) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// two fp32 values as an fp16 pair; saturating: a value beyond +-65504 becomes the largest finite half, not an inf that
// would poison every later layer
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---- packed fp32 pairs (FFMA2 / FADD2 / FMUL2: one issue slot for two lanes of math) -------------
typedef unsigned long long f2_t;
__device__ __forceinline__ f2_t pk(float lo, float hi) { f2_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk(f2_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f2_t fma2(f2_t a, f2_t b, f2_t c) { f2_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f2_t add2(f2_t a, f2_t b) { f2_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2_t mul2(f2_t a, f2_t b) { f2_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }


}  // namespace umma
