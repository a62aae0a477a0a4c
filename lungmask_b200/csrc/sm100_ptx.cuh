// sm_100a PTX wrappers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld).
// Hand-written for this repo; no CUTLASS dependency.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace lm {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug traps (launch failure on the host) instead of hanging the GPU.
#ifndef LM_MBAR_SPIN_LIMIT
#define LM_MBAR_SPIN_LIMIT (1u << 24)   // try_wait suspends ~1 us per failed try: ~10-20 s before trapping
#endif
// REGION: one copy of the out-of-line trap per register-allocation region of a kernel that uses setmaxnreg - ptxas gives
// every region that calls a common subroutine the smallest register budget among them (measured: a shared trap routine
// capped the epilogue warps at the producer's 96 registers).
template <int REGION>
static __device__ __noinline__ void mbar_timeout_trap(uint32_t bar, uint32_t parity) {
  printf("mbar_wait timeout: block %d thread %d bar 0x%x parity %u\n", (int)blockIdx.x, (int)threadIdx.x, bar, parity);
  __trap();
}
// The hot loop is try_wait only (the instruction itself suspends the thread until the phase flips or a
// hardware time limit expires); the watchdog is an iteration count, so no clock reads sit on the wake-up path.
template <int REGION = 0>
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > LM_MBAR_SPIN_LIMIT) mbar_timeout_trap<REGION>(bar, parity);
  }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar,
                                            int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* m, uint32_t bar,
                                            int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(dst),
      "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// TMA stores (shared -> global), bulk-group completion
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(m),
               "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(m),
               "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---------------------------------------------------------------- tcgen05
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_result),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// tcgen05.commit: arrives (count 1) on the mbarrier once all previously issued MMAs retire.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   bar)
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], kind::tf32, fp32 accumulate. Single-thread issue.
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Same with the accumulate flag fixed at compile time (no setp on the issuing thread's critical path).
template <bool ACC>
__device__ __forceinline__ void umma_tf32_c(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  if (ACC)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc)
                 : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc)
                 : "memory");
}

// D[tmem] (+)= A[smem] * B[smem], kind::f16 (fp16 operands), fp32 accumulate; accumulate flag fixed at compile time.
template <bool ACC>
__device__ __forceinline__ void umma_f16_c(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  if (ACC)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc)
                 : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc)
                 : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// K-major, 128B-swizzled operand tile: rows of 128 B (32 fp32), 8-row swizzle atoms 1024 B apart.
// Field layout follows the sm_100 shared-memory matrix descriptor (start>>4 | LBO | SBO | version=1
// | layout type 2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;               // LBO (ignored for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;     // SBO: 8 rows * 128 B
  d |= (uint64_t)1 << 46;               // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;               // SWIZZLE_128B
  return d;
}
// Instruction descriptor for kind::tf32, D=f32, A/B K-major.
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// Instruction descriptor for kind::f16 with fp16 A/B (format 0), D=f32, A/B K-major.
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Register reallocation between warpgroups (setmaxnreg: all four warps of a warpgroup execute it together).
template <int N> __device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// fp32 -> (fp16 hi, fp16 lo * 2^11): hi + lo * 2^-11 == x to ~2^-22 (x - hi is exact in fp32; the scaled
// residual keeps 11 significant bits even where x - hi would be an fp16 subnormal).  |x| must be <= 65504.
__device__ __forceinline__ void split_f16(float x, __half& hi, __half& lo) {
  hi = __float2half_rn(x);
  lo = __float2half_rn((x - __half2float(hi)) * 2048.f);
}
// two values at once with the packed conversions (cvt.rn.f16x2.f32): the same roundings as split_f16, fewer instructions
__device__ __forceinline__ void split_f16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);          // .x (low half) = a
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn((a - hf.x) * 2048.f, (b - hf.y) * 2048.f);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

}  // namespace lm
