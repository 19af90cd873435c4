// Thin inline-PTX wrappers for the Blackwell (sm_100a) tensor-core path: tcgen05.mma / TMEM / mbarrier / bulk copy.
// Layout conventions (validated on hardware by tools/probe_tc.cu):
//   * shared-memory operands use the no-swizzle K-major canonical layout: 8 rows x 16 bytes "core matrices" stored
//     contiguously (128 B); consecutive 8-row groups are SBO bytes apart, the two 16-byte K chunks of one MMA are LBO
//     bytes apart.  Images here use  offset(row, k) = ((k/8) * (ROWS/8) + row/8) * 128 B + (row%8) * 16 B + (k%8) * 2 B,
//     i.e. SBO = 128 B and LBO = ROWS/8 * 128 B;
//   * the A operand can instead live in tensor memory: lane = row, one 32-bit column = two consecutive bf16 of K;
//   * accumulators are fp32 in tensor memory: lane = row, column = n.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ecnf_tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__host__ __device__ __forceinline__ int canon_index(int row, int k, int rows) {  // in bf16 elements
  return ((k >> 3) * (rows >> 3) + (row >> 3)) * 64 + (row & 7) * 8 + (k & 7);
}

// ---- tensor memory management -----------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {  // whole warp, ncols power of 2 >= 32
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // whole warp (the allocating one)
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- mbarrier ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// same, letting the hardware park the warp for up to `ns` per attempt (far fewer polls issued while waiting)
__device__ __forceinline__ void mbar_wait_parked(uint64_t* bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// named barrier among `nthreads` threads (a multiple of 32) of the CTA; id 0 is __syncthreads
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// asynchronous prefetch of a contiguous global range into L2 (16-byte aligned, size multiple of 16)
__device__ __forceinline__ void prefetch_l2_bulk(const void* gsrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}

// ---- descriptors -------------------------------------------------------------------------------------------------
// shared-memory matrix descriptor, no swizzle, K-major (cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout_type=0 [61,64))
__device__ __forceinline__ uint64_t make_sdesc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         ((uint64_t)1 << 46);
}
// instruction descriptor for kind::f16, A = B = bf16 (K-major), D = fp32 (cute::UMMA::InstrDescriptor);
// OR in IDESC_B_MN for a B operand stored MN-major (validated by tools/probe_tc2.cu)
constexpr uint32_t IDESC_B_MN = 1u << 16;
__host__ __device__ __forceinline__ uint32_t make_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// one lane of a fully converged warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- MMA (issued by ONE thread) ------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// arrives on `bar` when every MMA issued so far by this thread has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- TMEM <-> registers: 32 lanes x 32 consecutive 32-bit columns per warp (warp w may touch lanes 32*(w%4)..+31) ----
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ uint32_t tmem_ld1(uint32_t taddr) {   // one column; pair with tmem_wait_ld()
  uint32_t v;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\n" : "=r"(v) : "r"(taddr) : "memory");
  return v;
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
      "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
      "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- packed fp32 pairs: one FFMA2 / FMUL2 / FADD2 does the two IEEE round-to-nearest operations of the scalar
// instructions it replaces (bit for bit), in one issue slot.  nvcc does not pair scalar code by itself. -------------------
__device__ __forceinline__ float2 fma2(float2 x, float2 y, float2 z) {    // (fmaf(x.x, y.x, z.x), fmaf(x.y, y.y, z.y))
  float2 d;
  asm("{\n\t.reg .b64 a, b, c, d;\n\t"
      "mov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tmov.b64 c, {%6, %7};\n\t"
      "fma.rn.f32x2 d, a, b, c;\n\tmov.b64 {%0, %1}, d;\n\t}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(x.x), "f"(x.y), "f"(y.x), "f"(y.y), "f"(z.x), "f"(z.y));
  return d;
}
__device__ __forceinline__ float2 mul2(float2 x, float2 y) {
  float2 d;
  asm("{\n\t.reg .b64 a, b, d;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tmul.rn.f32x2 d, a, b;\n\tmov.b64 {%0, %1}, d;\n\t}"
      : "=f"(d.x), "=f"(d.y) : "f"(x.x), "f"(x.y), "f"(y.x), "f"(y.y));
  return d;
}
__device__ __forceinline__ float2 add2(float2 x, float2 y) {
  float2 d;
  asm("{\n\t.reg .b64 a, b, d;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tadd.rn.f32x2 d, a, b;\n\tmov.b64 {%0, %1}, d;\n\t}"
      : "=f"(d.x), "=f"(d.y) : "f"(x.x), "f"(x.y), "f"(y.x), "f"(y.y));
  return d;
}
__device__ __forceinline__ float2 sub2(float2 x, float2 y) {
  float2 d;
  asm("{\n\t.reg .b64 a, b, d;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tsub.rn.f32x2 d, a, b;\n\tmov.b64 {%0, %1}, d;\n\t}"
      : "=f"(d.x), "=f"(d.y) : "f"(x.x), "f"(x.y), "f"(y.x), "f"(y.y));
  return d;
}
__device__ __forceinline__ float2 splat2(float x) { return make_float2(x, x); }

// ---- fp32 -> (hi, lo) bf16 split of two consecutive K elements, packed for a TMEM column (low half = even k) -------
// hi = round-to-nearest bf16 of x; lo = the same rounding of the exact residual x - float(hi).  The two halves of the
// packed hi word are widened back to fp32 by a shift and a mask (bf16 is the top half of an fp32).
__device__ __forceinline__ void split_pack(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);      // .x = x0 (low 16 bits), .y = x1
  hi = *reinterpret_cast<const uint32_t*>(&h);
  const float2 r = sub2(make_float2(x0, x1), make_float2(__uint_as_float(hi << 16), __uint_as_float(hi & 0xffff0000u)));
  const __nv_bfloat162 l = __floats2bfloat162_rn(r.x, r.y);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

}  // namespace ecnf_tc
