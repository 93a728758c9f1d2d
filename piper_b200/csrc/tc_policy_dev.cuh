// Device implementation of the primitive policy the policy-based kernel bodies (mrf_fused_body.inl, conv2_body.inl) are
// written against: inline PTX for tcgen05 / TMA / mbarrier.
// The CPU counterpart (a functional model used by tests) is tests/sim/sim_prim.h.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

#include "launch.cuh"

namespace pb200 {
namespace {

// ---- tcgen05 / TMA / mbarrier primitives -------------------------------------------------------------------------
struct DevPrim {
  static constexpr bool kSim = false;
  using Mbar = uint64_t;
  struct Ctx {
    __device__ __forceinline__ int tid() const { return threadIdx.x; }
    __device__ __forceinline__ int block() const { return blockIdx.x; }
    __device__ __forceinline__ int grid() const { return gridDim.x; }
  };
  static __device__ __forceinline__ uint32_t saddr(Ctx&, const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
  static __device__ __forceinline__ int bcast0(Ctx&, int v) { return __shfl_sync(0xffffffffu, v, 0); }
  static __device__ __forceinline__ void syncwarp() { __syncwarp(); }
  static __device__ __forceinline__ void syncthreads(Ctx&) { __syncthreads(); }
  // named barrier among `count` threads (a multiple of 32) of the CTA
  static __device__ __forceinline__ void bar_sync(Ctx&, int id, int count) { asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(count) : "memory"); }
  static __device__ __forceinline__ bool elect_one(Ctx&) {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
        "elect.sync rx|px, %1;\n\t"
        "@px mov.s32 %0, 1;\n\t}\n"
        : "+r"(pred)
        : "r"(0xFFFFFFFFu));
    return pred != 0;
  }
  static __device__ __forceinline__ long long clock() { return clock64(); }
  static __device__ __forceinline__ void prof_add(unsigned long long* p, long long v) { atomicAdd(p, (unsigned long long)v); }
  static __device__ __forceinline__ void pdl_launch() { pdl_launch_dependents(); }
  static __device__ __forceinline__ void pdl_sync() { pdl_wait(); }
  static __device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
  static __device__ __forceinline__ void fence_async_proxy() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
  static __device__ __forceinline__ void fence_tc_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
  static __device__ __forceinline__ void fence_tc_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
  static __device__ __forceinline__ void mbar_init(Ctx& c, Mbar* m, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(saddr(c, m)), "r"(count) : "memory");
  }
  static __device__ __forceinline__ void mbar_arrive(Ctx& c, Mbar* m) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(saddr(c, m)) : "memory");
  }
  static __device__ __forceinline__ void mbar_expect_tx(Ctx& c, Mbar* m, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(saddr(c, m)), "r"(bytes) : "memory");
  }
  // bounded: a protocol bug must end as a trap (launch failure), not as a hung GPU
  static __device__ __forceinline__ void mbar_wait(Ctx& c, Mbar* m, uint32_t parity) {
    const uint32_t a = saddr(c, m);
    const long long t0 = clock64();
    for (;;) {
      uint32_t done;
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}\n"
          : "=r"(done)
          : "r"(a), "r"(parity)
          : "memory");
      if (done) return;
      if (clock64() - t0 > 4000000000LL) __trap();
    }
  }
  // TMA 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier
  static __device__ __forceinline__ void bulk_g2s(Ctx& c, uint32_t dst_saddr, const void* gsrc, uint32_t bytes, Mbar* m) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst_saddr),
                 "l"(gsrc), "r"(bytes), "r"(saddr(c, m))
                 : "memory");
  }
  // TMA tensor copy (tiled mode, 3-D): one box [box2][box1][box0] global -> shared, dense, out-of-bounds elements zero;
  // the whole box is credited to the mbarrier.  SASS: UTMALDG.
  using TensorMap = CUtensorMap;
  static __device__ __forceinline__ void tma_load_3d(Ctx& c, uint32_t dst_saddr, const TensorMap* tm, int x, int y, int z, Mbar* m) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n" ::"r"(dst_saddr),
        "l"(tm), "r"(x), "r"(y), "r"(z), "r"(saddr(c, m))
        : "memory");
  }
  static __device__ __forceinline__ void tma_prefetch_desc(const TensorMap* tm) {
    asm volatile("prefetch.tensormap [%0];\n" ::"l"(tm) : "memory");
  }
  static __device__ __forceinline__ void tmem_alloc(Ctx& c, uint32_t* slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(saddr(c, slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  static __device__ __forceinline__ void tmem_dealloc(Ctx&, uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "r"(cols) : "memory");
  }
  // kind::f16: FP16 or BF16 operands, chosen by the instruction descriptor's format fields
  static __device__ __forceinline__ void mma_f16(Ctx&, uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t acc) {
    constexpr uint32_t HI = (128u >> 4) | (1u << 14);     // SBO = 128 bytes, descriptor version 1
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}\n" ::"r"(tmem_d),
        "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(acc), "r"(HI)
        : "memory");
  }
  static __device__ __forceinline__ void mma_tf32(Ctx&, uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t acc) {
    constexpr uint32_t HI = (128u >> 4) | (1u << 14);
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, p;\n\t}\n" ::"r"(tmem_d),
        "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(acc), "r"(HI)
        : "memory");
  }
  static __device__ __forceinline__ float to_tf32(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
  }
  static __device__ __forceinline__ float ldg(const float* p) { return __ldg(p); }
  static __device__ __forceinline__ void mma_commit(Ctx& c, Mbar* m) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(saddr(c, m)) : "memory");
  }
  static __device__ __forceinline__ void tmem_ld16(Ctx&, uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
  }
  // two 16-column loads in flight behind ONE tcgen05.wait::ld (the single form waits after every load: with 2 or 4
  // accumulators per chunk the epilogue paid the TMEM latency 2 - 4 times per item)
  static __device__ __forceinline__ void tmem_ld16x2(Ctx&, uint32_t taddr0, uint32_t taddr1, float (&v)[16], float (&w)[16]) {
    uint32_t r[16], s[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr0));
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]), "=r"(s[3]), "=r"(s[4]), "=r"(s[5]), "=r"(s[6]), "=r"(s[7]), "=r"(s[8]),
          "=r"(s[9]), "=r"(s[10]), "=r"(s[11]), "=r"(s[12]), "=r"(s[13]), "=r"(s[14]), "=r"(s[15])
        : "r"(taddr1));
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) { v[i] = __uint_as_float(r[i]); w[i] = __uint_as_float(s[i]); }
  }
  static __device__ __forceinline__ void tmem_st16(Ctx&, uint32_t taddr, const float* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
  }
  static __device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }
  // (a, b) -> packed hi pair and packed lo pair of the two-term split x = hi + lo: one cvt.rn.f16x2.f32 for the hi pair, two
  // cvt.f32.f16 to get it back, two subtractions, one cvt for the lo pair (the element-wise form spent 10 conversions here)
  static __device__ __forceinline__ void split2_f16(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(a, b);           // .x = a (low half)
    const __half2 l = __floats2half2_rn(a - __low2float(h), b - __high2float(h));
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
  }
  static __device__ __forceinline__ void split2_bf16(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    const __nv_bfloat162 l = __floats2bfloat162_rn(a - __low2float(h), b - __high2float(h));
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
  }
  static __device__ __forceinline__ float f16_round(float v) { return __half2float(__float2half_rn(v)); }
  static __device__ __forceinline__ uint32_t pack_f16(float a, float b) {
    __half2 v = __floats2half2_rn(a, b);                 // .x = a (low half), .y = b
    return *reinterpret_cast<uint32_t*>(&v);
  }
  static __device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
  static __device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);   // .x = a (low half), .y = b
    return *reinterpret_cast<uint32_t*>(&v);
  }
};

}  // namespace
}  // namespace pb200
