// Shared device helpers for the B200 (sm_100a) AWQ W4A16 kernels.
// Raw PTX wrappers only: mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05 (alloc/mma/commit/ld),
// int4 -> fp16 unpack tricks.  No CUTLASS/CuTe, no torch.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace b200awq {

#ifndef B200AWQ_SM_COUNT_FALLBACK
#define B200AWQ_SM_COUNT_FALLBACK 148
#endif

// ------------------------------------------------------------------------------------ misc
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// streaming 128-bit global load, read-only path, do not keep in L1
__device__ __forceinline__ uint4 ldg_stream_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ uint2 ldg_stream_u2(const void* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ uint32_t ldg_stream_u1(const void* p) {
  uint32_t r;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
// L2-only (coherent across SMs) loads for split-K partials written by other CTAs
__device__ __forceinline__ float4 ldcg_f4(const void* p) {
  float4 r;
  asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ float ldcg_f1(const void* p) {
  float r;
  asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}

// Split-K hand-off without sequentially-consistent fences (__threadfence() = fence.sc.gpu = MEMBAR.SC.GPU +
// L1 invalidate, measured at microseconds in the GEMV tail): contributors add with relaxed REDs, synchronise
// on a CTA barrier, ONE thread bumps the ticket with acq_rel at gpu scope (release is cumulative over what the
// barrier ordered before it); the thread that sees the final count acquires, and the barrier after it orders
// the rest of the CTA.
__device__ __forceinline__ void red_add_f32(float* p, float v) {
  asm volatile("red.relaxed.gpu.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ int atom_add_acq_rel(int* p, int v) {
  int old;
  asm volatile("atom.acq_rel.gpu.global.add.s32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
// Cross-CTA completion counters of the decode-program kernel: producers of a result release-add after a CTA
// barrier, consumers poll with an acquiring load (then a CTA barrier orders the rest of the CTA).
__device__ __forceinline__ void red_release_add_s32(int* p, int v) {
  asm volatile("red.release.gpu.global.add.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_s32(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint4 ldcg_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ float ld_relaxed_f32(const float* p) {
  float v;
  asm volatile("ld.relaxed.gpu.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}

// Programmatic dependent launch (PDL): a kernel launched with the programmatic-stream-serialization
// attribute may start while its predecessor is still running.  pdl_trigger() lets OUR successor start
// early; pdl_wait() blocks until the predecessor grid has completed and its writes are visible - it must
// precede every access to memory the predecessor may write (activations, workspace, outputs).  Loads of
// the packed weights (never written on the stream) are issued BEFORE pdl_wait(): consecutive linears
// then stream weights back to back.  Both are no-ops for a normally launched kernel.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ void sts_u4(uint32_t saddr, const uint4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ----------------------------------------------------------------------- int4 -> fp16 unpack
// (a & b) | c in one LOP3
__device__ __forceinline__ uint32_t lop3_and_or(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ __half2 u32_as_h2(uint32_t v) { return *reinterpret_cast<__half2*>(&v); }
__device__ __forceinline__ uint32_t h2_as_u32(__half2 v) { return *reinterpret_cast<uint32_t*>(&v); }

// f32 += f16 * f16 (exact product, single fp32 rounding); SASS: FHFMA (sm_100+)
__device__ __forceinline__ float fhfma(uint16_t a, uint16_t b, float c) {
  float d;
  asm("fma.rn.f32.f16 %0, %1, %2, %3;" : "=f"(d) : "h"(a), "h"(b), "f"(c));
  return d;
}
__device__ __forceinline__ uint16_t lo16(uint32_t v) { return static_cast<uint16_t>(v & 0xffffu); }
__device__ __forceinline__ uint16_t hi16(uint32_t v) { return static_cast<uint16_t>(v >> 16); }

// One AWQ GEMM-layout word holds 8 output columns of one k.  Pair t = columns (2t, 2t+1) sits in
// bits [4t, 4t+4) of the low / high half-word.  raw pairs as fp16 bit patterns:
//   kind A (t = 0, 2): 0x6400 | q        = 1024 + q
//   kind B (t = 1, 3): 0x6400 | (q << 4) = 1024 + 16 q
struct RawPairs {
  uint32_t p[4];
};
__device__ __forceinline__ RawPairs awq_raw_pairs(uint32_t w) {
  RawPairs r;
  const uint32_t w8 = w >> 8;
  r.p[0] = lop3_and_or(w, 0x000f000fu, 0x64006400u);
  r.p[1] = lop3_and_or(w, 0x00f000f0u, 0x64006400u);
  r.p[2] = lop3_and_or(w8, 0x000f000fu, 0x64006400u);
  r.p[3] = lop3_and_or(w8, 0x00f000f0u, 0x64006400u);
  return r;
}
// Zero-point operands for exact (q - z): kind A uses HSUB2 with (1024 + z); kind B uses
// HFMA2(raw, 1/16, -(64 + z)).  Both results are exact small integers in fp16.
struct ZeroPairs {
  __half2 z[4];
};
__device__ __forceinline__ ZeroPairs awq_zero_pairs(uint32_t zw) {
  RawPairs r = awq_raw_pairs(zw);
  ZeroPairs z;
  const __half2 m16 = __float2half2_rn(-0.0625f);
  z.z[0] = u32_as_h2(r.p[0]);
  z.z[1] = __hmul2(u32_as_h2(r.p[1]), m16);  // -(64 + z), exact
  z.z[2] = u32_as_h2(r.p[2]);
  z.z[3] = __hmul2(u32_as_h2(r.p[3]), m16);
  return z;
}
// Bit-exact dequant of one word: out[t] = fp16((q - z) * s) for column pair t, natural column order.
__device__ __forceinline__ uint4 awq_dequant_word(uint32_t w, const ZeroPairs& z, const uint4& s) {
  RawPairs r = awq_raw_pairs(w);
  const __half2 r16 = __float2half2_rn(0.0625f);
  __half2 d0 = __hsub2(u32_as_h2(r.p[0]), z.z[0]);
  __half2 d1 = __hfma2(u32_as_h2(r.p[1]), r16, z.z[1]);
  __half2 d2 = __hsub2(u32_as_h2(r.p[2]), z.z[2]);
  __half2 d3 = __hfma2(u32_as_h2(r.p[3]), r16, z.z[3]);
  uint4 o;
  o.x = h2_as_u32(__hmul2(d0, u32_as_h2(s.x)));
  o.y = h2_as_u32(__hmul2(d1, u32_as_h2(s.y)));
  o.z = h2_as_u32(__hmul2(d2, u32_as_h2(s.z)));
  o.w = h2_as_u32(__hmul2(d3, u32_as_h2(s.w)));
  return o;
}

// ---------------------------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// non-blocking probe (try_wait may suspend the calling thread for a system-dependent time; a warp whose lanes poll
// DIFFERENT barriers must not let one lane's suspension stall the others: see the converged producer loops)
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// generic-proxy smem writes -> visible to the async proxy (TMA / tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
// 2-D tiled load global -> smem, completion on mbarrier (bytes)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// L2 prefetch of a 2-D tile (no shared-memory destination, no completion tracking)
__device__ __forceinline__ void tma_prefetch_l2_2d(const void* tmap, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(tmap), "r"(c0), "r"(c1) : "memory");
}
// L2 prefetch hint for one 128-byte line (a hint: dropped, not faulted, if the address cannot be translated)
__device__ __forceinline__ void prefetch_l2_line(const void* gsrc) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(gsrc) : "memory");
}
// 1-D bulk copy global -> smem (no tensor map), completion on mbarrier (bytes); size % 16 == 0
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ------------------------------------------------------------------------------------ tcgen05
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], kind::f16 (fp16/bf16 inputs, fp32 accumulate)
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued tcgen05.mma of this thread arrive on the mbarrier when complete
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 columns of fp32: thread i of the warp gets lane (base_lane + i), 32 consecutive columns
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory matrix descriptor (sm_100): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout type [61,64) (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// kind::f16 instruction descriptor: D fp32, A/B fp16; majors: 0 = K-major, 1 = MN-major
__host__ __device__ constexpr uint32_t umma_idesc_f16(int m, int n, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (static_cast<uint32_t>(a_mn_major) << 15) | (static_cast<uint32_t>(b_mn_major) << 16) |
         (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

}  // namespace b200awq
