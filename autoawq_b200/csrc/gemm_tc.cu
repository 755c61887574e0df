// Tensor-core path (M > 8 tokens): Y[M, N] = X[M, K] . deq(W), fp16 x fp16 -> fp32 in TMEM (tcgen05).
//
// Orientation ("swap-AB"): the MMA's M dimension is the OUTPUT-FEATURE axis n (128 per tile, the only
// M the 1-CTA UMMA runs at full rate), the MMA's N dimension is the token axis (BT = 32..256 per tile).
//   A operand = W^T tile [128 n x 64 k]  - produced IN-KERNEL: 4 warps read packed int4 words, dequantise
//               in registers (bit-exact with the dequant kernel) and store fp16 into shared memory in the
//               UMMA canonical 128B-swizzled layout (MN-major for the GEMM layout, whose words hold 8
//               consecutive n of one k; K-major for the GEMV / GEMVFast layouts, whose words hold
//               consecutive k of one n).
//   B operand = X tile [BT tokens x 64 k], K-major, 128B swizzle, loaded by TMA (cp.async.bulk.tensor.2d).
//   D         = [128 lanes (n) x BT columns (tokens)] fp32 in tensor memory.
// Warp roles (448 threads): warp 0 = TMA producer, warp 1 = TMEM owner + single-thread MMA issuer,
// warps 2..5 = epilogue (tcgen05.ld -> +bias -> fp16 -> global), warps 6.. = dequant producers (16 for the GEMM layout).
// Pipeline: NS smem stages, one "full" mbarrier per stage (8 producer-warp arrivals + 1 TMA expect_tx),
// one "empty" mbarrier per stage (tcgen05.commit); two TMEM accumulator buffers with tmem_full /
// tmem_empty mbarriers, so the epilogue of one tile overlaps the main loop of the next.
// Persistent CTAs walk (n_tile, m_tile, k_split) work items.  Split-K (only for M <= 256 and fewer tiles than SMs, where
// the problem is HBM-bound and 148 SMs must all stream weights) reduces through fp32 atomics into the
// caller's zeroed workspace; the last CTA of a tile rounds to fp16 and restores the zeros.
#include <cuda.h>

#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "kernels.h"

namespace b200awq {

constexpr int kTileN = 128;  // output features per tile (UMMA M)
constexpr int kBK = 64;      // k per pipeline stage (one 128B swizzle row of fp16)
constexpr int kAStageBytes = kTileN * kBK * 2;  // 16 KB

struct TcParams {
  const int32_t* qweight;
  const __half* scales;
  const int32_t* qzeros;  // FAST layout: scaled zeros (fp16) reinterpret
  const __half* bias;
  __half* y;
  float* acc_ws;
  int* tickets;
  int M, K, N, G;
  int zw;          // GEMV layout: zeros width
  int n_tiles, m_tiles, ksplit;
  int has_tmq;     // GEMM layout: a tensor map over qweight is available for L2 prefetch
  int g_shift;     // log2(G) when G is a power of two, else 31 (G == K: one group) - no integer division on device
  int dbg;         // small-M kernel: record phase timestamps (knob 3 == 9)
};

template <int BT>
struct TcCfg {
  static constexpr int kXStageBytes = BT * kBK * 2;
  static constexpr int kStageBytes = kAStageBytes + kXStageBytes;
  static constexpr int kStages = (BT >= 256) ? 4 : (BT >= 128 ? 6 : 8);
  static constexpr int kTmemCols = 2 * (BT < 32 ? 32 : BT);  // two accumulator buffers
  static constexpr size_t kSmemBytes = (size_t)kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ------------------------------------------------------------------------------- A-tile producers
// 256 or 512 producer threads.  load() issues the global loads of one k-step (packed words plus,
// when the quantisation group changes, the group's zeros / scales) ONE STEP AHEAD of store(), which
// dequantises from registers and writes the swizzled fp16 tile: no global latency on the critical path.

// GEMM layout: thread dt owns word column c = dt % 16 (8 n) and rows kk = dt/16 + 16 j, j = 0..3.
// (A 512-thread variant with 2 rows per thread measured slower: 725 vs 838 TFLOP/s at M = 4096.)
// NG = quantisation groups per 64-row k-step: 1 for G >= 64, 2 for G == 32 (rows < 32 / >= 32).  Keeping the
// slot small (9 registers for NG = 1) is what allows a 6-deep register prefetch ring.
template <int NG>
struct GemmLayoutLoaderT {
  static constexpr int kThreads = 256;
  static constexpr int kDepth = NG == 1 ? 6 : 4;
  uint32_t q[4];
  uint32_t zq[NG];
  uint4 sc[NG];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int h = 0; h < NG; ++h) { zq[h] = 0; sc[h] = make_uint4(0, 0, 0, 0); }
  }
  __device__ __forceinline__ void load(const TcParams& p, int nt, int k0, int dt) {
    // 32-bit word offsets (K * N/8 < 2^32 for every real shape) keep the address arithmetic to a few
    // instructions per load; the first version spent ~90 instructions per k-step on 64-bit multiplies.
    const uint32_t NW = (uint32_t)p.N >> 3;
    const uint32_t c = dt & 15, rb = dt >> 4;
    const uint32_t wc = (uint32_t)nt * 16 + c;
    const bool ok = wc < NW;
    const uint32_t row0 = ((uint32_t)k0 + rb) * NW + wc;
    const uint32_t row16 = 16u * NW;
    const int32_t* src = p.qweight + row0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      q[j] = 0u;
      if (ok) q[j] = ldg_stream_u1(src + j * row16);
    }
#pragma unroll
    for (int h = 0; h < NG; ++h) {
      const int g = (k0 + (int)rb + 32 * h) >> p.g_shift;   // G is a power of two, or the single group G == K
      if (ok) {
        const uint32_t goff = (uint32_t)g * NW + wc;
        zq[h] = static_cast<uint32_t>(__ldg(p.qzeros + goff));
        sc[h] = __ldg(reinterpret_cast<const uint4*>(p.scales) + goff);  // 8 halves per word column
      }
    }
  }
  __device__ __forceinline__ void store(const TcParams& p, int nt, int k0, int dt, uint32_t a_stage) const {
    const int c = dt & 15, rb = dt >> 4;
    // columns past N keep q = 0, zeros = 0, scales = 0 from init(): they dequantise to exact zeros
    ZeroPairs zp[NG];
#pragma unroll
    for (int h = 0; h < NG; ++h) zp[h] = awq_zero_pairs(zq[h]);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int h = NG == 1 ? 0 : (j >> 1);
      const uint4 o = awq_dequant_word(q[j], zp[h], sc[h]);
      // MN-major SW128: (n/64)*8192 + (k/8)*1024 + (k%8)*128 + (((n%64)/8) ^ (k%8))*16 ; k = rb + 16 j
      const uint32_t off = (uint32_t)(c >> 3) * 8192u + (uint32_t)(2 * j + (rb >> 3)) * 1024u +
                           (uint32_t)(rb & 7) * 128u + (uint32_t)(((c & 7) ^ (rb & 7)) << 4);
      sts_u4(a_stage + off, o);
    }
  }
};

// GEMV layout: thread dt owns k-word cw = dt % 8 (8 consecutive k) and rows n = dt/8 + 32 j, j = 0..3.
struct GemvLayoutLoader {
  static constexpr int kThreads = 256;
  static constexpr int kDepth = 4;
  uint32_t q[4];
  uint32_t zs[4];  // per row: fp16 scale in the low half, zero-point (0..15) in the high half
  __device__ __forceinline__ void init() { zs[0] = zs[1] = zs[2] = zs[3] = 0; }
  __device__ __forceinline__ void load(const TcParams& p, int nt, int k0, int dt) {
    const int KW = p.K >> 3;
    const int cw = dt & 7, rb = dt >> 3;
    const int g = (k0 + cw * 8) >> p.g_shift;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = nt * kTileN + rb + 32 * j;
      q[j] = 0u;
      if (n < p.N) {
        q[j] = ldg_stream_u1(p.qweight + (int64_t)n * KW + (k0 >> 3) + cw);
        const uint32_t s = __half_as_ushort(__ldg(p.scales + (int64_t)n * (p.zw * 8) + g));
        const uint32_t zword = static_cast<uint32_t>(__ldg(p.qzeros + (int64_t)n * p.zw + (g >> 3)));
        zs[j] = s | (((zword >> (4 * (g & 7))) & 0xFu) << 16);
      }
    }
  }
  __device__ __forceinline__ void store(const TcParams& p, int nt, int k0, int dt, uint32_t a_stage) const {
    const int cw = dt & 7, rb = dt >> 3;
    const __half2 r16 = __float2half2_rn(0.0625f);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int nl = rb + 32 * j;
      const int n = nt * kTileN + nl;
      uint4 o = make_uint4(0, 0, 0, 0);
      if (n < p.N) {
        const float zf = static_cast<float>(zs[j] >> 16);
        const __half2 zA = __float2half2_rn(1024.f + zf);   // exact
        const __half2 zB = __float2half2_rn(-(64.f + zf));  // exact
        const __half2 s2 = __half2half2(__ushort_as_half(static_cast<unsigned short>(zs[j] & 0xffffu)));
        RawPairs r = awq_raw_pairs(q[j]);
        // pairs (k0,k4) (k1,k5) (k2,k6) (k3,k7)
        const uint32_t d0 = h2_as_u32(__hmul2(__hsub2(u32_as_h2(r.p[0]), zA), s2));
        const uint32_t d1 = h2_as_u32(__hmul2(__hfma2(u32_as_h2(r.p[1]), r16, zB), s2));
        const uint32_t d2 = h2_as_u32(__hmul2(__hsub2(u32_as_h2(r.p[2]), zA), s2));
        const uint32_t d3 = h2_as_u32(__hmul2(__hfma2(u32_as_h2(r.p[3]), r16, zB), s2));
        o.x = __byte_perm(d0, d1, 0x5410);  // (k0, k1)
        o.y = __byte_perm(d2, d3, 0x5410);  // (k2, k3)
        o.z = __byte_perm(d0, d1, 0x7632);  // (k4, k5)
        o.w = __byte_perm(d2, d3, 0x7632);  // (k6, k7)
      }
      // K-major SW128: row n * 128 B, 16-byte chunk (k/8) ^ (n % 8)
      const uint32_t off = (uint32_t)nl * 128u + (uint32_t)((cw ^ (nl & 7)) << 4);
      sts_u4(a_stage + off, o);
    }
  }
};

// GEMVFast layout: thread dt owns row n = dt/2 of the tile and the 32-k half h = dt%2 of the step.
struct FastLayoutLoader {
  static constexpr int kThreads = 256;
  static constexpr int kDepth = 4;
  uint4 q;
  uint32_t ss;  // scale (low half) | scaled zero (high half)
  __device__ __forceinline__ void init() { ss = 0; }
  __device__ __forceinline__ void load(const TcParams& p, int nt, int k0, int dt) {
    const int n = nt * kTileN + (dt >> 1), h = dt & 1;
    q = make_uint4(0, 0, 0, 0);
    const int g = (k0 + 32 * h) >> p.g_shift;
    if (n < p.N) {
      // 64-k block k0/64 of row group n/4 starts at int16 offset k0; run (n%4) * 16; half h * 8
      q = ldg_stream_u4(reinterpret_cast<const int16_t*>(p.qweight) + (int64_t)(n >> 2) * p.K + (int64_t)k0 +
                        (n & 3) * 16 + h * 8);
      const __half* sz_ptr = reinterpret_cast<const __half*>(p.qzeros);
      ss = static_cast<uint32_t>(__half_as_ushort(__ldg(p.scales + (int64_t)g * p.N + n))) |
           (static_cast<uint32_t>(__half_as_ushort(__ldg(sz_ptr + (int64_t)g * p.N + n))) << 16);
    }
  }
  __device__ __forceinline__ void store(const TcParams& p, int nt, int k0, int dt, uint32_t a_stage) const {
    const int nl = dt >> 1, h = dt & 1;
    const bool ok = nt * kTileN + nl < p.N;
    const __half2 r16 = __float2half2_rn(0.0625f);
    const __half2 m1024 = __float2half2_rn(1024.f), m64 = __float2half2_rn(-64.f);
    const __half2 s2 = __half2half2(__ushort_as_half(static_cast<unsigned short>(ss & 0xffffu)));
    const __half2 z2 = __half2half2(__ushort_as_half(static_cast<unsigned short>(ss >> 16)));
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
    uint32_t d[4][4];  // [word u][r'] : pair (k, k+1), k = 32h + 2u + 8r'
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      RawPairs r = awq_raw_pairs(w[u]);
      d[u][0] = h2_as_u32(__hfma2(__hsub2(u32_as_h2(r.p[0]), m1024), s2, z2));
      d[u][1] = h2_as_u32(__hfma2(__hfma2(u32_as_h2(r.p[1]), r16, m64), s2, z2));
      d[u][2] = h2_as_u32(__hfma2(__hsub2(u32_as_h2(r.p[2]), m1024), s2, z2));
      d[u][3] = h2_as_u32(__hfma2(__hfma2(u32_as_h2(r.p[3]), r16, m64), s2, z2));
    }
#pragma unroll
    for (int rp = 0; rp < 4; ++rp) {
      uint4 o = make_uint4(d[0][rp], d[1][rp], d[2][rp], d[3][rp]);  // k = 32h + 8rp + 0..7
      if (!ok) o = make_uint4(0, 0, 0, 0);
      const int cc = 4 * h + rp;
      const uint32_t off = (uint32_t)nl * 128u + (uint32_t)((cc ^ (nl & 7)) << 4);
      sts_u4(a_stage + off, o);
    }
  }
};

template <int LAYOUT>
struct LoaderOf;
template <> struct LoaderOf<0> { using T = GemmLayoutLoaderT<1>; };  // GEMM layout, G >= 64
template <> struct LoaderOf<3> { using T = GemmLayoutLoaderT<2>; };  // GEMM layout, G == 32
template <> struct LoaderOf<1> { using T = GemvLayoutLoader; };
template <> struct LoaderOf<2> { using T = FastLayoutLoader; };

// --------------------------------------------------------------------------------------- kernel
// warps: 0 = TMA producer, 1 = MMA issuer / TMEM owner, 2..5 = epilogue (TMEM lane quadrant = warp % 4),
// 6..13 = dequant producers.  Two TMEM accumulator buffers: the epilogue of tile i overlaps the main loop
// of tile i+1.
template <int LAYOUT>
constexpr int tc_threads() { return 64 + 128 + LoaderOf<LAYOUT>::T::kThreads; }

template <int BT, int LAYOUT>
__global__ void __launch_bounds__(tc_threads<LAYOUT>(), 1)
    gemm_tc_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmq,
                   const TcParams p) {
  using Cfg = TcCfg<BT>;
  constexpr int NS = Cfg::kStages;
  constexpr int NPROD = LoaderOf<LAYOUT>::T::kThreads;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_base = smem;                                  // NS x 16 KB
  uint8_t* x_base = smem + (size_t)NS * kAStageBytes;      // NS x BT*128 B
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)NS * Cfg::kStageBytes);
  uint64_t* full = bars;            // [NS]
  uint64_t* empty = bars + NS;      // [NS]
  uint64_t* tmem_full = bars + 2 * NS;       // [2]
  uint64_t* tmem_empty = bars + 2 * NS + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NS + 4);
  int* s_flag = reinterpret_cast<int*>(bars + 2 * NS + 5);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  pdl_trigger();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmx);
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], NPROD / 32 + 1);  // one elected arrival per producer warp + the TMA expect_tx
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], 128);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int KS = p.K / kBK;  // k-steps in total
  const int n_work = p.n_tiles * p.m_tiles * p.ksplit;

  if (warp == 0) {
    // ================================================================= TMA producer (X tiles)
    // The whole warp walks the loop and one elected lane issues (see the MMA warp below for why).
    {
      const bool leader = elect_one();
      // GEMM layout: pull the packed weights of the next kL2Ahead k-steps from HBM into L2 (TMA prefetch, no
      // smem destination) so that the producers' register prefetch only has to cover L2 latency.  Weights
      // do not depend on the predecessor kernel: this starts before the PDL wait.
      constexpr int kL2Ahead = 16;
      int wp = blockIdx.x, sp = 0, sp_end = 0;
      bool pf_valid = (LAYOUT == 0 || LAYOUT == 3) && p.has_tmq && wp < n_work;
      auto pf_range = [&]() {
        const int ks = wp % p.ksplit;
        sp = (int)((int64_t)KS * ks / p.ksplit);
        sp_end = (int)((int64_t)KS * (ks + 1) / p.ksplit);
      };
      auto pf_step = [&]() {
        const int nt = wp / (p.ksplit * p.m_tiles);
        if (leader) tma_prefetch_l2_2d(&tmq, nt * 16, sp * kBK);
        if (++sp == sp_end) {
          wp += gridDim.x;
          if (wp < n_work) pf_range(); else pf_valid = false;
        }
      };
      if (pf_valid) pf_range();
      for (int i = 0; i < kL2Ahead && pf_valid; ++i) pf_step();
      pdl_wait();  // the activations are the predecessor's output
      int stage = 0;
      uint32_t phase = 0;
      for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
        const int ks = w % p.ksplit;
        const int mt = (w / p.ksplit) % p.m_tiles;
        const int s_begin = (int)((int64_t)KS * ks / p.ksplit), s_end = (int)((int64_t)KS * (ks + 1) / p.ksplit);
        for (int s = s_begin; s < s_end; ++s) {
          mbar_wait(&empty[stage], phase ^ 1);
          if (leader) {
            mbar_arrive_expect_tx(&full[stage], Cfg::kXStageBytes);
            tma_load_2d(x_base + (size_t)stage * Cfg::kXStageBytes, &tmx, &full[stage], s * kBK, mt * BT);
          }
          __syncwarp();
          if (++stage == NS) { stage = 0; phase ^= 1; }
          if (pf_valid) pf_step();
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================= MMA issuer
    // The WHOLE warp walks the loop (waits, stage bookkeeping, descriptors) and one elected lane issues, so that every
    // operand of the tcgen05 instructions is warp-uniform for the compiler (uniform registers).  Under `if (lane == 0)`
    // the same operands are divergent values and each UTCHMMA / UTCBAR came wrapped in an ELECT + 5 x R2UR + retry loop:
    // ~130 instructions and ~700 clk per k-step on ONE thread, more than the 512 clk the four 128x256x16 MMAs of a
    // k-step take (r2 ncu: tensor pipe 57 % active at M = 4096) - the issue loop, not the tensor pipe, set the pace.
    {
      constexpr uint32_t idesc = umma_idesc_f16(kTileN, BT, (LAYOUT == 0 || LAYOUT == 3) ? 1 : 0, 0);
      constexpr bool kMnMajorA = (LAYOUT == 0 || LAYOUT == 3);
      const bool leader = elect_one();
      // MN-major, SW128: LBO = stride between 64-n atoms (8192), SBO = stride between 8-k atoms (1024); K-major SW128
      // otherwise.  Descriptors advance by adding (byte offset >> 4) to the start-address field (smem < 256 KB: no carry).
      const uint64_t da0 = kMnMajorA ? umma_smem_desc(smem_u32(a_base), 8192, 1024) : umma_smem_desc(smem_u32(a_base), 16, 1024);
      const uint64_t db0 = umma_smem_desc(smem_u32(x_base), 16, 1024);
      constexpr uint32_t kAStep = kMnMajorA ? (2048u >> 4) : (32u >> 4);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int w = blockIdx.x; w < n_work; w += gridDim.x, ++it) {
        const int ks = w % p.ksplit;
        const int s_begin = (int)((int64_t)KS * ks / p.ksplit), s_end = (int)((int64_t)KS * (ks + 1) / p.ksplit);
        const int buf = it & 1;
        const uint32_t use = (uint32_t)(it >> 1) & 1u;
        mbar_wait(&tmem_empty[buf], use ^ 1);  // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BT);
        for (int s = s_begin; s < s_end; ++s) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint64_t da = da0 + (uint64_t)((uint32_t)(stage * kAStageBytes) >> 4);
          const uint64_t db = db0 + (uint64_t)((uint32_t)(stage * Cfg::kXStageBytes) >> 4);
          if (leader) {
#pragma unroll
            for (int k16 = 0; k16 < kBK / 16; ++k16)
              umma_f16_ss(d_tmem, da + (uint64_t)(k16 * kAStep), db + (uint64_t)(k16 * (32 >> 4)), idesc,
                          (s > s_begin || k16 > 0) ? 1u : 0u);
            umma_commit(&empty[stage]);  // frees this smem stage when the MMAs above retire
          }
          __syncwarp();
          if (++stage == NS) { stage = 0; phase ^= 1; }
        }
        if (leader) umma_commit(&tmem_full[buf]);  // accumulator complete
        __syncwarp();
      }
    }
  } else if (warp < 6) {
    // ================================================================= epilogue (4 warps)
    const int et = threadIdx.x - 64;  // 0..127
    const int q4 = warp & 3;          // TMEM lane quadrant this warp may read
    pdl_wait();                       // outputs / workspace may alias memory the predecessor still uses
    int it = 0;
    for (int w = blockIdx.x; w < n_work; w += gridDim.x, ++it) {
      const int mt = (w / p.ksplit) % p.m_tiles;
      const int nt = w / (p.ksplit * p.m_tiles);
      const int buf = it & 1;
      const uint32_t use = (uint32_t)(it >> 1) & 1u;
      mbar_wait(&tmem_full[buf], use);
      tc_fence_after();
      const int n = nt * kTileN + q4 * 32 + lane;
      const bool n_ok = n < p.N;
      const float bias_v = (p.bias != nullptr && n_ok) ? __half2float(p.bias[n]) : 0.f;
      const int m0 = mt * BT;
#pragma unroll 1
      for (int c0 = 0; c0 < BT; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(buf * BT + c0), v);
        tmem_ld_wait();
        if (n_ok && m0 + c0 < p.M) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int m = m0 + c0 + j;
            if (m < p.M) {
              const float f = __uint_as_float(v[j]);
              if (p.ksplit == 1)
                p.y[(int64_t)m * p.N + n] = __float2half_rn(f + bias_v);
              else
                atomicAdd(&p.acc_ws[(int64_t)m * p.N + n], f);
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tmem_empty[buf]);
      if (p.ksplit > 1) {
        __threadfence();
        named_bar_sync(1, 128);
        if (et == 0) {
          const int prev = atomicAdd(&p.tickets[nt * p.m_tiles + mt], 1);
          *s_flag = (prev == p.ksplit - 1);
        }
        named_bar_sync(1, 128);
        const bool last = *s_flag != 0;
        named_bar_sync(1, 128);  // everyone has read the flag before a later item rewrites it
        if (last) {
          __threadfence();
          if (n_ok) {
            // 16 tokens per L2 round trip (loads first, then the stores): one token at a time cost ~0.45 us each
            for (int j0 = 0; j0 < BT && m0 + j0 < p.M; j0 += 16) {
              float f[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const int m = m0 + j0 + j;
                f[j] = m < p.M ? ld_relaxed_f32(&p.acc_ws[(int64_t)m * p.N + n]) : 0.f;
              }
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const int m = m0 + j0 + j;
                if (m < p.M) {
                  p.acc_ws[(int64_t)m * p.N + n] = 0.f;
                  p.y[(int64_t)m * p.N + n] = __float2half_rn(f[j] + bias_v);
                }
              }
            }
          }
          if (et == 0) p.tickets[nt * p.m_tiles + mt] = 0;
        }
      }
    }
  } else {
    // ================================================================= dequant producers (8 warps)
    // Global loads run kPrefetch k-steps ahead of the dequantisation (register ring): a k-step is only
    // ~500 MMA cycles, well below the DRAM / L2 latency a 1-deep prefetch would expose every step.
    constexpr int kPrefetch = LoaderOf<LAYOUT>::T::kDepth;
    const int dt = threadIdx.x - 192;  // 0..255
    const uint32_t a_base_s = smem_u32(a_base);
    typename LoaderOf<LAYOUT>::T ring[kPrefetch];
    // The (work item, k-step) sequence of this CTA is ONE stream: the load cursor runs kPrefetch steps ahead
    // of the store cursor straight through tile boundaries, so the ring never drains between tiles.
    struct Cursor {
      int w, s, s_end, nt;
      bool valid;
    };
    auto set_range = [&](Cursor& c) {
      const int ks = c.w % p.ksplit;
      c.nt = c.w / (p.ksplit * p.m_tiles);
      c.s = (int)((int64_t)KS * ks / p.ksplit);
      c.s_end = (int)((int64_t)KS * (ks + 1) / p.ksplit);
    };
    auto advance = [&](Cursor& c) {
      if (++c.s == c.s_end) {
        c.w += gridDim.x;
        c.valid = c.w < n_work;
        if (c.valid) set_range(c);
      }
    };
    Cursor L, S;
    L.w = S.w = blockIdx.x;
    L.valid = S.valid = blockIdx.x < n_work;
    if (L.valid) { set_range(L); set_range(S); }
#pragma unroll
    for (int d = 0; d < kPrefetch; ++d) {
      ring[d].init();
      if (L.valid) {
        ring[d].load(p, L.nt, L.s * kBK, dt);
        advance(L);
      }
    }
    int stage = 0;
    uint32_t phase = 0;
    while (S.valid) {
#pragma unroll
      for (int d = 0; d < kPrefetch; ++d) {
        if (S.valid) {
          mbar_wait(&empty[stage], phase ^ 1);
          ring[d].store(p, S.nt, S.s * kBK, dt, a_base_s + (uint32_t)stage * kAStageBytes);
          fence_proxy_async_smem();   // every writer: generic-proxy stores -> visible to the tensor core
          __syncwarp();
          if (lane == 0) mbar_arrive(&full[stage]);  // 8 arrivals per stage instead of 256
          if (++stage == NS) { stage = 0; phase ^= 1; }
          advance(S);
          if (L.valid) {
            ring[d].load(p, L.nt, L.s * kBK, dt);
            advance(L);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------ small-M kernel (TMA-staged packed weights)
// M <= 128 on the GEMM layout is HBM-bound; the kernel above is latency-bound there (its producers pull the packed
// words L2 -> registers through a 6-deep ring: ~500-900 clk per k-step whatever the token count, r2 M sweep).  This
// variant keeps the MMA / descriptor / epilogue machinery and changes what bounded it:
//   * the packed weights arrive by TMA in a deep shared-memory ring, one stage = a PAIR of k-steps (128 rows x 16 words
//     = 8 KB, plus the rows' group constants: 256 B of scales + 64 B of zeros per group), 11-14 stages = 96-123 KB in
//     flight per SM independent of registers (a read-only probe with the same ring moves 2.5 TB/s with 64 KB in flight
//     and 3.9 TB/s with 128 KB: profiles/r02_membw_box_shapes.log), issued by a dedicated warp that never waits for
//     activations (weights do not depend on the predecessor kernel);
//   * two producer teams of 8 warps: team t dequantises rows 64 t .. 64 t + 63 of every stage (conflict-free LDS, the
//     exact arithmetic of the dequant kernel: the A tile is bit-identical), one step ahead of its own stores, into its own
//     A stages; the activation tiles have their own ring (they come from L2 with ~1 us of latency);
//   * the MMA / TMA issue loops are walked by the whole warp with one elected lane issuing (uniform operands);
//   * work is cut into CONTIGUOUS RANGES of the linearised (n-tile, k-step pair) sequence, one range per SM: every SM
//     streams the same number of bytes whatever N / 128 is (the (tile, k-split) items of the kernel above leave
//     224 tiles on 148 SMs two waves deep).  A range crosses at most a few n-tiles = segments; a segment that holds a
//     whole K column stores fp16 directly, a partial one adds fp32 into the caller's zeroed workspace and bumps the
//     tile's ticket by its number of k-step pairs; the contributor that completes K rounds, adds the bias, restores
//     zeros.  Wherever N / 128 <= SM count (and from 64 tokens on) the ranges are tile-aligned instead: gemm_tcq_grid.
//   * no HBM -> L2 prefetch ahead of the ring: measured, no gain (profiles/r02_tcq_knob20.json).
template <int BT>
struct TcqCfg {
  static constexpr int kNS = 4;                                            // A stages (producers -> MMA), 2 per team
  static constexpr int kNX = BT <= 16 ? 16 : (BT == 32 ? 8 : (BT == 64 ? 8 : 4));   // X stages (TMA -> MMA), own ring
  static constexpr int kNQ = BT <= 32 ? 14 : 11;                           // packed-weight stages (TMA -> producers)
  static constexpr int kXStageBytes = BT * kBK * 2;
  static constexpr int kQRows = 2 * kBK;                                   // rows per packed stage: one k-step per team
  static constexpr int kQTileBytes = 16 * 4 * kQRows;                      // 128 rows x 16 words = 8 KB
  static constexpr int kQStageBytes = kQTileBytes + 2 * 256 + 2 * 64 + 128;   // up to 2 groups of constants; 128-B multiple
  static constexpr int kAccCols = BT < 32 ? 32 : BT;
  static constexpr int kTeams = 2;
  // One MMA-issuing warp per team, each with its own accumulator (the epilogue adds the two): the issue loop of ONE
  // warp (two barrier waits, descriptor arithmetic on the uniform datapath, 4 MMAs, 2 commits: ~55 dependent
  // instructions) takes ~300 ns per k-step however little the tensor pipe has to do - with every other stage removed
  // (no dequantisation, no MMAs) the kernel still ran at that pace (profiles/r02_tcq_experiments.md).
  static constexpr int kTmemCols = 2 * kTeams * kAccCols;                  // two buffers x one accumulator per team
  static_assert(kTmemCols <= 512 && (kTmemCols & (kTmemCols - 1)) == 0, "TMEM allocation: power of two <= 512");
  static constexpr int kThreads = 192 + 256 * kTeams + 64;   // X-TMA, MMA 0, 4 epilogue, 16 producer warps, Q-TMA, MMA 1
  static constexpr size_t kSmemBytes = (size_t)kNS * kAStageBytes + (size_t)kNX * kXStageBytes +
                                       (size_t)kNQ * kQStageBytes + 1024 /*align slack*/ + 1024 /*barriers*/;
  static_assert(kNS % kTeams == 0 && kNX % kTeams == 0, "team t owns A stages / X stages t, t + 2, ...");
  static_assert(kQStageBytes % 128 == 0, "TMA destination alignment");
  static_assert(kSmemBytes <= 232448, "shared memory per CTA");
};

__device__ __forceinline__ uint32_t lds_u1(uint32_t saddr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr) : "memory");
  return v;
}
__device__ __forceinline__ uint4 lds_u4(uint32_t saddr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr) : "memory");
  return v;
}

// Phase timestamps (globaltimer, ns) of the last small-M launch, 8 per CTA, written only when knob 3 == 9 (TcParams::dbg):
// [0] entry, [1] setup done (barriers, TMEM), [2] first packed stage landed, [3] producers done, [4] MMA issuer done,
// [5] last accumulator drained, [6] epilogue done (incl. finalisation), [7] number of segments.
__device__ unsigned long long g_tcq_dbg[256 * 8];
__device__ __forceinline__ unsigned long long tcq_timer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
cudaError_t gemm_tcq_debug_read(void* dst, size_t bytes) {
  return cudaMemcpyFromSymbol(dst, g_tcq_dbg, bytes < sizeof(g_tcq_dbg) ? bytes : sizeof(g_tcq_dbg));
}

// Work unit = a PAIR of k-steps (128 rows of one 128-column tile); p.K % 128 == 0.
template <int BT>
__global__ void __launch_bounds__(TcqCfg<BT>::kThreads, 1)
    gemm_tcq_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmq, const TcParams p) {
  using Cfg = TcqCfg<BT>;
  constexpr int NS = Cfg::kNS, NX = Cfg::kNX, NQ = Cfg::kNQ;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_base = smem;                                              // NS x 16 KB
  uint8_t* x_base = a_base + (size_t)NS * kAStageBytes;                // NX x BT*128 B
  uint8_t* q_base = x_base + (size_t)NX * Cfg::kXStageBytes;           // NQ x kQStageBytes
  uint64_t* bars = reinterpret_cast<uint64_t*>(q_base + (size_t)NQ * Cfg::kQStageBytes);
  uint64_t* full = bars;                     // [NS]  8 producer warps (one team)
  uint64_t* empty = full + NS;               // [NS]  tcgen05.commit
  uint64_t* xfull = empty + NS;              // [NX]  expect_tx of the activation tile
  uint64_t* xempty = xfull + NX;             // [NX]  tcgen05.commit
  uint64_t* qfull = xempty + NX;             // [NQ]  expect_tx of the packed stage
  uint64_t* qempty = qfull + NQ;             // [NQ]  16 producer warps (both teams)
  uint64_t* tmem_full = qempty + NQ;         // [2]
  uint64_t* tmem_empty = tmem_full + 2;      // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  int* s_flag = reinterpret_cast<int*>(tmem_empty + 3);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  pdl_trigger();
  const bool dbg = p.dbg != 0 && blockIdx.x < 256;
  unsigned long long* dbg_row = g_tcq_dbg + blockIdx.x * 8;
  if (dbg && threadIdx.x == 0) dbg_row[0] = tcq_timer();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmx);
    tma_prefetch_desc(&tmq);
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], 8);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < NX; ++s) {
      mbar_init(&xfull[s], 1);
      mbar_init(&xempty[s], 1);
    }
    for (int s = 0; s < NQ; ++s) {
      mbar_init(&qfull[s], 1);
      mbar_init(&qempty[s], 8 * Cfg::kTeams);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], Cfg::kTeams);   // one commit per MMA warp
      mbar_init(&tmem_empty[b], 128);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (dbg && threadIdx.x == 0) dbg_row[1] = tcq_timer();

  // this CTA's contiguous range of the linearised (n-tile, k-step pair) sequence
  const int KP = p.K / Cfg::kQRows;   // k-step pairs per tile
  const long long T = (long long)p.n_tiles * KP;
  const int t_begin = (int)(T * (long long)blockIdx.x / (long long)gridDim.x);
  const int t_end = (int)(T * (long long)(blockIdx.x + 1) / (long long)gridDim.x);
  constexpr int kQWarp = 6 + 8 * Cfg::kTeams;
  // groups of constants per packed stage: G = 64 -> one per k-step; G >= 128 (or one group per row) -> one per pair
  const int ng = p.g_shift == 6 ? 2 : 1;

  if (warp == kQWarp) {
    // ================================================================= Q-TMA: packed weights + group constants
    // (the whole warp walks the loop, one elected lane issues: uniform operands, no per-instruction retry loops)
    {
      const bool leader = elect_one();
      const uint32_t NW = (uint32_t)p.N >> 3;
      const uint32_t tx = (uint32_t)Cfg::kQTileBytes + (uint32_t)ng * 320u;
      int qs = 0;
      uint32_t qph = 0;
      for (int t = t_begin; t < t_end;) {
        const int nt = t / KP, d0 = t - nt * KP;
        const int d1 = (KP - d0 < t_end - t) ? KP : d0 + (t_end - t);
        for (int d = d0; d < d1; ++d) {
          mbar_wait(&qempty[qs], qph ^ 1);
          uint8_t* dst = q_base + (size_t)qs * Cfg::kQStageBytes;
          const uint32_t g = (uint32_t)(d * Cfg::kQRows) >> p.g_shift;
          if (leader) {
            mbar_arrive_expect_tx(&qfull[qs], tx);
            tma_load_2d(dst, &tmq, &qfull[qs], nt * 16, d * Cfg::kQRows);
            for (int h = 0; h < ng; ++h) {
              bulk_load_1d(dst + Cfg::kQTileBytes + h * 256, p.scales + (size_t)(g + h) * p.N + (size_t)nt * kTileN, 256,
                           &qfull[qs]);
              bulk_load_1d(dst + Cfg::kQTileBytes + 512 + h * 64, p.qzeros + (size_t)(g + h) * NW + (size_t)nt * 16, 64,
                           &qfull[qs]);
            }
          }
          __syncwarp();
          if (++qs == NQ) { qs = 0; qph ^= 1; }
        }
        t += d1 - d0;
      }
    }
  } else if (warp == 0) {
    // ================================================================= X-TMA: activation tiles, own ring (the tiles
    // come from L2 with ~1 us of latency: tying them to the A stages made that latency the k-step time)
    {
      const bool leader = elect_one();
      pdl_wait();  // the activations are the predecessor's output
      int xs = 0;
      uint32_t xph = 0;
      for (int t = t_begin; t < t_end;) {
        const int nt = t / KP, d0 = t - nt * KP;
        const int d1 = (KP - d0 < t_end - t) ? KP : d0 + (t_end - t);
        for (int s = 2 * d0; s < 2 * d1; ++s) {
          mbar_wait(&xempty[xs], xph ^ 1);
          if (leader) {
            mbar_arrive_expect_tx(&xfull[xs], Cfg::kXStageBytes);
            tma_load_2d(x_base + (size_t)xs * Cfg::kXStageBytes, &tmx, &xfull[xs], s * kBK, 0);
          }
          __syncwarp();
          if (++xs == NX) { xs = 0; xph ^= 1; }
        }
        t += d1 - d0;
      }
    }
  } else if (warp == 1 || warp == kQWarp + 1) {
    // ================================================================= MMA issuers (warp 1: team 0, last warp: team 1)
    // The WHOLE warp walks the loop (waits, stage bookkeeping, descriptors) and one elected lane issues: everything the
    // tcgen05 instructions consume is then warp-uniform for the compiler (uniform registers).  Under `if (lane == 0)`
    // the same operands are divergent values, and every UTCHMMA / UTCBAR came wrapped in an ELECT + 5 x R2UR + retry
    // loop: ~130 instructions and ~700 clk per k-step on ONE thread - the k-step time of the first version (ncu source
    // page: the producers' top stall was the wait for the MMA's stage release).
    // MMA warp w serves team w: k-step w of every pair (A stages w, w + 2; X stages w, w + 2, ...), accumulator w.
    {
      constexpr uint32_t idesc = umma_idesc_f16(kTileN, BT, 1, 0);
      const int mw = warp == 1 ? 0 : 1;
      const bool leader = elect_one();
      const uint32_t a_base_s = smem_u32(a_base), x_base_s = smem_u32(x_base);
      const uint64_t da0 = umma_smem_desc(a_base_s, 8192, 1024);   // MN-major SW128; start address in bits [0, 14)
      const uint64_t db0 = umma_smem_desc(x_base_s, 16, 1024);     // K-major SW128
      int stage = mw, xs = mw;
      uint32_t phase = 0, xph = 0;
      int it = 0;
      for (int t = t_begin; t < t_end; ++it) {
        const int nt = t / KP, d0 = t - nt * KP;
        const int d1 = (KP - d0 < t_end - t) ? KP : d0 + (t_end - t);
        const int buf = it & 1;
        const uint32_t use = (uint32_t)(it >> 1) & 1u;
        mbar_wait(&tmem_empty[buf], use ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)((buf * Cfg::kTeams + mw) * Cfg::kAccCols);
        for (int d = d0; d < d1; ++d) {
          mbar_wait(&xfull[xs], xph);
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          // descriptors advance by adding (byte offset >> 4) to the start-address field (no carry: smem < 256 KB)
          const uint64_t da = da0 + (uint64_t)((uint32_t)(stage * kAStageBytes) >> 4);
          const uint64_t db = db0 + (uint64_t)((uint32_t)(xs * Cfg::kXStageBytes) >> 4);
          if (leader) {
#pragma unroll
            for (int k16 = 0; k16 < kBK / 16; ++k16)
              umma_f16_ss(d_tmem, da + (uint64_t)(k16 * (2048 >> 4)), db + (uint64_t)(k16 * (32 >> 4)), idesc,
                          (d > d0 || k16 > 0) ? 1u : 0u);
            umma_commit(&empty[stage]);
            umma_commit(&xempty[xs]);
          }
          __syncwarp();
          stage += Cfg::kTeams;
          if (stage >= NS) { stage -= NS; phase ^= 1; }
          xs += Cfg::kTeams;
          if (xs >= NX) { xs -= NX; xph ^= 1; }
        }
        if (leader) umma_commit(&tmem_full[buf]);
        __syncwarp();
        t += d1 - d0;
      }
      if (dbg && leader && mw == 0) { dbg_row[4] = tcq_timer(); dbg_row[7] = (unsigned long long)it; }
    }
  } else if (warp < 6) {
    // ================================================================= epilogue (4 warps)
    const int et = threadIdx.x - 64;  // 0..127
    const int q4 = warp & 3;          // TMEM lane quadrant this warp may read
    pdl_wait();                       // outputs / workspace may alias memory the predecessor still uses
    int it = 0;
    for (int t = t_begin; t < t_end; ++it) {
      const int nt = t / KP, d0 = t - nt * KP;
      const int d1 = (KP - d0 < t_end - t) ? KP : d0 + (t_end - t);
      const bool whole = (d0 == 0 && d1 == KP);
      const int buf = it & 1;
      const uint32_t use = (uint32_t)(it >> 1) & 1u;
      mbar_wait(&tmem_full[buf], use);
      tc_fence_after();
      const int n = nt * kTileN + q4 * 32 + lane;   // N % 128 == 0: always in range
      const float bias_v = p.bias != nullptr ? __half2float(p.bias[n]) : 0.f;
      const uint32_t tbuf = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(buf * Cfg::kTeams * Cfg::kAccCols);
#pragma unroll 1
      for (int c0 = 0; c0 < BT; c0 += 16) {
        // the two teams' accumulators of 16 tokens, added in a fixed order
        uint32_t v[16], w[16];
        tmem_ld_32x16(tbuf + (uint32_t)c0, v);
        tmem_ld_32x16(tbuf + (uint32_t)(Cfg::kAccCols + c0), w);
        tmem_ld_wait();
        if (c0 < p.M) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int m = c0 + j;
            if (m < p.M) {
              const float f = __uint_as_float(v[j]) + __uint_as_float(w[j]);
              if (whole)
                p.y[(int64_t)m * p.N + n] = __float2half_rn(f + bias_v);
              else
                red_add_f32(&p.acc_ws[(int64_t)m * p.N + n], f);
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tmem_empty[buf]);
      if (dbg && et == 0) dbg_row[5] = tcq_timer();
      if (!whole) {
        // relaxed REDs -> CTA-scope barrier -> one acq_rel ticket (release is cumulative over what the barrier ordered)
        named_bar_sync(1, 128);
        if (et == 0) {
          const int prev = atom_add_acq_rel(&p.tickets[nt], d1 - d0);
          *s_flag = (prev + (d1 - d0) == KP);
        }
        named_bar_sync(1, 128);
        const bool last = *s_flag != 0;
        named_bar_sync(1, 128);  // everyone has read the flag before a later segment rewrites it
        if (last) {
          // all loads of a batch of 16 tokens are in flight before the first store (one L2 round trip per batch, not
          // one per token: the first version spent 0.45 us per token here)
          for (int m0 = 0; m0 < p.M; m0 += 16) {
            float f[16];
#pragma unroll
            for (int j = 0; j < 16; ++j)
              f[j] = (m0 + j < p.M) ? ld_relaxed_f32(&p.acc_ws[(int64_t)(m0 + j) * p.N + n]) : 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              if (m0 + j < p.M) {
                p.acc_ws[(int64_t)(m0 + j) * p.N + n] = 0.f;
                p.y[(int64_t)(m0 + j) * p.N + n] = __float2half_rn(f[j] + bias_v);
              }
            }
          }
          if (et == 0) p.tickets[nt] = 0;
        }
      }
      t += d1 - d0;
    }
    if (dbg && et == 0) dbg_row[6] = tcq_timer();
  } else {
    // ================================================================= dequant producers (2 teams x 8 warps)
    // Team t owns k-step t of every packed stage (rows 64 t ..): A stages t, t + 2.  The two teams' [wait, LDS, dequant,
    // STS, proxy fence, arrive] chains overlap.
    const int pt = threadIdx.x - 192;
    const int team = pt >> 8;
    const int dt = pt & 255;  // 0..255 within the team
    const uint32_t a_base_s = smem_u32(a_base);
    const uint32_t q_base_s = smem_u32(q_base);
    const uint32_t c = dt & 15, rb = dt >> 4;
    const uint32_t q_off = ((uint32_t)team * kBK + rb) * 64u + c * 4u;    // rows 64 team + rb + 16 j of word column c
    const uint32_t gh = ng == 2 ? (uint32_t)team : 0u;                      // which group of constants of the stage
    const uint32_t sc_off = Cfg::kQTileBytes + gh * 256u + c * 16u;         // 8 scales of word column c
    const uint32_t z_off = Cfg::kQTileBytes + 512u + gh * 64u + c * 4u;     // its 8 zero-points
    using L = GemmLayoutLoaderT<1>;
    auto fetch = [&](L& r, int qs) {
      const uint32_t qa = q_base_s + (uint32_t)qs * Cfg::kQStageBytes;
#pragma unroll
      for (int j = 0; j < 4; ++j) r.q[j] = lds_u1(qa + q_off + (uint32_t)j * 1024u);
      r.sc[0] = lds_u4(qa + sc_off);
      r.zq[0] = lds_u1(qa + z_off);
    };
    const int npairs = t_end - t_begin;
    L cur, nxt;
    cur.init();
    nxt.init();
    int qs = 0, stage = team;
    uint32_t qph = 0, phase = 0;
    if (npairs > 0) {
      mbar_wait(&qfull[0], 0);
      if (dbg && pt == 0) dbg_row[2] = tcq_timer();
      fetch(cur, 0);
    }
    for (int i = 0; i < npairs; ++i) {
      const int qs_n = (qs + 1 == NQ) ? 0 : qs + 1;
      const uint32_t qph_n = (qs + 1 == NQ) ? (qph ^ 1) : qph;
      if (i + 1 < npairs) {     // the next stage's packed words: in flight while this step is dequantised
        mbar_wait(&qfull[qs_n], qph_n);
        fetch(nxt, qs_n);
      }
      mbar_wait(&empty[stage], phase ^ 1);
      cur.store(p, 0, 0, dt, a_base_s + (uint32_t)stage * kAStageBytes);
      fence_proxy_async_smem();   // every writer: generic-proxy stores -> visible to the tensor core
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&full[stage]);
        mbar_arrive(&qempty[qs]);  // after the stores that consumed the stage's words (data dependence)
      }
      stage += Cfg::kTeams;
      if (stage >= NS) { stage -= NS; phase ^= 1; }
      cur = nxt;
      qs = qs_n;
      qph = qph_n;
    }
    if (dbg && pt == 0) dbg_row[3] = tcq_timer();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// -------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(f);
  });
  return fn;
}

struct TmapKey {
  const void* ptr;
  uint64_t inner, outer, pitch;
  uint32_t bi, bo;
  int kind;  // bit 0: element type, bit 1: 128B swizzle
  bool operator==(const TmapKey& o) const {
    return ptr == o.ptr && inner == o.inner && outer == o.outer && pitch == o.pitch && bi == o.bi && bo == o.bo &&
           kind == o.kind;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    h ^= (size_t)k.inner * 0x9E3779B97F4A7C15ull + (size_t)k.outer * 1315423911u + (size_t)k.pitch * 2654435761u +
         (size_t)k.bi * 31u + (size_t)k.bo * 131u + (size_t)k.kind;
    return h;
  }
};

cudaError_t make_tmap_2d(const void* ptr, int elem_kind, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                         uint32_t box_inner, uint32_t box_outer, CUtensorMap* out, bool swizzle128) {
  static std::mutex mu;
  static std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> cache;
  TmapKey key{ptr, inner, outer, pitch_bytes, box_inner, box_outer, elem_kind | (swizzle128 ? 2 : 0)};
  {
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    if (it != cache.end()) {
      *out = it->second;
      return cudaSuccess;
    }
  }
  EncodeTiledFn enc = get_encode_fn();
  if (enc == nullptr) return cudaErrorNotSupported;
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)pitch_bytes};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = elem_kind == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_INT32;
  CUresult r = enc(out, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
  std::lock_guard<std::mutex> lk(mu);
  if (cache.size() > 8192) cache.clear();
  cache.emplace(key, *out);
  return cudaSuccess;
}

// X[M, K] fp16 (row pitch ld elements) -> box {64 k, BT rows}
static cudaError_t make_x_tmap(const void* x, int64_t ld, int M, int K, int BT, CUtensorMap* out) {
  return make_tmap_2d(x, 0, (uint64_t)K, (uint64_t)M, (uint64_t)ld * 2, kBK, (uint32_t)BT, out);
}

static int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = B200AWQ_SM_COUNT_FALLBACK;
  }
  return n;
}

template <int BT, int LAYOUT>
static cudaError_t launch_tc(const CUtensorMap& tm, const CUtensorMap& tmq, const TcParams& p, cudaStream_t st) {
  using Cfg = TcCfg<BT>;
  auto kern = gemm_tc_kernel<BT, LAYOUT>;
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  const int n_work = p.n_tiles * p.m_tiles * p.ksplit;
  const int grid = n_work < sm_count() ? n_work : sm_count();
  return launch_kernel(kern, dim3(grid), dim3(tc_threads<LAYOUT>()), Cfg::kSmemBytes, st, tm, tmq, p);
}

template <int LAYOUT>
static cudaError_t dispatch_bt(int BT, const CUtensorMap& tm, const CUtensorMap& tmq, const TcParams& p,
                               cudaStream_t st) {
  switch (BT) {
    case 32: return launch_tc<32, LAYOUT>(tm, tmq, p, st);
    case 64: return launch_tc<64, LAYOUT>(tm, tmq, p, st);
    case 128: return launch_tc<128, LAYOUT>(tm, tmq, p, st);
    default: return launch_tc<256, LAYOUT>(tm, tmq, p, st);
  }
}

// Grid of the small-M kernel = how the linearised (n-tile, k-step pair) sequence is cut (CTA b owns the pairs
// [T b / grid, T (b + 1) / grid), T = n_tiles * KP).  mode = knob 21.
int gemm_tcq_grid(int n_tiles, int KP, int M, int sms, int mode) {
  const long long T = (long long)n_tiles * KP;
  long long grid = T / 2;   // balanced ranges: every CTA streams the same bytes; at least 2 pairs per CTA
  if (grid < 1) grid = 1;
  if (grid > sms) grid = sms;
  // Tile-aligned ranges (knob 21: 1 = never, 2 = always): a range that never straddles an n-tile has ONE segment, and a
  // range that is a whole tile stores fp16 directly - no fp32 REDs, no ticket, no read-back (M * 128 REDs per segment,
  // M / 16 L2 round trips per finalised tile).
  if (mode != 1) {
    long long g = 0;
    if (n_tiles <= sms) {
      // every tile is cut into ks ranges (boundaries b * KP / ks never cross a tile since the grid is a multiple of
      // n_tiles); ks = 1 stores whole tiles directly.  Measured better than the balanced cut at every M <= 128 on the
      // shapes with N / 128 <= 148 (profiles/r02_tcq_sweep.json).
      int ks = sms / n_tiles;
      if (ks > KP / 2) ks = KP / 2;
      if (ks < 1) ks = 1;
      g = (long long)n_tiles * ks;
    } else if (mode == 2 || M >= 64) {
      // more tiles than SMs: whole tiles per CTA when they divide evenly (224 tiles -> 112 CTAs x 2); below 64 tokens
      // the balanced cut wins there (all 148 SMs stream, the split-K traffic is small)
      const int tpc = (n_tiles + sms - 1) / sms;
      if (n_tiles % tpc == 0) g = n_tiles / tpc;
    }
    if (g > 0) grid = g;
  }
  return (int)grid;
}

template <int BT>
static cudaError_t launch_tcq(const CUtensorMap& tm, const CUtensorMap& tmq, const TcParams& p, cudaStream_t st) {
  using Cfg = TcqCfg<BT>;
  auto kern = gemm_tcq_kernel<BT>;
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  const int grid = gemm_tcq_grid(p.n_tiles, p.K / Cfg::kQRows, p.M, sm_count(), knob(21));
  return launch_kernel(kern, dim3((unsigned)grid), dim3(Cfg::kThreads), Cfg::kSmemBytes, st, tm, tmq, p);
}

// Small-M path (M <= kTcqMaxM, GEMM layout, G >= 64, N % 128 == 0): see gemm_tcq_kernel.  The fp32 split-K scratch is
// the caller's workspace: M * N floats fit the documented min(M, 128) * N * 8 bytes.
constexpr int kTcqMaxM = 128;
bool gemm_tcq_shape_ok(int M, int K, int N, int G) {
  return M >= 1 && M <= kTcqMaxM && G >= 64 && (K % 128) == 0 && (N % kTileN) == 0 && N / kTileN <= 4096;
}
bool gemm_tcq_applicable(const GemmArgs& a, const float* acc_ws, const int* tickets) {
  if (knob(19) == 1) return false;
  if (!gemm_tcq_shape_ok(a.M, a.K, a.N, a.G)) return false;
  if (acc_ws == nullptr || tickets == nullptr) return false;
  if (((reinterpret_cast<uintptr_t>(a.qweight) | reinterpret_cast<uintptr_t>(a.scales) |
        reinterpret_cast<uintptr_t>(a.qzeros)) & 15) != 0)
    return false;
  return true;
}

static int zeros_width_tc(int K, int G) {
  const int mult = G >= 128 ? 1 : (G == 64 ? 2 : 4);
  int base = ((K / G) + 7) / 8;
  return ((base + mult - 1) / mult) * mult;
}

cudaError_t gemm_tc(const GemmArgs& a, int layout, float* acc_ws, int* tickets, cudaStream_t st) {
  if (a.K % kBK != 0 || a.G % 32 != 0) return cudaErrorNotSupported;
  const bool g_pow2 = (a.G & (a.G - 1)) == 0;
  if (!g_pow2 && a.G != a.K) return cudaErrorNotSupported;  // AWQ group sizes: 32 / 64 / 128 / whole row
  if ((reinterpret_cast<uintptr_t>(a.x) & 15) != 0 || (a.ldx % 8) != 0) return cudaErrorMisalignedAddress;
  const int BT = a.M <= 32 ? 32 : (a.M <= 64 ? 64 : (a.M <= 128 ? 128 : 256));
  TcParams p;
  p.qweight = a.qweight;
  p.scales = reinterpret_cast<const __half*>(a.scales);
  p.qzeros = a.qzeros;
  p.bias = reinterpret_cast<const __half*>(a.bias);
  p.y = reinterpret_cast<__half*>(a.y);
  p.acc_ws = acc_ws;
  p.tickets = tickets;
  p.M = a.M; p.K = a.K; p.N = a.N; p.G = a.G;
  p.dbg = 0;
  p.zw = zeros_width_tc(a.K, a.G);
  p.g_shift = 31;
  if (g_pow2) {
    p.g_shift = 0;
    while ((1 << p.g_shift) < a.G) ++p.g_shift;
  }
  p.n_tiles = (a.N + kTileN - 1) / kTileN;
  if (layout == 0 && gemm_tcq_applicable(a, acc_ws, tickets)) {
    const int BQ = a.M <= 16 ? 16 : (a.M <= 32 ? 32 : (a.M <= 64 ? 64 : 128));
    CUtensorMap tmxq, tmwq;
    p.m_tiles = 1;
    p.has_tmq = 1;
    p.dbg = knob(3) == 9 ? 1 : 0;
    cudaError_t eq = make_x_tmap(a.x, a.ldx, a.M, a.K, BQ, &tmxq);
    if (eq == cudaSuccess)
      eq = make_tmap_2d(a.qweight, 1, (uint64_t)(a.N / 8), (uint64_t)a.K, (uint64_t)(a.N / 8) * 4, 16, 2 * kBK, &tmwq, false);
    if (eq == cudaSuccess) {
      switch (BQ) {
        case 16: return launch_tcq<16>(tmxq, tmwq, p, st);
        case 32: return launch_tcq<32>(tmxq, tmwq, p, st);
        case 64: return launch_tcq<64>(tmxq, tmwq, p, st);
        default: return launch_tcq<128>(tmxq, tmwq, p, st);
      }
    }
    // a tensor map that cannot be encoded: fall through to the register-staged kernel
  }
  p.m_tiles = (a.M + BT - 1) / BT;
  const int KS = a.K / kBK;
  int ksplit = 1;
  const int tiles = p.n_tiles * p.m_tiles;
  // fp32 partial sums: the workspace holds min(M, kMaxSplitM) * N 8-byte words = room for 2 * kMaxSplitM token rows
  if (a.M <= 2 * kMaxSplitM && acc_ws != nullptr && tickets != nullptr && tiles < sm_count() && tiles <= 4096) {
    ksplit = sm_count() / tiles;
    if (ksplit < 1) ksplit = 1;
    while (ksplit > 1 && KS / ksplit < 4) --ksplit;  // at least 4 k-steps per slice
  }
  // Above 64 tokens the reduction is no longer free: ~0.15 us per token (M * 128 fp32 REDs per CTA, M / 16 L2 round trips
  // for the finaliser) against ~0.5 us per k-step saved on the critical path (profiles/r02_m_sweep_final.json: 14336 x
  // 4096 at M = 256 114 -> 66 us with 4 slices, 4096 x 4096 45 -> 47 us) - split only when it pays.
  if (a.M > 64 && ksplit > 1 && (float)(KS - KS / ksplit) * 0.5f < 0.15f * (float)a.M) ksplit = 1;
  const int forced = knob(1);
  if (forced > 0 && a.M <= 2 * kMaxSplitM && acc_ws != nullptr && tickets != nullptr) ksplit = forced > KS ? KS : forced;
  p.ksplit = ksplit;
  CUtensorMap tm, tmq;
  cudaError_t e = make_x_tmap(a.x, a.ldx, a.M, a.K, BT, &tm);
  if (e != cudaSuccess) return e;
  tmq = tm;
  p.has_tmq = 0;
  if (layout == 0 && (a.N % 4) == 0 && (reinterpret_cast<uintptr_t>(a.qweight) & 15) == 0 && (a.N / 8) % 4 == 0) {
    // qweight [K, N/8] int32 -> box {16 words = one 128-column tile, 64 rows}; only used for L2 prefetch
    if (make_tmap_2d(a.qweight, 1, (uint64_t)(a.N / 8), (uint64_t)a.K, (uint64_t)(a.N / 8) * 4, 16, kBK, &tmq, false) ==
        cudaSuccess)
      p.has_tmq = 1;
  }
  switch (layout) {
    case 0: return a.G >= 64 ? dispatch_bt<0>(BT, tm, tmq, p, st) : dispatch_bt<3>(BT, tm, tmq, p, st);
    case 1: return dispatch_bt<1>(BT, tm, tmq, p, st);
    default: return dispatch_bt<2>(BT, tm, tmq, p, st);
  }
}

}  // namespace b200awq
