// CUDA-core GEMV path (M <= 8 tokens) for the three AWQ layouts.  HBM-bound: the job of these kernels
// is to stream the packed int4 weights once, with 128-bit coalesced loads and enough bytes in flight
// to cover DRAM latency, and to keep the ALU cost per weight below the issue budget that 6.5+ TB/s
// leaves (about 46 weights / clock / SM on a 148-SM B200).
//
// Arithmetic (all layouts): the 4-bit code q is used directly as an fp16 *subnormal* bit pattern
// (q * 2^-24, or q * 2^-20 for the nibbles that sit 4 bits higher), multiplied with the fp16 activation
// and accumulated in fp32 by FHFMA (fma.rn.f32.f16: exact product, one fp32 rounding) - one ALU op per
// weight plus 5/8 op of LOP3/SHF unpack.  Zero-point and scale are applied once per (group, column):
//     y[n] += s[g,n] * ( 2^24 * sum_k x[k] q[k,n]  -  z[g,n] * sum_k x[k] )
// The cross-thread / cross-CTA (split-K) reduction is fp32; the result is rounded to fp16 once.
#include <cuda.h>

#include <atomic>
#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "gemv_tile.cuh"
#include "kernels.h"

namespace b200awq {

constexpr float kScaleA = 16777216.0f;  // 2^24: code read through mask 0x000f000f
constexpr float kScaleB = 1048576.0f;   // 2^20: code read through mask 0x00f000f0

// ======================================================================= GEMM layout [K, N/8]
// v2: the dot products run on the tensor pipe through mma.sync.m16n8k16 with REGISTER-resident fragments.
// Why: measured on B200, FHFMA issues at ~16 lanes/clk/SM (quarter rate), which caps a CUDA-core fp32
// GEMV at ~1.7 TB/s (26% of HBM peak); feeding the same registers to HMMA costs 0.75 ALU op per weight.
//
// Fragment construction without a transpose: one AWQ word = 8 columns of ONE k, low half-word = even
// columns, high half-word = odd columns.  For two consecutive rows (k, k+1) of the same word column
//     lo = PRMT(w_k, w_k+1, 0x5410)   = [even cols of k | even cols of k+1]
//     hi = PRMT(w_k, w_k+1, 0x7632)   = [odd  cols of k | odd  cols of k+1]
// and  (lo >> 4t') & 0x000f000f | 0x64006400  is the fp16 pair (col 2t' @ k, col 2t' @ k+1) = 1024 + q,
// i.e. a pair ALONG K, which is what the A fragment wants.  Nibbles sitting 4 bits higher are read with
// mask 0x00f000f0 as 1024 + 16 q (kind B).  No per-weight zero/scale work at all: the tensor core
// accumulates S = sum_k x_k * (1024 + c*q_k) in fp32 and the epilogue folds, per (group, column),
//     y += s * ( S - (1024 + c*z) * sum_k x_k ) / c ,     c = 1 (kind A) or 16 (kind B).
// The 1024 offset costs ~10 bits of the fp32 accumulator's 24: the result keeps >= 13 bits, above fp16.
//
// Warp tile = 256 columns x 16 rows: lane (g = lane/4, tig = lane%4) loads uint4 (4 words, 32 columns) at
// word column 4g for rows 4 tig .. 4 tig + 3 (128 B contiguous per row across the 8 g's).  MMA (w, t)
// takes A rows {g: column 8w+2t, g+8: column 8w+2t+1} of the lane's word w, A cols {2tig,2tig+1: rows
// 0,1 of the lane; 2tig+8,+9: rows 2,3}; B = activations x[token g][those rows]; D row g / g+8, cols =
// tokens 2tig, 2tig+1.  All M <= 8 tokens ride along for free.
// CTA = NWARP warps sharing the column block, each walking its own k16-blocks; KC rows per CTA
// (grid.y = K / KC slices, fp32 atomics into the zeroed workspace, last CTA rounds + re-zeroes).

// Lean by construction - a 4096x4096 GEMV is ~59 KB per SM (~1 us of HBM time), so every prologue /
// epilogue instruction shows: no shared-memory staging of x (B fragments come straight from global, issued
// with the weight loads), sum_k x_k comes out of one extra MMA against an all-ones A fragment, no runtime
// divisions, one __syncthreads.  RW (rows per warp, 32/64/128) divides G, so a warp's rows sit in ONE
// quantisation group and its accumulators are folded once.
template <int MT, int RW>
__global__ void __launch_bounds__(kGvWarps * 32, 2)
    gemv_gemm_layout_kernel(const __half* __restrict__ x, int64_t ldx, const int32_t* __restrict__ qweight,
                            const __half* __restrict__ scales, const int32_t* __restrict__ qzeros,
                            const __half* __restrict__ bias, __half* __restrict__ y, float* __restrict__ acc_ws,
                            int* __restrict__ tickets, int M, int K, int N, int G) {
  constexpr int NB = RW / 16;                  // k16-blocks per warp
  constexpr int KC = kGvWarps * RW;            // rows per CTA
  extern __shared__ __align__(16) float gv_dyn[];
  float (*red)[MT][kGvRedStride] = reinterpret_cast<float (*)[MT][kGvRedStride]>(gv_dyn);
  float (*xsum_s)[MT] = reinterpret_cast<float (*)[MT]>(gv_dyn + kGvWarps * MT * kGvRedStride);
  __shared__ int s_last;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, tig = lane & 3;
  const int NW = N >> 3;
  const int k0 = blockIdx.y * KC;
  const int n_base = blockIdx.x * kGvTN;
  const int wc = (n_base >> 3) + 4 * g;        // first word column of this lane
  const bool col_ok = wc < NW;                 // N % 32 == 0 on this path
  const int wrow = k0 + warp * RW;             // first row of this warp
  const bool tok_ok = g < M;                   // this lane feeds token g into the B fragment

  // ---- software pipeline: two k16-blocks of weights (+ activations) in flight per lane ---------------
  uint4 q[2][4];
  uint2 xb[2];
  auto issue_w = [&](int slot, int b) {
    const int kr = wrow + 16 * b + 4 * tig;    // this lane's 4 rows of block b
    const int32_t* src = qweight + (int64_t)kr * NW + wc;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      q[slot][r] = make_uint4(0, 0, 0, 0);
      if (col_ok && kr + r < K) q[slot][r] = ldg_stream_u4(src + (int64_t)r * NW);
    }
  };
  auto issue_x = [&](int slot, int b) {
    const int kr = wrow + 16 * b + 4 * tig;
    xb[slot] = make_uint2(0, 0);
    if (tok_ok && kr + 3 < K) {
      xb[slot] = *reinterpret_cast<const uint2*>(x + (int64_t)g * ldx + kr);
    } else if (tok_ok && kr < K) {             // ragged K tail
      __half t[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) t[r] = (kr + r < K) ? x[(int64_t)g * ldx + kr + r] : __float2half(0.f);
      xb[slot] = *reinterpret_cast<uint2*>(t);
    }
  };
  pdl_trigger();                 // the next kernel on the stream may start its own weight prefetch
  issue_w(0, 0);                 // weights never depend on the predecessor: in flight before the wait
  if (NB > 1) issue_w(1, 1);
  pdl_wait();                    // activations / workspace / outputs: only after the predecessor is done
  issue_x(0, 0);
  if (NB > 1) issue_x(1, 1);

  float acc[4][4][4];  // [word][t][d-reg]: d0/d1 = column 8w+2t, tokens 2tig / 2tig+1 ; d2/d3 = column 8w+2t+1
  float xs_acc[4] = {0.f, 0.f, 0.f, 0.f};      // ones-row MMA: d0/d1 = sum_k x[token 2tig / 2tig+1][k]
#pragma unroll
  for (int w = 0; w < 4; ++w)
#pragma unroll
    for (int t = 0; t < 4; ++t)
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[w][t][r] = 0.f;

#pragma unroll
  for (int b = 0; b < NB; ++b) {
    const int sl = b & 1;
    constexpr uint32_t MA = 0x000f000fu, MB = 0x00f000f0u, MG = 0x64006400u, ONES = 0x3C003C00u;
    mma_16816(xs_acc, ONES, ONES, ONES, ONES, xb[sl].x, xb[sl].y);
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const uint32_t wa = (&q[sl][0].x)[w], wb = (&q[sl][1].x)[w], wc_ = (&q[sl][2].x)[w], wd = (&q[sl][3].x)[w];
      const uint32_t lo01 = __byte_perm(wa, wb, 0x5410), hi01 = __byte_perm(wa, wb, 0x7632);
      const uint32_t lo23 = __byte_perm(wc_, wd, 0x5410), hi23 = __byte_perm(wc_, wd, 0x7632);
      const uint32_t lo01s = lo01 >> 8, hi01s = hi01 >> 8, lo23s = lo23 >> 8, hi23s = hi23 >> 8;
      // t = 0: columns 0,1 (kind A) ; t = 1: columns 2,3 (kind B) ; t = 2: columns 4,5 (A) ; t = 3: 6,7 (B)
      mma_16816(acc[w][0], lop3_and_or(lo01, MA, MG), lop3_and_or(hi01, MA, MG), lop3_and_or(lo23, MA, MG),
                lop3_and_or(hi23, MA, MG), xb[sl].x, xb[sl].y);
      mma_16816(acc[w][1], lop3_and_or(lo01, MB, MG), lop3_and_or(hi01, MB, MG), lop3_and_or(lo23, MB, MG),
                lop3_and_or(hi23, MB, MG), xb[sl].x, xb[sl].y);
      mma_16816(acc[w][2], lop3_and_or(lo01s, MA, MG), lop3_and_or(hi01s, MA, MG), lop3_and_or(lo23s, MA, MG),
                lop3_and_or(hi23s, MA, MG), xb[sl].x, xb[sl].y);
      mma_16816(acc[w][3], lop3_and_or(lo01s, MB, MG), lop3_and_or(hi01s, MB, MG), lop3_and_or(lo23s, MB, MG),
                lop3_and_or(hi23s, MB, MG), xb[sl].x, xb[sl].y);
    }
    if (b + 2 < NB) {
      issue_w(sl, b + 2);
      issue_x(sl, b + 2);
    }
  }

  // ---- raw per-warp sums -> shared memory -----------------------------------------------------------
#pragma unroll
  for (int w = 0; w < 4; ++w)
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int pc = gv_pos(32 * g + 8 * w + 2 * t);
      if (2 * tig < MT) *reinterpret_cast<float2*>(&red[warp][2 * tig][pc]) = make_float2(acc[w][t][0], acc[w][t][2]);
      if (2 * tig + 1 < MT)
        *reinterpret_cast<float2*>(&red[warp][2 * tig + 1][pc]) = make_float2(acc[w][t][1], acc[w][t][3]);
    }
  if (g == 0) {
    if (2 * tig < MT) xsum_s[warp][2 * tig] = xs_acc[0];
    if (2 * tig + 1 < MT) xsum_s[warp][2 * tig + 1] = xs_acc[1];
  }
  __syncthreads();

  // ---- fold zero-point / scale per (group, column): thread c owns column n_base + c ------------------
  const bool split = gridDim.y > 1;
  const int c = tid;
  const int n = n_base + c;
  if (n < N) {
    const int j = c & 7;
    const bool kindB = ((j >> 1) & 1) != 0;
    const int zshift = 4 * ((j >> 1) + 4 * (j & 1));  // 4 * AWQ_REVERSE_ORDER[j]
    const int pc = gv_pos(c);
    float val[MT];
#pragma unroll
    for (int m = 0; m < MT; ++m) val[m] = 0.f;
    // warps sharing a quantisation group are summed raw, then folded once
    int w = 0;
#pragma unroll 1
    while (w < kGvWarps) {
      const int krow = k0 + w * RW;
      if (krow >= K) break;
      const int gabs = krow / G;
      float s = __half2float(__ldg(scales + (int64_t)gabs * N + n));
      const float z = static_cast<float>((static_cast<uint32_t>(__ldg(qzeros + (int64_t)gabs * NW + (n >> 3))) >> zshift) & 0xFu);
      const float zoff = kindB ? 1024.f + 16.f * z : 1024.f + z;
      if (kindB) s *= 0.0625f;
      float S[MT], X[MT];
#pragma unroll
      for (int m = 0; m < MT; ++m) S[m] = X[m] = 0.f;
      const int gend = (gabs + 1) * G;
      for (; w < kGvWarps && k0 + w * RW < gend && k0 + w * RW < K; ++w) {
#pragma unroll
        for (int m = 0; m < MT; ++m) {
          S[m] += red[w][m][pc];
          X[m] += xsum_s[w][m];
        }
      }
#pragma unroll
      for (int m = 0; m < MT; ++m) val[m] += s * (S[m] - zoff * X[m]);
    }
#pragma unroll
    for (int m = 0; m < MT; ++m) {
      if (m < M) {
        if (!split) {
          float v = val[m];
          if (bias != nullptr) v += __half2float(bias[n]);
          y[(int64_t)m * N + n] = __float2half_rn(v);
        } else {
          atomicAdd(&acc_ws[(int64_t)m * N + n], val[m]);
        }
      }
    }
  }
  if (!split) return;

  // ---- split-K: the last CTA of this column block rounds, adds bias, and re-zeroes the scratch -------
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const int prev = atomicAdd(&tickets[blockIdx.x], 1);
    s_last = (prev == static_cast<int>(gridDim.y) - 1);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (n < N) {
    const float bv = (bias != nullptr) ? __half2float(bias[n]) : 0.f;
#pragma unroll
    for (int m = 0; m < MT; ++m) {
      if (m < M) {
        float* p = &acc_ws[(int64_t)m * N + n];
        const float v = ldcg_f1(p);
        *p = 0.f;
        y[(int64_t)m * N + n] = __float2half_rn(v + bv);
      }
    }
  }
  if (tid == 0) tickets[blockIdx.x] = 0;
}

template <int MT, int RW>
static cudaError_t launch_gemv_gemm_layout(const GemmArgs& a, float* acc_ws, int* tickets, cudaStream_t st) {
  constexpr int KC = kGvWarps * RW;
  constexpr size_t smem = (size_t)(kGvWarps * MT * kGvRedStride + kGvWarps * MT) * sizeof(float);
  auto kern = gemv_gemm_layout_kernel<MT, RW>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
  }
  dim3 grid((a.N + kGvTN - 1) / kGvTN, (a.K + KC - 1) / KC);
  return launch_kernel(kern, grid, dim3(kGvWarps * 32), smem, st, reinterpret_cast<const __half*>(a.x), a.ldx,
                       a.qweight, reinterpret_cast<const __half*>(a.scales), a.qzeros,
                       reinterpret_cast<const __half*>(a.bias), reinterpret_cast<__half*>(a.y), acc_ws, tickets, a.M,
                       a.K, a.N, a.G);
}

// Rows per warp: the largest of {128, 64, 32} that divides G and still leaves >= 2 CTAs per SM.
static int pick_rw(int K, int N, int G) {
  const int forced = knob(0);
  if (forced == 32 || forced == 64 || forced == 128) return (G % forced == 0) ? forced : 32;
  const int colblk = (N + kGvTN - 1) / kGvTN;
  for (int rw = 128; rw > 32; rw >>= 1) {
    if (G % rw != 0) continue;
    const int kc = kGvWarps * rw;
    if ((int64_t)colblk * ((K + kc - 1) / kc) >= 2 * 148) return rw;
  }
  return 32;
}

// N % 32 == 0, G % 32 == 0 (every AWQ checkpoint: G in {32, 64, 128, K}) and 8-byte aligned activation rows
// take the tensor-pipe GEMV; other shapes are routed to the tcgen05 kernel by the C-ABI layer.
bool gemv_gemm_layout_supported(const GemmArgs& a) {
  return (a.N % 32) == 0 && (a.G % 32) == 0 && (reinterpret_cast<uintptr_t>(a.qweight) % 16) == 0 && a.M <= 8 &&
         (a.ldx % 4) == 0 && (reinterpret_cast<uintptr_t>(a.x) % 8) == 0;
}

template <int MT>
static cudaError_t dispatch_rw(const GemmArgs& a, float* acc_ws, int* tickets, int rw, cudaStream_t st) {
  if (rw == 128) return launch_gemv_gemm_layout<MT, 128>(a, acc_ws, tickets, st);
  if (rw == 64) return launch_gemv_gemm_layout<MT, 64>(a, acc_ws, tickets, st);
  return launch_gemv_gemm_layout<MT, 32>(a, acc_ws, tickets, st);
}

cudaError_t gemv_gemm_layout(const GemmArgs& a, float* acc_ws, int* tickets, cudaStream_t st) {
  const int rw = pick_rw(a.K, a.N, a.G);
  if (a.M <= 1) return dispatch_rw<1>(a, acc_ws, tickets, rw, st);
  if (a.M <= 2) return dispatch_rw<2>(a, acc_ws, tickets, rw, st);
  if (a.M <= 4) return dispatch_rw<4>(a, acc_ws, tickets, rw, st);
  return dispatch_rw<8>(a, acc_ws, tickets, rw, st);
}

}  // namespace b200awq

// ======================================================================= GEMM layout, persistent TMA-ring GEMV
// v3/v4.  What the register-staged kernel above taught (ncu, B200): with loads staged in REGISTERS a CTA
// keeps ~50 KB per SM in flight and every short-lived CTA pays its own chain of dependent latencies
// (DRAM -> MMA -> fold constants -> atomics -> fence -> ticket): DRAM sat at 9-29 % busy.  A first
// ring-buffer version with four warps sharing each 16-row block spent 2/3 of its instructions on
// per-block flush / fold / barriers.  This version:
//   * ONE persistent CTA per SM; a producer warp streams 8 KB weight tiles (64 rows x 256 columns, TMA 2-D,
//     128B swizzle) plus the tile's group scales / zeros (bulk copies) into shared memory; every consumer
//     warp owns TWO ring stages (8 warps x 2 x 9 KB = 147 KB in flight per SM, independent of registers,
//     running ahead across tile and - under PDL - KERNEL boundaries: weights never depend on the
//     predecessor);
//   * consumer warps are INDEPENDENT: warp w walks its own contiguous run of tiles, keeps the 64 + 4
//     accumulators in registers across the 4 k16-blocks of a tile and across the tiles of a quantisation
//     group, folds zero-point / scale inside the warp (lane l owns word-column l: its 8 columns' scales
//     are one LDS.128, their zeros one LDS.32) into a per-warp column accumulator in shared memory;
//   * one CTA-level reduction at the end (or a warp-level push when a warp's run crosses a 256-column
//     block), fp32 atomics into the zeroed workspace, tickets count TILES so the last contributor of a
//     column block is known without any host-side schedule.
namespace b200awq {

// Phase timestamps (globaltimer, ns) of the last persistent-GEMV launch, one row of 8 per CTA; written only when
// knob 3 is set.  Read back with b200awq_debug_read().
__device__ unsigned long long g_v3_dbg[256 * 8];
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
cudaError_t gemv_v3_debug_read(void* dst, size_t bytes) {
  return cudaMemcpyFromSymbol(dst, g_v3_dbg, bytes < sizeof(g_v3_dbg) ? bytes : sizeof(g_v3_dbg));
}


// Grouped (MoE) variant, template flag MOE: blockIdx.y = job = eight sorted slots of one expert
// (awq/modules/fused/moe.py:60-89).  The stacked expert weights [E, K, N/8] are ONE 2-D tensor map of E*K rows, so the
// expert is a row offset in the tile coordinate; activations are gathered and outputs scattered through the sorted
// slot ids; split-K scratch and tickets are per job.
struct V3Moe {
  const int* sorted_ids;
  const int* expert_ids;
  const int* num_post_pad;
  const float* topk_w;     // routing weights [n_slots] or nullptr (mul_weights = false)
  int n_slots, topk, x_per_slot, block_size;
};

template <int MT, int SPW, bool MOE = false>
__global__ void __launch_bounds__(kV3Threads, 1)
    gemv_v3_kernel(const __grid_constant__ CUtensorMap tmw, const __half* __restrict__ x, int64_t ldx,
                   const __half* __restrict__ scales, const int32_t* __restrict__ qzeros,
                   const __half* __restrict__ bias, __half* __restrict__ y, float* __restrict__ acc_ws,
                   int* __restrict__ tickets, int M, int K, int N, int G, int g_shift,
                   const uint8_t* __restrict__ next_w, long long next_bytes, int dbg, const V3Moe moe,
                   int packed) {
  constexpr int NS = V3Smem<MT, SPW>::kStages;
  __shared__ int s_slot[8];       // MOE: output row of each of the job's slots (-1 = padding)
  int row_off = 0;                // MOE: first row of the job's expert in the stacked tensor
  if (MOE) {
    // The routing tables (num_post_pad, sorted_ids, expert_ids) are the PREDECESSOR's output (moe_align): under
    // programmatic dependent launch this kernel may start before that kernel has finished, so nothing of them may be read
    // before the wait - not even to decide that the job is padding (a CTA that exits without waiting would also let the
    // grid "complete" early and break the chain for the successor).  The expert's weights depend on the routing, so
    // unlike the dense GEMV there is nothing to prefetch ahead of the wait.  (Found by bench.py's Mixtral leg: with
    // knob 4 the step ran in 1.8 ms instead of 3.3 ms - jobs saw stale tables and returned as padding.)
    pdl_wait();
    const int job = blockIdx.y;
    if (job * 8 >= *moe.num_post_pad) return;
    if (threadIdx.x < 8) {
      const int id = moe.sorted_ids[job * 8 + threadIdx.x];
      s_slot[threadIdx.x] = id < moe.n_slots ? id : -1;
    }
    const int e = moe.expert_ids[(job * 8) / moe.block_size];
    row_off = e * K;
    scales += (int64_t)e * (K / G) * N;
    qzeros += (int64_t)e * (K / G) * (N >> 3);
    acc_ws += (int64_t)job * 8 * N;
    tickets += job * (N / kV3TileCols);
  }
  extern __shared__ __align__(1024) uint8_t v3_smem[];
  uint8_t* ring = v3_smem;                                   // NS x 8 KB weight tiles (1 KB aligned: swizzle atoms)
  uint8_t* aux = v3_smem + (size_t)NS * kV3TileBytes;        // NS x (256 scales + 32 zero words)
  float* red = reinterpret_cast<float*>(aux + (size_t)NS * kV3AuxBytes);
  uint64_t* full = reinterpret_cast<uint64_t*>(red + V3Smem<MT, SPW>::red_floats);
  uint64_t* empty = full + NS;
  int* flags = reinterpret_cast<int*>(empty + NS);   // [0..7] per-warp push flags, [8] CTA flag,
  int* warp_cb = flags + 16;                         // [8] column block of each warp's pending sums
  int* warp_ntl = warp_cb + 8;                       // [8] tiles those sums cover

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NW = N >> 3;
  const int TPC = K / kV3TileRows;                 // tiles per column block
  const int T = (N / kV3TileCols) * TPC;           // all tiles, column-block major
  const int t0 = (int)((int64_t)T * blockIdx.x / gridDim.x);
  const int t1 = (int)((int64_t)T * (blockIdx.x + 1) / gridDim.x);
  const int ntile = t1 - t0;

  pdl_trigger();
  if (dbg && tid == 0 && blockIdx.x < 256) g_v3_dbg[blockIdx.x * 8 + 0] = gtimer();
  if (tid == 0) {
    if ((smem_u32(v3_smem) & 1023u) != 0) __trap();  // the 128B-swizzle read pattern assumes 1 KB aligned stages
    tma_prefetch_desc(&tmw);
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    fence_mbar_init();
  }
  __syncthreads();
  if (MOE) {
    bool any = false;
#pragma unroll
    for (int m = 0; m < 8; ++m) any = any || s_slot[m] >= 0;
    if (!any) return;   // pure padding (uniform)
  }

  if (warp == 0) {
    // ============================================================ producer: weights never wait for PDL
    // lane w feeds consumer warp w's private stages: no head-of-line blocking between consumers
    if (lane < kV3Warps) {
      const int w = lane;
      const int a = t0 + (int)((int64_t)ntile * w / kV3Warps);
      const int bnd = t0 + (int)((int64_t)ntile * (w + 1) / kV3Warps);
      // No HBM -> L2 prefetch ahead of the ring: the 24-stage ring already saturates what the consumers can drain
      // (19.5 us without vs 20.7 us with one on 4096 x 28672, profiles/r01_gemv_v3_ring_sweep.json).
      int cb = a / TPC, kt = a - cb * TPC;
      int stage_i = 0;
      uint32_t ph = 0;
      for (int t = a; t < bnd; ++t) {
        const int stage = w * SPW + stage_i;
        mbar_wait(&empty[stage], ph ^ 1);
        const int grp_abs = (kt * kV3TileRows) >> g_shift;
        uint8_t* st = ring + (size_t)stage * kV3TileBytes;
        uint8_t* sa = aux + (size_t)stage * kV3AuxBytes;
        mbar_arrive_expect_tx(&full[stage], kV3TileBytes + kV3AuxBytes);
        tma_load_2d(st, &tmw, &full[stage], cb * (kV3TileCols / 8), row_off + kt * kV3TileRows);
        bulk_load_1d(sa, scales + (int64_t)grp_abs * N + cb * kV3TileCols, kV3ScaleBytes, &full[stage]);
        bulk_load_1d(sa + kV3ScaleBytes, qzeros + (int64_t)grp_abs * NW + cb * (kV3TileCols / 8), kV3ZeroBytes,
                     &full[stage]);
        if (++kt == TPC) { kt = 0; ++cb; }
        if (++stage_i == SPW) { stage_i = 0; ph ^= 1; }
      }
    }
    __syncwarp();
    // All of this CTA's tiles are requested: HBM would now idle while the consumers finish and the split-K
    // epilogue runs.  Use the gap to pull this CTA's share of the NEXT linear's packed weights (the library
    // learns the call sequence of a decode step) from HBM into L2: the successor kernel starts on L2 hits.
    if (next_w != nullptr) {
      const long long nline = (next_bytes + 127) / 128;
      const long long c0 = nline * blockIdx.x / gridDim.x, c1 = nline * (blockIdx.x + 1) / gridDim.x;
      for (long long c = c0 + lane; c < c1; c += 32) prefetch_l2_line(next_w + c * 128);
    }
    return;
  }

  // ================================================================ consumers (independent warps)
  const int cw = warp - 1;             // 0..7
  const int ct = tid - 32;             // 0..255
  const int g = lane >> 2, tig = lane & 3;
  const int my_slot = MOE ? s_slot[g] : 0;
  const bool tok_ok = MOE ? my_slot >= 0 : g < M;
  // this lane's token row: row g of x, or (MOE) the row the slot's id names
  const __half* xrow = MOE ? x + (int64_t)(tok_ok ? (moe.x_per_slot ? my_slot : my_slot / moe.topk) : 0) * K
                           : x + (int64_t)g * ldx;
  V3Scatter scat;
  if (MOE) {
    scat.ids = s_slot;
    scat.tw = moe.topk_w;
  }
  float* my_red = red + (size_t)cw * MT * kGvRedStride;
  float ycol[MT][8];          // this lane's folded column sums: word-column `lane` (8 columns) x MT tokens
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int j = 0; j < 8; ++j) ycol[m][j] = 0.f;
  const int a_w = t0 + (int)((int64_t)ntile * cw / kV3Warps);
  const int b_w = t0 + (int)((int64_t)ntile * (cw + 1) / kV3Warps);

  pdl_wait();  // activations, workspace, tickets, outputs belong to the stream order
  if (dbg && ct == 0 && blockIdx.x < 256) g_v3_dbg[blockIdx.x * 8 + 1] = gtimer();

  // activations of tile t, block b: rows 16b + {2tig, 2tig+1} and 16b + {2tig+8, 2tig+9}
  auto load_x = [&](int t, int ktile, uint32_t (&xb)[4][2]) {
#pragma unroll
    for (int bb = 0; bb < 4; ++bb) xb[bb][0] = xb[bb][1] = 0u;
    if (t < b_w && tok_ok) {
      const __half* px = xrow + ktile * kV3TileRows + 2 * tig;
#pragma unroll
      for (int bb = 0; bb < 4; ++bb) {
        xb[bb][0] = *reinterpret_cast<const uint32_t*>(px + 16 * bb);
        xb[bb][1] = *reinterpret_cast<const uint32_t*>(px + 16 * bb + 8);
      }
    }
  };

  float acc[4][4][4];
  float xs_acc[4];
  auto zero_acc = [&]() {
#pragma unroll
    for (int w = 0; w < 4; ++w)
#pragma unroll
      for (int tt = 0; tt < 4; ++tt)
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[w][tt][r] = 0.f;
    xs_acc[0] = xs_acc[1] = xs_acc[2] = xs_acc[3] = 0.f;
  };
  zero_acc();

  int cur_cb = -1, ntl = 0;
  uint32_t xcur[4][2], xnext[4][2];
  int cb = a_w / TPC, kt = a_w - cb * TPC;
  load_x(a_w, kt, xcur);
  int stage_i = 0;
  uint32_t ph = 0;
  for (int t = a_w; t < b_w; ++t) {
    const int stage = cw * SPW + stage_i;
    if (cb != cur_cb) {
      if (cur_cb >= 0 && ntl > 0) {
        // this warp's run crosses a column block: push its pending sums alone (rare)
        v3_dump_cols<MT>(my_red, ycol, lane);
        if (packed)
          v3_atom_cols<MT, 32>(my_red, 1, 0, cur_cb, ntl, TPC, lane, bias, y, reinterpret_cast<unsigned long long*>(acc_ws),
                               M, N, scat);
        else
          v3_push_warp<MT>(my_red, cur_cb, ntl, TPC, lane, bias, y, acc_ws, tickets, M, N, scat);
      }
      cur_cb = cb;
      ntl = 0;
    }
    ++ntl;
    load_x(t + 1, (kt + 1 == TPC) ? 0 : kt + 1, xnext);  // next tile's activations in flight meanwhile
    mbar_wait(&full[stage], ph);
    if (dbg && ct == 0 && t == a_w && blockIdx.x < 256) g_v3_dbg[blockIdx.x * 8 + 2] = gtimer();
    const uint8_t* st = ring + (size_t)stage * kV3TileBytes;
    const uint8_t* sa = aux + (size_t)stage * kV3AuxBytes;

    v3_tile_mma(st, g, tig, xcur, acc, xs_acc);

    // ---- fold when the quantisation group (or this warp's run) ends with this tile -----------------
    const bool group_end = g_shift < 31 ? ((((kt + 1) * kV3TileRows) & (G - 1)) == 0) : (kt + 1 == TPC);
    if (group_end || t + 1 == b_w) {
      v3_fold_reg<MT>(sa, my_red, ycol, lane, g, tig, acc, xs_acc);
      zero_acc();
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[stage]);   // the whole warp is done reading this stage
#pragma unroll
    for (int bb = 0; bb < 4; ++bb) {
      xcur[bb][0] = xnext[bb][0];
      xcur[bb][1] = xnext[bb][1];
    }
    if (++kt == TPC) { kt = 0; ++cb; }
    if (++stage_i == SPW) { stage_i = 0; ph ^= 1; }
  }

  // ---- CTA-level reduction of the per-warp column sums, grouped by column block --------------------
  if (dbg && ct == 0 && blockIdx.x < 256) g_v3_dbg[blockIdx.x * 8 + 3] = gtimer();
  v3_dump_cols<MT>(my_red, ycol, lane);   // the staging area now carries the warp's column sums [MT][256]
  if (lane == 0) {
    warp_cb[cw] = (ntl > 0) ? cur_cb : -1;
    warp_ntl[cw] = ntl;
  }
  named_bar_sync_gv(1, kV3Warps * 32);
  if (dbg && ct == 0 && blockIdx.x < 256) g_v3_dbg[blockIdx.x * 8 + 4] = gtimer();
  if (packed) {
    // packed epilogue: one returning atomic per (token, column) and column-block group; whoever completes a column
    // finalises it on the spot - no ticket pass, no read-back pass (gemv_tile.cuh)
    int w0 = 0;
    while (w0 < kV3Warps) {
      const int cbg = warp_cb[w0];
      int w1 = w0 + 1, tiles = warp_ntl[w0];
      while (w1 < kV3Warps && warp_cb[w1] == cbg) tiles += warp_ntl[w1++];
      if (cbg >= 0)
        v3_atom_cols<MT, kV3Warps * 32>(red + (size_t)w0 * MT * kGvRedStride, w1 - w0, MT * kGvRedStride, cbg, tiles, TPC,
                                        ct, bias, y, reinterpret_cast<unsigned long long*>(acc_ws), M, N, scat);
      w0 = w1;
    }
    if (dbg && ct == 0 && blockIdx.x < 256) g_v3_dbg[blockIdx.x * 8 + 7] = gtimer();
    return;
  }
  // pass 1: all column-block groups of this CTA (consecutive warps with the same block) -> workspace
  {
    int w0 = 0;
    while (w0 < kV3Warps) {
      const int cbg = warp_cb[w0];
      int w1 = w0 + 1;
      while (w1 < kV3Warps && warp_cb[w1] == cbg) ++w1;
      if (cbg >= 0)
        v3_add_cols<MT, kV3Warps * 32>(red + (size_t)w0 * MT * kGvRedStride, w1 - w0, MT * kGvRedStride, cbg, ct, acc_ws,
                                       M, N, scat);
      w0 = w1;
    }
  }
  named_bar_sync_gv(1, kV3Warps * 32);
  if (dbg && ct == 0 && blockIdx.x < 256) g_v3_dbg[blockIdx.x * 8 + 5] = gtimer();
  // pass 2: thread w bumps the ticket of the group that STARTS at warp w (tickets in parallel, one round trip)
  if (ct < kV3Warps) {
    const int w = ct;
    const int cbg = warp_cb[w];
    int is_last = 0;
    if (cbg >= 0 && (w == 0 || warp_cb[w - 1] != cbg)) {
      int tiles = 0;
      for (int w1 = w; w1 < kV3Warps && warp_cb[w1] == cbg; ++w1) tiles += warp_ntl[w1];
      is_last = (atom_add_acq_rel(&tickets[cbg], tiles) + tiles == TPC);
    }
    flags[w] = is_last;
  }
  named_bar_sync_gv(1, kV3Warps * 32);
  if (dbg && ct == 0 && blockIdx.x < 256) g_v3_dbg[blockIdx.x * 8 + 6] = gtimer();
  // pass 3: finalise the blocks for which this CTA was the last contributor
#pragma unroll 1
  for (int w = 0; w < kV3Warps; ++w)
    if (flags[w]) v3_finalize<MT, kV3Warps * 32>(warp_cb[w], ct, bias, y, acc_ws, tickets, M, N, scat);
  if (dbg && ct == 0 && blockIdx.x < 256) g_v3_dbg[blockIdx.x * 8 + 7] = gtimer();
}

static int v3_sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = B200AWQ_SM_COUNT_FALLBACK;
  }
  return n;
}

// Successor table: decode calls the same linears in the same order every token; remember, per weight
// tensor, which weight tensor was used next, and let the kernel prefetch it into L2.  Measured on B200 (r1):
// 478.6 vs 498.7 tok/s decode with / without it - HBM is not idle enough in the kernel tails for the extra
// L2 traffic to pay, so it is OFF by default (knob 6 = 1 enables it for experiments).
struct NextW {
  const void* ptr;
  long long bytes;
};
static NextW learn_successor(const void* w, long long bytes) {
  if (knob(6) == 0) return NextW{nullptr, 0};   // (the default: no lock, no table on the launch path)
  static std::mutex mu;
  static std::unordered_map<const void*, NextW> succ;
  static const void* prev = nullptr;
  std::lock_guard<std::mutex> lk(mu);
  if (prev != nullptr && prev != w) succ[prev] = NextW{w, bytes};
  prev = w;
  if (succ.size() > 65536) succ.clear();
  auto it = succ.find(w);
  if (it == succ.end() || knob(6) == 0) return NextW{nullptr, 0};
  return it->second;
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device) instead of on every launch (it is a
// driver call of a few microseconds; the per-op path makes 160 launches per token).  `done` is one word per kernel
// instantiation (a function-local static at the call site), bit d = device d.
template <typename Kern>
static cudaError_t ensure_smem_attr(Kern kern, size_t smem, std::atomic<uint64_t>& done) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const uint64_t bit = 1ull << (dev & 63);
  if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
  return e;
}

template <int MT, int SPW>
static cudaError_t launch_v3(const GemmArgs& a, float* acc_ws, int* tickets, cudaStream_t st) {
  const NextW nx = learn_successor(a.qweight, (long long)a.K * (a.N / 8) * 4);
  int g_shift = 31;  // G == K: a single group
  if ((a.G & (a.G - 1)) == 0) {
    g_shift = 0;
    while ((1 << g_shift) < a.G) ++g_shift;
  }
  CUtensorMap tm;
  // qweight [K, N/8] int32 -> box {32 words = 128 B, 64 rows}, 128B swizzle
  cudaError_t e = make_tmap_2d(a.qweight, /*int32*/ 1, (uint64_t)(a.N / 8), (uint64_t)a.K, (uint64_t)(a.N / 8) * 4, 32,
                               kV3TileRows, &tm);
  if (e != cudaSuccess) return e;
  auto kern = gemv_v3_kernel<MT, SPW>;
  const size_t smem = V3Smem<MT, SPW>::bytes;
  static std::atomic<uint64_t> attr_done{0};
  e = ensure_smem_attr(kern, smem, attr_done);
  if (e != cudaSuccess) return e;
  const int T = (a.N / kV3TileCols) * (a.K / kV3TileRows);
  const int grid = T < v3_sm_count() ? T : v3_sm_count();
  return launch_kernel(kern, dim3(grid), dim3(kV3Threads), smem, st, tm, reinterpret_cast<const __half*>(a.x), a.ldx,
                       reinterpret_cast<const __half*>(a.scales), a.qzeros, reinterpret_cast<const __half*>(a.bias),
                       reinterpret_cast<__half*>(a.y), acc_ws, tickets, a.M, a.K, a.N, a.G, g_shift,
                       reinterpret_cast<const uint8_t*>(nx.ptr), nx.bytes, knob(3) == 1 ? 1 : 0,
                       // packed epilogue at M = 1 only: there it saves the ticket and read-back round trips (4096 x 4096:
                       // 8.75 -> 7.18 us); for M >= 2 the returning 64-bit atomics cost more than they save on the
                       // larger shapes (4096 x 14336, M = 8: 32 -> 49 us), so those keep fp32 REDs + tickets.
                       V3Moe{}, (MT == 1 && a.K / kV3TileRows < 256) ? 1 : 0);
}

// Grouped launch: grid.y = sorted_len / 8 jobs (most of them padding: they exit at once).  Needs hbs * 8 rows of fp32
// scratch and hbs * N/256 tickets; the caller checks that.
cudaError_t gemv_v3_moe(const void* x, int x_per_slot, const int32_t* qweight, const void* scales, const int32_t* qzeros,
                        const float* topk_w, const int* sorted_ids, const int* expert_ids, const int* num_post_pad,
                        void* y, int n_slots, int topk, int hbs, int E, int K, int N, int G, int block_size,
                        float* acc_ws, int* tickets, cudaStream_t st) {
  int g_shift = 31;
  if ((G & (G - 1)) == 0) {
    g_shift = 0;
    while ((1 << g_shift) < G) ++g_shift;
  }
  CUtensorMap tm;
  cudaError_t e = make_tmap_2d(qweight, /*int32*/ 1, (uint64_t)(N / 8), (uint64_t)E * K, (uint64_t)(N / 8) * 4, 32,
                               kV3TileRows, &tm);
  if (e != cudaSuccess) return e;
  const int T = (N / kV3TileCols) * (K / kV3TileRows);
  const int grid = T < v3_sm_count() ? T : v3_sm_count();
  V3Moe moe{sorted_ids, expert_ids, num_post_pad, topk_w, n_slots, topk, x_per_slot, block_size};
  // a job holds at most min(8, tokens) real slots (a token picks an expert once) and they are a prefix of the job:
  // few tokens -> the narrow variants, which afford more ring stages per warp
  const int tokens = n_slots / (topk > 0 ? topk : 1);
  auto go = [&](auto kern, size_t smem, int mt) -> cudaError_t {
    cudaError_t e2 = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e2 != cudaSuccess) return e2;
    return launch_kernel(kern, dim3(grid, hbs), dim3(kV3Threads), smem, st, tm, reinterpret_cast<const __half*>(x),
                         (int64_t)K, reinterpret_cast<const __half*>(scales), qzeros, static_cast<const __half*>(nullptr),
                         reinterpret_cast<__half*>(y), acc_ws, tickets, mt, K, N, G, g_shift,
                         static_cast<const uint8_t*>(nullptr), 0LL, 0, moe, 0);   // (grouped jobs keep the ticket epilogue)
  };
  if (tokens <= 1) return go(gemv_v3_kernel<1, 3, true>, V3Smem<1, 3>::bytes, 1);
  if (tokens <= 2) return go(gemv_v3_kernel<2, 2, true>, V3Smem<2, 2>::bytes, 2);
  if (tokens <= 4) return go(gemv_v3_kernel<4, 2, true>, V3Smem<4, 2>::bytes, 4);
  return go(gemv_v3_kernel<8, 2, true>, V3Smem<8, 2>::bytes, 8);
}

bool gemv_v3_moe_supported(int K, int N, int G, int hbs) {
  const bool g_ok = ((G & (G - 1)) == 0) || G == K;
  return (N % kV3TileCols) == 0 && (K % kV3TileRows) == 0 && (G % kV3TileRows) == 0 && (K % G) == 0 && g_ok &&
         (int64_t)hbs * (N / kV3TileCols) <= (int64_t)(kTicketBytes / sizeof(int));
}

// Shapes the persistent TMA-ring kernel takes: whole 64 x 256 tiles inside one quantisation group.
bool gemv_v3_supported(const GemmArgs& a) {
  const bool g_ok = ((a.G & (a.G - 1)) == 0) || a.G == a.K;  // power of two, or one group per column
  return gemv_gemm_layout_supported(a) && (a.N % kV3TileCols) == 0 && (a.K % kV3TileRows) == 0 &&
         (a.G % kV3TileRows) == 0 && g_ok && a.N / kV3TileCols <= 4096;
}

cudaError_t gemv_v3(const GemmArgs& a, float* acc_ws, int* tickets, cudaStream_t st) {
  // M = 1: three ring stages per warp (profiles/r01_gemv_v3_ring_sweep.json); activations come straight from global
  // memory - staging them in shared memory cost the third stage and measured 477 vs 498 tok/s
  if (a.M <= 1) return launch_v3<1, 3>(a, acc_ws, tickets, st);
  if (a.M <= 2) return launch_v3<2, 2>(a, acc_ws, tickets, st);
  if (a.M <= 4) return launch_v3<4, 2>(a, acc_ws, tickets, st);
  return launch_v3<8, 2>(a, acc_ws, tickets, st);   // (column sums in registers: two ring stages also at MT = 8)
}

}  // namespace b200awq

// ======================================================================= GEMV layout [N, K/8]
// Output row n is a contiguous K/2-byte run: a warp streams it 512 B per instruction (lane = 32
// consecutive k), keeps two fp32 accumulators per (row, token) (the two nibble scale classes), folds
// scale / zero once per 32-k chunk (always inside one quantisation group since G % 32 == 0) and finishes
// with a 5-step warp-shuffle reduction.  No split-K, deterministic.  Activations live in shared memory,
// permuted so that the four 16-byte pieces a lane needs for one chunk are each a conflict-free
// 512-byte warp access:  piece c of chunk (it, lane)  ->  slot (it * 4 + c) * 32 + lane.
namespace b200awq {

template <int MT, int RW>
__global__ void __launch_bounds__(256)
    gemv_gemv_layout_kernel(const __half* __restrict__ x, int64_t ldx, const int32_t* __restrict__ qweight,
                            const __half* __restrict__ scales, const int32_t* __restrict__ qzeros,
                            const __half* __restrict__ bias, __half* __restrict__ y, int M, int K, int N, int G,
                            int zw) {
  extern __shared__ __align__(16) uint4 xs_perm[];  // [MT][nit*128] uint4
  pdl_trigger();
  pdl_wait();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nit = (K + 1023) / 1024;                 // 1024-k passes per row
  const int slots = nit * 128;                       // uint4 slots per token
  // prologue: stage x (8 halves per slot)
  for (int i = tid; i < MT * slots; i += blockDim.x) {
    const int m = i / slots, s = i % slots;
    const int it = s / 128, c = (s % 128) / 32, l = s % 32;
    const int k = it * 1024 + l * 32 + c * 8;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (m < M && k < K) {
      const __half* src = x + (int64_t)m * ldx + k;
      if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        v = *reinterpret_cast<const uint4*>(src);
      } else {
        __half t[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = src[j];
        v = *reinterpret_cast<uint4*>(t);
      }
    }
    xs_perm[i] = v;
  }
  __syncthreads();

  const int KW = K >> 3;
  const int n0 = (blockIdx.x * 8 + warp) * RW;
  float val[RW][MT];
#pragma unroll
  for (int r = 0; r < RW; ++r)
#pragma unroll
    for (int m = 0; m < MT; ++m) val[r][m] = 0.f;

  for (int it = 0; it < nit; ++it) {
    const int kc = it * 1024 + lane * 32;  // first k of this lane's chunk
    const bool k_ok = kc < K;
    uint4 q[RW];
#pragma unroll
    for (int r = 0; r < RW; ++r) {
      q[r] = make_uint4(0, 0, 0, 0);
      if (k_ok && n0 + r < N) q[r] = ldg_stream_u4(qweight + (int64_t)(n0 + r) * KW + (kc >> 3));
    }
    const int g = k_ok ? kc / G : 0;
#pragma unroll
    for (int m = 0; m < MT; ++m) {
      // 32 activations of this chunk
      uint32_t xr[16];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint4 v = xs_perm[m * slots + (it * 4 + c) * 32 + lane];
        xr[4 * c + 0] = v.x; xr[4 * c + 1] = v.y; xr[4 * c + 2] = v.z; xr[4 * c + 3] = v.w;
      }
      float xsum = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float2 f = __half22float2(u32_as_h2(xr[i]));
        xsum += f.x + f.y;
      }
#pragma unroll
      for (int r = 0; r < RW; ++r) {
        float aA = 0.f, aB = 0.f;
        const uint32_t w[4] = {q[r].x, q[r].y, q[r].z, q[r].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          // word j: k = kc + 8j + i at nibble i; x pairs xr[4j + i/2]
          const uint32_t w8 = w[j] >> 8;
          const uint32_t p0 = w[j] & 0x000f000fu;  // (k0, k4)  class A
          const uint32_t p1 = w[j] & 0x00f000f0u;  // (k1, k5)  class B
          const uint32_t p2 = w8 & 0x000f000fu;    // (k2, k6)  class A
          const uint32_t p3 = w8 & 0x00f000f0u;    // (k3, k7)  class B
          const uint32_t x01 = xr[4 * j + 0], x23 = xr[4 * j + 1], x45 = xr[4 * j + 2], x67 = xr[4 * j + 3];
          aA = fhfma(lo16(p0), lo16(x01), aA);
          aA = fhfma(hi16(p0), lo16(x45), aA);
          aB = fhfma(lo16(p1), hi16(x01), aB);
          aB = fhfma(hi16(p1), hi16(x45), aB);
          aA = fhfma(lo16(p2), lo16(x23), aA);
          aA = fhfma(hi16(p2), lo16(x67), aA);
          aB = fhfma(lo16(p3), hi16(x23), aB);
          aB = fhfma(hi16(p3), hi16(x67), aB);
        }
        if (k_ok && n0 + r < N) {
          const float s = __half2float(scales[(int64_t)(n0 + r) * (zw * 8) + g]);
          const uint32_t zword = static_cast<uint32_t>(qzeros[(int64_t)(n0 + r) * zw + (g >> 3)]);
          const float z = static_cast<float>((zword >> (4 * (g & 7))) & 0xFu);
          val[r][m] += s * (kScaleA * aA + kScaleB * aB - z * xsum);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < RW; ++r)
#pragma unroll
    for (int m = 0; m < MT; ++m) {
      float v = val[r][m];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0 && n0 + r < N && m < M) {
        if (bias != nullptr) v += __half2float(bias[n0 + r]);
        y[(int64_t)m * N + n0 + r] = __float2half_rn(v);
      }
    }
}

template <int MT, int RW>
static cudaError_t launch_gemv_gemv_layout(const GemmArgs& a, int zw, cudaStream_t st) {
  const int nit = (a.K + 1023) / 1024;
  const size_t smem = (size_t)MT * nit * 128 * sizeof(uint4);
  auto kern = gemv_gemv_layout_kernel<MT, RW>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
  }
  const int rows_per_cta = 8 * RW;
  return launch_kernel(kern, dim3((a.N + rows_per_cta - 1) / rows_per_cta), dim3(256), smem, st,
                       reinterpret_cast<const __half*>(a.x), a.ldx, a.qweight, reinterpret_cast<const __half*>(a.scales),
                       a.qzeros, reinterpret_cast<const __half*>(a.bias), reinterpret_cast<__half*>(a.y), a.M, a.K, a.N,
                       a.G, zw);
}

static int zeros_width(int K, int G) {  // awq/modules/linear/gemv.py:12-24
  const int mult = G >= 128 ? 1 : (G == 64 ? 2 : 4);
  int base = ((K / G) + 7) / 8;
  return ((base + mult - 1) / mult) * mult;
}

cudaError_t gemv_gemv_layout(const GemmArgs& a0, cudaStream_t st) {
  const int zw = zeros_width(a0.K, a0.G);
  // keep the staged activations under ~200 KB of shared memory: at most `cap` tokens per pass
  const int nit = (a0.K + 1023) / 1024;
  const size_t per_tok = (size_t)nit * 128 * 16;
  int done = 0;
  while (done < a0.M) {
    GemmArgs a = a0;
    int m = a0.M - done;
    int mt = m <= 1 ? 1 : (m <= 2 ? 2 : (m <= 4 ? 4 : 8));
    while (mt > 1 && per_tok * mt > 200 * 1024) mt >>= 1;
    if (m > mt) m = mt;
    a.M = m;
    a.x = reinterpret_cast<const __half*>(a0.x) + (int64_t)done * a0.ldx;
    a.y = reinterpret_cast<__half*>(a0.y) + (int64_t)done * a0.N;
    cudaError_t e;
    if (mt == 1) e = launch_gemv_gemv_layout<1, 2>(a, zw, st);
    else if (mt == 2) e = launch_gemv_gemv_layout<2, 2>(a, zw, st);
    else if (mt == 4) e = launch_gemv_gemv_layout<4, 1>(a, zw, st);
    else e = launch_gemv_gemv_layout<8, 1>(a, zw, st);
    if (e != cudaSuccess) return e;
    done += m;
  }
  return cudaSuccess;
}

}  // namespace b200awq

// ======================================================================= GEMVFast layout
// qweight int16 [N/4, K] (awq/modules/linear/gemv_fast.py:26-65).  Decoded structure: for the 4-row
// group R and the 64-k block b, the 64 int16 at [R, 64b .. 64b+63] are 4 runs of 16 (one per row
// r = 0..3); in a run, int16 i (i = 0..15) nibble r' holds k = 64b + 32(i/8) + (i%8) + 8r'.  Hence a 16-byte
// piece is 32 consecutive-in-k weights of ONE row, and (word >> 4r') & 0x000f000f is the natural pair
// (k, k+1) with k = base + 2u + 8r' - the layout was built for exactly this unpack.
// scales / scaled zeros are [groups(padded), N] fp16 with W = q*s + sz, sz = -(z*s) rounded to fp16.
// A warp streams one row group: 512 B per instruction = 4 blocks x 4 rows; lane l -> block l/8, row
// (l%8)/2, half l%2.  Reduction over the 8 lanes of a row by shuffles (xor 1, 8, 16).
namespace b200awq {

template <int MT>
__global__ void __launch_bounds__(128)
    gemv_fast_layout_kernel(const __half* __restrict__ x, int64_t ldx, const int16_t* __restrict__ qweight,
                            const __half* __restrict__ scales, const __half* __restrict__ szeros,
                            const __half* __restrict__ bias, __half* __restrict__ y, int M, int K, int N, int G) {
  extern __shared__ __align__(16) uint4 xs4[];  // [MT][K/8] uint4, natural order
  pdl_trigger();
  pdl_wait();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int KV = K >> 3;
  for (int i = tid; i < MT * KV; i += blockDim.x) {
    const int m = i / KV, k = (i % KV) * 8;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (m < M) {
      const __half* src = x + (int64_t)m * ldx + k;
      if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        v = *reinterpret_cast<const uint4*>(src);
      } else {
        __half t[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = src[j];
        v = *reinterpret_cast<uint4*>(t);
      }
    }
    xs4[i] = v;
  }
  __syncthreads();

  const int R = blockIdx.x * 4 + warp;           // row group
  if (R * 4 >= N) return;
  const int bo = lane >> 3, r = (lane & 7) >> 1, h = lane & 1;
  const int n = R * 4 + r;
  const int16_t* wrow = qweight + (int64_t)R * K;  // K int16 per row group... (N/4 rows of K int16)
  float val[MT];
#pragma unroll
  for (int m = 0; m < MT; ++m) val[m] = 0.f;
  const int nit = (K + 255) / 256;
  constexpr int UN = 4;
  for (int it0 = 0; it0 < nit; it0 += UN) {
    uint4 q[UN];
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const int it = it0 + u;
      const int kc = it * 256 + bo * 64 + h * 32;
      q[u] = make_uint4(0, 0, 0, 0);
      // int16 offset inside the row group: block (it*4+bo)*64 + run r*16 + half h*8
      if (it < nit && kc < K) q[u] = ldg_stream_u4(wrow + (int64_t)(it * 4 + bo) * 64 + r * 16 + h * 8);
    }
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const int it = it0 + u;
      const int kc = it * 256 + bo * 64 + h * 32;
      if (it >= nit || kc >= K) continue;
      const int g = kc / G;
      const float s = __half2float(scales[(int64_t)g * N + n]);
      const float sz = __half2float(szeros[(int64_t)g * N + n]);
      const uint32_t w[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        uint32_t xr[16];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint4 v = xs4[m * KV + (kc >> 3) + c];
          xr[4 * c + 0] = v.x; xr[4 * c + 1] = v.y; xr[4 * c + 2] = v.z; xr[4 * c + 3] = v.w;
        }
        float xsum = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float2 f = __half22float2(u32_as_h2(xr[i]));
          xsum += f.x + f.y;
        }
        float aA = 0.f, aB = 0.f;
#pragma unroll
        for (int uu = 0; uu < 4; ++uu) {
          const uint32_t w8 = w[uu] >> 8;
          const uint32_t p0 = w[uu] & 0x000f000fu, p1 = w[uu] & 0x00f000f0u;
          const uint32_t p2 = w8 & 0x000f000fu, p3 = w8 & 0x00f000f0u;
          aA = fhfma(lo16(p0), lo16(xr[uu]), aA);
          aA = fhfma(hi16(p0), hi16(xr[uu]), aA);
          aB = fhfma(lo16(p1), lo16(xr[uu + 4]), aB);
          aB = fhfma(hi16(p1), hi16(xr[uu + 4]), aB);
          aA = fhfma(lo16(p2), lo16(xr[uu + 8]), aA);
          aA = fhfma(hi16(p2), hi16(xr[uu + 8]), aA);
          aB = fhfma(lo16(p3), lo16(xr[uu + 12]), aB);
          aB = fhfma(hi16(p3), hi16(xr[uu + 12]), aB);
        }
        val[m] += s * (kScaleA * aA + kScaleB * aB) + sz * xsum;
      }
    }
  }
#pragma unroll
  for (int m = 0; m < MT; ++m) {
    float v = val[m];
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    if ((lane & 0x19) == 0 && m < M && n < N) {  // lanes 0, 2, 4, 6: one per row
      if (bias != nullptr) v += __half2float(bias[n]);
      y[(int64_t)m * N + n] = __float2half_rn(v);
    }
  }
}

template <int MT>
static cudaError_t launch_gemv_fast(const FastArgs& a, cudaStream_t st) {
  const size_t smem = (size_t)MT * (a.K / 8) * sizeof(uint4);
  auto kern = gemv_fast_layout_kernel<MT>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e != cudaSuccess) return e;
  }
  const int groups = a.N / 4;
  return launch_kernel(kern, dim3((groups + 3) / 4), dim3(128), smem, st, reinterpret_cast<const __half*>(a.x), a.ldx,
                       a.qweight, reinterpret_cast<const __half*>(a.scales), reinterpret_cast<const __half*>(a.szeros),
                       reinterpret_cast<const __half*>(a.bias), reinterpret_cast<__half*>(a.y), a.M, a.K, a.N, a.G);
}

cudaError_t gemv_fast_layout(const FastArgs& a0, cudaStream_t st) {
  const size_t per_tok = (size_t)(a0.K / 8) * 16;
  int done = 0;
  while (done < a0.M) {
    FastArgs a = a0;
    int m = a0.M - done;
    int mt = m <= 1 ? 1 : (m <= 2 ? 2 : (m <= 4 ? 4 : 8));
    while (mt > 1 && per_tok * mt > 200 * 1024) mt >>= 1;
    if (m > mt) m = mt;
    a.M = m;
    a.x = reinterpret_cast<const __half*>(a0.x) + (int64_t)done * a0.ldx;
    a.y = reinterpret_cast<__half*>(a0.y) + (int64_t)done * a0.N;
    cudaError_t e;
    if (mt == 1) e = launch_gemv_fast<1>(a, st);
    else if (mt == 2) e = launch_gemv_fast<2>(a, st);
    else if (mt == 4) e = launch_gemv_fast<4>(a, st);
    else e = launch_gemv_fast<8>(a, st);
    if (e != cudaSuccess) return e;
    done += m;
  }
  return cudaSuccess;
}

}  // namespace b200awq
