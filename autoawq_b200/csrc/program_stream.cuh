// Decode program, stream variant: the persistent kernel of program.cu re-built around a ONE-TIME RE-LAYOUT of the
// packed weights (the "stream format", restated in numpy in oracle/stream_format.py; the reference's precedent for
// a post-load re-layout is awq/modules/linear/exllama.py:66-79) so that the grid-wide hand-off between two
// dependent linears shrinks to "store, poll".
//
// Why (round-1 measurements, profiles/r01_program_phase_timeline.log): with the checkpoint's GEMM layout
// [K, N/8] a DRAM-efficient tile is >= 128 bytes = 256 columns wide, so N = 4096 has only 16 column blocks for 148
// CTAs: split-K with a fan-in of ~9 CTAs per column block is forced, and its cost - ~110 k 64-bit REDs per op into
// L2, every CTA polling 64-bit sums, a reclamation protocol for the accumulator rows - was ~6 us per op boundary
// against ~4 us of weight streaming.  In the stream format ANY partition is contiguous in memory, so the work is
// cut OUTPUT-STATIONARY: a CTA owns whole 16-column sets (all of K), its 8 consumer warps split the CTA's units
// (set, 128 rows of K) evenly, partial sums meet in shared memory, and the CTA publishes FINISHED fp16 outputs:
//   * no cross-CTA reduction, no atomics, no fixed-point packing, nothing to zero or reclaim, no duty warp;
//   * the hand-off word is (fp16 value | 16-bit tag): one plain 32-bit store by the owner, polled by the consumers
//     with ld.relaxed.gpu - a word is valid when its tag equals the tag of (run, op), so buffers never need
//     clearing and a run is bit-reproducible (fixed summation order);
//   * every CTA reads the whole activation row (K x 4 bytes from L2), RMSNorm needs no second grid-wide pass;
//   * SiLU*mul is fused into the PRODUCER: the stream format of a gate|up linear pairs gate column j and up
//     column j in one lane, so the consumer of `down` polls d words instead of 2 d.
// The weight stream itself is as before: a producer warp keeps a shared-memory ring of bulk copies
// (cp.async.bulk, plain 1-D: every warp's byte range is contiguous) full ACROSS op boundaries.
//
// Included by program.cu (one translation unit: shares the watchdog / debug symbols).
#pragma once

namespace b200awq {

constexpr int kSpStageWarps = 8;                  // warps that stage the activations (thread -> k mapping of aux.cu's
                                                  // rmsnorm_kernel: 256 threads x 8 consecutive k per pass)
constexpr int kSpStagePass = kSpStageWarps * 32 * 8;   // k covered by one staging pass
constexpr int kSpStageBytes = 4288;               // 4 units of G >= 128 (4 x 1072), 7 of G = 64, 14 of G = 32
constexpr int kSpAux = 48;                        // group constants per unit: 32 B scales + 8 B zeros + 8 B pad
constexpr int kSpLMax = 32;                       // 16-column sets one CTA may touch in one op
constexpr int kSpRows = 4;                        // hand-off rows in rotation (op i publishes into row i % 4)
constexpr int kSpXsumMax = 1024;                  // units along K (K / UK) an op may have

struct __align__(128) SpOp {
  const uint8_t* wstream;      // stream-format weights
  const uint32_t* cta_begin;   // [grid + 1] first unit of every CTA (unit = set * NU + j)
  const __half* bias;
  __half* y;                   // fp16 output of the per-op path (every buffer holds the same values after a run)
  const __half* src;           // source in plain global memory (src_op < 0)
  const __half* norm_w;        // RMSNorm weight [K]
  __half* xout;                // RMSNorm prologue: where the recorded norm wanted its output, or null
  __half* act_out;             // mode 1: where the recorded SiLU*mul wanted its output, or null
  int K, N;
  int uk_shift, F, NU, unit_bytes, ups;
  int mode;                    // 0: plain sets, 1: gate|up pairs (publishes silu(gate) * up, N / 2 columns)
  int prologue;                // kProCopy / kProRmsnorm
  int src_op, src_off;         // >= 0: the source is op src_op's published row, from column src_off
  float eps;
  int pad_[4];
};
static_assert(sizeof(SpOp) == 128, "SpOp layout");

__host__ __device__ constexpr size_t sp_fixed_smem(int nw, int spw) {
  return (size_t)nw * spw * kSpStageBytes + (size_t)kSpLMax * nw * 16 * 4 + (size_t)kSpXsumMax * 4 +
         (size_t)2 * nw * spw * 8 + 2 * 128 + 256;
}
static_assert(sp_fixed_smem(8, 4) % 16 == 0, "xs must stay 16-byte aligned");

__device__ __forceinline__ uint4 ld_relaxed_u4(const void* p) {
  uint4 r;
  asm volatile("ld.relaxed.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ void st_relaxed_u32(void* p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t sp_tag(int base, int op) { return (uint32_t)((base + op) % 65535 + 1); }

// set -> original columns (oracle/stream_format.py:set_columns)
__device__ __forceinline__ void sp_cols(int mode, int N, int s, int g, int& lo, int& hi) {
  if (mode == 0) {
    lo = 16 * s + g;
    hi = lo + 8;
  } else {
    lo = 8 * s + g;
    hi = (N >> 1) + lo;
  }
}

// ------------------------------------------------------------------------------------------ re-layout kernel
// One thread per output word / per group-constant slot; run once per linear at program creation.
__global__ void __launch_bounds__(256)
    stream_pack_kernel(const int32_t* __restrict__ qweight, const __half* __restrict__ scales,
                       const int32_t* __restrict__ qzeros, uint8_t* __restrict__ out, int K, int N, int G, int mode) {
  const int UK = G < 128 ? G : 128, F = UK >> 4, NU = K / UK, UB = F * 128 + kSpAux;
  const int NW = N >> 3;
  const int wpu = F * 32 + 12;   // 32-bit slots per unit: fragment words + 8 scale pairs + 2 zero words + 2 pad
  const int64_t total = (int64_t)(N >> 4) * NU * wpu;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int slot = (int)(i % wpu);
    const int64_t unit = i / wpu;
    const int j = (int)(unit % NU), s = (int)(unit / NU);
    uint8_t* ub = out + unit * UB;
    auto nib = [&](int k, int col) -> uint32_t {
      const uint32_t w = (uint32_t)qweight[(int64_t)k * NW + (col >> 3)];
      const int jj = col & 7;
      return (w >> (4 * ((jj >> 1) + 4 * (jj & 1)))) & 0xFu;   // 4 * AWQ_REVERSE_ORDER[jj]
    };
    if (slot < F * 32) {
      int f, lane;
      if (F >= 4) {          // [quad][lane][4]
        const int quad = slot >> 7, r = slot & 127;
        lane = r >> 2;
        f = quad * 4 + (r & 3);
      } else {               // [lane][2]
        lane = slot >> 1;
        f = slot & 1;
      }
      const int g = lane >> 2, tig = lane & 3;
      int lo, hi;
      sp_cols(mode, N, s, g, lo, hi);
      const int k0 = j * UK + 16 * f + 2 * tig;
      const uint32_t w = nib(k0, lo) | nib(k0, hi) << 4 | nib(k0 + 8, lo) << 8 | nib(k0 + 8, hi) << 12 |
                         nib(k0 + 1, lo) << 16 | nib(k0 + 1, hi) << 20 | nib(k0 + 9, lo) << 24 | nib(k0 + 9, hi) << 28;
      reinterpret_cast<uint32_t*>(ub)[slot] = w;
    } else {
      const int a = slot - F * 32;      // 0..7 scale pairs, 8..9 zero words, 10..11 pad
      const int grp = (j * UK) / G;
      uint32_t v = 0;
      if (a < 8) {
        int lo, hi;
        sp_cols(mode, N, s, a, lo, hi);
        const __half sl = scales[(int64_t)grp * N + lo], sh = scales[(int64_t)grp * N + hi];
        v = (uint32_t)__half_as_ushort(sl) | (uint32_t)__half_as_ushort(sh) << 16;
      } else if (a < 10) {
        for (int b = 0; b < 4; ++b) {
          const int g = (a - 8) * 4 + b;
          int lo, hi;
          sp_cols(mode, N, s, g, lo, hi);
          auto znib = [&](int col) -> uint32_t {
            const uint32_t w = (uint32_t)qzeros[(int64_t)grp * NW + (col >> 3)];
            const int jj = col & 7;
            return (w >> (4 * ((jj >> 1) + 4 * (jj & 1)))) & 0xFu;
          };
          v |= (znib(lo) | znib(hi) << 4) << (8 * b);
        }
      }
      reinterpret_cast<uint32_t*>(ub + F * 128)[a] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------ the kernel
// One unit (one 16-column set, UK = 16 F rows of K) times the activations, folded with the unit's group constants:
// returns the unit's contribution to the lo / hi column of lane group g (token 0).
//   raw sums:  S = sum_k x_k (1024 + c q)   (mma.sync on the raw codes, two accumulator chains: even / odd fragments)
//   fold:      s (S - (1024 + c z) X) / c   with X = sum_k x_k of the unit   (csrc/gemv_tile.cuh:v3_fold)
// NU units in flight per call (sp_units<F, NU>): a single unit is one long dependency chain (LDS -> unpack -> 4
// chained HMMA -> fold, ~250 cycles) and a warp has nothing else to overlap it with - measured: unit-at-a-time the
// kernel was bound by exactly that latency at 4.5 TB/s (tools/stream_experiments.py: 759 us per step without the
// math, 1510 with), while the tensor pipe itself sustains 0.33 HMMA/clk/SM = 12.5 TB/s of int4 weights
// (tools/hmma_rate.cu).  Four units interleaved give eight independent chains per warp.
template <int F, int NUQ>
__device__ __forceinline__ void sp_units(const uint8_t* __restrict__ st, int UB, const uint32_t* __restrict__ xs,
                                         const float* __restrict__ xsum, const int (&ju)[NUQ], int lane, bool xl,
                                         float (&tlo)[NUQ], float (&thi)[NUQ]) {
  constexpr uint32_t MA = 0x000f000fu, MB = 0x00f000f0u, MG = 0x64006400u;
  const int g = lane >> 2, tig = lane & 3;
  uint32_t wq[NUQ][F];
#pragma unroll
  for (int i = 0; i < NUQ; ++i) {
    const uint8_t* up = st + (size_t)i * UB;
    if constexpr (F >= 4) {
#pragma unroll
      for (int qd = 0; qd < F / 4; ++qd) {
        const uint4 q = *reinterpret_cast<const uint4*>(up + qd * 512 + lane * 16);
        wq[i][qd * 4 + 0] = q.x;
        wq[i][qd * 4 + 1] = q.y;
        wq[i][qd * 4 + 2] = q.z;
        wq[i][qd * 4 + 3] = q.w;
      }
    } else {
      const uint2 q = *reinterpret_cast<const uint2*>(up + lane * 8);
      wq[i][0] = q.x;
      wq[i][1] = q.y;
    }
  }
  float acc[NUQ][2][4];
#pragma unroll
  for (int i = 0; i < NUQ; ++i)
#pragma unroll
    for (int c = 0; c < 2; ++c) acc[i][c][0] = acc[i][c][1] = acc[i][c][2] = acc[i][c][3] = 0.f;
#pragma unroll
  for (int f = 0; f < F; ++f) {
#pragma unroll
    for (int i = 0; i < NUQ; ++i) {
      uint2 xb = make_uint2(0u, 0u);
      if (xl) xb = *reinterpret_cast<const uint2*>(xs + ((size_t)ju[i] * F + f) * 8 + tig * 2);
      const uint32_t w = wq[i][f], w8 = w >> 8;
      mma_16816(acc[i][f & 1], lop3_and_or(w, MA, MG), lop3_and_or(w, MB, MG), lop3_and_or(w8, MA, MG),
                lop3_and_or(w8, MB, MG), xb.x, xb.y);
    }
  }
#pragma unroll
  for (int i = 0; i < NUQ; ++i) {
    const uint8_t* ax = st + (size_t)i * UB + F * 128;
    const float2 sc = __half22float2(u32_as_h2(*reinterpret_cast<const uint32_t*>(ax + 4 * g)));
    const uint32_t zb = ax[32 + g];
    const float X = xsum[ju[i]];
    const float s_lo = acc[i][0][0] + acc[i][1][0], s_hi = acc[i][0][2] + acc[i][1][2];
    tlo[i] = sc.x * (s_lo - (1024.f + static_cast<float>(zb & 0xFu)) * X);
    thi[i] = (sc.y * 0.0625f) * (s_hi - (1024.f + 16.f * static_cast<float>(zb >> 4)) * X);
  }
}

// a chunk of n units starting at unit j (within its set): apply(t_lo, t_hi) is called once per unit, in unit order
// (so the sums do not depend on how the chunk was cut into groups of four)
template <int F, int GR, typename Apply>
__device__ __forceinline__ void sp_chunk(const uint8_t* __restrict__ st, int UB, int n, const uint32_t* __restrict__ xs,
                                         const float* __restrict__ xsum, int j, int NU, int lane, bool xl, Apply&& apply) {
  int i = 0;
  for (; i + GR <= n; i += GR) {
    int ju[GR];
#pragma unroll
    for (int q = 0; q < GR; ++q) {
      ju[q] = j + i + q;
      if (ju[q] >= NU) ju[q] -= NU;      // the chunk may run across a set boundary (at most one: NU >= units per chunk)
    }
    float a[GR], b[GR];
    sp_units<F, GR>(st + (size_t)i * UB, UB, xs, xsum, ju, lane, xl, a, b);
#pragma unroll
    for (int q = 0; q < GR; ++q) apply(a[q], b[q]);
  }
  for (; i < n; ++i) {
    int ju[1] = {j + i >= NU ? j + i - NU : j + i};
    float a[1], b[1];
    sp_units<F, 1>(st + (size_t)i * UB, UB, xs, xsum, ju, lane, xl, a, b);
    apply(a[0], b[0]);
  }
}

// debug stamps (knob 3 = 2), per op and CTA (first 8 CTAs, first 32 ops):
// [0] op begin, [1] source row complete (poll over), [2] activations staged, [3] warp 0's first chunk landed,
// [4] warp 0 finished its units, [5] all warps finished, [6] outputs published, [7] unused
// knob 3 = 8: per-WARP stamps of the first 8 CTAs / 16 ops: g_sp_dbg[op][cta][warp][slot], slots: 0 op begin, 1 own
// polls done, 2 staged (past the barrier), 3 first chunk landed, 4 own units done, 5 past the post-loop barrier,
// 6 own finish stores issued.  (A timer read right after bar.sync captures the ARRIVAL: the barrier blocks at the next
// instruction that touches barrier-protected state - hence the shared-memory read in front of slots 2 and 5.)
__device__ unsigned long long g_sp_dbg[16 * 8 * 8 * 8];
cudaError_t stream_debug_read(void* dst, size_t bytes) {
  return cudaMemcpyFromSymbol(dst, g_sp_dbg, bytes < sizeof(g_sp_dbg) ? bytes : sizeof(g_sp_dbg));
}
#define SP_WSTAMP(slot)                                                                                          \
  do {                                                                                                           \
    if (dbg == 8 && blockIdx.x < 8 && op < 16) {                                                                 \
      __syncwarp();                                                                                              \
      if (lane == 0) g_sp_dbg[((op * 8 + blockIdx.x) * 8 + cw) * 8 + (slot)] = prog_timer();                    \
    }                                                                                                            \
  } while (0)
#define SP_TOUCH_SMEM()                                                                      \
  do {                                                                                       \
    if (dbg == 8) {                                                                          \
      int tv_;                                                                               \
      asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(tv_) : "r"(smem_u32(wfirst)) : "memory"); \
      if (tv_ == 0x7fffffff) __trap();                                                       \
    }                                                                                        \
  } while (0)
#define SP_STAMP(slot)                                                                                       \
  do {                                                                                                       \
    if (dbg == 2 && ct == 0 && blockIdx.x < 8 && op < 32) g_prog_dbg[(op * 8 + blockIdx.x) * 8 + (slot)] = prog_timer(); \
  } while (0)

__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

template <int NW, int SPW, int GR>
__global__ void __launch_bounds__(32 + NW * 32, 1)
    stream_program_kernel(const SpOp* __restrict__ ops, const uint32_t* __restrict__ cta_all, int n_ops,
                          uint32_t* __restrict__ rows, int row_stride, int* __restrict__ state, int dbg) {
  extern __shared__ __align__(1024) uint8_t sp_smem[];
  uint8_t* ring = sp_smem;
  float* part = reinterpret_cast<float*>(sp_smem + (size_t)(NW * SPW) * kSpStageBytes);   // [LMax][8 warps][16]
  float* xsum = part + kSpLMax * NW * 16;                                           // [K / UK]
  uint64_t* full = reinterpret_cast<uint64_t*>(xsum + kSpXsumMax);
  uint64_t* empty = full + (NW * SPW);
  SpOp* sdesc = reinterpret_cast<SpOp*>(empty + (NW * SPW));      // [2] op descriptors, prefetched one op ahead
  int* misc = reinterpret_cast<int*>(sdesc + 2);
  float* wsum = reinterpret_cast<float*>(misc);        // [8]
  int* wfirst = misc + 8;                              // [NW] first local set each warp touched (-1: none)
  int* wlast = misc + 8 + NW;                    // [NW]
  uint32_t* scta = reinterpret_cast<uint32_t*>(misc + 8 + 2 * NW);   // [2][2] this CTA's unit range (with sdesc)
  static_assert((12 + 2 * NW) * 4 <= 256, "misc area");
  uint32_t* xs = reinterpret_cast<uint32_t*>(sp_smem + sp_fixed_smem(NW, SPW));   // activations in B-fragment order

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nblk = gridDim.x, bid = blockIdx.x;
  const int base = state[0];     // tag base of this run (advanced by the last CTA to leave, see the end)

  if (tid == 0) {
    for (int s = 0; s < (NW * SPW); ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) {   // op 0's descriptor
    reinterpret_cast<uint32_t*>(sdesc)[lane] = reinterpret_cast<const uint32_t*>(ops)[lane];
    if (lane < 2) scta[lane] = cta_all[bid + lane];
  }
  __syncthreads();

  if (warp == 0) {
    // ============================================================ producer: the weight stream of ALL ops
    // Lane w feeds consumer warp w's private ring.  The eight lanes run ONE converged loop and probe their
    // "slot free" barriers with the non-blocking mbarrier.test_wait: with a blocking try_wait per lane (round 1, and
    // the first version of this kernel) a lane waiting for a slot that frees up late suspended the whole warp, so
    // slots that were free long ago were refilled microseconds late and the ring ran dry at every op boundary.
    // Descriptor fields of the next op are fetched one op ahead into registers (global loads, off the critical path).
    {
      const int w = lane < NW ? lane : 0;
      bool active = lane < NW;
      struct Run {
        uint32_t u, ub;
        int UB, ups;
        const uint8_t* src;
      };
      auto fetch = [&](int op, Run& r) {
        r.u = r.ub = 0;
        r.UB = r.ups = 1;
        r.src = nullptr;
        if (op < n_ops && lane < NW) {
          const uint32_t u0 = cta_all[(size_t)op * (nblk + 1) + bid], u1 = cta_all[(size_t)op * (nblk + 1) + bid + 1];
          const uint32_t nu = u1 - u0;
          r.u = u0 + (uint32_t)((uint64_t)nu * w / NW);
          r.ub = u0 + (uint32_t)((uint64_t)nu * (w + 1) / NW);
          r.UB = ops[op].unit_bytes;
          r.ups = ops[op].ups;
          r.src = ops[op].wstream;
        }
      };
      Run cur, nxt;
      int op = 0;
      fetch(0, cur);
      fetch(1, nxt);
      // Loads are neither gated on the consumers' staging nor preceded by an HBM -> L2 prefetch: both measured slower
      // here (DESIGN.md §3.5b, profiles/r02_stream_experiments.md).
      int stage_i = 0;
      uint32_t ph = 0;
      ProgWatch wd;
      for (;;) {
        while (active && cur.u >= cur.ub) {        // this lane's run of the op is requested: next op
          if (++op >= n_ops) {
            active = false;
            break;
          }
          cur = nxt;
          fetch(op + 1, nxt);
        }
        if (!__any_sync(0xffffffffu, active)) break;
        bool issued = false;
        if (active) {
          const int stage = w * SPW + stage_i;
          if (mbar_test_wait(&empty[stage], ph ^ 1)) {
            const int n = (int)(cur.ub - cur.u) < cur.ups ? (int)(cur.ub - cur.u) : cur.ups;
            mbar_arrive_expect_tx(&full[stage], (uint32_t)(n * cur.UB));
            bulk_load_1d(ring + (size_t)stage * kSpStageBytes, cur.src + (size_t)cur.u * cur.UB, (uint32_t)(n * cur.UB),
                         &full[stage]);
            cur.u += (uint32_t)cur.ups;
            if (++stage_i == SPW) { stage_i = 0; ph ^= 1; }
            issued = true;
          }
        }
        if (!__any_sync(0xffffffffu, issued)) {   // nothing to load: leave the issue slots alone
          if (__any_sync(0xffffffffu, wd.tick(kWEmpty, op))) break;   // watchdog (warp-uniform): never hang the GPU
          __nanosleep(32);
        }
      }
    }
  } else {
    // ================================================================ consumers
    const int cw = warp - 1;
    const int ct = tid - 32;
    const int g = lane >> 2, tig = lane & 3;
    const bool xl = g == 0;       // M = 1: token 0 is column n = 0 of the MMA's B operand, supplied by the g = 0 lanes
    int stage_i = 0;
    uint32_t ph = 0;

    for (int op = 0; op < n_ops; ++op) {
      const SpOp* o = sdesc + (op & 1);                            // shared memory (prefetched during op - 1)
      const int K = o->K, N = o->N, NU = o->NU, F = o->F, UB = o->unit_bytes, ups = o->ups, mode = o->mode;
      const uint32_t u0 = scta[(op & 1) * 2], u1 = scta[(op & 1) * 2 + 1];
      const uint32_t nu = u1 - u0;
      const uint32_t ua = u0 + (uint32_t)((uint64_t)nu * cw / NW), ub = u0 + (uint32_t)((uint64_t)nu * (cw + 1) / NW);
      const int set0 = (int)(u0 / NU);                            // first set of the CTA
      const __half* bias = o->bias;
      __half* y = o->y;
      __half* act_out = o->act_out;
      SP_STAMP(0);
      SP_WSTAMP(0);

      // ---- stage the activations (whole row, every CTA): poll the producer's published row / read global memory,
      //      apply the recorded RMSNorm, write them in B-fragment order and keep the per-unit sums sum_k x_k.
      //      Thread t takes 8 consecutive k per pass (k = 2048 pass + 8 t) and sums squares in the order of
      //      aux.cu's rmsnorm_kernel, so the norm reproduces the stand-alone kernel bit for bit.
      {
        const int uk_shift = o->uk_shift;
        const int seg = (1 << uk_shift) >> 3;                      // lanes per unit (each lane holds 8 consecutive k)
        const bool from_row = o->src_op >= 0;
        const uint32_t* row = from_row ? rows + (size_t)(o->src_op % kSpRows) * row_stride + o->src_off : nullptr;
        const uint32_t want = from_row ? sp_tag(base, o->src_op) : 0u;
        const __half* src = o->src;
        const bool norm = o->prologue == kProRmsnorm;
        const __half* nw = o->norm_w;
        float ss = 0.f;
        // the norm weights of the first batch of passes depend on nothing: in flight before the polls
        uint4 nwv[4];
        if (norm) {
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            const int c = cw * 256 + b * kSpStagePass + lane * 8;
            if (cw < kSpStageWarps && c < K) nwv[b] = __ldg(reinterpret_cast<const uint4*>(nw + c));
          }
        }
        // fragment order: k = 16 ks + j -> word ks * 8 + ((j & 7) >> 1) * 2 + (j >> 3)   (a word = the pair (j, j + 1))
        auto frag_ptr = [&](int c) { return xs + (c >> 4) * 8 + ((c >> 3) & 1); };   // + 2 * pair index
        auto unit_sums = [&](int c, bool ok, const uint32_t (&h)[4]) {
          float sx = 0.f;
          if (ok) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float2 f = __half22float2(u32_as_h2(h[q]));
              sx += f.x + f.y;
            }
          }
          for (int d = 1; d < seg; d <<= 1) sx += __shfl_xor_sync(0xffffffffu, sx, d);
          if (ok && (lane & (seg - 1)) == 0) xsum[c >> uk_shift] = sx;
        };
        // passes are taken in batches of 4: every load of a batch is in flight before the first tag is looked at
        // (a poll is an L2 round trip of ~1 us under load; K = 14336 has 7 passes)
        // (the first kSpStageWarps warps stage; the others wait at the barriers)
        const int cb_first = cw < kSpStageWarps ? cw * 256 : K;
        for (int cb0 = cb_first; cb0 < K; cb0 += 4 * kSpStagePass) {      // warp-uniform trip counts
          uint4 v0[4], v1[4];
          if (from_row) {
#pragma unroll
            for (int b = 0; b < 4; ++b) {
              const int c = cb0 + b * kSpStagePass + lane * 8;
              if (c < K) {
                v0[b] = ld_relaxed_u4(row + c);
                v1[b] = ld_relaxed_u4(row + c + 4);
              }
            }
          }
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            const int cb = cb0 + b * kSpStagePass;
            if (cb >= K) break;                                          // warp-uniform
            const int c = cb + lane * 8;
            const bool ok = c < K;
            uint32_t h[4] = {0u, 0u, 0u, 0u};                            // the eight fp16 values as four pairs
            if (ok) {
              if (from_row) {
                ProgWatch wd;
                for (;;) {
                  const uint4 a = v0[b], d = v1[b];
                  if ((a.x >> 16) == want && (a.y >> 16) == want && (a.z >> 16) == want && (a.w >> 16) == want &&
                      (d.x >> 16) == want && (d.y >> 16) == want && (d.z >> 16) == want && (d.w >> 16) == want)
                    break;
                  if (wd.tick(kWCopy, op)) break;
                  v0[b] = ld_relaxed_u4(row + c);
                  v1[b] = ld_relaxed_u4(row + c + 4);
                }
                h[0] = (v0[b].x & 0xffffu) | (v0[b].y << 16);
                h[1] = (v0[b].z & 0xffffu) | (v0[b].w << 16);
                h[2] = (v1[b].x & 0xffffu) | (v1[b].y << 16);
                h[3] = (v1[b].z & 0xffffu) | (v1[b].w << 16);
              } else {
                const uint4 v = ldg_stream_u4(src + c);
                h[0] = v.x; h[1] = v.y; h[2] = v.z; h[3] = v.w;
              }
              uint32_t* dst = frag_ptr(c);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                dst[2 * q] = h[q];
                const float2 f = __half22float2(u32_as_h2(h[q]));
                ss += f.x * f.x + f.y * f.y;
              }
            }
            if (!norm) unit_sums(c, ok, h);
          }
        }
        SP_STAMP(1);
        SP_WSTAMP(1);
        if (norm) {
          ss = prog_warp_sum(ss);
          if (lane == 0 && cw < kSpStageWarps) wsum[cw] = ss;
          named_bar_sync_gv(1, (NW * 32));
          float tot = 0.f;
#pragma unroll
          for (int i = 0; i < kSpStageWarps; ++i) tot += wsum[i];
          const float rs = rsqrtf(tot / static_cast<float>(K) + o->eps);
          __half* xout = o->xout;
          int xlo = 0, xhi = 0;
          if (xout != nullptr) {       // this CTA's share of the norm's recorded output buffer
            const int u8 = K >> 3;
            xlo = (int)((int64_t)u8 * bid / nblk) << 3;
            xhi = (int)((int64_t)u8 * (bid + 1) / nblk) << 3;
          }
          for (int cb0 = cb_first; cb0 < K; cb0 += 4 * kSpStagePass) {   // the thread's own chunks again
#pragma unroll
            for (int b = 0; b < 4; ++b) {
              const int cb = cb0 + b * kSpStagePass;
              if (cb >= K) break;
              const int c = cb + lane * 8;
              const bool ok = c < K;
              uint32_t h[4] = {0u, 0u, 0u, 0u};
              if (ok) {
                uint32_t* dst = frag_ptr(c);
                const uint4 wv = cb0 == cb_first ? nwv[b] : __ldg(reinterpret_cast<const uint4*>(nw + c));
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const float2 a = __half22float2(u32_as_h2(dst[2 * q]));
                  const float2 wq = __half22float2(u32_as_h2((&wv.x)[q]));
                  // arithmetic of aux.cu's rmsnorm_kernel: fp16(x * rs * w)
                  h[q] = h2_as_u32(__halves2half2(__float2half_rn(a.x * rs * wq.x), __float2half_rn(a.y * rs * wq.y)));
                  dst[2 * q] = h[q];
                }
                if (c >= xlo && c < xhi) *reinterpret_cast<uint4*>(xout + c) = make_uint4(h[0], h[1], h[2], h[3]);
              }
              unit_sums(c, ok, h);
            }
          }
        }
        named_bar_sync_gv(1, (NW * 32));
      }
      SP_STAMP(2);
      SP_TOUCH_SMEM();
      SP_WSTAMP(2);
      // every warp is past op - 1's finish phase (it read sdesc[(op - 1) & 1]): fetch op + 1's descriptor into that
      // slot, asynchronously - it lands during this op's unit loop
      if (cw == 0 && op + 1 < n_ops) {
        SpOp* dn = sdesc + ((op + 1) & 1);
        if (lane < 8) cp_async_16(reinterpret_cast<uint8_t*>(dn) + lane * 16, reinterpret_cast<const uint8_t*>(ops + op + 1) + lane * 16);
        else if (lane < 10)
          cp_async_4(scta + ((op + 1) & 1) * 2 + (lane - 8), cta_all + (size_t)(op + 1) * (nblk + 1) + bid + (lane - 8));
      }

      // ---- this warp's run of units
      {
        int s_cur = (int)(ua / NU), j = (int)(ua - (uint32_t)s_cur * NU);
        float ylo = 0.f, yhi = 0.f;
        int first_ls = -1, last_ls = -1;
        auto flush = [&]() {
          const int ls = s_cur - set0;
          if (tig == 0) {
            float* p = part + ((size_t)ls * NW + cw) * 16;
            p[g] = ylo;
            p[g + 8] = yhi;
          }
          if (first_ls < 0) first_ls = ls;
          last_ls = ls;
          ylo = yhi = 0.f;
        };
        for (uint32_t u = ua; u < ub; u += ups) {
          const int n = (int)(ub - u) < ups ? (int)(ub - u) : ups;
          const int stage = cw * SPW + stage_i;
          prog_mbar_wait(&full[stage], ph, kWFull, op);
          if (u == ua) {
            SP_STAMP(3);
            SP_WSTAMP(3);
          }
          const uint8_t* st = ring + (size_t)stage * kSpStageBytes;
          auto apply = [&](float t_lo, float t_hi) {
            ylo += t_lo;
            yhi += t_hi;
            if (++j == NU) {
              flush();
              j = 0;
              ++s_cur;
            }
          };
          const int j0 = j;
          if (F == 8) sp_chunk<8, GR>(st, UB, n, xs, xsum, j0, NU, lane, xl, apply);
          else if (F == 4) sp_chunk<4, GR>(st, UB, n, xs, xsum, j0, NU, lane, xl, apply);
          else sp_chunk<2, GR>(st, UB, n, xs, xsum, j0, NU, lane, xl, apply);
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty[stage]);
          if (++stage_i == SPW) { stage_i = 0; ph ^= 1; }
        }
        if (j != 0 && ua < ub) flush();     // the run ended inside a set
        if (lane == 0) {                    // (written by every warp for every op: nothing to reset)
          wfirst[cw] = first_ls;
          wlast[cw] = last_ls;
        }
      }
      SP_STAMP(4);
      SP_WSTAMP(4);
      if (cw == 0) cp_async_wait_all();     // op + 1's descriptor has landed (issued a whole unit loop ago)
      named_bar_sync_gv(1, (NW * 32));
      SP_STAMP(5);
      SP_TOUCH_SMEM();
      SP_WSTAMP(5);

      // ---- finish: sum the warps' partial sums in a fixed order, publish (fp16 | tag) and the per-op-path tensors
      {
        const int nsets = nu == 0 ? 0 : (int)((u1 - 1) / NU) - set0 + 1;
        const uint32_t tagw = sp_tag(base, op) << 16;
        uint32_t* out_row = rows + (size_t)(op % kSpRows) * row_stride;
        for (int t = ct; t < nsets * 8; t += (NW * 32)) {
          const int ls = t >> 3, gg = t & 7;
          float lo = 0.f, hi = 0.f;
#pragma unroll
          for (int w = 0; w < NW; ++w) {
            if (wfirst[w] >= 0 && wfirst[w] <= ls && ls <= wlast[w]) {
              const float* p = part + ((size_t)ls * NW + w) * 16;
              lo += p[gg];
              hi += p[gg + 8];
            }
          }
          int clo, chi;
          sp_cols(mode, N, set0 + ls, gg, clo, chi);
          if (bias != nullptr) {
            lo += __half2float(bias[clo]);
            hi += __half2float(bias[chi]);
          }
          const __half hlo = __float2half_rn(lo), hhi = __float2half_rn(hi);
          if (mode == 0) {
            st_relaxed_u32(out_row + clo, tagw | __half_as_ushort(hlo));
            st_relaxed_u32(out_row + chi, tagw | __half_as_ushort(hhi));
          } else {
            // fused SiLU*mul with the arithmetic of aux.cu's silu_mul_kernel
            const float gf = __half2float(hlo), uf = __half2float(hhi);
            const __half a = __float2half_rn(gf / (1.f + __expf(-gf)) * uf);
            st_relaxed_u32(out_row + clo, tagw | __half_as_ushort(a));
            if (act_out != nullptr) act_out[clo] = a;
          }
          y[clo] = hlo;      // the per-op path's tensors: nobody inside the kernel reads them
          y[chi] = hhi;
        }
      }
      SP_STAMP(6);
      SP_WSTAMP(6);
      // (the next op's staging barriers separate these reads of part[] / wfirst[] from the next writes; the
      // descriptor slot this op used is overwritten only after the next op's staging barrier)
    }
  }

  // ---- the last CTA to leave advances the tag base for the next run (every CTA read it before doing anything)
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(&state[1], 1) == nblk - 1) {
      state[1] = 0;
      state[0] = (base + n_ops) % 65535;
    }
  }
}

}  // namespace b200awq
