// Decode program: the whole chain of M = 1 operator calls of a decode step (RMSNorm -> W4A16 linear -> ... ->
// SiLU*mul -> linear) recorded once and executed by ONE persistent kernel launch.
//
// Why (measured, B200, profiles/r01_gemv_v3_phase_timeline.log): a stand-alone GEMV launch spends ~5 us of its
// 7-20 us outside the weight stream - launch + ring fill (the first tile lands after ~5 us of loaded HBM latency),
// the split-K tail, the ticket round trip - and HBM idles through every one of those gaps, 128 times per decode
// step.  The packed weights never depend on the activations, so here the producer warp of every CTA walks the
// WHOLE op list and keeps its shared-memory ring full across op boundaries: while the consumers of op i reduce,
// publish and wait for the grid-wide completion of op i, the tiles of op i+1 are already landing.
//
// Structure (one CTA per SM, launched cooperatively so that all CTAs are co-resident; 10 warps per CTA):
//   * producer warp: as in the persistent GEMV (gemv.cu) - lane w feeds consumer warp w's private stages with
//     8 KB weight tiles (TMA 2-D, 128B swizzle) + the tile's group scales / zeros - but over all ops back to back;
//     the tensor maps live in the device-resident op table;
//   * 8 consumer warps, per op: (1) poll the columns they need of the previous op's PACKED row until complete (each
//     64-bit word carries the split-K sum and the number of tiles that contributed - see "packed split-K hand-off"
//     below), (2) build the op's activations in shared memory from it - fp16(sum + bias) is exactly what the
//     per-op path stores - applying the recorded glue op on the fly (RMSNorm: every CTA recomputes the row's norm
//     from L2; SiLU*mul: only the k-range of the CTA's own tiles) with the arithmetic of the stand-alone kernels
//     (aux.cu); (3) the tile loop and per-group fold of the persistent GEMV, unchanged (gemv_tile.cuh); (4) one
//     packed RED per column of each column block the CTA touched.  Nothing to publish, nothing to acknowledge;
//   * duty warp: off the critical path, stores this CTA's slice of every op's fp16 output (and of the SiLU*mul
//     output), so every tensor of the per-op path holds the same values after a run, and recycles the four rotating
//     rows (staged[] / zeroed[] counters, see program_kernel).
//   History (profiles/r01_program_l2ahead_sweep.md, DESIGN.md 3.5): tickets + last-arriver finalisation: ~10 us per
//   op boundary, 529 tok/s; fp32 row + one release/acquire counter per op: ~8 us, 652 tok/s; packed rows: 734-744.
//
// Reference call sequence this replaces: awq/modules/fused/block.py:117-170 (norm -> qkv -> ... -> o -> norm ->
// mlp) with awq/modules/fused/mlp.py:41-55 (gate/up GEMM, silu*mul, down GEMM), each a separate awq_ext call.
#include <cuda.h>

#include <algorithm>
#include <cstring>
#include <vector>

#include "../../include/b200awq.h"
#include "common.cuh"
#include "gemv_tile.cuh"
#include "kernels.h"

namespace b200awq {

enum { kProCopy = 0, kProRmsnorm = 1, kProSilu = 2 };

struct __align__(128) ProgOp {
  CUtensorMap tmw;        // qweight [K, N/8] int32, box 32 words x 64 rows, 128B swizzle
  const __half* scales;
  const int32_t* qzeros;
  const __half* bias;
  __half* y;
  const __half* src;      // external source (fp16, global) when !src_prev: COPY x, RMSNORM row, SILU gate|up
  const __half* norm_w;   // RMSNORM weight [K]
  __half* xout;           // where the recorded glue op wanted its result, or null
  int src_off;            // src_prev: first column of the previous op's output this op reads
  int src_prev;           // 1: the source is the previous op's output, taken from its fp32 accumulators
  int K, N, G, g_shift;
  int prologue;
  float eps;
  int ext_dep;            // >= 0: the external source was written by that (older) op of this program
  const int32_t* qw_src;  // the checkpoint-format qweight (host-side use: the stream variant re-lays it out)
};
static_assert(sizeof(ProgOp) == 256, "ProgOp layout");

constexpr int kProgMT = 1;
__host__ __device__ constexpr size_t prog_fixed_smem(int spw) {
  return (size_t)kV3Warps * spw * (kV3TileBytes + kV3AuxBytes) +
         (size_t)(kV3Warps * kProgMT * kGvRedStride + kV3Warps * kProgMT * kV3TileCols) * 4 +
         2 * kV3Warps * spw * 8 + 128 + 64;
}
static_assert(prog_fixed_smem(2) % 16 == 0, "xs must stay 16-byte aligned");

// knob 3 = 2: per-op phase timestamps (globaltimer ns) of the first 8 CTAs for the first 32 kernel ops:
// [0] op begin, [1] previous op complete (wait over), [2] activations staged, [3] first tile landed (warp 0),
// [4] warp 0 finished its tiles, [5] all warps finished, [6] partial sums added, [7] published.
__device__ unsigned long long g_prog_dbg[32 * 8 * 8];
__device__ __forceinline__ unsigned long long prog_timer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
cudaError_t program_debug_read(void* dst, size_t bytes) {
  return cudaMemcpyFromSymbol(dst, g_prog_dbg, bytes < sizeof(g_prog_dbg) ? bytes : sizeof(g_prog_dbg));
}
#define PROG_STAMP(slot)                                                                    \
  do {                                                                                      \
    if (dbg == 2 && ct == 0 && blockIdx.x < 8 && op < 32) g_prog_dbg[(op * 8 + blockIdx.x) * 8 + (slot)] = prog_timer(); \
  } while (0)

__device__ __forceinline__ float prog_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------------- packed split-K hand-off
// One 64-bit word per output column carries the sum AND its own completion state:
//     word = (tiles contributed << 48) | sum of (v_fixed + tiles * 2^39),   v_fixed = round(v * 2^24)
// Every push is a single red.add.u64, so a reader that sees tiles == K/64 holds the complete sum - no counter to
// publish after the data, no acknowledgement to wait for, no acquire before reading it: the chain between two
// ops is one RED (one way) plus one polling load.  Integer addition also makes the result independent of the
// order in which CTAs arrive: a program run is bit-reproducible.
// Range: |partial sum| is clamped to tiles * 32768 (fp16 outputs beyond that are inf anyway); resolution 2^-24
// (one fp16 subnormal step, below the fp32 rounding of the per-op path for |y| >= 1); K/64 < 256 tiles per column.
constexpr int kProgRows = 4;              // accumulator rows in rotation (see the reclamation protocol below)
static_assert(kProgRows == 4, "prog_wait_row_clean hard-codes the rotation depth");
constexpr float kFixScale = 16777216.0f;  // 2^24
__device__ __forceinline__ unsigned long long prog_pack(float v, int ntl) {
  long long f = __float2ll_rn(v * kFixScale);
  const long long lim = ((long long)ntl << 39) - 1;
  f = f > lim ? lim : (f < -lim ? -lim : f);
  return ((unsigned long long)ntl << 48) + (unsigned long long)(((long long)ntl << 39) + f);
}
__device__ __forceinline__ void red_add_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("red.relaxed.gpu.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// Polling load: STRONG (relaxed at gpu scope), not a weak load with a cache hint - the rows are polled without any
// acquire in front, and a weak ld.cg may keep returning a stale copy from the near L2 partition for ever (seen on
// B200: the duty warps spun on complete rows).
__device__ __forceinline__ ulonglong2 ldcg_u64x2(const unsigned long long* p) {
  ulonglong2 r;
  asm volatile("ld.relaxed.gpu.global.v2.u64 {%0,%1}, [%2];" : "=l"(r.x), "=l"(r.y) : "l"(p) : "memory");
  return r;
}
// 8 consecutive outputs of the previous op as the per-op path would have stored them, fp16(sum + bias);
// ok = false while any of the 8 columns is still missing contributions (TPC = the previous op's K / 64)
__device__ __forceinline__ bool prog_prev8(const unsigned long long* __restrict__ row, const __half* __restrict__ bias,
                                           int c, int TPC, uint4& out) {
  const ulonglong2 w0 = ldcg_u64x2(row + c), w1 = ldcg_u64x2(row + c + 2), w2 = ldcg_u64x2(row + c + 4),
                   w3 = ldcg_u64x2(row + c + 6);
  const unsigned long long w[8] = {w0.x, w0.y, w1.x, w1.y, w2.x, w2.y, w3.x, w3.y};
  bool ok = true;
  float v[8];
  const long long off = (long long)TPC << 39;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    ok = ok && (int)(w[j] >> 48) == TPC;
    v[j] = __ll2float_rn((long long)(w[j] & 0xFFFFFFFFFFFFull) - off) * (1.0f / kFixScale);
  }
  if (bias != nullptr) {
    const uint4 bv = *reinterpret_cast<const uint4*>(bias + c);
    const __half* bh = reinterpret_cast<const __half*>(&bv);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] += __half2float(bh[j]);
  }
  __half* rh = reinterpret_cast<__half*>(&out);
#pragma unroll
  for (int j = 0; j < 8; ++j) rh[j] = __float2half_rn(v[j]);
  return ok;
}

// Watchdog for every spin in this kernel: a lost completion must never hang the GPU.  The first wait that exceeds
// the limit records {code, op, CTA, 1} in g_prog_abort and every spin loop bails out once that is set: the kernel
// terminates (with garbage results) and the host reads the record with b200awq_debug_read under knob 3 = 3.
// [0..3] = first record; [4 + cta * 10 + warp] = (code << 16 | op) of the wait each warp abandoned (0 = none)
__device__ int g_prog_abort[4 + 256 * 10];
cudaError_t program_abort_read(void* dst, size_t bytes) {
  return cudaMemcpyFromSymbol(dst, g_prog_abort, bytes < sizeof(g_prog_abort) ? bytes : sizeof(g_prog_abort));
}
cudaError_t program_abort_clear(cudaStream_t st) {
  void* p = nullptr;
  cudaError_t e = cudaGetSymbolAddress(&p, g_prog_abort);
  return e != cudaSuccess ? e : cudaMemsetAsync(p, 0, sizeof(g_prog_abort), st);
}
// watchdog limit in ns (default 0.5 s; knob 16 = seconds, for runs under compute-sanitizer / cuda-gdb where a kernel
// is orders of magnitude slower and a healthy wait would be mistaken for a lost completion)
__device__ unsigned long long g_prog_watch_ns = 500000000ull;
cudaError_t program_set_watchdog_seconds(int seconds) {
  const unsigned long long ns = seconds > 0 ? (unsigned long long)seconds * 1000000000ull : 500000000ull;
  return cudaMemcpyToSymbol(g_prog_watch_ns, &ns, sizeof(ns));
}
struct ProgWatch {
  unsigned long long t_start = 0;
  int spins = 0;
  // returns true when the caller must give up
  __device__ __forceinline__ bool tick(int code, int op) {
    if ((++spins & 255) == 0) {
      if (*reinterpret_cast<volatile int*>(&g_prog_abort[3]) != 0) {
        if (blockIdx.x < 256 && g_prog_abort[4 + blockIdx.x * 10 + (threadIdx.x >> 5)] == 0)
          g_prog_abort[4 + blockIdx.x * 10 + (threadIdx.x >> 5)] = (code << 16) | (op & 0xffff);
        return true;
      }
      const unsigned long long now = prog_timer();
      if (t_start == 0) t_start = now;
      else if (now - t_start > g_prog_watch_ns) {
        if (atomicCAS(&g_prog_abort[3], 0, 1) == 0) {
          g_prog_abort[0] = code;
          g_prog_abort[1] = op;
          g_prog_abort[2] = blockIdx.x;
        }
        if (blockIdx.x < 256 && g_prog_abort[4 + blockIdx.x * 10 + (threadIdx.x >> 5)] == 0)
          g_prog_abort[4 + blockIdx.x * 10 + (threadIdx.x >> 5)] = (code << 16) | (op & 0xffff);
        return true;
      }
    }
    return false;
  }
};
enum { kWStaged = 1, kWExtDep = 2, kWEmpty = 3, kWFull = 4, kWGate = 5, kWRedOk = 6, kWStagedOp = 7, kWDutyY = 8,
       kWDutySilu = 9, kWCopy = 10, kWSilu = 11, kWNorm = 12 };
__device__ __forceinline__ void prog_wait(const int* cnt, int target, int code, int op) {
  ProgWatch wd;
  while (ld_acquire_s32(cnt) < target)
    if (wd.tick(code, op)) break;
}
// returns false when the wait was abandoned (abort): the caller must not touch the barrier's stage any more
__device__ __forceinline__ bool prog_mbar_wait(uint64_t* bar, uint32_t parity, int code, int op) {
  ProgWatch wd;
  while (!mbar_try_wait(bar, parity))
    if (wd.tick(code, op)) return false;
  return true;
}
__device__ __forceinline__ void prog_wait_smem(volatile int* flag, int target, int code, int op) {
  ProgWatch wd;
  while (*flag < target)
    if (wd.tick(code, op)) break;
}

// "Row op % 4 is clean": normally read from the shared-memory flag the duty warp keeps ahead.  The duty warps are
// within one iteration of each other (each waits for staged[i] of ALL CTAs), so the flag cannot lag behind what the
// consumers need (tests/test_program_protocol_model.py); the direct check of the global counter is a defensive
// fall-back that costs nothing on the fast path.
__device__ __forceinline__ void prog_wait_row_clean(volatile int* red_ok, const int* zeroed, int op, int nblk) {
  ProgWatch wd;
  while (*red_ok < op) {
    if (op < 4 || ld_acquire_s32(&zeroed[op - 4]) >= nblk) break;
    if (wd.tick(kWRedOk, op)) break;
  }
}

}  // namespace b200awq
#include "program_stream.cuh"
namespace b200awq {

constexpr int kProgThreads = kV3Threads + 32;   // producer warp + 8 consumer warps + duty warp

// Reclamation of the accumulator rows (off the critical path, run by the duty warp of every CTA):
//   op i adds into row i % 4; its sums are read while op i+1 stages its activations.
//   staged[i]  counts CTAs whose consumers finished staging op i (= finished reading row i-1);
//   zeroed[j]  counts CTAs whose duty warp stored its slice of op j's fp16 output and zeroed its slice of row j.
//   Duty warp, iteration i = 1..n_ops: make sure row i % 4 is clean for this CTA's REDs of op i (zeroed[i-4]),
//   wait for its slice of row i-1, store y[i-1] (and the SiLU*mul output of op i), publish staged[i] for the CTA,
//   wait until every CTA has staged op i, zero its slice of row i-1, publish zeroed[i-1].
template <int SPW>
__global__ void __launch_bounds__(kProgThreads, 1)
    program_kernel(const ProgOp* __restrict__ ops, int n_ops, unsigned long long* __restrict__ rows, int acc_stride,
                   int* __restrict__ staged, int* __restrict__ zeroed, int M, int dbg) {
  constexpr int MT = kProgMT, NS = kV3Warps * SPW;
  extern __shared__ __align__(1024) uint8_t pg_smem[];
  uint8_t* ring = pg_smem;
  uint8_t* aux = pg_smem + (size_t)NS * kV3TileBytes;
  float* red = reinterpret_cast<float*>(aux + (size_t)NS * kV3AuxBytes);
  float* colacc = red + kV3Warps * MT * kGvRedStride;
  uint64_t* full = reinterpret_cast<uint64_t*>(colacc + kV3Warps * MT * kV3TileCols);
  uint64_t* empty = full + NS;
  int* flags = reinterpret_cast<int*>(empty + NS);
  int* warp_cb = flags;                 // [8] column block of each warp's pending sums
  int* warp_ntl = flags + 8;            // [8] tiles those sums cover
  volatile int* pub_op = reinterpret_cast<volatile int*>(flags + 16);     // ops whose sums this CTA has pushed
  volatile int* red_ok = reinterpret_cast<volatile int*>(flags + 17);     // highest op whose row is clean for REDs
  volatile int* staged_op = reinterpret_cast<volatile int*>(flags + 18);  // ops this CTA's consumers have staged
  float* wsum = reinterpret_cast<float*>(flags + 32);  // 8 floats (+ pad)
  __half* xs = reinterpret_cast<__half*>(pg_smem + prog_fixed_smem(SPW));

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nblk = gridDim.x, bid = blockIdx.x;

  if (tid == 0) {
    if ((smem_u32(pg_smem) & 1023u) != 0) __trap();
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    fence_mbar_init();
    *pub_op = 0;
    *red_ok = 0;
    *staged_op = 0;
  }
  for (int i = tid; i < kV3Warps * MT * kV3TileCols; i += kProgThreads) colacc[i] = 0.f;
  __syncthreads();

  // this CTA's share of an n-element row, in units of 8 elements
  auto slice8 = [&](int n, int& lo, int& hi) {
    const int u = n >> 3;
    lo = (int)((int64_t)u * bid / nblk) << 3;
    hi = (int)((int64_t)u * (bid + 1) / nblk) << 3;
  };

  if (warp == 0) {
    // ============================================================ producer: the weight stream of ALL ops
    // lane w feeds consumer warp w's private stages, op after op: the ring never drains at an op boundary
    if (lane < kV3Warps) {
      const int w = lane;
      int stage_i = 0;
      uint32_t ph = 0;
      for (int op = 0; op < n_ops; ++op) {
        const ProgOp* o = ops + op;
        const int K = o->K, N = o->N, g_shift = o->g_shift;
        const __half* scales = o->scales;
        const int32_t* qzeros = o->qzeros;
        const int NW = N >> 3;
        const int TPC = K / kV3TileRows;
        const int T = (N / kV3TileCols) * TPC;
        const int t0 = (int)((int64_t)T * bid / nblk);
        const int t1 = (int)((int64_t)T * (bid + 1) / nblk);
        const int ntile = t1 - t0;
        const int a = t0 + (int)((int64_t)ntile * w / kV3Warps);
        const int bnd = t0 + (int)((int64_t)ntile * (w + 1) / kV3Warps);
        int cb = a / TPC, kt = a - cb * TPC;
        // gate: hold the next op's loads back until this CTA's sums of the previous op are on their way
        // (measured +9 %: the REDs do not queue behind a fresh burst of bulk loads; the ring refills while the
        // consumers poll and stage)
        if (op > 0) prog_wait_smem(pub_op, op, kWGate, op);
        for (int t = a; t < bnd; ++t) {
          const int stage = w * SPW + stage_i;
          if (!prog_mbar_wait(&empty[stage], ph ^ 1, kWEmpty, op)) return;
          const int grp_abs = (kt * kV3TileRows) >> g_shift;
          uint8_t* st = ring + (size_t)stage * kV3TileBytes;
          uint8_t* sa = aux + (size_t)stage * kV3AuxBytes;
          mbar_arrive_expect_tx(&full[stage], kV3TileBytes + kV3AuxBytes);
          tma_load_2d(st, &o->tmw, &full[stage], cb * (kV3TileCols / 8), kt * kV3TileRows);
          bulk_load_1d(sa, scales + (int64_t)grp_abs * N + cb * kV3TileCols, kV3ScaleBytes, &full[stage]);
          bulk_load_1d(sa + kV3ScaleBytes, qzeros + (int64_t)grp_abs * NW + cb * (kV3TileCols / 8), kV3ZeroBytes,
                       &full[stage]);
          if (++kt == TPC) { kt = 0; ++cb; }
          if (++stage_i == SPW) { stage_i = 0; ph ^= 1; }
        }
      }
    }
    return;
  }

  if (warp == kV3Warps + 1) {
    // ============================================================ duty warp: outputs + row reclamation
    // red_ok runs ahead of the reclamation: op j may add into row j % 4 as soon as every CTA has zeroed its slice
    // after op j-4 (zeroed[j-4] complete); checked without blocking at every step so the consumers never wait for it
    int rk = 0;
    auto advance_red_ok = [&]() {
      if (lane == 0) {
        int r = rk;
        while (r + 1 < n_ops && (r + 1 < kProgRows || ld_acquire_s32(&zeroed[r + 1 - kProgRows]) >= nblk)) ++r;
        if (r != rk)
          asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"(smem_u32(const_cast<int*>(red_ok))), "r"(r) : "memory");
        rk = r;
      }
    };
    for (int i = 1; i <= n_ops; ++i) {
      const ProgOp* po = ops + i - 1;
      unsigned long long* R_prev = rows + (size_t)((i - 1) % kProgRows) * acc_stride;
      advance_red_ok();
      // ---- this CTA's slice of op i-1's fp16 output (polls until the slice is complete)
      const int TPCp = po->K / kV3TileRows;
      int ylo, yhi;
      slice8(po->N, ylo, yhi);
      for (int c = ylo + lane * 8; c < yhi; c += 32 * 8) {
        uint4 v;
        ProgWatch wd;
        while (!prog_prev8(R_prev, po->bias, c, TPCp, v)) {
          if (wd.tick(kWDutyY, i)) break;
          __nanosleep(400);   // off the critical path: do not hammer the lines the REDs are landing on
        }
        *reinterpret_cast<uint4*>(po->y + c) = v;
      }
      if (i < n_ops) {
        const ProgOp* o = ops + i;
        // ---- this CTA's slice of the SiLU*mul output op i's prologue stands for
        if (o->prologue == kProSilu && o->xout != nullptr) {
          const bool from_prev = o->src_prev != 0;
          const unsigned long long* pr = R_prev + o->src_off;
          const __half* pbias = (from_prev && po->bias != nullptr) ? po->bias + o->src_off : nullptr;
          const int K = o->K;
          int xlo, xhi;
          slice8(K, xlo, xhi);
          for (int c = xlo + lane * 8; c < xhi; c += 32 * 8) {
            uint4 gv, uv;
            if (from_prev) {
              ProgWatch wd;
              while (!prog_prev8(pr, pbias, c, TPCp, gv)) {
                if (wd.tick(kWDutySilu, i)) break;
                __nanosleep(400);
              }
              while (!prog_prev8(pr, pbias, K + c, TPCp, uv)) {
                if (wd.tick(kWDutySilu, i)) break;
                __nanosleep(400);
              }
            } else {
              gv = ldcg_u4(o->src + c);
              uv = ldcg_u4(o->src + K + c);
            }
            const __half* gh = reinterpret_cast<const __half*>(&gv);
            const __half* uh = reinterpret_cast<const __half*>(&uv);
            uint4 ov;
            __half* oh = reinterpret_cast<__half*>(&ov);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float gf = __half2float(gh[j]), uf = __half2float(uh[j]);
              oh[j] = __float2half_rn(gf / (1.f + __expf(-gf)) * uf);
            }
            *reinterpret_cast<uint4*>(o->xout + c) = ov;
          }
        }
        // ---- publish "this CTA has staged op i", wait for everybody, recycle row i-1
        __syncwarp();   // EVERY lane is done polling row i-1 (lane 0 alone publishing let other CTAs zero the row
                        // under this warp's slower lanes: they then polled zeros for ever)
        if (lane == 0) {
          ProgWatch wd;
          int sv;
          do {
            asm volatile("ld.acquire.cta.shared.s32 %0, [%1];" : "=r"(sv) : "r"(smem_u32(const_cast<int*>(staged_op))) : "memory");
            if (wd.tick(kWStagedOp, i)) break;
          } while (sv < i);
          red_release_add_s32(&staged[i], 1);
        }
        advance_red_ok();
        if (lane == 0) prog_wait(&staged[i], nblk, kWStaged, i);
        __syncwarp();
        int zlo, zhi;
        slice8(acc_stride, zlo, zhi);
        for (int c = zlo + lane * 2; c < zhi && dbg != 4; c += 32 * 2)   // (knob 3 = 4 keeps the rows for inspection)
          *reinterpret_cast<ulonglong2*>(R_prev + c) = make_ulonglong2(0ull, 0ull);
        __syncwarp();
        if (lane == 0) red_release_add_s32(&zeroed[i - 1], 1);
      } else {
        // epilogue: every CTA read only its own slice of the last row - zero exactly that slice (columns >= N are
        // never written); all rows are zero again when the kernel exits
        __syncwarp();
        for (int c = ylo + lane * 2; c < yhi && dbg != 4; c += 32 * 2)
          *reinterpret_cast<ulonglong2*>(R_prev + c) = make_ulonglong2(0ull, 0ull);
      }
    }
    return;
  }

  // ================================================================ consumers
  const int cw = warp - 1;
  const int ct = tid - 32;
  const int g = lane >> 2, tig = lane & 3;
  const bool tok_ok = g < M;
  float* my_red = red + (size_t)cw * MT * kGvRedStride;
  float* my_col = colacc + (size_t)cw * MT * kV3TileCols;
  constexpr int NCT = kV3Warps * 32;

  // add `cols` [256] (shared memory, summed over nsrc sources src_stride floats apart) covering ntl tiles into
  // column block cb of the op's packed row
  auto push_cols = [&](float* cols, int nsrc, int src_stride, int cb, int ntl, int t, int nthreads,
                       unsigned long long* R_cur) {
    for (int c = t; c < kV3TileCols; c += nthreads) {
      float v = 0.f;
      for (int sidx = 0; sidx < nsrc; ++sidx) {
        v += cols[sidx * src_stride + c];
        cols[sidx * src_stride + c] = 0.f;
      }
      red_add_u64(R_cur + cb * kV3TileCols + c, prog_pack(v, ntl));
    }
  };

  int stage_i = 0;
  uint32_t ph = 0;
  for (int op = 0; op < n_ops; ++op) {
    const ProgOp* o = ops + op;
    unsigned long long* R_cur = rows + (size_t)(op % kProgRows) * acc_stride;
    const unsigned long long* R_prev = rows + (size_t)((op + kProgRows - 1) % kProgRows) * acc_stride;
    const int K = o->K, N = o->N, G = o->G, g_shift = o->g_shift;
    const int TPC = K / kV3TileRows;
    const int T = (N / kV3TileCols) * TPC;
    const int t0 = (int)((int64_t)T * bid / nblk);
    const int t1 = (int)((int64_t)T * (bid + 1) / nblk);
    const int ntile = t1 - t0;
    const int a_w = t0 + (int)((int64_t)ntile * cw / kV3Warps);
    const int b_w = t0 + (int)((int64_t)ntile * (cw + 1) / kV3Warps);

    PROG_STAMP(0);
    // an external source written by an older op of this program: its duty-warp stores must all be visible
    if (o->ext_dep >= 0) {
      if (ct == 0) prog_wait(&zeroed[o->ext_dep], nblk, kWExtDep, op);
      named_bar_sync_gv(1, NCT);
    }
    PROG_STAMP(1);

    // ---- stage (and transform) the activations this CTA's tiles need; arithmetic mirrors aux.cu exactly.  A source
    // inside the previous op's output is polled from its packed row until every needed column is complete.
    {
      const bool from_prev = o->src_prev != 0;
      const unsigned long long* pr = R_prev + o->src_off;
      const __half* pbias = (from_prev && ops[op - 1].bias != nullptr) ? ops[op - 1].bias + o->src_off : nullptr;
      const int TPCp = from_prev ? ops[op - 1].K / kV3TileRows : 0;
      const __half* src = o->src;
      auto load8 = [&](int c, uint4& v) -> bool {
        if (from_prev) return prog_prev8(pr, pbias, c, TPCp, v);
        v = ldcg_u4(src + c);
        return true;
      };
      __half* xout = o->xout;
      int xlo = 0, xhi = 0;
      if (xout != nullptr) slice8(K, xlo, xhi);
      const int pro = o->prologue;
      // k-range of this CTA's tiles: tiles are column-block major, so the range is contiguous modulo K
      const int k_start = (t0 % TPC) * kV3TileRows;
      const int k_len = ntile * kV3TileRows < K ? ntile * kV3TileRows : K;
      if (pro == kProCopy) {
        for (int i = ct * 8; i < k_len; i += NCT * 8) {
          int k = k_start + i;
          if (k >= K) k -= K;
          uint4 v;
          ProgWatch wd;
          while (!load8(k, v))
            if (wd.tick(kWCopy, op)) break;
          *reinterpret_cast<uint4*>(xs + k) = v;
        }
      } else if (pro == kProSilu) {
        for (int i = ct * 8; i < k_len; i += NCT * 8) {
          int k = k_start + i;
          if (k >= K) k -= K;
          uint4 gv, uv;
          ProgWatch wd;
          for (;;) {
            const bool okg = load8(k, gv), oku = load8(K + k, uv);
            if (okg && oku) break;
            if (wd.tick(kWSilu, op)) break;
          }
          const __half* gh = reinterpret_cast<const __half*>(&gv);
          const __half* uh = reinterpret_cast<const __half*>(&uv);
          uint4 ov;
          __half* oh = reinterpret_cast<__half*>(&ov);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float gf = __half2float(gh[j]), uf = __half2float(uh[j]);
            oh[j] = __float2half_rn(gf / (1.f + __expf(-gf)) * uf);
          }
          *reinterpret_cast<uint4*>(xs + k) = ov;
        }
      } else {
        // RMSNorm: the whole row.  Both chunks of a thread (and their norm weights) are in flight together.
        float ss = 0.f;
        uint4 nwa = make_uint4(0u, 0u, 0u, 0u), nwb = nwa;
        for (int i = ct * 8; i < K; i += NCT * 16) {
          const int i2 = i + NCT * 8;
          const bool two = i2 < K;
          uint4 va, vb = make_uint4(0u, 0u, 0u, 0u);
          if (i < NCT * 16) {
            nwa = __ldg(reinterpret_cast<const uint4*>(o->norm_w + i));
            if (two) nwb = __ldg(reinterpret_cast<const uint4*>(o->norm_w + i2));
          }
          ProgWatch wd;
          for (;;) {
            const bool oka = load8(i, va);
            const bool okb = two ? load8(i2, vb) : true;
            if (oka && okb) break;
            if (wd.tick(kWNorm, op)) break;
          }
          const __half2* ha = reinterpret_cast<const __half2*>(&va);
          const __half2* hb = reinterpret_cast<const __half2*>(&vb);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(ha[j]);
            ss += f.x * f.x + f.y * f.y;
          }
          *reinterpret_cast<uint4*>(xs + i) = va;
          if (two) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 f = __half22float2(hb[j]);
              ss += f.x * f.x + f.y * f.y;
            }
            *reinterpret_cast<uint4*>(xs + i2) = vb;
          }
        }
        ss = prog_warp_sum(ss);
        if (lane == 0) wsum[cw] = ss;
        named_bar_sync_gv(1, NCT);
        float tot = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) tot += wsum[i];
        const float rs = rsqrtf(tot / static_cast<float>(K) + o->eps);
        const __half* nw = o->norm_w;
        for (int i = ct * 8; i < K; i += NCT * 8) {   // the thread's own chunks again
          uint4 v = *reinterpret_cast<const uint4*>(xs + i);
          const uint4 wv = i == ct * 8 ? nwa : (i == ct * 8 + NCT * 8 ? nwb : __ldg(reinterpret_cast<const uint4*>(nw + i)));
          __half* vh = reinterpret_cast<__half*>(&v);
          const __half* wh = reinterpret_cast<const __half*>(&wv);
#pragma unroll
          for (int j = 0; j < 8; ++j) vh[j] = __float2half_rn(__half2float(vh[j]) * rs * __half2float(wh[j]));
          *reinterpret_cast<uint4*>(xs + i) = v;
          if (i >= xlo && i < xhi) *reinterpret_cast<uint4*>(xout + i) = v;
        }
      }
      named_bar_sync_gv(1, NCT);
      // this CTA is done reading the previous op's row: tell the duty warp (it publishes staged[op])
      if (ct == 0)
        asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"(smem_u32(const_cast<int*>(staged_op))), "r"(op) : "memory");
    }
    PROG_STAMP(2);

    // ---- the persistent-GEMV tile loop over this warp's run of tiles
    auto load_x = [&](int t, int ktile, uint32_t (&xb)[4][2]) {
#pragma unroll
      for (int bb = 0; bb < 4; ++bb) xb[bb][0] = xb[bb][1] = 0u;
      if (t < b_w && tok_ok) {
        const __half* px = xs + ktile * kV3TileRows + 2 * tig;   // M = 1: token g = 0
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
    for (int t = a_w; t < b_w; ++t) {
      const int stage = cw * SPW + stage_i;
      if (cb != cur_cb) {
        if (cur_cb >= 0 && ntl > 0) {
          // this warp's run crosses a column block: push its pending sums alone (rare)
          __syncwarp();
          if (op > 0) prog_wait_row_clean(red_ok, zeroed, op, nblk);
          push_cols(my_col, 1, 0, cur_cb, ntl, lane, 32, R_cur);
        }
        cur_cb = cb;
        ntl = 0;
      }
      ++ntl;
      load_x(t + 1, (kt + 1 == TPC) ? 0 : kt + 1, xnext);
      prog_mbar_wait(&full[stage], ph, kWFull, op);
      if (t == a_w) PROG_STAMP(3);
      const uint8_t* st = ring + (size_t)stage * kV3TileBytes;
      const uint8_t* sa = aux + (size_t)stage * kV3AuxBytes;
      v3_tile_mma(st, g, tig, xcur, acc, xs_acc);
      const bool group_end = g_shift < 31 ? ((((kt + 1) * kV3TileRows) & (G - 1)) == 0) : (kt + 1 == TPC);
      if (group_end || t + 1 == b_w) {
        v3_fold<MT>(sa, my_red, my_col, lane, g, tig, acc, xs_acc);
        zero_acc();
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[stage]);
#pragma unroll
      for (int bb = 0; bb < 4; ++bb) {
        xcur[bb][0] = xnext[bb][0];
        xcur[bb][1] = xnext[bb][1];
      }
      if (++kt == TPC) { kt = 0; ++cb; }
      if (++stage_i == SPW) { stage_i = 0; ph ^= 1; }
    }

    // ---- CTA-level reduction of the per-warp column sums, one packed RED per column; nothing to publish
    PROG_STAMP(4);
    if (lane == 0) {
      warp_cb[cw] = (ntl > 0) ? cur_cb : -1;
      warp_ntl[cw] = ntl;
    }
    if (op > 0 && ct == 0) prog_wait_row_clean(red_ok, zeroed, op, nblk);   // the op's row is clean (duty warp, long since)
    named_bar_sync_gv(1, NCT);
    PROG_STAMP(5);
    {
      // one push per column block this CTA touched: consecutive warps with the same block, empty warps (-1, their
      // column sums are zero) in between included
      int w0 = 0;
      while (w0 < kV3Warps) {
        const int cbg = warp_cb[w0];
        if (cbg < 0) { ++w0; continue; }
        int w1 = w0 + 1, tiles = warp_ntl[w0];
        while (w1 < kV3Warps && (warp_cb[w1] == cbg || warp_cb[w1] < 0)) tiles += warp_cb[w1] < 0 ? 0 : warp_ntl[w1], ++w1;
        push_cols(colacc + (size_t)w0 * MT * kV3TileCols, w1 - w0, MT * kV3TileCols, cbg, tiles, ct, NCT, R_cur);
        w0 = w1;
      }
    }
    PROG_STAMP(6);
    if (ct == 0) *pub_op = op + 1;
    PROG_STAMP(7);
    // (the next op's staging barrier separates these shared-memory reads from the next fold's writes; the last op's
    // sums are stored by the duty warps)
  }
}

// ------------------------------------------------------------------------------------------------ host side
struct Program {
  ProgOp* d_ops = nullptr;
  int* d_done = nullptr;
  int n_ops = 0;
  int M = 0;
  int max_N = 0;
  int acc_stride = 0;   // floats per accumulator row (3 rows rotate through the ops)
  size_t xs_bytes = 0;
  int device = 0;
  // stream variant (program_stream.cuh): re-laid-out weights, per-op CTA partition, hand-off rows, tag state
  bool stream = false;
  SpOp* d_sp_ops = nullptr;
  uint8_t* d_stream = nullptr;
  uint32_t* d_cta = nullptr;
  uint32_t* d_rows = nullptr;
  int* d_state = nullptr;
  int row_stride = 0;
  size_t stream_bytes = 0;
};

size_t stream_format_bytes(int K, int N, int G) {
  if (K <= 0 || N <= 0 || G <= 0) return 0;
  const int UK = G < 128 ? G : 128;
  return (size_t)(N / 16) * (K / UK) * ((size_t)(UK / 16) * 128 + kSpAux);
}
bool stream_format_supported(int K, int N, int G, int mode) {
  if (K <= 0 || N <= 0 || G <= 0 || (K % G) != 0 || (N % 16) != 0 || (K % 128) != 0) return false;
  if (!(G == 32 || G == 64 || (G % 128) == 0)) return false;
  if (mode == 1 && ((N / 2) % 8) != 0) return false;
  return mode == 0 || mode == 1;
}
cudaError_t stream_pack(const int32_t* qweight, const void* scales, const int32_t* qzeros, void* out, int K, int N, int G,
                        int mode, cudaStream_t st) {
  if (!stream_format_supported(K, N, G, mode)) return cudaErrorNotSupported;
  const int UK = G < 128 ? G : 128;
  const int64_t total = (int64_t)(N / 16) * (K / UK) * ((UK / 16) * 32 + 12);
  const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  stream_pack_kernel<<<blocks, 256, 0, st>>>(qweight, static_cast<const __half*>(scales), qzeros,
                                             static_cast<uint8_t*>(out), K, N, G, mode);
  return cudaGetLastError();
}

// Builds the stream variant from the folded op table.  Returns false when the sequence is outside its envelope
// (the caller then tries the split-K kernel).  *err != cudaSuccess reports a CUDA failure.
static bool stream_build(Program* pr, const std::vector<ProgOp>& table, int grid, cudaError_t* err) {
  *err = cudaSuccess;
  const int n = static_cast<int>(table.size());
  if (n >= 60000) return false;
  // creation is a load-time step (not capturable): whatever produced the checkpoint tensors on any stream is done
  // before the re-layout reads them
  if ((*err = cudaDeviceSynchronize()) != cudaSuccess) return false;
  std::vector<SpOp> ops(n);
  std::vector<int> mode(n, 0);
  // producer-side SiLU*mul: a SILU prologue whose source is the whole output of the previous linear
  for (int i = 0; i < n; ++i)
    if (table[i].prologue == kProSilu) {
      if (i == 0 || !table[i].src_prev || table[i].src_off != 0 || table[i - 1].N != 2 * table[i].K) {
        // a later consumer of an already fused gate|up output (ext_dep) is fine, anything else is not
        const int j = table[i].ext_dep;
        if (!(j >= 0 && mode[j] == 1 && table[i].src == table[j].y && table[j].N == 2 * table[i].K)) return false;
      } else {
        mode[i - 1] = 1;
      }
    }
  size_t wbytes = 0, max_cols = 0;
  int max_K = 0;
  std::vector<size_t> woff(n);
  for (int i = 0; i < n; ++i) {
    const ProgOp& p = table[i];
    if (!stream_format_supported(p.K, p.N, p.G, mode[i])) return false;
    const int UK = p.G < 128 ? p.G : 128;
    if (p.K / UK > kSpXsumMax) return false;
    if ((p.N / 16 + grid - 1) / grid > kSpLMax) return false;
    woff[i] = wbytes;
    wbytes += (stream_format_bytes(p.K, p.N, p.G) + 255) & ~(size_t)255;
    max_cols = std::max(max_cols, (size_t)(mode[i] ? p.N / 2 : p.N));
    max_K = std::max(max_K, p.K);
  }
  // K <= 24160: the envelope is sized for 12 consumer warps x 3 stages, more than the 8-warp kernel needs
  if (sp_fixed_smem(12, 3) + (size_t)max_K * 2 > (size_t)227 * 1024) return false;
  for (int i = 0; i < n; ++i) {
    const ProgOp& p = table[i];
    SpOp& o = ops[i];
    std::memset(&o, 0, sizeof(o));
    o.bias = p.bias;
    o.y = p.y;
    o.K = p.K;
    o.N = p.N;
    const int UK = p.G < 128 ? p.G : 128;
    o.uk_shift = UK == 32 ? 5 : (UK == 64 ? 6 : 7);
    o.F = UK / 16;
    o.NU = p.K / UK;
    o.unit_bytes = o.F * 128 + kSpAux;
    o.ups = kSpStageBytes / o.unit_bytes;
    o.mode = mode[i];
    o.eps = p.eps;
    o.norm_w = p.norm_w;
    o.src_op = -1;
    if (p.prologue == kProSilu) {
      // the SiLU*mul itself runs in the producer (mode 1); this op copies the published product
      const int j = p.src_prev ? i - 1 : p.ext_dep;
      if (i - j >= kSpRows) return false;
      o.prologue = kProCopy;
      o.src_op = j;
      o.src_off = 0;
      if (p.xout != nullptr) ops[j].act_out = p.xout;
    } else {
      o.prologue = p.prologue;
      o.xout = p.prologue == kProRmsnorm ? p.xout : nullptr;
      if (p.prologue == kProCopy && p.xout != nullptr) return false;
      int j = -1;
      if (p.src_prev) j = i - 1;
      else if (p.ext_dep >= 0) j = p.ext_dep;
      if (j >= 0) {
        if (mode[j] == 1 || i - j >= kSpRows) return false;   // raw gate|up columns of a fused producer / row recycled
        const uintptr_t y0 = reinterpret_cast<uintptr_t>(table[j].y), s0 = reinterpret_cast<uintptr_t>(p.src);
        if (s0 < y0 || s0 + (size_t)p.K * 2 > y0 + (size_t)table[j].N * 2 || ((s0 - y0) & 7) != 0) return false;
        o.src_op = j;
        o.src_off = static_cast<int>((s0 - y0) / 2);
      } else {
        o.src = p.src;
        if ((reinterpret_cast<uintptr_t>(p.src) & 7) != 0) return false;
      }
    }
  }
  // CTA partition: whole 16-column sets, as even as the set count allows
  std::vector<uint32_t> cta((size_t)n * (grid + 1));
  for (int i = 0; i < n; ++i) {
    const int64_t S = table[i].N / 16;
    for (int c = 0; c <= grid; ++c) cta[(size_t)i * (grid + 1) + c] = (uint32_t)((S * c / grid) * ops[i].NU);
  }
  pr->row_stride = (int)((max_cols + 63) & ~(size_t)63);
  cudaError_t e = cudaMalloc(&pr->d_stream, wbytes);
  if (e == cudaSuccess) e = cudaMalloc(&pr->d_sp_ops, (size_t)n * sizeof(SpOp));
  if (e == cudaSuccess) e = cudaMalloc(&pr->d_cta, cta.size() * sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMalloc(&pr->d_rows, (size_t)kSpRows * pr->row_stride * sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMalloc(&pr->d_state, 2 * sizeof(int));
  if (e == cudaSuccess) e = cudaMemset(pr->d_rows, 0, (size_t)kSpRows * pr->row_stride * sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMemset(pr->d_state, 0, 2 * sizeof(int));
  for (int i = 0; i < n && e == cudaSuccess; ++i) {
    ops[i].wstream = pr->d_stream + woff[i];
    ops[i].cta_begin = pr->d_cta + (size_t)i * (grid + 1);
    e = stream_pack(table[i].qw_src, table[i].scales, table[i].qzeros, pr->d_stream + woff[i], table[i].K, table[i].N,
                    table[i].G, mode[i], nullptr);
  }
  if (e == cudaSuccess) e = cudaMemcpy(pr->d_sp_ops, ops.data(), (size_t)n * sizeof(SpOp), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(pr->d_cta, cta.data(), cta.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(stream_program_kernel<8, 4, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024));
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    cudaFree(pr->d_stream);
    cudaFree(pr->d_sp_ops);
    cudaFree(pr->d_cta);
    cudaFree(pr->d_rows);
    cudaFree(pr->d_state);
    pr->d_stream = nullptr;
    pr->d_sp_ops = nullptr;
    pr->d_cta = nullptr;
    pr->d_rows = nullptr;
    pr->d_state = nullptr;
    *err = e;
    return false;
  }
  pr->stream = true;
  pr->stream_bytes = wbytes;
  pr->xs_bytes = (size_t)max_K * 2;
  return true;
}

static int prog_sm_count() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
    n = B200AWQ_SM_COUNT_FALLBACK;
  return n;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
static bool overlaps(const void* a, size_t na, const void* b, size_t nb) {
  const uintptr_t a0 = reinterpret_cast<uintptr_t>(a), b0 = reinterpret_cast<uintptr_t>(b);
  return a0 < b0 + nb && b0 < a0 + na;
}

// Folds the recorded call sequence into linear ops with an activation prologue.  Returns a B200AWQ_* code;
// *cuda_err carries the CUDA error behind B200AWQ_ECUDA.
//
// Hazard rules (the kernel orders ops only through "every CTA has added its sums of op i-1"; the fp16 output of
// op i-1 and the glue output of op i are stored, in per-CTA slices, while op i stages its activations):
//   * a glue op (RMSNorm / SiLU*mul) is executed as the prologue of every later linear that reads its output
//     buffer; that buffer is written as a side effect, nobody inside the kernel may READ it;
//   * a source inside the previous op's output is read from that op's fp32 accumulators (src_prev); any other
//     overlap with the previous op's output is rejected; outputs older than that are ordinary global reads;
//   * a linear must not write (y) what it reads (src) or what its own prologue publishes (xout);
//   * a buffer that a pending glue record depends on must not be overwritten before the record's last use.
int program_create(const b200awq_op_t* ops, int n, Program** out, cudaError_t* cuda_err) {
  *cuda_err = cudaSuccess;
  *out = nullptr;
  if (ops == nullptr || n <= 0) return B200AWQ_EINVAL;
  std::vector<ProgOp> table;
  struct Glue {
    int kind;
    const void* src;
    const void* w;
    void* out;
    int width;
    float eps;
    bool used;
    bool live;
  };
  std::vector<Glue> glues;
  const int grid = prog_sm_count();
  int max_K = 0, max_N = 0, M = -1;
  bool v3_ok = true;
  for (int i = 0; i < n; ++i) {
    const b200awq_op_t& op = ops[i];
    if (M < 0) M = op.M;
    if (op.M != M) return B200AWQ_EUNSUPPORTED;
    if (op.kind == B200AWQ_OP_RMSNORM || op.kind == B200AWQ_OP_SILU_AND_MUL) {
      if (op.x == nullptr || op.y == nullptr || op.K <= 0) return B200AWQ_EINVAL;
      if (op.kind == B200AWQ_OP_RMSNORM && op.weight == nullptr) return B200AWQ_EINVAL;
      if ((op.K % 8) != 0 || !aligned16(op.x) || !aligned16(op.y) || (op.weight != nullptr && !aligned16(op.weight)))
        return B200AWQ_EUNSUPPORTED;
      const size_t in_bytes = (size_t)(op.kind == B200AWQ_OP_SILU_AND_MUL ? 2 : 1) * op.K * 2;
      if (overlaps(op.y, (size_t)op.K * 2, op.x, in_bytes)) return B200AWQ_EUNSUPPORTED;  // in-place glue op
      for (Glue& gl : glues)
        if (gl.live && (overlaps(gl.out, (size_t)gl.width * 2, op.y, (size_t)op.K * 2) ||
                        overlaps(gl.src, (size_t)(gl.kind == kProSilu ? 2 : 1) * gl.width * 2, op.y, (size_t)op.K * 2))) {
          if (!gl.used) return B200AWQ_EUNSUPPORTED;
          gl.live = false;
        }
      // its input must not be a buffer only CTA 0 publishes
      for (const Glue& gl : glues)
        if (overlaps(gl.out, (size_t)gl.width * 2, op.x, in_bytes)) return B200AWQ_EUNSUPPORTED;
      glues.push_back(Glue{op.kind == B200AWQ_OP_RMSNORM ? kProRmsnorm : kProSilu, op.x, op.weight, op.y, op.K, op.eps,
                           false, true});
      continue;
    }
    if (op.kind != B200AWQ_OP_LINEAR_GEMM) return B200AWQ_EINVAL;
    if (op.x == nullptr || op.qweight == nullptr || op.scales == nullptr || op.qzeros == nullptr || op.y == nullptr ||
        op.K <= 0 || op.N <= 0 || op.group_size <= 0 || (op.K % op.group_size) != 0)
      return B200AWQ_EINVAL;
    GemmArgs a{op.x, op.ldx, static_cast<const int32_t*>(op.qweight), op.scales, static_cast<const int32_t*>(op.qzeros),
               op.bias, op.y, op.M, op.K, op.N, op.group_size};
    if (M != 1) return B200AWQ_EUNSUPPORTED;
    // envelope of the split-K kernel (the stream variant has its own, checked in stream_build)
    if (!gemv_v3_supported(a) || (op.N / kV3TileCols) * (op.K / kV3TileRows) < grid ||   // every CTA owns tiles
        op.K / kV3TileRows >= 256)                                                       // tiles per column fit the packed word
      v3_ok = false;
    ProgOp p;
    std::memset(&p, 0, sizeof(p));
    p.ext_dep = -1;
    p.qw_src = a.qweight;
    if (v3_ok) {
      cudaError_t e = make_tmap_2d(a.qweight, /*int32*/ 1, (uint64_t)(a.N / 8), (uint64_t)a.K, (uint64_t)(a.N / 8) * 4, 32,
                                   kV3TileRows, &p.tmw);
      if (e != cudaSuccess) {
        *cuda_err = e;
        return B200AWQ_ECUDA;
      }
    }
    p.scales = static_cast<const __half*>(op.scales);
    p.qzeros = static_cast<const int32_t*>(op.qzeros);
    p.bias = static_cast<const __half*>(op.bias);
    p.y = static_cast<__half*>(op.y);
    p.K = op.K;
    p.N = op.N;
    p.G = op.group_size;
    p.g_shift = 31;
    if ((p.G & (p.G - 1)) == 0) {
      p.g_shift = 0;
      while ((1 << p.g_shift) < p.G) ++p.g_shift;
    }
    Glue* hit = nullptr;
    for (Glue& gl : glues)
      if (gl.live && gl.out == op.x && gl.width == op.K) hit = &gl;
    if (hit != nullptr) {
      p.prologue = hit->kind;
      p.src = static_cast<const __half*>(hit->src);
      p.norm_w = static_cast<const __half*>(hit->w);
      p.xout = hit->used ? nullptr : static_cast<__half*>(hit->out);   // published once, by its first consumer
      p.eps = hit->eps;
      hit->used = true;
    } else {
      p.prologue = kProCopy;
      p.src = static_cast<const __half*>(op.x);
      if (!aligned16(op.x)) return B200AWQ_EUNSUPPORTED;
      for (const Glue& gl : glues)   // reading a buffer only CTA 0 publishes (a dead or mismatching record)
        if (overlaps(gl.out, (size_t)gl.width * 2, op.x, (size_t)op.K * 2)) return B200AWQ_EUNSUPPORTED;
    }
    const size_t src_bytes = (size_t)(p.prologue == kProSilu ? 2 : 1) * op.K * 2;
    if (overlaps(p.y, (size_t)op.N * 2, p.src, src_bytes)) return B200AWQ_EUNSUPPORTED;
    if (p.xout != nullptr && overlaps(p.xout, (size_t)op.K * 2, p.y, (size_t)op.N * 2)) return B200AWQ_EUNSUPPORTED;
    if (!table.empty()) {
      // the previous op's fp16 output reaches memory only while THIS op stages its activations: a source inside it
      // is taken from the previous op's fp32 accumulators instead (same values), anything else touching it is a race
      const ProgOp& pv = table.back();
      const uintptr_t y0 = reinterpret_cast<uintptr_t>(pv.y), s0 = reinterpret_cast<uintptr_t>(p.src);
      if (s0 >= y0 && s0 + src_bytes <= y0 + (size_t)pv.N * 2) {
        if (((s0 - y0) & 15) != 0) return B200AWQ_EUNSUPPORTED;
        p.src_prev = 1;
        p.src_off = static_cast<int>((s0 - y0) / 2);
      } else if (overlaps(pv.y, (size_t)pv.N * 2, p.src, src_bytes)) {
        return B200AWQ_EUNSUPPORTED;
      } else {
        // a source written by an older op of this program: wait for that op's duty-warp stores
        for (int j = static_cast<int>(table.size()) - 2; j >= 0; --j)
          if (overlaps(table[j].y, (size_t)table[j].N * 2, p.src, src_bytes)) {
            p.ext_dep = j;
            break;
          }
      }
      if (p.xout != nullptr && overlaps(p.xout, (size_t)op.K * 2, pv.y, (size_t)pv.N * 2)) return B200AWQ_EUNSUPPORTED;
    }
    // writing y over something a live glue record still needs ends that record
    for (Glue& gl : glues)
      if (gl.live && &gl != hit &&
          (overlaps(gl.out, (size_t)gl.width * 2, p.y, (size_t)op.N * 2) ||
           overlaps(gl.src, (size_t)(gl.kind == kProSilu ? 2 : 1) * gl.width * 2, p.y, (size_t)op.N * 2))) {
        if (!gl.used) return B200AWQ_EUNSUPPORTED;
        gl.live = false;
      }
    max_K = op.K > max_K ? op.K : max_K;
    max_N = op.N > max_N ? op.N : max_N;
    table.push_back(p);
  }
  for (const Glue& gl : glues)
    if (!gl.used) return B200AWQ_EUNSUPPORTED;   // a glue op nobody consumes would never run
  if (table.empty()) return B200AWQ_EUNSUPPORTED;

  Program* pr = new Program();
  pr->n_ops = static_cast<int>(table.size());
  pr->M = M;
  pr->max_N = max_N;
  cudaError_t e = cudaGetDevice(&pr->device);
  // first choice: the stream variant (one-time re-layout, output-stationary partition); knob 14 = 1 skips it
  if (e == cudaSuccess && knob(14) != 1 && stream_build(pr, table, grid, &e)) {
    *out = pr;
    return B200AWQ_OK;
  }
  if (e != cudaSuccess) {
    delete pr;
    *cuda_err = e;
    return B200AWQ_ECUDA;
  }
  const size_t smem = prog_fixed_smem(2) + (size_t)(max_K + 8) * 2 * kProgMT;
  if (!v3_ok || knob(14) == 2 || smem > (size_t)227 * 1024) {
    delete pr;
    return B200AWQ_EUNSUPPORTED;
  }
  pr->acc_stride = (max_N + 7) & ~7;
  pr->xs_bytes = (size_t)(max_K + 8) * 2 * kProgMT;
  if (e == cudaSuccess) e = cudaMalloc(&pr->d_ops, table.size() * sizeof(ProgOp));
  if (e == cudaSuccess) e = cudaMalloc(&pr->d_done, 2 * (table.size() + 1) * sizeof(int));
  if (e == cudaSuccess) e = cudaMemcpy(pr->d_ops, table.data(), table.size() * sizeof(ProgOp), cudaMemcpyHostToDevice);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(program_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024));
  if (e != cudaSuccess) {
    cudaFree(pr->d_ops);
    cudaFree(pr->d_done);
    delete pr;
    *cuda_err = e;
    return B200AWQ_ECUDA;
  }
  *out = pr;
  return B200AWQ_OK;
}

int program_max_n(const Program* p) { return p->max_N; }
int program_m(const Program* p) { return p->M; }
int program_num_ops(const Program* p) { return p->n_ops; }

int program_is_stream(const Program* p) { return p->stream ? 1 : 0; }
size_t program_stream_bytes(const Program* p) { return p->stream_bytes; }

cudaError_t program_run(Program* p, float* acc_ws, cudaStream_t st) {
  // staged[] and zeroed[] counters (see program_kernel)
  cudaError_t e = program_abort_clear(st);
  if (e != cudaSuccess) return e;
  if (p->stream) {
    // 8 consumer warps, 4 ring stages each, 4 units in flight (measured 1.50 / 1.59 / 1.73 ms per Llama-3-8B step with
    // 8 / 12 / 16 warps)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(prog_sm_count());
    cfg.blockDim = dim3(32 + 8 * 32);
    cfg.dynamicSmemBytes = sp_fixed_smem(8, 4) + p->xs_bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;   // all CTAs co-resident: the hand-off polls are grid-wide waits
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const SpOp* sops = p->d_sp_ops;
    const uint32_t* cta = p->d_cta;
    return cudaLaunchKernelEx(&cfg, stream_program_kernel<8, 4, 4>, sops, cta, p->n_ops, p->d_rows, p->row_stride,
                              p->d_state, knob(3));
  }
  e = cudaMemsetAsync(p->d_done, 0, (size_t)2 * (p->n_ops + 1) * sizeof(int), st);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(prog_sm_count());
  cfg.blockDim = dim3(kProgThreads);
  cfg.dynamicSmemBytes = prog_fixed_smem(2) + p->xs_bytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;   // all CTAs co-resident: the completion counters are grid-wide waits
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const ProgOp* ops = p->d_ops;
  const int dbg = knob(3);
  unsigned long long* rows = reinterpret_cast<unsigned long long*>(acc_ws);
  int* staged = p->d_done;
  int* zeroed = p->d_done + (p->n_ops + 1);
  return cudaLaunchKernelEx(&cfg, program_kernel<2>, ops, p->n_ops, rows, p->acc_stride, staged, zeroed, p->M, dbg);
}

void program_destroy(Program* p) {
  if (p == nullptr) return;
  cudaFree(p->d_ops);
  cudaFree(p->d_done);
  cudaFree(p->d_sp_ops);
  cudaFree(p->d_stream);
  cudaFree(p->d_cta);
  cudaFree(p->d_rows);
  cudaFree(p->d_state);
  delete p;
}

}  // namespace b200awq
