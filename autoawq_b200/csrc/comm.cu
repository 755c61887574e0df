// One-shot all-reduce over NVLink peer memory for the tensor-parallel decode path (SURVEY.md 8e).
//
// A row-parallel linear (o_proj / down_proj split along K, autoawq_b200/shard.py) leaves a PARTIAL fp16 [M, hidden]
// output on every GPU; the block's result is their sum.  At decode that is 16 KB per collective, 160 collectives per
// token for Llama-3-70B: pure latency.  ncclAllReduce inside a CUDA graph measured 22.8 us per call on 2 x B200
// (profiles/r02_tp70b_n2.json) - 3.6 ms of a 9.9 ms step.  This kernel does the same sum in one launch of one CTA:
//
//   every rank owns a SYMMETRIC buffer (cudaMalloc + CUDA IPC: each process maps all peers' buffers):
//       inbox[2 parities][world slots][max_elems / 2] LL words of 8 bytes = {two fp16 values, 32-bit call number}
//   call number e (a device-resident counter: CUDA-graph replay safe), parity p = e & 1, rank r:
//     1. push: store my partial, as LL words tagged e, into slot r of EVERY rank's inbox[p] (P2P stores over NVLink /
//        NVSwitch; the own copy is a local store),
//     2. wait and reduce: every thread polls its words of each slot of my inbox[p] until they carry e, and sums them in
//        RANK ORDER (fp32 accumulation, one rounding): the result is bit-identical on all ranks, and written over the
//        partial in place.
//   Every word carries its own validity (NCCL's LL idea): ONE NVLink hop, no barrier, no fence, no flag.  8-byte
//   aligned stores do not tear; 16-byte vectors (two words) are used on both sides.  (A flag protocol - push, CTA
//   barrier, fence.sys, flag store, flag poll, reduce - measured 8.1 us at N = 2 against 5.2 us for LL,
//   profiles/r02_tp70b_n2.json.)
//   Two parities: a rank can start call e + 1 (writing inbox[(e + 1) & 1]) while a slower peer still reads
//   inbox[e & 1]; it cannot start e + 2 before every peer has pushed e + 1, i.e. finished reading e.
//   No memset, no host round trip, nothing to reset.  A spin gives up after 2 s (dead peer) and raises the comm's
//   error flag instead of hanging the GPU.
//
// Messages larger than the buffer (prefill) stay on NCCL (autoawq_b200/comm.py decides).
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstring>

#include "../../include/b200awq.h"
#include "common.cuh"
#include "kernels.h"

namespace b200awq {

constexpr int kCommMaxWorld = 8;
constexpr int kCommThreads = 1024;

struct CommPeers {
  uint8_t* base[kCommMaxWorld];
};

struct Comm {
  int rank = 0, world = 1, max_elems = 0, device = 0;
  uint8_t* local = nullptr;      // this rank's symmetric buffer
  int* d_state = nullptr;        // [0] call counter, [1] error flag (local only)
  CommPeers peers{};
  bool opened = false;
  size_t bytes = 0;
};

static size_t comm_bytes(int world, int max_elems) {
  return (size_t)2 * world * max_elems * 4;   // inbox[2][world][max_elems / 2] words of 8 bytes
}

__device__ __forceinline__ void st_relaxed_sys_u4(void* p, const uint4& v) {
  asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_relaxed_sys_u4(const void* p) {
  uint4 r;
  asm volatile("ld.relaxed.sys.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
  return r;
}

__global__ void __launch_bounds__(kCommThreads, 1)
    ll_allreduce_kernel(CommPeers peers, int rank, int world, int max_elems, __half* __restrict__ y, int n,
                        int* __restrict__ state) {
  const int tid = threadIdx.x;
  const uint32_t e = (uint32_t)state[0] + 1u;
  const int par = (int)(e & 1u);
  const int nv = n >> 2;                                      // vectors of 4 halves = two LL words = 16 bytes on the wire
  const size_t slot_bytes = (size_t)max_elems * 4;            // 2 halves -> 8 bytes
  const size_t inbox_off = (size_t)par * world * slot_bytes;
  const uint2* src = reinterpret_cast<const uint2*>(y);
  for (int v = tid; v < nv; v += kCommThreads) {
    const uint2 d = src[v];
    const uint4 w = make_uint4(d.x, e, d.y, e);
    for (int p = 0; p < world; ++p)
      st_relaxed_sys_u4(peers.base[p] + inbox_off + (size_t)rank * slot_bytes + (size_t)v * 16, w);
  }
  const uint8_t* mine = peers.base[rank] + inbox_off;
  uint2* dst = reinterpret_cast<uint2*>(y);
  unsigned long long t0 = 0;
  bool dead = false;
  for (int v = tid; v < nv; v += kCommThreads) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int q = 0; q < world; ++q) {
      const uint8_t* a = mine + (size_t)q * slot_bytes + (size_t)v * 16;
      uint4 w = ld_relaxed_sys_u4(a);
      int spins = 0;
      while (!dead && (w.y != e || w.w != e)) {
        if ((++spins & 1023) == 0) {
          unsigned long long now;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
          if (t0 == 0) t0 = now;
          else if (now - t0 > 2000000000ull) {   // 2 s: a peer is gone - do not hang the GPU
            state[1] = 1;
            dead = true;
          }
        }
        w = ld_relaxed_sys_u4(a);
      }
      const float2 f0 = __half22float2(u32_as_h2(w.x)), f1 = __half22float2(u32_as_h2(w.z));
      acc[0] += f0.x;
      acc[1] += f0.y;
      acc[2] += f1.x;
      acc[3] += f1.y;
    }
    dst[v] = make_uint2(h2_as_u32(__floats2half2_rn(acc[0], acc[1])), h2_as_u32(__floats2half2_rn(acc[2], acc[3])));
  }
  __syncthreads();
  if (tid == 0) state[0] = (int)e;
}

int comm_create(int rank, int world, int max_elems, Comm** out, cudaError_t* err) {
  *out = nullptr;
  *err = cudaSuccess;
  if (world < 1 || world > kCommMaxWorld || rank < 0 || rank >= world || max_elems <= 0 || (max_elems % 8) != 0)
    return B200AWQ_EINVAL;
  Comm* c = new Comm();
  c->rank = rank;
  c->world = world;
  c->max_elems = max_elems;
  c->bytes = comm_bytes(world, max_elems);
  cudaError_t e = cudaGetDevice(&c->device);
  if (e == cudaSuccess) e = cudaMalloc(&c->local, c->bytes);
  if (e == cudaSuccess) e = cudaMemset(c->local, 0, c->bytes);
  if (e == cudaSuccess) e = cudaMalloc(&c->d_state, 2 * sizeof(int));
  if (e == cudaSuccess) e = cudaMemset(c->d_state, 0, 2 * sizeof(int));
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    cudaFree(c->local);
    cudaFree(c->d_state);
    delete c;
    *err = e;
    return B200AWQ_ECUDA;
  }
  c->peers.base[rank] = c->local;
  if (world == 1) c->opened = true;
  *out = c;
  return B200AWQ_OK;
}

cudaError_t comm_ipc_handle(Comm* c, void* out64) {
  cudaIpcMemHandle_t h;
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  cudaError_t e = cudaIpcGetMemHandle(&h, c->local);
  if (e == cudaSuccess) std::memcpy(out64, &h, sizeof(h));
  return e;
}

cudaError_t comm_open(Comm* c, const void* handles) {
  for (int p = 0; p < c->world; ++p) {
    if (p == c->rank) continue;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, static_cast<const uint8_t*>(handles) + (size_t)p * 64, sizeof(h));
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return e;
    c->peers.base[p] = static_cast<uint8_t*>(ptr);
  }
  c->opened = true;
  return cudaSuccess;
}

cudaError_t comm_all_reduce(Comm* c, void* y, int n, cudaStream_t st) {
  ll_allreduce_kernel<<<1, kCommThreads, 0, st>>>(c->peers, c->rank, c->world, c->max_elems, static_cast<__half*>(y), n,
                                                  c->d_state);
  return cudaGetLastError();
}

bool comm_ready(const Comm* c) { return c->opened; }
int comm_max_elems(const Comm* c) { return c->max_elems; }

cudaError_t comm_error_flag(Comm* c, int* out) {
  return cudaMemcpy(out, c->d_state + 1, sizeof(int), cudaMemcpyDeviceToHost);
}

void comm_destroy(Comm* c) {
  if (c == nullptr) return;
  for (int p = 0; p < c->world; ++p)
    if (p != c->rank && c->peers.base[p] != nullptr) cudaIpcCloseMemHandle(c->peers.base[p]);
  cudaFree(c->local);
  cudaFree(c->d_state);
  delete c;
}

}  // namespace b200awq
