// extern "C" surface of libb200awq.so (include/b200awq.h): argument validation, path selection,
// error translation.  Kernels live in dequant.cu / gemv.cu / gemm_tc.cu / aux.cu.
#include <atomic>
#include <cstdio>
#include <cstring>

#include <nvtx3/nvToolsExt.h>   // header-only (the tools library is loaded lazily, and only when a profiler is attached)

#include "../../include/b200awq.h"
#include "kernels.h"

namespace b200awq {

// NVTX range around one operator call when knob 15 is set (SURVEY 5: "NVTX ranges per WQLinear call"): the ranges
// show up in Nsight Systems / ncu --nvtx timelines; off (the default) costs one relaxed atomic load.
struct NvtxScope {
  bool on;
  explicit NvtxScope(const char* name);
  ~NvtxScope() {
    if (on) nvtxRangePop();
  }
};

static std::atomic<int> g_knobs[32] = {{0}, {0}, {8}};   // (the rest value-initialise to 0)
int knob(int key) { return (key >= 0 && key < 32) ? g_knobs[key].load(std::memory_order_relaxed) : 0; }
// keys b200awq_set_knob accepts (include/b200awq.h lists them); any other key is an error rather than a silent no-op
static constexpr uint32_t kLiveKnobs = 0x7fu /* 0-6 */ | 1u << 12 | 1u << 14 | 1u << 15 | 1u << 16 | 1u << 19 | 1u << 21;

NvtxScope::NvtxScope(const char* name) : on(knob(15) != 0) {
  if (on) nvtxRangePushA(name);
}

static thread_local char g_cuda_err[256] = "";

static int fold(cudaError_t e) {
  if (e == cudaSuccess) return B200AWQ_OK;
  std::snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", cudaGetErrorName(e), cudaGetErrorString(e));
  (void)cudaGetLastError();  // clear sticky launch-config errors
  if (e == cudaErrorNotSupported) return B200AWQ_EUNSUPPORTED;
  if (e == cudaErrorMisalignedAddress || e == cudaErrorInvalidValue) return B200AWQ_EINVAL;
  return B200AWQ_ECUDA;
}

static bool shape_ok(int M, int K, int N, int G) {
  return M >= 0 && K > 0 && N > 0 && G > 0 && (K % G) == 0 && (N % 8) == 0;
}

struct Ws {
  int* tickets;
  float* acc;
};
static bool carve(void* ws, size_t bytes, int M, int N, Ws* out) {
  out->tickets = nullptr;
  out->acc = nullptr;
  if (ws == nullptr) return false;
  const int rows = M < kMaxSplitM ? M : kMaxSplitM;
  const size_t need = kTicketBytes + (size_t)rows * N * 8;   // one 64-bit packed word (or two floats) per element
  if (bytes < need || (reinterpret_cast<uintptr_t>(ws) & 15) != 0) return false;
  out->tickets = reinterpret_cast<int*>(ws);
  out->acc = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + kTicketBytes);
  return true;
}

}  // namespace b200awq

using namespace b200awq;

extern "C" {

int b200awq_abi_version(void) { return B200AWQ_ABI_VERSION; }

const char* b200awq_error_string(int code) {
  switch (code) {
    case B200AWQ_OK: return "ok";
    case B200AWQ_EINVAL: return "invalid argument (shape, null or misaligned pointer)";
    case B200AWQ_EUNSUPPORTED: return "shape not supported by this path";
    case B200AWQ_EWORKSPACE: return "workspace missing or too small (see b200awq_workspace_bytes)";
    case B200AWQ_ECUDA: return "CUDA error (see b200awq_last_cuda_error)";
    case B200AWQ_EARCH: return "device is not sm_100";
    default: return "unknown error code";
  }
}

const char* b200awq_last_cuda_error(void) { return g_cuda_err; }

size_t b200awq_workspace_bytes(int M, int K, int N) {
  (void)K;
  if (M < 0 || N <= 0) return 0;
  const int rows = M < kMaxSplitM ? M : kMaxSplitM;
  return kTicketBytes + (size_t)rows * N * 8;
}

int b200awq_set_knob(int key, int value) {
  if (key < 0 || key >= 32 || ((kLiveKnobs >> key) & 1u) == 0) return B200AWQ_EINVAL;
  g_knobs[key].store(value, std::memory_order_relaxed);
  if (key == 16) return fold(program_set_watchdog_seconds(value));   // decode-program watchdog (device-side constant)
  return B200AWQ_OK;
}
int b200awq_get_knob(int key) { return knob(key); }

int b200awq_debug_read(void* host_dst, size_t bytes) {
  if (knob(3) == 2) return fold(program_debug_read(host_dst, bytes));
  if (knob(3) == 3) return fold(program_abort_read(host_dst, bytes));
  if (knob(3) == 8) return fold(stream_debug_read(host_dst, bytes));
  if (knob(3) == 9) return fold(gemm_tcq_debug_read(host_dst, bytes));
  return fold(gemv_v3_debug_read(host_dst, bytes));
}

int b200awq_dequantize_gemm(const int32_t* qweight, const void* scales, const int32_t* qzeros, void* out_f16, int K,
                            int N, int group_size, b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_dequantize_gemm");
  const int G = group_size <= 0 ? K : group_size;
  if (!qweight || !scales || !qzeros || !out_f16 || !shape_ok(1, K, N, G)) return B200AWQ_EINVAL;
  return fold(dequantize_gemm(qweight, scales, qzeros, out_f16, K, N, G, static_cast<cudaStream_t>(stream)));
}

int b200awq_gemm_forward(const void* x, int64_t ldx, const int32_t* qweight, const void* scales,
                         const int32_t* qzeros, const void* bias, void* y, int M, int K, int N, int group_size,
                         void* workspace, size_t workspace_bytes, b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_gemm_forward");
  const int G = group_size <= 0 ? K : group_size;
  if (!shape_ok(M, K, N, G) || ldx < K) return B200AWQ_EINVAL;
  if (M == 0) return B200AWQ_OK;
  if (!x || !qweight || !scales || !qzeros || !y) return B200AWQ_EINVAL;
  GemmArgs a{x, ldx, qweight, scales, qzeros, bias, y, M, K, N, G};
  Ws ws;
  const bool have_ws = carve(workspace, workspace_bytes, M, N, &ws);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // M <= 8 (knob 2): the persistent TMA-ring GEMV.  At its default the threshold drops to 4 where the small-M tensor-core
  // kernel applies: from 5 tokens on it is faster on every Llama shape (profiles/r02_tcq_sweep.json: 13 vs 20 us on
  // 4096 x 4096, 33 vs 47 us on 4096 x 28672 at M = 8; at M = 4 the GEMV still wins on three of four shapes).
  int gemv_max = knob(2);
  if (gemv_max == 8 && M > 4 && have_ws && gemm_tcq_applicable(a, ws.acc, ws.tickets)) gemv_max = 4;
  if (M <= gemv_max && M <= 8 && gemv_gemm_layout_supported(a)) {
    if (!have_ws) return B200AWQ_EWORKSPACE;  // the GEMV splits K across CTAs
    if ((N + 255) / 256 > 4096) return B200AWQ_EUNSUPPORTED;
    if (knob(5) == 0 && gemv_v3_supported(a)) return fold(gemv_v3(a, ws.acc, ws.tickets, st));
    return fold(gemv_gemm_layout(a, ws.acc, ws.tickets, st));
  }
  return fold(gemm_tc(a, 0, ws.acc, ws.tickets, st));
}

int b200awq_tcq_plan(int M, int K, int N, int group_size, int sm_count, int mode, int* grid, int* pairs_per_tile) {
  const int G = group_size <= 0 ? K : group_size;
  if (!grid || !pairs_per_tile || sm_count <= 0 || !shape_ok(M, K, N, G)) return B200AWQ_EINVAL;
  if (!gemm_tcq_shape_ok(M, K, N, G)) return B200AWQ_EUNSUPPORTED;
  *pairs_per_tile = K / 128;
  *grid = gemm_tcq_grid(N / 128, K / 128, M, sm_count, mode);
  return B200AWQ_OK;
}

int b200awq_gemv_forward(const void* x, int64_t ldx, const int32_t* qweight, const void* scales,
                         const int32_t* qzeros, const void* bias, void* y, int M, int K, int N, int group_size,
                         void* workspace, size_t workspace_bytes, b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_gemv_forward");
  const int G = group_size <= 0 ? K : group_size;
  if (!shape_ok(M, K, N, G) || ldx < K || (K % 32) != 0) return B200AWQ_EINVAL;
  if (G != 32 && G != 64 && G < 128) return B200AWQ_EUNSUPPORTED;  // calculate_zeros_width's domain
  if (M == 0) return B200AWQ_OK;
  if (!x || !qweight || !scales || !qzeros || !y) return B200AWQ_EINVAL;
  GemmArgs a{x, ldx, qweight, scales, qzeros, bias, y, M, K, N, G};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // the warp-per-row FHFMA kernel does M x the FMA work (7.5 us at M = 1, 35 us at M = 8 on 4096 x 4096, 135 us on
  // 14336 x 4096): beyond two tokens the tcgen05 kernel with the GEMV-layout loader is faster (it needs K % 64 == 0)
  if (M <= knob(2) && (M <= 2 || (K % 64) != 0)) return fold(gemv_gemv_layout(a, st));
  Ws ws;
  carve(workspace, workspace_bytes, M, N, &ws);
  return fold(gemm_tc(a, 1, ws.acc, ws.tickets, st));
}

int b200awq_fast_forward(const void* x, int64_t ldx, const int16_t* qweight, const void* scales,
                         const void* scaled_zeros, const void* bias, void* y, int M, int K, int N, int group_size,
                         void* workspace, size_t workspace_bytes, b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_fast_forward");
  const int G = group_size <= 0 ? K : group_size;
  if (!shape_ok(M, K, N, G) || ldx < K || (K % 64) != 0 || (G % 32) != 0) return B200AWQ_EINVAL;
  if (M == 0) return B200AWQ_OK;
  if (!x || !qweight || !scales || !scaled_zeros || !y) return B200AWQ_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // the warp-per-row FHFMA kernel does M x the FMA work (measured: 10 us at M = 1, 35 us at M = 8 on 4096 x 4096,
  // 124 us on 14336 x 4096): beyond two tokens the tcgen05 kernel with the FAST-layout loader is faster
  if (M <= (knob(2) < 2 ? knob(2) : 2)) {
    FastArgs f{x, ldx, qweight, scales, scaled_zeros, bias, y, M, K, N, G};
    return fold(gemv_fast_layout(f, st));
  }
  GemmArgs a{x, ldx, reinterpret_cast<const int32_t*>(qweight), scales,
             reinterpret_cast<const int32_t*>(scaled_zeros), bias, y, M, K, N, G};
  Ws ws;
  carve(workspace, workspace_bytes, M, N, &ws);
  return fold(gemm_tc(a, 2, ws.acc, ws.tickets, st));
}

int b200awq_rmsnorm(const void* x, const void* weight, void* out, int rows, int hidden, float eps,
                    b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_rmsnorm");
  if (!x || !weight || !out || rows < 0 || hidden <= 0) return B200AWQ_EINVAL;
  if (rows == 0) return B200AWQ_OK;
  return fold(rmsnorm(x, weight, out, rows, hidden, eps, static_cast<cudaStream_t>(stream)));
}

int b200awq_silu_and_mul(const void* gate_up, void* out, int rows, int d, b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_silu_and_mul");
  if (!gate_up || !out || rows < 0 || d <= 0) return B200AWQ_EINVAL;
  if (rows == 0) return B200AWQ_OK;
  return fold(silu_and_mul(gate_up, out, rows, d, static_cast<cudaStream_t>(stream)));
}


int b200awq_program_create(const b200awq_op_t* ops, int n_ops, b200awq_program_t* out) {
  if (out == nullptr) return B200AWQ_EINVAL;
  *out = nullptr;
  Program* p = nullptr;
  cudaError_t ce = cudaSuccess;
  const int rc = program_create(ops, n_ops, &p, &ce);
  if (rc == B200AWQ_ECUDA) return fold(ce);
  if (rc != B200AWQ_OK) return rc;
  *out = reinterpret_cast<b200awq_program_t>(p);
  return B200AWQ_OK;
}

int b200awq_program_num_ops(b200awq_program_t prog) {
  return prog == nullptr ? 0 : program_num_ops(reinterpret_cast<Program*>(prog));
}

int b200awq_program_kind(b200awq_program_t prog) {
  return prog == nullptr ? 0 : (program_is_stream(reinterpret_cast<Program*>(prog)) ? 2 : 1);
}

size_t b200awq_stream_bytes(int K, int N, int group_size) {
  return stream_format_supported(K, N, group_size, 0) ? stream_format_bytes(K, N, group_size) : 0;
}

int b200awq_stream_pack(const int32_t* qweight, const void* scales, const int32_t* qzeros, void* out, int K, int N,
                        int group_size, int mode, b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_stream_pack");
  if (!qweight || !scales || !qzeros || !out) return B200AWQ_EINVAL;
  if (!shape_ok(1, K, N, group_size)) return B200AWQ_EINVAL;
  if (!stream_format_supported(K, N, group_size, mode)) return B200AWQ_EUNSUPPORTED;
  return fold(stream_pack(qweight, scales, qzeros, out, K, N, group_size, mode, static_cast<cudaStream_t>(stream)));
}

int b200awq_program_run(b200awq_program_t prog, void* workspace, size_t workspace_bytes, b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_program_run");
  if (prog == nullptr) return B200AWQ_EINVAL;
  Program* p = reinterpret_cast<Program*>(prog);
  if (program_is_stream(p)) return fold(program_run(p, nullptr, static_cast<cudaStream_t>(stream)));   // owns its rows
  Ws ws;
  // four rows of 64-bit packed sums (= 8 floats per column), max-N columns rounded up to 8, rotate through the ops
  if (!carve(workspace, workspace_bytes, 8, (program_max_n(p) + 7) & ~7, &ws)) return B200AWQ_EWORKSPACE;
  return fold(program_run(p, ws.acc, static_cast<cudaStream_t>(stream)));
}

int b200awq_program_destroy(b200awq_program_t prog) {
  program_destroy(reinterpret_cast<Program*>(prog));
  return B200AWQ_OK;
}

int b200awq_comm_create(int rank, int world, int max_elems, b200awq_comm_t* out) {
  if (out == nullptr) return B200AWQ_EINVAL;
  Comm* c = nullptr;
  cudaError_t ce = cudaSuccess;
  const int rc = comm_create(rank, world, max_elems, &c, &ce);
  if (rc == B200AWQ_ECUDA) return fold(ce);
  if (rc != B200AWQ_OK) return rc;
  *out = reinterpret_cast<b200awq_comm_t>(c);
  return B200AWQ_OK;
}
int b200awq_comm_ipc_handle(b200awq_comm_t comm, void* out64) {
  if (comm == nullptr || out64 == nullptr) return B200AWQ_EINVAL;
  return fold(comm_ipc_handle(reinterpret_cast<Comm*>(comm), out64));
}
int b200awq_comm_open(b200awq_comm_t comm, const void* handles) {
  if (comm == nullptr || handles == nullptr) return B200AWQ_EINVAL;
  return fold(comm_open(reinterpret_cast<Comm*>(comm), handles));
}
int b200awq_comm_all_reduce(b200awq_comm_t comm, void* y, int n, b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_comm_all_reduce");
  Comm* c = reinterpret_cast<Comm*>(comm);
  if (c == nullptr || y == nullptr || n <= 0 || (n % 8) != 0 || (reinterpret_cast<uintptr_t>(y) & 15) != 0) return B200AWQ_EINVAL;
  if (!comm_ready(c)) return B200AWQ_EINVAL;
  if (n > comm_max_elems(c)) return B200AWQ_EUNSUPPORTED;
  return fold(comm_all_reduce(c, y, n, static_cast<cudaStream_t>(stream)));
}
int b200awq_comm_error(b200awq_comm_t comm) {
  if (comm == nullptr) return B200AWQ_EINVAL;
  int f = 0;
  const int rc = fold(comm_error_flag(reinterpret_cast<Comm*>(comm), &f));
  return rc != B200AWQ_OK ? rc : (f != 0 ? B200AWQ_ECUDA : B200AWQ_OK);
}
int b200awq_comm_destroy(b200awq_comm_t comm) {
  comm_destroy(reinterpret_cast<Comm*>(comm));
  return B200AWQ_OK;
}

int b200awq_topk_softmax(const float* gating_output, float* topk_weights, int32_t* topk_ids,
                         int32_t* token_expert_indices, int M, int E, int topk, b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_topk_softmax");
  if (M < 0 || E <= 0 || topk <= 0 || topk > E) return B200AWQ_EINVAL;
  if (M == 0) return B200AWQ_OK;
  if (!gating_output || !topk_weights || !topk_ids || !token_expert_indices) return B200AWQ_EINVAL;
  if (E > 4096) return B200AWQ_EUNSUPPORTED;
  return fold(topk_softmax(gating_output, topk_weights, topk_ids, token_expert_indices, M, E, topk,
                           static_cast<cudaStream_t>(stream)));
}

int b200awq_moe_align_block_size(const int32_t* topk_ids, int numel, int num_experts, int block_size,
                                 int32_t* sorted_ids, int32_t* expert_ids, int32_t* num_tokens_post_pad,
                                 b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_moe_align_block_size");
  if (numel < 0 || num_experts <= 0 || block_size <= 0) return B200AWQ_EINVAL;
  if (!topk_ids || !sorted_ids || !expert_ids || !num_tokens_post_pad) return B200AWQ_EINVAL;
  return fold(moe_align_block_size(topk_ids, numel, num_experts, block_size, sorted_ids, expert_ids, num_tokens_post_pad,
                                   static_cast<cudaStream_t>(stream)));
}

int b200awq_grouped_gemm_forward(const void* x, int x_rows_per_token, const int32_t* qweight, const void* scales,
                                 const int32_t* qzeros, const float* topk_weights, const int32_t* sorted_ids,
                                 const int32_t* expert_ids, const int32_t* num_tokens_post_pad, void* y, int T, int topk,
                                 int sorted_len, int E, int K, int N, int group_size, int mul_weights, int block_size,
                                 void* workspace, size_t workspace_bytes, b200awq_stream_t stream) {
  NvtxScope nvtx_("b200awq_grouped_gemm_forward");
  const int G = group_size <= 0 ? K : group_size;
  if (T < 0 || topk <= 0 || sorted_len < 0 || E <= 0 || !shape_ok(1, K, N, G) || block_size <= 0) return B200AWQ_EINVAL;
  if (x_rows_per_token != 1 && x_rows_per_token != topk) return B200AWQ_EINVAL;
  if (T == 0) return B200AWQ_OK;
  if (!x || !qweight || !scales || !qzeros || !topk_weights || !sorted_ids || !expert_ids || !num_tokens_post_pad || !y)
    return B200AWQ_EINVAL;
  if ((block_size % 8) != 0) return B200AWQ_EUNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int hbs = sorted_len / 8;
  // decode-sized problems: the persistent TMA-ring GEMV, one job per 8 sorted slots (needs 8 rows of fp32 scratch
  // per job); anything larger, or without a workspace: the register-staged grouped kernel
  const size_t need = kTicketBytes + (size_t)hbs * 8 * N * sizeof(float);
  if (knob(12) != 2 && hbs > 0 && workspace != nullptr && workspace_bytes >= need &&
      (reinterpret_cast<uintptr_t>(workspace) & 15) == 0 && gemv_v3_moe_supported(K, N, G, hbs)) {
    int* tickets = reinterpret_cast<int*>(workspace);
    float* acc = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + kTicketBytes);
    return fold(gemv_v3_moe(x, x_rows_per_token == 1 ? 0 : 1, qweight, scales, qzeros, mul_weights ? topk_weights : nullptr,
                            sorted_ids, expert_ids, num_tokens_post_pad, y, T * topk, topk, hbs, E, K, N, G, block_size,
                            acc, tickets, st));
  }
  if (!moe_grouped_supported(K, N, G)) return B200AWQ_EUNSUPPORTED;
  return fold(moe_grouped_gemm(x, x_rows_per_token == 1 ? 0 : 1, qweight, scales, qzeros, topk_weights, sorted_ids,
                               expert_ids, num_tokens_post_pad, y, T * topk, topk, sorted_len, K, N, G, mul_weights,
                               block_size, st));
}
}  // extern "C"
