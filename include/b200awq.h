/* b200awq.h - C ABI of the B200 (sm_100a) AWQ W4A16 linear path.
 *
 * This is the drop-in boundary: a plain C shared library (libb200awq.so) whose entry points are what a
 * replacement for the reference's `awq_ext` / `awq_v2_ext` pybind modules binds.  No torch types: device
 * pointers, sizes, a CUDA stream.  All pointers are DEVICE pointers unless stated; fp16 tensors are passed
 * as `const void*` (IEEE binary16).  Every function launches asynchronously on `stream`, never
 * synchronises, never allocates (CUDA-graph capturable) and returns 0 on success or a B200AWQ_E* code
 * (b200awq_error_string() explains it; `cudaGetLastError` state is folded into B200AWQ_ECUDA).
 *
 * Reference interface each entry point replaces (file:line under casper-hansen/AutoAWQ @ 88e4c76):
 *   b200awq_dequantize_gemm ...... awq_ext.dequantize_weights_cuda  awq/modules/linear/gemm.py:51-53,100-102
 *                                                                   tests/test_dequantization.py:40-49
 *   b200awq_gemm_forward ......... awq_ext.gemm_forward_cuda        awq/modules/linear/gemm.py:56-58
 *                                   (+ the dequant+matmul branch)   awq/modules/linear/gemm.py:50-54
 *   b200awq_gemv_forward ......... awq_ext.gemv_forward_cuda        awq/modules/linear/gemv.py:177-180
 *                                   awq_ext.gemmv2_forward_cuda     awq/modules/linear/gemv.py:168-176
 *   b200awq_fast_forward ......... awq_v2_ext.gemv_forward_cuda_decode   awq/modules/linear/gemv_fast.py:192-201
 *                                   awq_v2_ext.gemm_forward_cuda_prefill  awq/modules/linear/gemv_fast.py:203-205
 *   b200awq_rmsnorm .............. awq_ext.layernorm_forward_cuda   awq/modules/fused/norm.py:33-36
 *   b200awq_silu_and_mul ......... awq_ext.silu_and_mul             awq/modules/fused/moe.py:76
 *
 * Tensor layouts (SURVEY.md Appendix A):
 *   GEMM  : qweight [K, N/8] i32 (AWQ interleave), qzeros [K/G, N/8] i32, scales [K/G, N] f16
 *   GEMV  : qweight [N, K/8] i32 (sequential),     qzeros [N, zw] i32,    scales [N, 8*zw] f16
 *   FAST  : qweight [N/4, K] i16,                  szeros [8*zw, N] f16 (= -z*s), scales [8*zw, N] f16
 */
#ifndef B200AWQ_H_
#define B200AWQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200AWQ_ABI_VERSION 1

typedef void* b200awq_stream_t; /* cudaStream_t */

enum {
  B200AWQ_OK = 0,
  B200AWQ_EINVAL = 1,      /* bad shape / null pointer / misaligned pointer */
  B200AWQ_EUNSUPPORTED = 2,/* shape outside the implemented envelope (e.g. K % 64 != 0 on the tensor-core path) */
  B200AWQ_EWORKSPACE = 3,  /* workspace missing or too small */
  B200AWQ_ECUDA = 4,       /* a CUDA runtime / driver call failed */
  B200AWQ_EARCH = 5        /* device is not sm_100 */
};

int b200awq_abi_version(void);
const char* b200awq_error_string(int code);
/* last CUDA error text seen by this library on the calling thread ("" if none) */
const char* b200awq_last_cuda_error(void);

/* Bytes of scratch the forward entry points may need for (M, K, N): 16 KB of tickets + min(M, 128) * N 64-bit words
 * (split-K partials: packed fixed-point sum + tile count per element for the M <= 8 GEMV, fp32 sums of up to 256 token
 * rows otherwise).
 * The caller allocates once (zero-initialised!) and passes it to every call; the library restores the
 * all-zero ticket state before each kernel exits, so one buffer serves any number of calls on one stream. */
size_t b200awq_workspace_bytes(int M, int K, int N);

/* W[K, N] f16 = (nibble - zero_nibble) * scale, bit-exact with awq/utils/packing_utils.py:87-102. */
int b200awq_dequantize_gemm(const int32_t* qweight, const void* scales, const int32_t* qzeros, void* out_f16,
                            int K, int N, int group_size, b200awq_stream_t stream);

/* Y[M, N] f16 = X[M, K] f16 . deq(W) (+ bias[N] f16 if non-null), GEMM layout.  ldx = row pitch of X in
 * elements (>= K).  M <= 4 runs the persistent tensor-core GEMV (M <= 8 where the small-M kernel does not apply),
 * 5 <= M <= 128 the small-M tcgen05 kernel with TMA-staged packed weights, larger M the tcgen05 GEMM. */
int b200awq_gemm_forward(const void* x, int64_t ldx, const int32_t* qweight, const void* scales,
                         const int32_t* qzeros, const void* bias, void* y, int M, int K, int N, int group_size,
                         void* workspace, size_t workspace_bytes, b200awq_stream_t stream);

/* Same contraction on the GEMV layout (WQLinear_GEMV buffers). */
int b200awq_gemv_forward(const void* x, int64_t ldx, const int32_t* qweight, const void* scales,
                         const int32_t* qzeros, const void* bias, void* y, int M, int K, int N, int group_size,
                         void* workspace, size_t workspace_bytes, b200awq_stream_t stream);

/* Same contraction on the GEMVFast layout (WQLinear_GEMVFast buffers; W = q*s + szeros). */
int b200awq_fast_forward(const void* x, int64_t ldx, const int16_t* qweight, const void* scales,
                         const void* scaled_zeros, const void* bias, void* y, int M, int K, int N, int group_size,
                         void* workspace, size_t workspace_bytes, b200awq_stream_t stream);

/* out[r, :] = x[r, :] * rsqrt(mean(x[r, :]^2) + eps) * weight   (fp32 math, fp16 in/out; out may alias x) */
int b200awq_rmsnorm(const void* x, const void* weight, void* out, int rows, int hidden, float eps,
                    b200awq_stream_t stream);

/* out[r, j] = silu(gate_up[r, j]) * gate_up[r, d + j], j < d  (fp32 math, fp16 in/out) */
int b200awq_silu_and_mul(const void* gate_up, void* out, int rows, int d, b200awq_stream_t stream);

/* ---- MoE (awq/modules/fused/moe.py:45-171; Mixtral: awq/models/mixtral.py:129-158) ------------------------------
 * b200awq_topk_softmax ............ awq_ext.topk_softmax        moe.py:162-167 (fused_topk)
 * b200awq_moe_align_block_size .... awq_ext.moe_alig_block_size moe.py:131-133
 * b200awq_grouped_gemm_forward .... awq_ext.grouped_gemm_forward moe.py:60-89
 *
 * topk_softmax: softmax over the E experts (fp32), the topk largest probabilities per token (ties: lower expert),
 * not renormalised; token_expert_indices[m, k] = k * M + m.
 * moe_align_block_size: flattened slot indices (token * topk + k) grouped by expert in ascending order, every
 * expert's run padded with `numel` to a multiple of block_size; expert_ids[b] = expert of block b;
 * *num_tokens_post_pad = total padded length.  sorted_ids holds numel + E * (block_size - 1) entries, expert_ids
 * numel + E.
 * grouped_gemm_forward: y [T * topk, N] f16; for every real slot id in sorted_ids[0 .. *num_tokens_post_pad),
 * y[id] = x_row(id) . deq(W[expert_ids[pos / block_size]]) (* topk_weights[id] if mul_weights), x_row(id) = x[id /
 * topk] when x_rows_per_token == 1 (x [T, 1, K]) and x[id] when x_rows_per_token == topk (x [T, topk, K]).
 * qweight [E, K, N/8], scales [E, K/G, N], qzeros [E, K/G, N/8] (stacked GEMM layout).  block_size is 16 at the
 * reference's call site (moe.py:54-56) and must be a multiple of 8 here.  Two kernels: with a workspace of
 * b200awq_workspace_bytes(sorted_len, K, N) bytes (zero-initialised, left zero; the per-op workspace serves) and
 * N % 256 == 0, K % 64 == 0, G in {64, 128, K} the persistent TMA-ring GEMV runs one job per 8 sorted slots (the
 * decode case); otherwise a register-staged grouped kernel (K % 512 == 0, N % 32 == 0, G % 64 == 0), else
 * B200AWQ_EUNSUPPORTED.  Knob 12 = 2 forces the second kernel. */
int b200awq_topk_softmax(const float* gating_output, float* topk_weights, int32_t* topk_ids,
                         int32_t* token_expert_indices, int M, int E, int topk, b200awq_stream_t stream);
int b200awq_moe_align_block_size(const int32_t* topk_ids, int numel, int num_experts, int block_size,
                                 int32_t* sorted_ids, int32_t* expert_ids, int32_t* num_tokens_post_pad,
                                 b200awq_stream_t stream);
int b200awq_grouped_gemm_forward(const void* x, int x_rows_per_token, const int32_t* qweight, const void* scales,
                                 const int32_t* qzeros, const float* topk_weights, const int32_t* sorted_ids,
                                 const int32_t* expert_ids, const int32_t* num_tokens_post_pad, void* y, int T, int topk,
                                 int sorted_len, int E, int K, int N, int group_size, int mul_weights, int block_size,
                                 void* workspace, size_t workspace_bytes, b200awq_stream_t stream);

/* Host-side plan of the small-M tensor-core kernel (no GPU needed): for a GEMM-layout call of this shape on a device with
 * `sm_count` SMs, *grid = number of CTAs and *pairs_per_tile = K / 128; CTA b owns the contiguous range
 * [T b / grid, T (b + 1) / grid) of the linearised (128-column tile, 128-row pair) sequence, T = (N / 128) * (K / 128).
 * `mode` as knob 21.  B200AWQ_EUNSUPPORTED when the shape is outside that kernel's envelope
 * (M <= 128, G >= 64, K % 128 == 0, N % 128 == 0). */
int b200awq_tcq_plan(int M, int K, int N, int group_size, int sm_count, int mode, int* grid, int* pairs_per_tile);

/* Tuning / debug knobs (process-global; used by the micro-benchmarks and layout self-tests).  Keys not listed here
 * are rejected with B200AWQ_EINVAL.
 *   key 0: GEMV rows per warp override: 32 / 64 / 128 (0 = heuristic)
 *   key 1: tensor-core path split-K override (0 = heuristic)
 *   key 2: M threshold at or below which the GEMV kernels are used (default 8; the GEMM-layout entry point lowers it to 4
 *          wherever the small-M tensor-core kernel of key 19 applies: it is faster from 5 tokens on)
 *   key 3: 1 = the persistent GEMV records per-CTA phase timestamps (read with b200awq_debug_read);
 *          2 = the decode-program kernel records per-op phase timestamps of its first 8 CTAs / 32 ops
 *          (b200awq_debug_read then returns [op][cta][8] uint64 ns: op begin, previous op complete, activations
 *          staged, first tile landed, warp 0 done, all warps done, partial sums pushed, next op's loads released);
 *          3 = b200awq_debug_read returns the decode-program kernel's abort record instead: int32 [0..3] = {code, op,
 *          CTA, aborted} of the first wait that exceeded 0.5 s (every spin loop of that kernel gives up rather than
 *          hang the GPU), then per CTA 10 ints = (code << 16 | op) of the wait each warp abandoned;
 *          4 = the decode-program kernel does not recycle its accumulator rows (inspection with tools/program_debug.py)
 *          9 = the small-M tensor-core kernel (9 <= M <= 128, GEMM layout) records per-CTA phase timestamps
 *          (b200awq_debug_read returns [cta][8] uint64 ns: entry, setup done, first packed stage landed, producers
 *          done, MMA issuer done, last accumulator drained, epilogue done, number of segments)
 *   key 4: 1 = launch every kernel with the programmatic-dependent-launch attribute (the kernels issue
 *          their weight loads before griddepcontrol.wait, so consecutive linears overlap); default 0
 *   key 5: 1 = disable the persistent TMA-ring GEMV (use the register-staged GEMV for every M <= 8 shape)
 *   key 6: 1 = enable the learned next-weight L2 prefetch (the M <= 8 path remembers which weight tensor
 *          followed which in the call sequence and prefetches the successor's packed weights into L2 at the
 *          tail of each kernel); default 0 - it measured slightly slower on B200
 *   key 12: 2 = grouped_gemm_forward always uses the register-staged grouped kernel
 *   key 16: decode-program watchdog in seconds (0 = the default 0.5 s): every spin of the program kernels gives up
 *           after this long; raise it under compute-sanitizer / a debugger, where kernels run orders of magnitude slower
 *   key 15: 1 = wrap every launching entry point in an NVTX range named after it (profiler timelines); default 0
 *   key 19: 1 = never use the small-M kernel with TMA-staged packed weights (gemm_tcq_kernel; default: every GEMM-layout
 *           call with 5 <= M <= 128 (M above key 2's threshold), G >= 64, K % 128 == 0, N % 128 == 0 runs it)
 *   key 21: small-M kernel work cut: 0 = tile-aligned ranges when N / 128 <= SM count (or from 64 tokens on), balanced
 *           (n-tile, k-step pair) ranges otherwise; 1 = always balanced; 2 = tile-aligned whenever possible
 *   key 14: decode program kind (read at b200awq_program_create): 0 = stream variant when the sequence fits it,
 *           else the split-K kernel; 1 = split-K kernel only; 2 = stream variant only
 */
int b200awq_set_knob(int key, int value);
int b200awq_get_knob(int key);
/* Copies the phase timestamps of the last persistent-GEMV launch (knob 3) to HOST memory: per CTA 8 x uint64 ns
 * (globaltimer): [0] kernel entry, [1] after the PDL wait, [2] first tile landed, [3] consumer warp 0 done,
 * [4] all consumer warps done, [5] partial sums added (REDs issued), [6] tickets bumped, [7] finalisation done.
 * Synchronises the device. */
int b200awq_debug_read(void* host_dst, size_t bytes);

/* ---------------------------------------------------------------------------------------------------------
 * Decode programs: the chain of operator calls of one decode step (M = 1), recorded once and executed by ONE
 * persistent kernel whose weight stream runs across op boundaries (csrc/program.cu).  The op list is exactly
 * the sequence of calls the reference's fused block makes through awq_ext (awq/modules/fused/block.py:117-170,
 * awq/modules/fused/mlp.py:41-55): RMSNorm -> linear -> ... -> SiLU*mul -> linear.  After a run every buffer
 * named by the ops holds what the per-op entry points above would have left there.
 *
 *   RMSNORM       : x = input row [K], weight [K], y = output [K], eps           (K = hidden)
 *   SILU_AND_MUL  : x = gate|up [2K], y = output [K]                             (K = d)
 *   LINEAR_GEMM   : as b200awq_gemm_forward (GEMM layout)
 * b200awq_program_create returns B200AWQ_EUNSUPPORTED when the sequence does not fit the fused kernel (M != 1,
 * a shape outside the persistent GEMV's envelope, a glue op whose output no later linear reads, aliasing the
 * kernel's ordering cannot honour); the caller then issues the ops one by one.  Pointers are captured, not
 * copied: the tensors must stay alive and in place for the life of the program.  Create / destroy allocate and
 * copy (not capturable); run only enqueues a memset + one kernel on `stream` (capturable).  A program is not
 * re-entrant: one run in flight at a time. */
enum { B200AWQ_OP_RMSNORM = 1, B200AWQ_OP_LINEAR_GEMM = 2, B200AWQ_OP_SILU_AND_MUL = 3 };

typedef struct b200awq_op {
  int32_t kind;
  int32_t M, K, N, group_size;
  float eps;
  int64_t ldx;
  const void* x;
  const void* qweight;
  const void* scales;
  const void* qzeros;
  const void* bias;
  const void* weight;
  void* y;
} b200awq_op_t;

typedef struct b200awq_program* b200awq_program_t;

int b200awq_program_create(const b200awq_op_t* ops, int n_ops, b200awq_program_t* out);
/* 0: null handle; 1: split-K kernel on the checkpoint layout (round 1); 2: stream variant - at creation every
 * linear of the program was re-laid-out once into the stream format (below), the kernel partitions the work
 * output-stationary and hands activations from op to op as tagged fp16 words (csrc/program_stream.cuh).  Creation
 * prefers 2 and falls back to 1 (shapes / aliasing outside its envelope; knob 14 = 1 forces 1, 2 forbids 1). */
int b200awq_program_kind(b200awq_program_t prog);
/* number of fused kernel ops (= linear ops) of the program; 0 for a null handle */
int b200awq_program_num_ops(b200awq_program_t prog);
/* workspace: b200awq_workspace_bytes(8, K, max N over the program's linears rounded up to 8): four rows of 64-bit
 * packed split-K sums; zero-initialised and left all-zero like the per-op workspace (the same buffer may serve both) */
int b200awq_program_run(b200awq_program_t prog, void* workspace, size_t workspace_bytes, b200awq_stream_t stream);
int b200awq_program_destroy(b200awq_program_t prog);

/* ---------------------------------------------------------------------------------------------------------
 * One-shot all-reduce over NVLink peer memory (csrc/comm.cu; SURVEY 8e: the reference has no collective at all -
 * multi-GPU there is accelerate layer placement, awq/models/base.py:527-535).  For the tensor-parallel decode path:
 * the fp16 partial outputs of a row-parallel linear (o_proj / down_proj split along K) are summed across the GPUs
 * of one box in ONE kernel launch per call: push into every rank's inbox as words tagged with the call number (P2P
 * stores), wait for the peers' words, reduce in rank order (bit-identical results on all ranks).  One process per GPU: create -> exchange the 64-byte IPC handles by
 * any means (autoawq_b200/comm.py uses torch.distributed.all_gather_object) -> open -> all_reduce any number of
 * times (asynchronous on `stream`, CUDA-graph capturable: the call counter lives on the device).  n % 8 == 0,
 * n <= max_elems (larger messages: use NCCL), world <= 8, y 16-byte aligned; in place.  b200awq_comm_error
 * synchronises and returns B200AWQ_ECUDA if a wait ever timed out (2 s: dead peer). */
typedef struct b200awq_comm* b200awq_comm_t;
int b200awq_comm_create(int rank, int world, int max_elems, b200awq_comm_t* out);
int b200awq_comm_ipc_handle(b200awq_comm_t comm, void* out_64_bytes);
int b200awq_comm_open(b200awq_comm_t comm, const void* handles_world_x_64_bytes);
int b200awq_comm_all_reduce(b200awq_comm_t comm, void* y_f16, int n, b200awq_stream_t stream);
int b200awq_comm_error(b200awq_comm_t comm);
int b200awq_comm_destroy(b200awq_comm_t comm);

/* ---------------------------------------------------------------------------------------------------------
 * Stream format: the one-time, load-time re-layout of a GEMM-layout linear that the decode-program kernel
 * streams (SURVEY 8f #4; the reference's precedent for a post-load re-layout is WQLinear_Exllama.post_init,
 * awq/modules/linear/exllama.py:66-79; the checkpoint format and the module API stay the reference's).  Layout:
 * oracle/stream_format.py (numpy restatement, bit-compared with this entry point in the tests).  Columns are taken
 * in sets of 16, K in units of min(G, 128) rows; a unit is contiguous (fragments in mma.m16n8k16 A-operand order +
 * the unit's scales / zeros), the buffer is set-major, so any partition of the work is a contiguous byte range.
 * mode 0: set s = columns 16 s .. 16 s + 15; mode 1 (a fused gate|up linear): gate column j and up column j share
 * a lane, so SiLU*mul happens in the producer.  Requires N % 16 == 0, K % 128 == 0, G in {32, 64} or G % 128 == 0.
 * b200awq_stream_bytes returns 0 for unsupported shapes. */
size_t b200awq_stream_bytes(int K, int N, int group_size);
int b200awq_stream_pack(const int32_t* qweight, const void* scales, const int32_t* qzeros, void* out, int K, int N,
                        int group_size, int mode, b200awq_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200AWQ_H_ */
