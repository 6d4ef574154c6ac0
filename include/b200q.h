/*
 * b200q.h -- C ABI of libb200q.so: the B200 (sm_100a) replacement for blazr's quantized linear-layer
 * operator.  Plain pointers and sizes only; no torch / C++ types cross this boundary.
 *
 * What each entry point replaces in the reference (ml-rust/blazr, paths relative to /root/reference):
 *
 *   blazr reaches the operator only through trait bounds on the backend client
 *   (`boostr::quant::QuantMatmulOps<R>` / `boostr::quant::DequantOps<R>`: src/loader/api.rs:25,45,67,90;
 *   src/engine/generate_text.rs:32-33; src/engine/scheduler.rs:110-111) and through the weights its
 *   loaders build.  The trait bodies live in the un-vendored `boostr` crate, so this ABI is shaped by the
 *   data blazr hands over:
 *
 *   b200q_weight_from_ggml   <- GGUF upload: VarMap::from_gguf keeps raw ggml blocks tagged with their
 *                               ggml type (src/loader/gguf.rs:33,38,40; type tag :365-372).
 *   b200q_weight_from_awq    <- DecomposedQuantTensor::new(qweight u32[K,N/8], scales f32[K/gs,N],
 *                               zeros f32[K/gs,N], None, Awq{group_size}, [N,K])
 *                               (src/loader/safetensors/awq.rs:190-226, zeros unpack :242-263).
 *   b200q_weight_from_gptq   <- DecomposedQuantTensor::new(qweight u32[K/8,N], scales f32[G,N],
 *                               qzeros u32[G,N/8] packed, g_idx i32[K], Gptq{group_size}, [N,K]) + bias
 *                               (src/loader/safetensors/gptq.rs:198-259).
 *   b200q_matmul             <- QuantMatmulOps: Y[M,N] = X[M,K] . dequant(W)[N,K]^T (+bias) issued 7L+1
 *                               times per forward (src/engine/executor_generate.rs:357,372; batched
 *                               decode M = N_seq src/engine/batch_decode.rs:115-147); must be CUDA-graph
 *                               capturable (src/engine/cuda_graphs.rs:101-130).
 *   b200q_dequantize         <- DequantOps: packed blocks -> dense tensor (src/loader/gguf.rs:25,53,77).
 *   b200q_shard_range /
 *   b200q_weight_*_shard     <- TensorParallelState::shard_range (src/engine/tensor_parallel.rs:61-67),
 *                               load_model_tp (src/loader/api.rs:39-56).
 *
 * Conventions
 *   - Every function returns 0 on success or a negative b200q_status; it never throws or aborts.
 *     b200q_last_error() returns a thread-local message for the last failure on the calling thread.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - Weight handles are immutable after creation: share them freely across threads and streams.
 *   - Compute entry points do no allocation, no host synchronisation and read no host scalars after
 *     launch, so they may be captured into CUDA graphs.  Scratch comes from the caller's `workspace`
 *     (>= b200q_workspace_bytes(w, M) bytes, 256-byte aligned, ZERO-FILLED before its first use; one
 *     workspace must not be used by two in-flight calls at once).
 *   - There is NO CPU fallback: an unsupported format/shape is an error code.
 */
#ifndef B200Q_H
#define B200Q_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum b200q_status {
    B200Q_OK = 0,
    B200Q_ERR_INVALID_ARG = -1,
    B200Q_ERR_UNSUPPORTED = -2,
    B200Q_ERR_CUDA = -3,
    B200Q_ERR_WORKSPACE = -4,
    B200Q_ERR_NO_DEVICE = -5
} b200q_status;

typedef enum b200q_dtype { B200Q_F32 = 0, B200Q_F16 = 1, B200Q_BF16 = 2, B200Q_F64 = 3 /* b200q_matmul_q8 output only: un-rounded partial sums */ } b200q_dtype;

/* internal format families, reported by b200q_weight_info */
typedef enum b200q_family {
    B200Q_FAM_Q4_K = 1, B200Q_FAM_Q6_K = 2, B200Q_FAM_Q8_0 = 3, B200Q_FAM_G4 = 4 /* AWQ/GPTQ */,
    B200Q_FAM_Q5_K = 5, B200Q_FAM_Q4_0 = 6, B200Q_FAM_Q4_1 = 7, B200Q_FAM_Q5_0 = 8, B200Q_FAM_Q5_1 = 9,
    B200Q_FAM_Q2_K = 10, B200Q_FAM_Q3_K = 11, B200Q_FAM_IQ4_NL = 12, B200Q_FAM_IQ4_XS = 13, B200Q_FAM_TQ2_0 = 14, B200Q_FAM_I8S = 15 /* decoded family of the grid-coded IQ formats */
} b200q_family;

/* source kinds */
#define B200Q_SRC_GGML 0
#define B200Q_SRC_AWQ 1
#define B200Q_SRC_GPTQ 2

typedef struct b200q_weight b200q_weight; /* opaque */

typedef struct b200q_weight_info_t {
    int64_t N, K;          /* logical [out_features, in_features] */
    int64_t N_pad, K_pad;  /* padded to the 128 x 256 tile grid */
    int32_t family;        /* b200q_family */
    int32_t source;        /* B200Q_SRC_* */
    int32_t ggml_type;     /* ggml type id for GGML sources, else -1 */
    int32_t group_size;    /* AWQ/GPTQ group size, else 0 */
    int32_t sub;           /* width of the integer-partial sub-block: 16 or 32 */
    int32_t has_bias, has_perm;
    int32_t device;
    int64_t device_bytes;    /* bytes of the repacked device buffer */
    int64_t canonical_bytes; /* bytes of the canonical (on-disk) packed weight: the roofline's algorithmic bytes */
    int32_t chunk_bytes;     /* bytes of one 128-row x 256-k tile */
} b200q_weight_info_t;

int32_t b200q_version(void);
const char* b200q_last_error(void);
int32_t b200q_device_count(void);

/* ---- weight upload (one-off; synchronises `stream` before returning; host source may be freed) ---- */
/* host_blocks: N rows of K/block ggml blocks, row-major, exactly as stored in a GGUF file.
 * src_on_device != 0 means `blocks` is already a device pointer on `device`. */
int32_t b200q_weight_from_ggml(int32_t ggml_type, const void* blocks, int32_t src_on_device, int64_t N, int64_t K,
                               int32_t device, void* stream, b200q_weight** out);
/* Same, keeping only rows [n0,n1) and columns [k0,k1) of the logical [N,K] weight (TP sharding at block
 * granularity: k0,k1 must be multiples of the ggml block size). */
int32_t b200q_weight_from_ggml_shard(int32_t ggml_type, const void* blocks, int32_t src_on_device, int64_t N, int64_t K,
                                     int64_t n0, int64_t n1, int64_t k0, int64_t k1, int32_t device, void* stream,
                                     b200q_weight** out);
/* AWQ triplet as blazr's loader builds it.  Scales must be f16-representable, zeros integers in [0,15]. */
int32_t b200q_weight_from_awq(const uint32_t* qweight, const float* scales, const float* zeros, int32_t src_on_device,
                              int32_t group_size, int64_t N, int64_t K, int32_t device, void* stream, b200q_weight** out);
/* GPTQ group as blazr's loader builds it.  g_idx and bias may be NULL.  zero_plus_one selects the
 * AutoGPTQ-v1 convention (stored zero = z-1); blazr does not reveal which one boostr uses. */
int32_t b200q_weight_from_gptq(const uint32_t* qweight, const float* scales, const uint32_t* qzeros, const int32_t* g_idx,
                               const float* bias, int32_t src_on_device, int32_t group_size, int32_t zero_plus_one,
                               int64_t N, int64_t K, int32_t device, void* stream, b200q_weight** out);
/* TP shards of the INT4 layouts: rows [n0,n1) (multiple of 8) and columns [k0,k1) (multiple of group_size;
 * GPTQ act-order weights cannot be split along K). */
int32_t b200q_weight_from_awq_shard(const uint32_t* qweight, const float* scales, const float* zeros, int32_t src_on_device,
                                    int32_t group_size, int64_t N, int64_t K, int64_t n0, int64_t n1, int64_t k0, int64_t k1,
                                    int32_t device, void* stream, b200q_weight** out);
/* GPTQ shard: same ranges; bias is sliced to [n0,n1).  An act-order weight (non-trivial g_idx) can be split along N only. */
int32_t b200q_weight_from_gptq_shard(const uint32_t* qweight, const float* scales, const uint32_t* qzeros, const int32_t* g_idx, const float* bias,
                                     int32_t src_on_device, int32_t group_size, int32_t zero_plus_one, int64_t N, int64_t K, int64_t n0, int64_t n1,
                                     int64_t k0, int64_t k1, int32_t device, void* stream, b200q_weight** out);
int32_t b200q_weight_free(b200q_weight* w);
int32_t b200q_weight_info(const b200q_weight* w, b200q_weight_info_t* info);
/* optional f32 bias [N] (device copy is made) added in every matmul epilogue */
int32_t b200q_weight_set_bias(b200q_weight* w, const float* bias, int32_t src_on_device, void* stream);
/* Streaming-order hint (performance only; results never depend on it): `next` is the weight the caller will run through
 * b200q_matmul_q8 right after `w` (the model's projection order: qkv -> o -> gate|up -> down -> next layer's qkv ...).
 * A decode matvec on `w` then prefetches the first chunks of `next` into L2 once its own weight stream is fully requested,
 * so HBM keeps streaming across the kernel boundary and the glue operators in between.  `next` is not owned: clear the
 * hint (next = NULL) before freeing it.  The one mutable field of a handle; set it before the handle is shared. */
int32_t b200q_weight_set_next(b200q_weight* w, const b200q_weight* next);
/* Dual-format pairing: `second` (same K, same device, no bias / permutation) is a projection of ANOTHER format that reads the same
 * activations as `w` and whose output columns directly follow w's (y[:, N1 : N1 + N2], N1 % 128 == 0) -- the q|k (Q4_K) and v
 * (Q6_K) projections of a Q4_K_M file (reference src/loader/gguf.rs:365-372 tags every tensor with its own ggml type).  Every decode
 * matvec on `w` (b200q_matmul_q8 / b200q_matmul_norm, M <= 4) then computes BOTH in one launch: ldy and the output buffer must
 * cover N1 + N2 columns; the fused-exchange, SwiGLU and tcgen05 (M >= 5) forms refuse / ignore the pairing.  Built for Q4_K + Q6_K;
 * other combinations return B200Q_ERR_UNSUPPORTED (launch them separately).  `second` is not owned: clear the pairing
 * (second = NULL) before freeing it.  Set it before the handle is shared. */
int32_t b200q_weight_set_pair(b200q_weight* w, const b200q_weight* second);

/* reference src/engine/tensor_parallel.rs:61-67 */
int32_t b200q_shard_range(int64_t total, int64_t rank, int64_t world, int64_t* start, int64_t* end);
/* shard_range applied at `granule` granularity (rows of 1 / blocks of 32,128,256 ...) */
int32_t b200q_shard_range_blocks(int64_t total, int64_t granule, int64_t rank, int64_t world, int64_t* start, int64_t* end);

/* ---- compute ---- */
size_t b200q_workspace_bytes(const b200q_weight* w, int64_t M);
/* Y[M,N] (ldy elements between rows) = X[M,K] (ldx) . dequant(W)^T (+bias).  x,y,workspace: device memory.
 * M == 1..4 : dp4a stream-K matvec on int8-quantised activations (decode);
 * M >= 5    : tcgen05/TMEM dequant-GEMM on bf16 activations (batched decode and prefill). */
int32_t b200q_matmul(const b200q_weight* w, const void* x, int32_t x_dtype, int64_t M, int64_t ldx, void* y, int32_t y_dtype,
                     int64_t ldy, void* workspace, size_t workspace_bytes, void* stream);
/* Split form for callers that share one quantised activation among several weights (q,k,v / gate,up):
 * quantise once into `xq` (b200q_act_bytes(K, M) bytes), then b200q_matmul_q8 for each weight (M <= 4). */
size_t b200q_act_bytes(int64_t K, int64_t M);
int32_t b200q_quantize_act(const void* x, int32_t x_dtype, int64_t M, int64_t K, int64_t ldx, const int32_t* perm /*nullable, device*/,
                           void* xq, void* stream);
int32_t b200q_matmul_q8(const b200q_weight* w, const void* xq, int64_t M, void* y, int32_t y_dtype, int64_t ldy,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- expert banks (MoE): reference boostr::ExpertWeights{gate_proj, up_proj, down_proj}, stacked
 * [num_experts, dim_in, dim_out] and sliced per expert (src/engine/executor_cache.rs:19,218-228,260,283,344-348).
 * A bank is a device-resident table of E weights of one format and shape; b200q_bank_set is the
 * set_expert_weights analogue (placement changes swap one table entry, members are not owned).
 * b200q_moe_matmul_q8 runs n_slots independent M = 1 matvecs in ONE stream-K launch: slot s uses expert
 * sel[s] (device int32, produced by the router just ahead in the stream), the quantised activation row
 * s / x_slot_div of xq (an activation buffer of x_rows rows, b200q_act_bytes(K, x_rows) layout) and writes
 * y[s * y_slot_stride + n].  x_slot_div = top_k shares one token's activation among its experts (gate/up);
 * x_slot_div = 1 gives every slot its own row (down).  Same arithmetic, bit for bit, as b200q_matmul_q8 per slot. */
typedef struct b200q_bank b200q_bank;
int32_t b200q_bank_create(const b200q_weight* const* experts, int32_t E, b200q_bank** out);
int32_t b200q_bank_free(b200q_bank* b);
int32_t b200q_bank_set(b200q_bank* b, int32_t e, const b200q_weight* w, void* stream);
const b200q_weight* b200q_bank_get(const b200q_bank* b, int32_t e);
size_t b200q_bank_workspace_bytes(const b200q_bank* b, int64_t n_slots);
int32_t b200q_moe_matmul_q8(const b200q_bank* b, const int32_t* sel_dev, int64_t n_slots, const void* xq, int64_t x_rows,
                            int64_t x_slot_div, void* y, int32_t y_dtype, int64_t y_slot_stride, void* workspace,
                            size_t workspace_bytes, void* stream);

/* weighted combine of the selected experts' outputs (MoE decode): out[T, H] = sum_j gate_w[t, j] * y[t * top_k + j, :], j ascending,
 * f32 multiply then add (fixed order: expert-parallel partial sums are reproducible) */
int32_t b200q_moe_combine(const float* y, const float* gate_w, int64_t T, int64_t top_k, int64_t H, float* out, void* stream);

/* ---- tensor-parallel exchange over NVLink peer memory, FUSED into the kernels on both sides of it (replaces the NCCL
 * all-reduce blazr's TP issues after the row-parallel o_proj / down_proj, reference src/engine/tensor_parallel.rs:125-163;
 * SURVEY.md sections 5 and 8b/8e).  One process per GPU: create on every rank, all-gather the 64-byte IPC handles, connect.
 *   producer  b200q_matmul_q8_rowpar : the row-parallel matvec stores its exact f64 row sums [M, ld] straight into a slot of
 *             every rank's buffer (8-byte peer stores from the kernel's flush paths) and nothing else: the slot elements are
 *             their own ready flags (empty = +0.0 bits; an exact zero travels as -0.0), no fence, no flag, no extra launch.
 *   consumer  b200q_allreduce_add_rmsnorm_quant : every thread polls the `world` slot elements of its column in local memory,
 *             empties them, sums in rank order in f64, rounds once (identical bits on every rank and equal to the 1-GPU
 *             output), adds the residual, RMS-norms and quantises -- the reduced vector never exists in HBM.
 *             b200q_allreduce_finish is the stand-alone consumer (reduced f32 vector) for other callers.
 *   lm_head   b200q_matmul_q8_gather (column-parallel over the vocabulary) stores f32 logits [M, ld] into region `rank` of
 *             every rank's gather area; b200q_argmax_gathered consumes them (vocabulary id = rank * ld + column).
 *   b200q_allreduce : stand-alone one-shot push all-reduce of a device vector (expert-parallel partial outputs).
 * Every producer call must be followed by exactly one consumer call on every rank before the next producer call of the same
 * kind.  All entry points are graph-capturable (epochs live in device memory). */
typedef struct b200q_comm b200q_comm;
/* max_elems: doubles per all-reduce slot (>= M * hidden); gather_elems: floats per rank in the gather area (>= M * ld, 0 = none) */
int32_t b200q_comm_create(int32_t rank, int32_t world, int64_t max_elems, int64_t gather_elems, int32_t device, b200q_comm** out);
int32_t b200q_comm_handle(const b200q_comm* c, void* out64);
int32_t b200q_comm_connect(b200q_comm* c, const void* handles /* world x 64 bytes, rank order */);
int32_t b200q_comm_free(b200q_comm* c);
/* device pointer of this rank's gather area: f32 [world][elems_per_rank] */
int32_t b200q_comm_gather_ptr(const b200q_comm* c, void** ptr, int64_t* elems_per_rank);
int32_t b200q_matmul_q8_rowpar(const b200q_weight* w, const void* xq, int64_t M, b200q_comm* c, int64_t ld, void* workspace, size_t workspace_bytes,
                               void* stream);
int32_t b200q_allreduce_add_rmsnorm_quant(b200q_comm* c, const float* h_in, float* h_out, const float* norm_w, float eps, int64_t H, int64_t M,
                                          void* xq, float* xnorm, void* stream);
int32_t b200q_allreduce_finish(b200q_comm* c, float* dst, int64_t n, void* stream);
int32_t b200q_matmul_q8_gather(const b200q_weight* w, const void* xq, int64_t M, b200q_comm* c, int64_t ld, void* workspace, size_t workspace_bytes,
                               void* stream);
int32_t b200q_argmax_gathered(b200q_comm* c, int64_t ld, int64_t M, int64_t* out_ids, int32_t* pos_inc, void* stream);
int32_t b200q_allreduce(b200q_comm* c, const void* src, int32_t src_dtype /* B200Q_F32 | B200Q_F64 */, float* dst, int64_t n, void* stream);
int32_t b200q_allreduce_f64(b200q_comm* c, const double* src, float* dst, int64_t n, void* stream); /* = b200q_allreduce(.., B200Q_F64, ..) */

/* Decode matmuls with a fused activation producer (M <= 4): the consumer warps build the quantised activation in
 * shared memory while the first weight chunks are in flight, so no separate norm / SwiGLU kernel runs.
 *   norm  : h = h_in (+ delta, nullable); h_out (nullable; written once) = h; x = quant(rmsnorm(h) * norm_w); y = x . W^T
 *   swiglu: x = quant(silu(gate) * up) for gate_up[M, 2K] (gate first);           y = x . W^T
 * Same arithmetic (bit for bit) as b200q_add_rmsnorm_quant / b200q_swiglu_quant followed by b200q_matmul_q8. */
int32_t b200q_matmul_norm(const b200q_weight* w, const float* h_in, const float* delta, float* h_out, const float* norm_w, float eps, int64_t M,
                          void* y, int32_t y_dtype, int64_t ldy, void* workspace, size_t workspace_bytes, void* stream);
int32_t b200q_matmul_swiglu(const b200q_weight* w, const float* gate_up, int64_t M, void* y, int32_t y_dtype, int64_t ldy, void* workspace,
                            size_t workspace_bytes, void* stream);
/* Fused SwiGLU epilogue (M <= 4): `w` is the gate|up projection uploaded with its 2 F rows INTERLEAVED per 128-row tile --
 * row r of the uploaded matrix is row b200q_gate_up_row(F, r) of the concatenated [gate (F rows); up (F rows)] matrix, i.e.
 * tile t holds gate/up rows 64 t .. 64 t + 63 with the pair (gate j, up j) in one thread's accumulators (F % 64 == 0).
 * Every finished tile is activated (silu(gate) * up) and quantised straight into the activation records of the following
 * down projection (xq_out, b200q_act_bytes(F, M) layout, zero-filled once by the caller): neither the gate|up output nor a
 * separate SwiGLU launch exists.  Same bits as b200q_matmul_q8 + b200q_swiglu_quant on the un-interleaved weight.
 * b200q_matmul_norm_swiglu additionally fuses the add + RMSNorm + quantise producer (see b200q_matmul_norm);
 * b200q_moe_matmul_q8_swiglu is the grouped (expert-bank) form: slot s writes record row s of xq_out (n_slots rows). */
int64_t b200q_gate_up_row(int64_t F, int64_t r);
int32_t b200q_matmul_q8_swiglu(const b200q_weight* w, const void* xq, int64_t M, void* xq_out, void* workspace, size_t workspace_bytes, void* stream);
int32_t b200q_matmul_norm_swiglu(const b200q_weight* w, const float* h_in, const float* delta, float* h_out, const float* norm_w, float eps, int64_t M,
                                 void* xq_out, void* workspace, size_t workspace_bytes, void* stream);
int32_t b200q_moe_matmul_q8_swiglu(const b200q_bank* b, const int32_t* sel_dev, int64_t n_slots, const void* xq, int64_t x_rows, int64_t x_slot_div,
                                   void* xq_out, void* workspace, size_t workspace_bytes, void* stream);
/* Force a path (testing / benchmarking): 0 = auto, 1 = dp4a matvec, 2 = tcgen05 GEMM */
int32_t b200q_matmul_path(const b200q_weight* w, int32_t path, const void* x, int32_t x_dtype, int64_t M, int64_t ldx, void* y,
                          int32_t y_dtype, int64_t ldy, void* workspace, size_t workspace_bytes, void* stream);

/* dense dequantisation: out[N,K] row-major in `dtype` (f32 is bit-exact: a*q - b, no FMA) */
int32_t b200q_dequantize(const b200q_weight* w, void* out, int32_t dtype, void* stream);
/* test hooks for the bit-exact contracts: activation quantiser planes and integer dot partials.
 * q int8[M,K_pad], d f32[M,K_pad/32], bsum16 i32[M,K_pad/16]; partials i32[M,N,K_pad/sub]. */
int32_t b200q_act_unpack(const void* xq, int64_t M, int64_t K, int8_t* q, float* d, int32_t* bsum16, void* stream);
int32_t b200q_int_partials(const b200q_weight* w, const void* xq, int64_t M, int32_t* partials, void* stream);


/* ---- decode-step glue operators (outside the quantized-matmul path; SURVEY.md section 8f "next") ----
 * They let one whole decode step be captured in a CUDA graph: each emits the int8 activation records
 * (b200q_act_bytes layout) that the following b200q_matmul_q8 consumes, so no separate quantise pass runs.
 * Reference call sites: src/engine/cuda_graphs.rs:101-130 (captured forward + argmax_to_buf). */
/* h_out[M,H] = h_in (+ delta, nullable); xq = quant(rmsnorm(h_out) * w); xnorm (nullable) receives the f32 normalised
 * row.  h_in and h_out must differ when delta != NULL.  H <= 8192 runs as one thread-block cluster per row (the row is read
 * once, the sum of squares is combined through distributed shared memory); larger H runs H/256 CTAs wide. */
int32_t b200q_add_rmsnorm_quant(const float* h_in, const float* delta, float* h_out, const float* w, float eps, int64_t H, int64_t M,
                                void* xq, float* xnorm, void* stream);
/* xq = quant(silu(gate) * up) for gate_up[M, 2F] (gate first) */
int32_t b200q_swiglu_quant(const float* gate_up, int64_t F, int64_t M, void* xq, void* stream);
/* batched decode (M > 4, tcgen05 path takes f32 activations): act[M, F] = silu(gate) * up.  The norm and attention
 * operators likewise accept xq == NULL when their f32 output (xnorm / attn_out) is requested instead. */
int32_t b200q_swiglu_f32(const float* gate_up, int64_t F, int64_t M, float* act, void* stream);
/* same, for gate_up columns in the SwiGLU-epilogue row order of an interleaved gate|up weight (b200q_gate_up_row) */
int32_t b200q_swiglu_f32_interleaved(const float* gate_up, int64_t F, int64_t M, float* act, void* stream);
/* RoPE (adjacent pairs; cos/sin from rope_table [max_ctx][hd/2][2] f32) on q and the new k, KV append at pos[m],
 * single-query attention (f64 reductions, deterministic exp), quantised output.
 * qkv[M,(nh+2nkv)*hd] f32; caches [M][max_ctx][nkv][hd] f32; attn_out (nullable) receives the f32 result */
int32_t b200q_attn_decode(const float* qkv, const int32_t* pos, float* cache_k, float* cache_v, const float* rope_table, int32_t n_heads,
                          int32_t n_kv_heads, int32_t head_dim, int32_t max_ctx, int64_t M, void* xq, float* attn_out, void* stream);
/* Paged-KV form (reference forward_with_paged_kv_cache + the slot_mapping / block_table tensors process_decode_batch builds,
 * src/engine/batch_decode.rs:77-147): k_pool / v_pool are [num_blocks][block_size][nkv][hd] f32 pools shared by all sequences;
 * block_table int32 [M][max_blocks] (entries beyond a sequence's length are never read), slot_mapping int32 [M] = block *
 * block_size + offset of the NEW token (nullable: derived from block_table and pos); pos[m] = sequence length - 1.  Same
 * arithmetic, bit for bit, as the contiguous form.  slot -1 / a position >= max_blocks * block_size -> b200q_decode_error. */
int32_t b200q_attn_decode_paged(const float* qkv, const int32_t* pos, float* k_pool, float* v_pool, const int32_t* block_table, const int32_t* slot_mapping,
                                int32_t block_size, int32_t max_blocks, const float* rope_table, int32_t n_heads, int32_t n_kv_heads, int32_t head_dim,
                                int64_t M, void* xq, float* attn_out, void* stream);
/* Largest max_ctx b200q_attn_decode / b200q_attn_decode_paged accept (40960): their one CTA per (head, sequence) keeps every
 * score of the context in shared memory.  Beyond it, use the split-context forms below. */
int32_t b200q_attn_decode_max_ctx(void);
/* Workspace the split-context forms need for this shape (0 for a head_dim other than 64 / 128 or non-positive sizes):
 * f32 scores [M][nh][max_ctx] plus per-split maxima and f64 partial sums.  One workspace serves every layer of a model whose
 * attention calls run in sequence on one stream. */
size_t b200q_attn_split_workspace_bytes(int32_t n_heads, int32_t n_kv_heads, int32_t head_dim, int32_t max_ctx, int64_t M);
/* Split-context decode attention for any max_ctx >= 1: the arguments and results of b200q_attn_decode / _paged, computed by
 * three kernels that split the positions of each (kv head, sequence) over up to 128 CTAs, each serving all query heads of its kv
 * head.  Scores are bit-identical to the single-CTA kernel's; only the order of the f64 sums of the weighted sum differs.
 * Launch shape depends on max_ctx only (graph-capturable).  A short workspace -> B200Q_ERR_WORKSPACE.  Out-of-range positions
 * and slot -1 write nothing and raise b200q_decode_error, as in the single-CTA forms. */
int32_t b200q_attn_decode_split(const float* qkv, const int32_t* pos, float* cache_k, float* cache_v, const float* rope_table, int32_t n_heads,
                                int32_t n_kv_heads, int32_t head_dim, int32_t max_ctx, int64_t M, void* xq, float* attn_out, void* workspace,
                                size_t workspace_bytes, void* stream);
int32_t b200q_attn_decode_paged_split(const float* qkv, const int32_t* pos, float* k_pool, float* v_pool, const int32_t* block_table, const int32_t* slot_mapping,
                                      int32_t block_size, int32_t max_blocks, const float* rope_table, int32_t n_heads, int32_t n_kv_heads, int32_t head_dim,
                                      int64_t M, void* xq, float* attn_out, void* workspace, size_t workspace_bytes, void* stream);
/* The four attention forms above with the KV cache in a chosen element type: cache_k / cache_v (k_pool / v_pool) are arrays
 * of kv_dtype elements in the same layouts, followed by the same arguments.  kv_dtype B200Q_F32 is exactly the f32-named
 * function (they are its B200Q_F32 case); B200Q_F16 halves the cache.  An f16 element is stored as
 * f16_rn(clamp(x, -65504, 65504)) of the f32 value the f32 form would store (the rotated k, the raw v; NaN stores -65504), and
 * the step that appends row p scores and weights its own k / v from those rounded values, so a row reads the same at every
 * step.  Every loaded element widens exactly to f32; all arithmetic after the load is that of the f32 forms.  Another kv_dtype
 * -> B200Q_ERR_UNSUPPORTED; cache pointers not 16-byte aligned -> B200Q_ERR_INVALID_ARG (both before any launch).  The split
 * workspace does not depend on kv_dtype. */
int32_t b200q_attn_decode_kv(const float* qkv, const int32_t* pos, void* cache_k, void* cache_v, int32_t kv_dtype, const float* rope_table, int32_t n_heads,
                             int32_t n_kv_heads, int32_t head_dim, int32_t max_ctx, int64_t M, void* xq, float* attn_out, void* stream);
int32_t b200q_attn_decode_paged_kv(const float* qkv, const int32_t* pos, void* k_pool, void* v_pool, int32_t kv_dtype, const int32_t* block_table,
                                   const int32_t* slot_mapping, int32_t block_size, int32_t max_blocks, const float* rope_table, int32_t n_heads,
                                   int32_t n_kv_heads, int32_t head_dim, int64_t M, void* xq, float* attn_out, void* stream);
int32_t b200q_attn_decode_split_kv(const float* qkv, const int32_t* pos, void* cache_k, void* cache_v, int32_t kv_dtype, const float* rope_table,
                                   int32_t n_heads, int32_t n_kv_heads, int32_t head_dim, int32_t max_ctx, int64_t M, void* xq, float* attn_out,
                                   void* workspace, size_t workspace_bytes, void* stream);
int32_t b200q_attn_decode_paged_split_kv(const float* qkv, const int32_t* pos, void* k_pool, void* v_pool, int32_t kv_dtype, const int32_t* block_table,
                                         const int32_t* slot_mapping, int32_t block_size, int32_t max_blocks, const float* rope_table, int32_t n_heads,
                                         int32_t n_kv_heads, int32_t head_dim, int64_t M, void* xq, float* attn_out, void* workspace, size_t workspace_bytes,
                                         void* stream);
/* A position pos[m] outside [0, max_ctx) makes b200q_attn_decode write nothing and raise a sticky per-device error
 * word instead of indexing past the KV cache.  b200q_decode_error reads and clears it for the current device
 * (synchronises the device: not capturable; call it after a generate loop).  bit 0 = position out of range. */
int32_t b200q_decode_error(int32_t* out_flags);
/* greedy token: argmax over V, lowest index wins ties; pos_inc (nullable) is incremented per row (graph replay) */
int32_t b200q_argmax(const float* logits, int64_t V, int64_t M, int64_t* out_ids, int32_t* pos_inc, void* stream);
/* h[m,:] = f16 table[ids[m],:] */
int32_t b200q_embed(const void* table_f16, const int64_t* ids, int64_t H, int64_t M, float* h, void* stream);

/* number of kernels the library has launched on this process (all threads); for bench accounting */
int64_t b200q_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* B200Q_H */
