// internal.h -- host-side structures and launcher prototypes shared by the translation units of libb200q.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200q.h"

struct b200q_weight {
    int64_t N, K, N_pad, K_pad;
    int family, source, ggml_type, group_size, sub, gpc;
    int device;
    int chunk_bytes;
    int64_t T, KC;  // tiles along N, chunks along K
    uint8_t* data;  // repacked tiles [T][KC][chunk_bytes]
    int64_t device_bytes, canonical_bytes;
    float* bias;    // device f32 [N] or null
    int32_t* perm;  // device i32 [K] (GPTQ act-order) or null
    int num_sms;
    const b200q_weight* next;  // successor hint (b200q_weight_set_next), not owned; null = none
    const b200q_weight* pair;  // dual-format partner (b200q_weight_set_pair), not owned: its rows follow this weight's in y; null = none
};

// Expert bank (SURVEY 8a row a9: boostr::ExpertWeights stacked [num_experts, ...]): E weights of one format and shape
// addressed through a device-resident pointer table, so one grouped launch streams the selected experts.
struct b200q_bank {
    int E;
    b200q_weight proto;              // shape / format of every member (data = null)
    const uint8_t** table_dev;       // device array [E] of repacked weight buffers
    const b200q_weight** members;    // host array [E] (not owned)
};

namespace b200q {

void count_launch(int n = 1);

// ---- kernels_aux.cu ----
cudaError_t launch_repack_ggml(int family, const uint8_t* src_dev, int64_t src_row_bytes, int64_t n0, int64_t k0, const b200q_weight* w,
                               cudaStream_t st);
cudaError_t launch_repack_awq(const uint32_t* qweight, const float* scales, const float* zeros, int64_t N_full, int64_t n0, int64_t k0,
                              const b200q_weight* w, int* err_flag, cudaStream_t st);
cudaError_t launch_repack_gptq(const uint32_t* qweight, const float* scales, const uint32_t* qzeros, const int32_t* perm, int zpo,
                               int64_t N_full, int64_t n0, int64_t k0, const b200q_weight* w, int* err_flag, cudaStream_t st);
cudaError_t launch_dequantize(const b200q_weight* w, void* out, int dtype, cudaStream_t st);
cudaError_t launch_act_quant(const void* x, int x_dtype, int64_t M, int64_t K, int64_t K_pad, int64_t ldx, const int32_t* perm, uint8_t* xq,
                             cudaStream_t st);
cudaError_t launch_act_unpack(const uint8_t* xq, int64_t M, int64_t K_pad, int8_t* q, float* d, int32_t* bsum16, cudaStream_t st);
cudaError_t launch_int_partials(const b200q_weight* w, const uint8_t* xq, int64_t M, int32_t* out, cudaStream_t st);
cudaError_t launch_to_bf16(const void* x, int x_dtype, int64_t M, int64_t K, int64_t K_pad, int64_t M_pad, int64_t ldx, const int32_t* perm,
                           void* out_bf16, cudaStream_t st);

// ---- matvec.cu ----
struct MatvecPlan {
    int grid, nstages, stage_bytes, smem_bytes, mb, xhat_bytes;
};
struct FusedPrologue {
    int mode;  // 1 = add + rmsnorm + quant, 2 = swiglu + quant
    const float* h_in;
    const float* delta;
    float* h_out;
    const float* norm_w;
    float eps;
    const float* gate_up;
};
cudaError_t matvec_plan(const b200q_weight* w, int64_t M, MatvecPlan* plan, int pro = 0);
size_t matvec_ws_bytes(const b200q_weight* w, int64_t M);  // counters + partials (excludes the activation buffer)
void set_matvec_trace(long long* dev_buf);
struct RemoteOut;  // fused TP exchange target (comm_dev.cuh: mode + CommDev)
cudaError_t launch_matvec(const b200q_weight* w, const uint8_t* xq, int64_t M, void* y, int y_dtype, int64_t ldy, uint8_t* ws, cudaStream_t st,
                          const FusedPrologue* fp = nullptr, const RemoteOut* ro = nullptr, void* swiglu_xq_out = nullptr);
size_t matvec_grouped_ws_bytes(const b200q_bank* b, int64_t n_slots);
cudaError_t launch_matvec_grouped(const b200q_bank* b, const int32_t* sel_dev, int64_t n_slots, const uint8_t* xq, int64_t x_rows, int64_t x_slot_div,
                                  void* y, int y_dtype, int64_t y_slot_stride, uint8_t* ws, cudaStream_t st, void* swiglu_xq_out = nullptr);

// ---- comm.cu ----
struct CommDev;
bool comm_dev(const b200q_comm* c, CommDev* d);  // false when a peer is not connected yet
int64_t comm_slot_elems(const b200q_comm* c);
int64_t comm_gather_elems(const b200q_comm* c);
int comm_device(const b200q_comm* c);
int32_t set_error(int32_t code, const char* fmt, ...);  // api.cu: thread-local b200q_last_error message

// ---- gemm_tc.cu ----
size_t gemm_ws_bytes(const b200q_weight* w, int64_t M);
cudaError_t launch_gemm_tc(const b200q_weight* w, const void* x, int x_dtype, int64_t M, int64_t ldx, void* y, int y_dtype, int64_t ldy,
                           uint8_t* ws, size_t ws_bytes, cudaStream_t st);

}  // namespace b200q
