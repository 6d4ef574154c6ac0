// api.cu -- the extern "C" boundary of libb200q.so (include/b200q.h).  No exceptions cross it: every entry
// point returns a status code and records a thread-local message.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

#include "comm_dev.cuh"
#include "common.cuh"
#include "internal.h"

namespace b200q {
static std::atomic<long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
}  // namespace b200q

using namespace b200q;

static thread_local char g_err[512] = "";

static int32_t fail(int32_t code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
namespace b200q {
// the same thread-local message for the other translation units (comm.cu, decode_ops.cu)
int32_t set_error(int32_t code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
}  // namespace b200q
static int32_t cuda_fail(cudaError_t e, const char* what) {
    return fail(B200Q_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}
#define CUDA_TRY(expr)                                      \
    do {                                                    \
        cudaError_t _e = (expr);                            \
        if (_e != cudaSuccess) return cuda_fail(_e, #expr); \
    } while (0)

struct FamilyInfo {
    int family, block_elems, block_bytes, sub, chunk_bytes;
};
static bool ggml_family(int ggml_type, FamilyInfo* fi) {
    switch (ggml_type) {
        case 12: *fi = {B200Q_FAM_Q4_K, 256, 144, 32, 128 * 144}; return true;
        case 14: *fi = {B200Q_FAM_Q6_K, 256, 210, 16, 128 * 210}; return true;
        case 8: *fi = {B200Q_FAM_Q8_0, 32, 34, 32, 128 * 272}; return true;
        case 13: *fi = {B200Q_FAM_Q5_K, 256, 176, 32, 128 * 176}; return true;
        case 3: *fi = {B200Q_FAM_Q4_1, 32, 20, 32, 128 * 160}; return true;
        case 7: *fi = {B200Q_FAM_Q5_1, 32, 24, 32, 128 * 192}; return true;
        case 10: *fi = {B200Q_FAM_Q2_K, 256, 84, 16, 128 * 84}; return true;
        case 11: *fi = {B200Q_FAM_Q3_K, 256, 110, 16, 128 * 110}; return true;
        case 23: *fi = {B200Q_FAM_IQ4_XS, 256, 136, 32, 128 * 136}; return true;
        case 35: *fi = {B200Q_FAM_TQ2_0, 256, 66, 32, 128 * 66}; return true;
        // grid-coded IQ formats -> the decoded I8S family (int8 values + integer scale multipliers), sub-block 16
        case 16: *fi = {B200Q_FAM_I8S, 256, 66, 16, 128 * 274}; return true;   // IQ2_XXS
        case 17: *fi = {B200Q_FAM_I8S, 256, 74, 16, 128 * 274}; return true;   // IQ2_XS
        case 18: *fi = {B200Q_FAM_I8S, 256, 98, 16, 128 * 274}; return true;   // IQ3_XXS
        case 22: *fi = {B200Q_FAM_I8S, 256, 82, 16, 128 * 274}; return true;   // IQ2_S
        case 21: *fi = {B200Q_FAM_I8S, 256, 110, 16, 128 * 274}; return true;  // IQ3_S
        case 19: *fi = {B200Q_FAM_I8S, 256, 50, 16, 128 * 274}; return true;   // IQ1_S
        case 29: *fi = {B200Q_FAM_I8S, 256, 56, 16, 128 * 274}; return true;   // IQ1_M
        case 34: *fi = {B200Q_FAM_TQ2_0, 256, 54, 32, 128 * 66}; return true;              // TQ1_0 -> TQ2_0 layout (source adaptor)
        // source adaptors (formats.cuh): exact re-encodings into an existing family at upload
        case 2: *fi = {B200Q_FAM_G4, 32, 18, 32, 128 * 128 + 128 * 8 * 3}; return true;   // Q4_0  -> G4, 32-wide groups
        case 6: *fi = {B200Q_FAM_Q8_0, 32, 22, 32, 128 * 272}; return true;               // Q5_0  -> Q8_0 family
        case 20: *fi = {B200Q_FAM_Q8_0, 32, 18, 32, 128 * 272}; return true;              // IQ4_NL -> Q8_0 family
        default: return false;
    }
}

static int32_t alloc_weight(b200q_weight* w, int device) {
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(B200Q_ERR_NO_DEVICE, "device %d is sm_%d%d; libb200q is built for sm_100a only (no fallback)", device, prop.major, prop.minor);
    w->num_sms = prop.multiProcessorCount;
    w->device = device;
    w->N_pad = (w->N + TILE_ROWS - 1) / TILE_ROWS * TILE_ROWS;
    w->K_pad = (w->K + CHUNK_K - 1) / CHUNK_K * CHUNK_K;
    w->T = w->N_pad / TILE_ROWS;
    w->KC = w->K_pad / CHUNK_K;
    w->device_bytes = w->T * w->KC * (int64_t)w->chunk_bytes;
    CUDA_TRY(cudaMalloc(&w->data, (size_t)w->device_bytes));
    return B200Q_OK;
}

static void free_weight(b200q_weight* w) {
    if (!w) return;
    if (w->data) cudaFree(w->data);
    if (w->bias) cudaFree(w->bias);
    if (w->perm) cudaFree(w->perm);
    delete w;
}

static int gpc_for(int gs) {
    if (gs >= 256) return (gs % 256 == 0) ? 1 : 0;
    if (gs == 128) return 2;
    if (gs == 64) return 4;
    if (gs == 32) return 8;
    return 0;
}

template <typename T>
static cudaError_t to_device(const T* src, size_t count, int on_device, cudaStream_t st, const T** dev, std::vector<void*>& temps) {
    if (on_device || !src) { *dev = src; return cudaSuccess; }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, count * sizeof(T));
    if (e != cudaSuccess) return e;
    temps.push_back(p);
    e = cudaMemcpyAsync(p, src, count * sizeof(T), cudaMemcpyHostToDevice, st);
    *dev = (const T*)p;
    return e;
}

static int32_t finish_g4(b200q_weight* w, int* err_dev, std::vector<void*>& temps, cudaError_t e, cudaStream_t st, b200q_weight** out) {
    int herr = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&herr, err_dev, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    for (void* p : temps) cudaFree(p);
    if (e != cudaSuccess) { free_weight(w); return cuda_fail(e, "INT4 repack"); }
    if (herr & 1) { free_weight(w); return fail(B200Q_ERR_UNSUPPORTED, "scales are not f16-representable (blazr casts f16->f32 at load; anything else is unsupported)"); }
    if (herr & 2) { free_weight(w); return fail(B200Q_ERR_UNSUPPORTED, "zero points are not integers in [0,255]"); }
    *out = w;
    return B200Q_OK;
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

extern "C" {

int32_t b200q_version(void) { return 100; }
const char* b200q_last_error(void) { return g_err; }
int64_t b200q_launch_count(void) { return (int64_t)g_launches.load(); }

int32_t b200q_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int32_t b200q_shard_range(int64_t total, int64_t rank, int64_t world, int64_t* start, int64_t* end) {
    // reference src/engine/tensor_parallel.rs:61-67: even split, remainder spread over the low ranks
    if (!start || !end || world <= 0 || rank < 0 || rank >= world || total < 0) return fail(B200Q_ERR_INVALID_ARG, "shard_range: bad arguments");
    int64_t per = total / world, rem = total % world;
    *start = rank * per + (rank < rem ? rank : rem);
    *end = *start + per + (rank < rem ? 1 : 0);
    return B200Q_OK;
}
int32_t b200q_shard_range_blocks(int64_t total, int64_t granule, int64_t rank, int64_t world, int64_t* start, int64_t* end) {
    if (granule <= 0 || total % granule != 0) return fail(B200Q_ERR_INVALID_ARG, "shard_range_blocks: total %lld not a multiple of %lld", (long long)total, (long long)granule);
    int64_t s, e;
    int32_t rc = b200q_shard_range(total / granule, rank, world, &s, &e);
    if (rc) return rc;
    *start = s * granule;
    *end = e * granule;
    return B200Q_OK;
}

int32_t b200q_weight_from_ggml_shard(int32_t ggml_type, const void* blocks, int32_t src_on_device, int64_t N, int64_t K, int64_t n0,
                                     int64_t n1, int64_t k0, int64_t k1, int32_t device, void* stream, b200q_weight** out) {
    if (!out) return fail(B200Q_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    FamilyInfo fi;
    if (!ggml_family(ggml_type, &fi)) return fail(B200Q_ERR_UNSUPPORTED, "ggml type %d has no sm_100a kernel (no CPU fallback)", ggml_type);
    if (!blocks || N <= 0 || K <= 0) return fail(B200Q_ERR_INVALID_ARG, "bad blocks/N/K");
    if (K % fi.block_elems) return fail(B200Q_ERR_INVALID_ARG, "K=%lld is not a multiple of the block size %d", (long long)K, fi.block_elems);
    if (n0 < 0 || n1 > N || n0 >= n1 || k0 < 0 || k1 > K || k0 >= k1) return fail(B200Q_ERR_INVALID_ARG, "bad shard range");
    if (k0 % fi.block_elems || k1 % fi.block_elems) return fail(B200Q_ERR_INVALID_ARG, "K shard [%lld,%lld) must be block (%d) aligned", (long long)k0, (long long)k1, fi.block_elems);
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(device));
    b200q_weight* w = new (std::nothrow) b200q_weight();
    if (!w) return fail(B200Q_ERR_CUDA, "out of host memory");
    memset(w, 0, sizeof(*w));
    w->N = n1 - n0;
    w->K = k1 - k0;
    w->family = fi.family;
    w->source = B200Q_SRC_GGML;
    w->ggml_type = ggml_type;
    w->sub = fi.sub;
    w->gpc = ggml_type == 2 ? 8 : 1;
    if (ggml_type == 16 || ggml_type == 17) w->gpc = 3;  // I8S: scale exponent (w = d * m * 2^-gpc * v)
    if (ggml_type == 18) w->gpc = 2;
    if (ggml_type == 22) w->gpc = 3;
    if (ggml_type == 21) w->gpc = 0;
    if (ggml_type == 19 || ggml_type == 29) w->gpc = 3;
    w->group_size = ggml_type == 2 ? 32 : 0;
    w->chunk_bytes = fi.chunk_bytes;
    w->canonical_bytes = w->N * (w->K / fi.block_elems) * fi.block_bytes;
    int32_t rc = alloc_weight(w, device);
    if (rc) { free_weight(w); return rc; }
    int64_t src_row_bytes = K / fi.block_elems * fi.block_bytes;
    const uint8_t* src_dev = (const uint8_t*)blocks;
    uint8_t* staging = nullptr;
    if (!src_on_device) {
        // stage only the rows of this shard
        size_t bytes = (size_t)(n1 - n0) * src_row_bytes;
        cudaError_t e = cudaMalloc(&staging, bytes);
        if (e != cudaSuccess) { free_weight(w); return cuda_fail(e, "cudaMalloc(staging)"); }
        e = cudaMemcpyAsync(staging, (const uint8_t*)blocks + n0 * src_row_bytes, bytes, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) { cudaFree(staging); free_weight(w); return cuda_fail(e, "cudaMemcpyAsync(H2D blocks)"); }
        src_dev = staging;
    }
    cudaError_t e = launch_repack_ggml(fi.family, src_dev, src_row_bytes, src_on_device ? n0 : 0, k0, w, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (staging) cudaFree(staging);
    if (e != cudaSuccess) { free_weight(w); return cuda_fail(e, "repack"); }
    *out = w;
    return B200Q_OK;
}

int32_t b200q_weight_from_ggml(int32_t ggml_type, const void* blocks, int32_t src_on_device, int64_t N, int64_t K, int32_t device,
                               void* stream, b200q_weight** out) {
    return b200q_weight_from_ggml_shard(ggml_type, blocks, src_on_device, N, K, 0, N, 0, K, device, stream, out);
}

int32_t b200q_weight_from_awq_shard(const uint32_t* qweight, const float* scales, const float* zeros, int32_t src_on_device,
                                    int32_t group_size, int64_t N, int64_t K, int64_t n0, int64_t n1, int64_t k0, int64_t k1, int32_t device,
                                    void* stream, b200q_weight** out) {
    if (!out) return fail(B200Q_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    if (!qweight || !scales || !zeros || N <= 0 || K <= 0) return fail(B200Q_ERR_INVALID_ARG, "bad AWQ arguments");
    int gpc = gpc_for(group_size);
    if (!gpc) return fail(B200Q_ERR_UNSUPPORTED, "AWQ group_size %d unsupported (32, 64, 128 or a multiple of 256)", group_size);
    if (N % 8 || K % group_size) return fail(B200Q_ERR_INVALID_ARG, "AWQ needs N %% 8 == 0 and K %% group_size == 0");
    if (n0 < 0 || n1 > N || n0 >= n1 || k0 < 0 || k1 > K || k0 >= k1 || k0 % group_size || k1 % group_size || k0 % 32)
        return fail(B200Q_ERR_INVALID_ARG, "bad AWQ shard range (K shards must be group aligned)");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(device));
    b200q_weight* w = new (std::nothrow) b200q_weight();
    if (!w) return fail(B200Q_ERR_CUDA, "out of host memory");
    memset(w, 0, sizeof(*w));
    w->N = n1 - n0; w->K = k1 - k0;
    w->family = B200Q_FAM_G4; w->source = B200Q_SRC_AWQ; w->ggml_type = -1; w->group_size = group_size; w->sub = 32; w->gpc = gpc;
    w->chunk_bytes = 128 * 128 + 128 * gpc * 3;
    // canonical on-disk bytes: 4-bit weights + f16 scale + 4-bit zero per group (SURVEY.md section 8d)
    w->canonical_bytes = w->N * w->K / 2 + w->N * (w->K / group_size) * 2 + w->N * (w->K / group_size) / 2;
    int32_t rc = alloc_weight(w, device);
    if (rc) { free_weight(w); return rc; }
    std::vector<void*> temps;
    const uint32_t* qd; const float *sd, *zd;
    int64_t G = K / group_size;
    cudaError_t e = to_device(qweight, (size_t)K * (N / 8), src_on_device, st, &qd, temps);
    if (e == cudaSuccess) e = to_device(scales, (size_t)G * N, src_on_device, st, &sd, temps);
    if (e == cudaSuccess) e = to_device(zeros, (size_t)G * N, src_on_device, st, &zd, temps);
    int* err_dev = nullptr;
    if (e == cudaSuccess) { e = cudaMalloc((void**)&err_dev, sizeof(int)); if (e == cudaSuccess) temps.push_back(err_dev); }
    if (e == cudaSuccess) e = cudaMemsetAsync(err_dev, 0, sizeof(int), st);
    if (e == cudaSuccess) e = launch_repack_awq(qd, sd, zd, N, n0, k0, w, err_dev, st);
    return finish_g4(w, err_dev, temps, e, st, out);
}

int32_t b200q_weight_from_awq(const uint32_t* qweight, const float* scales, const float* zeros, int32_t src_on_device, int32_t group_size,
                              int64_t N, int64_t K, int32_t device, void* stream, b200q_weight** out) {
    return b200q_weight_from_awq_shard(qweight, scales, zeros, src_on_device, group_size, N, K, 0, N, 0, K, device, stream, out);
}

int32_t b200q_weight_from_gptq_shard(const uint32_t* qweight, const float* scales, const uint32_t* qzeros, const int32_t* g_idx, const float* bias,
                                     int32_t src_on_device, int32_t group_size, int32_t zero_plus_one, int64_t N, int64_t K, int64_t n0, int64_t n1,
                                     int64_t k0, int64_t k1, int32_t device, void* stream, b200q_weight** out) {
    if (!out) return fail(B200Q_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    if (!qweight || !scales || !qzeros || N <= 0 || K <= 0) return fail(B200Q_ERR_INVALID_ARG, "bad GPTQ arguments");
    if (n0 < 0 || n1 > N || n0 >= n1 || n0 % 8 || n1 % 8 || k0 < 0 || k1 > K || k0 >= k1 || k0 % group_size || k1 % group_size || k0 % 32)
        return fail(B200Q_ERR_INVALID_ARG, "bad GPTQ shard range (rows in multiples of 8, K shards group aligned)");
    const bool k_sharded = k0 != 0 || k1 != K;
    int gpc = gpc_for(group_size);
    if (!gpc) return fail(B200Q_ERR_UNSUPPORTED, "GPTQ group_size %d unsupported (32, 64, 128 or a multiple of 256)", group_size);
    if (N % 8 || K % group_size || K % 8) return fail(B200Q_ERR_INVALID_ARG, "GPTQ needs N %% 8 == 0 and K %% group_size == 0");
    if (zero_plus_one != 0 && zero_plus_one != 1) return fail(B200Q_ERR_INVALID_ARG, "zero_plus_one must be 0 or 1");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(device));
    // g_idx -> group-sorting permutation (host); identity g_idx needs none
    std::vector<int32_t> perm;
    bool need_perm = false;
    if (g_idx) {
        std::vector<int32_t> gi((size_t)K);
        if (src_on_device) { CUDA_TRY(cudaMemcpy(gi.data(), g_idx, (size_t)K * 4, cudaMemcpyDeviceToHost)); }
        else memcpy(gi.data(), g_idx, (size_t)K * 4);
        int64_t G = K / group_size;
        std::vector<int64_t> cnt((size_t)G + 1, 0);
        for (int64_t k = 0; k < K; k++) {
            if (gi[k] < 0 || gi[k] >= G) return fail(B200Q_ERR_INVALID_ARG, "g_idx[%lld]=%d out of range", (long long)k, gi[k]);
            if (gi[k] != k / group_size) need_perm = true;
            cnt[gi[k] + 1]++;
        }
        if (need_perm) {
            for (int64_t g = 0; g < G; g++)
                if (cnt[g + 1] != group_size) return fail(B200Q_ERR_UNSUPPORTED, "g_idx group %lld has %lld members, expected %d", (long long)g, (long long)cnt[g + 1], group_size);
            for (int64_t g = 0; g < G; g++) cnt[g + 1] += cnt[g];
            perm.resize((size_t)K);
            for (int64_t k = 0; k < K; k++) perm[cnt[gi[k]]++] = (int32_t)k;
        }
    }
    // act-order scatters every group over the whole K axis: a contiguous K slice of the weight does not correspond to a
    // contiguous slice of the activations (SURVEY.md section 7 "GPTQ act-order g_idx defeats contiguous K-splits")
    if (need_perm && k_sharded) return fail(B200Q_ERR_UNSUPPORTED, "GPTQ act-order (non-trivial g_idx) weights cannot be split along K");
    b200q_weight* w = new (std::nothrow) b200q_weight();
    if (!w) return fail(B200Q_ERR_CUDA, "out of host memory");
    memset(w, 0, sizeof(*w));
    w->N = n1 - n0; w->K = k1 - k0;
    w->family = B200Q_FAM_G4; w->source = B200Q_SRC_GPTQ; w->ggml_type = -1; w->group_size = group_size; w->sub = 32; w->gpc = gpc;
    w->chunk_bytes = 128 * 128 + 128 * gpc * 3;
    w->canonical_bytes = w->N * w->K / 2 + w->N * (w->K / group_size) * 2 + w->N * (w->K / group_size) / 2 + (g_idx ? w->K * 4 : 0);
    int32_t rc = alloc_weight(w, device);
    if (rc) { free_weight(w); return rc; }
    std::vector<void*> temps;
    cudaError_t e = cudaSuccess;
    if (need_perm) {
        e = cudaMalloc((void**)&w->perm, (size_t)K * 4);
        if (e == cudaSuccess) e = cudaMemcpyAsync(w->perm, perm.data(), (size_t)K * 4, cudaMemcpyHostToDevice, st);
    }
    if (e == cudaSuccess && bias) {
        e = cudaMalloc((void**)&w->bias, (size_t)w->N * 4);
        if (e == cudaSuccess) e = cudaMemcpyAsync(w->bias, bias + n0, (size_t)w->N * 4, src_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st);
    }
    const uint32_t *qd = nullptr, *zd = nullptr; const float* sd = nullptr;
    int64_t G = K / group_size;
    if (e == cudaSuccess) e = to_device(qweight, (size_t)(K / 8) * N, src_on_device, st, &qd, temps);
    if (e == cudaSuccess) e = to_device(scales, (size_t)G * N, src_on_device, st, &sd, temps);
    if (e == cudaSuccess) e = to_device(qzeros, (size_t)G * (N / 8), src_on_device, st, &zd, temps);
    int* err_dev = nullptr;
    if (e == cudaSuccess) { e = cudaMalloc((void**)&err_dev, sizeof(int)); if (e == cudaSuccess) temps.push_back(err_dev); }
    if (e == cudaSuccess) e = cudaMemsetAsync(err_dev, 0, sizeof(int), st);
    if (e == cudaSuccess) e = launch_repack_gptq(qd, sd, zd, w->perm, zero_plus_one, N, n0, k0, w, err_dev, st);
    return finish_g4(w, err_dev, temps, e, st, out);
}

int32_t b200q_weight_from_gptq(const uint32_t* qweight, const float* scales, const uint32_t* qzeros, const int32_t* g_idx, const float* bias,
                               int32_t src_on_device, int32_t group_size, int32_t zero_plus_one, int64_t N, int64_t K, int32_t device,
                               void* stream, b200q_weight** out) {
    return b200q_weight_from_gptq_shard(qweight, scales, qzeros, g_idx, bias, src_on_device, group_size, zero_plus_one, N, K, 0, N, 0, K, device, stream, out);
}

int32_t b200q_weight_free(b200q_weight* w) {
    if (!w) return B200Q_OK;
    cudaSetDevice(w->device);
    free_weight(w);
    return B200Q_OK;
}

int32_t b200q_weight_info(const b200q_weight* w, b200q_weight_info_t* info) {
    if (!w || !info) return fail(B200Q_ERR_INVALID_ARG, "null argument");
    info->N = w->N; info->K = w->K; info->N_pad = w->N_pad; info->K_pad = w->K_pad;
    info->family = w->family; info->source = w->source; info->ggml_type = w->ggml_type; info->group_size = w->group_size;
    info->sub = w->sub; info->has_bias = w->bias != nullptr; info->has_perm = w->perm != nullptr; info->device = w->device;
    info->device_bytes = w->device_bytes; info->canonical_bytes = w->canonical_bytes; info->chunk_bytes = w->chunk_bytes;
    return B200Q_OK;
}

int32_t b200q_weight_set_bias(b200q_weight* w, const float* bias, int32_t src_on_device, void* stream) {
    if (!w) return fail(B200Q_ERR_INVALID_ARG, "null weight");
    CUDA_TRY(cudaSetDevice(w->device));
    if (w->bias) { cudaFree(w->bias); w->bias = nullptr; }
    if (!bias) return B200Q_OK;
    CUDA_TRY(cudaMalloc((void**)&w->bias, (size_t)w->N * 4));
    CUDA_TRY(cudaMemcpyAsync(w->bias, bias, (size_t)w->N * 4, src_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    return B200Q_OK;
}

int32_t b200q_weight_set_next(b200q_weight* w, const b200q_weight* next) {
    if (!w) return fail(B200Q_ERR_INVALID_ARG, "null weight");
    if (next && next->device != w->device) return fail(B200Q_ERR_INVALID_ARG, "successor lives on device %d, weight on device %d", next->device, w->device);
    w->next = next;
    return B200Q_OK;
}

int32_t b200q_weight_set_pair(b200q_weight* w, const b200q_weight* second) {
    if (!w) return fail(B200Q_ERR_INVALID_ARG, "null weight");
    if (!second) { w->pair = nullptr; return B200Q_OK; }
    if (second == w || second->pair) return fail(B200Q_ERR_INVALID_ARG, "a weight cannot be paired with itself or with a weight that has a partner");
    if (second->device != w->device) return fail(B200Q_ERR_INVALID_ARG, "partner lives on device %d, weight on device %d", second->device, w->device);
    if (second->K != w->K || second->KC != w->KC) return fail(B200Q_ERR_INVALID_ARG, "partner K = %lld differs from K = %lld", (long long)second->K, (long long)w->K);
    if (w->N % TILE_ROWS) return fail(B200Q_ERR_UNSUPPORTED, "the first weight of a pair needs N %% 128 == 0 (got %lld): its partner's rows follow it tile-aligned", (long long)w->N);
    if (w->bias || second->bias || w->perm || second->perm) return fail(B200Q_ERR_UNSUPPORTED, "paired weights carry neither a bias nor an act-order permutation");
    if (!(w->family == B200Q_FAM_Q4_K && second->family == B200Q_FAM_Q6_K))
        return fail(B200Q_ERR_UNSUPPORTED, "dual-format launch is built for a Q4_K weight followed by a Q6_K one (families %d, %d)", w->family, second->family);
    w->pair = second;
    return B200Q_OK;
}

// ---- compute ----
size_t b200q_act_bytes(int64_t K, int64_t M) {
    int64_t kc = (K + CHUNK_K - 1) / CHUNK_K;
    return (size_t)kc * (size_t)M * ACT_REC_BYTES;
}

size_t b200q_workspace_bytes(const b200q_weight* w, int64_t M) {
    if (!w || M <= 0) return 0;
    size_t mv = align256(matvec_ws_bytes(w, M));
    size_t act = align256(b200q_act_bytes(w->K, M <= 4 ? M : 4));
    size_t gm = align256(gemm_ws_bytes(w, M));
    size_t a = mv + act;
    return a > gm ? a : gm;
}

int32_t b200q_quantize_act(const void* x, int32_t x_dtype, int64_t M, int64_t K, int64_t ldx, const int32_t* perm, void* xq, void* stream) {
    if (!x || !xq || M <= 0 || K <= 0 || ldx < K || x_dtype < 0 || x_dtype > 2) return fail(B200Q_ERR_INVALID_ARG, "bad quantize_act arguments");
    int64_t K_pad = (K + CHUNK_K - 1) / CHUNK_K * CHUNK_K;
    CUDA_TRY(launch_act_quant(x, x_dtype, M, K, K_pad, ldx, perm, (uint8_t*)xq, (cudaStream_t)stream));
    return B200Q_OK;
}

int32_t b200q_matmul_q8(const b200q_weight* w, const void* xq, int64_t M, void* y, int32_t y_dtype, int64_t ldy, void* workspace,
                        size_t workspace_bytes, void* stream) {
    if (!w || !xq || !y || !workspace) return fail(B200Q_ERR_INVALID_ARG, "null argument");
    if (M < 1 || M > 4) return fail(B200Q_ERR_UNSUPPORTED, "matmul_q8 handles M in [1,4] (got %lld); use b200q_matmul", (long long)M);
    if (ldy < w->N || y_dtype < 0 || y_dtype > 3) return fail(B200Q_ERR_INVALID_ARG, "bad ldy / y_dtype");  // 3 = f64 partial sums (TP)
    if (workspace_bytes < align256(matvec_ws_bytes(w, M))) return fail(B200Q_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, align256(matvec_ws_bytes(w, M)));
    CUDA_TRY(launch_matvec(w, (const uint8_t*)xq, M, y, y_dtype, ldy, (uint8_t*)workspace, (cudaStream_t)stream));
    return B200Q_OK;
}

// ---- fused tensor-parallel exchange, producer side (comm_dev.cuh): the matvec stores its finished row sums into every rank's buffer ----
static int32_t matmul_q8_remote(const b200q_weight* w, const void* xq, int64_t M, b200q_comm* c, int mode, int64_t ld, void* workspace, size_t workspace_bytes,
                                void* stream) {
    if (!w || !xq || !c || !workspace) return fail(B200Q_ERR_INVALID_ARG, "null argument");
    if (M < 1 || M > 4) return fail(B200Q_ERR_UNSUPPORTED, "fused-exchange matvec handles M in [1,4] (got %lld)", (long long)M);
    if (ld < w->N) return fail(B200Q_ERR_INVALID_ARG, "row stride %lld < N = %lld", (long long)ld, (long long)w->N);
    const int64_t cap = mode == RP_ALLREDUCE ? comm_slot_elems(c) : comm_gather_elems(c);
    if (M * ld > cap) return fail(B200Q_ERR_INVALID_ARG, "M * ld = %lld exceeds the communicator's %s capacity %lld", (long long)(M * ld), mode == RP_ALLREDUCE ? "slot" : "gather", (long long)cap);
    if (comm_device(c) != w->device) return fail(B200Q_ERR_INVALID_ARG, "communicator on device %d, weight on device %d", comm_device(c), w->device);
    if (workspace_bytes < align256(matvec_ws_bytes(w, M))) return fail(B200Q_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, align256(matvec_ws_bytes(w, M)));
    RemoteOut ro;
    ro.mode = mode;
    if (!comm_dev(c, &ro.comm)) return fail(B200Q_ERR_INVALID_ARG, "communicator not connected");
    CUDA_TRY(launch_matvec(w, (const uint8_t*)xq, M, nullptr, B200Q_F64, ld, (uint8_t*)workspace, (cudaStream_t)stream, nullptr, &ro));
    return B200Q_OK;
}

int32_t b200q_matmul_q8_rowpar(const b200q_weight* w, const void* xq, int64_t M, b200q_comm* c, int64_t ld, void* workspace, size_t workspace_bytes, void* stream) {
    return matmul_q8_remote(w, xq, M, c, RP_ALLREDUCE, ld, workspace, workspace_bytes, stream);
}

int32_t b200q_matmul_q8_gather(const b200q_weight* w, const void* xq, int64_t M, b200q_comm* c, int64_t ld, void* workspace, size_t workspace_bytes, void* stream) {
    return matmul_q8_remote(w, xq, M, c, RP_ALLGATHER, ld, workspace, workspace_bytes, stream);
}

// ---- expert banks (MoE) ----
int32_t b200q_bank_create(const b200q_weight* const* experts, int32_t E, b200q_bank** out) {
    if (!experts || !out || E < 1) return fail(B200Q_ERR_INVALID_ARG, "bad bank arguments");
    const b200q_weight* w0 = experts[0];
    if (!w0) return fail(B200Q_ERR_INVALID_ARG, "null expert 0");
    for (int e = 0; e < E; e++) {
        const b200q_weight* w = experts[e];
        if (!w) return fail(B200Q_ERR_INVALID_ARG, "null expert %d", e);
        if (w->family != w0->family || w->N != w0->N || w->K != w0->K || w->chunk_bytes != w0->chunk_bytes || w->gpc != w0->gpc || w->device != w0->device)
            return fail(B200Q_ERR_INVALID_ARG, "expert %d differs from expert 0 in format, shape or device", e);
        if (w->bias || w->perm) return fail(B200Q_ERR_UNSUPPORTED, "bank members must not carry a bias or an act-order permutation");
    }
    b200q_bank* b = new b200q_bank();
    b->E = E;
    b->proto = *w0;
    b->proto.data = nullptr;
    b->members = new const b200q_weight*[E];
    std::vector<const uint8_t*> tab(E);
    for (int e = 0; e < E; e++) { b->members[e] = experts[e]; tab[e] = experts[e]->data; }
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(w0->device);
    cudaError_t ce = cudaMalloc((void**)&b->table_dev, sizeof(uint8_t*) * (size_t)E);
    if (ce == cudaSuccess) ce = cudaMemcpy((void*)b->table_dev, tab.data(), sizeof(uint8_t*) * (size_t)E, cudaMemcpyHostToDevice);
    cudaSetDevice(prev);
    if (ce != cudaSuccess) { delete[] b->members; delete b; return cuda_fail(ce, "bank table upload"); }
    *out = b;
    return B200Q_OK;
}

int32_t b200q_bank_free(b200q_bank* b) {
    if (!b) return B200Q_OK;
    if (b->table_dev) cudaFree((void*)b->table_dev);
    delete[] b->members;
    delete b;
    return B200Q_OK;
}

int32_t b200q_bank_set(b200q_bank* b, int32_t e, const b200q_weight* w, void* stream) {
    if (!b || !w || e < 0 || e >= b->E) return fail(B200Q_ERR_INVALID_ARG, "bad bank_set arguments");
    const b200q_weight& p0 = b->proto;
    if (w->family != p0.family || w->N != p0.N || w->K != p0.K || w->chunk_bytes != p0.chunk_bytes || w->gpc != p0.gpc || w->device != p0.device || w->bias || w->perm)
        return fail(B200Q_ERR_INVALID_ARG, "replacement expert differs from the bank's format, shape or device");
    b->members[e] = w;
    CUDA_TRY(cudaMemcpyAsync((void*)(b->table_dev + e), &w->data, sizeof(uint8_t*), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));  // &w->data is host stack/heap memory: finish before returning
    return B200Q_OK;
}

const b200q_weight* b200q_bank_get(const b200q_bank* b, int32_t e) {
    if (!b || e < 0 || e >= b->E) return nullptr;
    return b->members[e];
}

size_t b200q_bank_workspace_bytes(const b200q_bank* b, int64_t n_slots) {
    if (!b || n_slots < 1) return 0;
    return align256(matvec_grouped_ws_bytes(b, n_slots));
}

int32_t b200q_moe_matmul_q8(const b200q_bank* b, const int32_t* sel_dev, int64_t n_slots, const void* xq, int64_t x_rows, int64_t x_slot_div, void* y,
                            int32_t y_dtype, int64_t y_slot_stride, void* workspace, size_t workspace_bytes, void* stream) {
    if (!b || !sel_dev || !xq || !y || !workspace) return fail(B200Q_ERR_INVALID_ARG, "null argument");
    if (n_slots < 1 || n_slots > 65536) return fail(B200Q_ERR_INVALID_ARG, "n_slots out of range");
    if (x_slot_div < 1 || x_rows < 1 || (n_slots + x_slot_div - 1) / x_slot_div > x_rows) return fail(B200Q_ERR_INVALID_ARG, "activation rows do not cover the slots");
    if (y_slot_stride < b->proto.N || y_dtype < 0 || y_dtype > 2) return fail(B200Q_ERR_INVALID_ARG, "bad y_slot_stride / y_dtype");
    if (workspace_bytes < b200q_bank_workspace_bytes(b, n_slots)) return fail(B200Q_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, b200q_bank_workspace_bytes(b, n_slots));
    CUDA_TRY(launch_matvec_grouped(b, sel_dev, n_slots, (const uint8_t*)xq, x_rows, x_slot_div, y, y_dtype, y_slot_stride, (uint8_t*)workspace, (cudaStream_t)stream));
    return B200Q_OK;
}

/* grouped gate|up with the fused SwiGLU epilogue: slot s writes the quantised activation row s of xq_out (n_slots rows) */
int32_t b200q_moe_matmul_q8_swiglu(const b200q_bank* b, const int32_t* sel_dev, int64_t n_slots, const void* xq, int64_t x_rows, int64_t x_slot_div,
                                   void* xq_out, void* workspace, size_t workspace_bytes, void* stream) {
    if (!b || !sel_dev || !xq || !xq_out || !workspace) return fail(B200Q_ERR_INVALID_ARG, "null argument");
    if (n_slots < 1 || n_slots > 65536) return fail(B200Q_ERR_INVALID_ARG, "n_slots out of range");
    if (x_slot_div < 1 || x_rows < 1 || (n_slots + x_slot_div - 1) / x_slot_div > x_rows) return fail(B200Q_ERR_INVALID_ARG, "activation rows do not cover the slots");
    if (b->proto.N % 128) return fail(B200Q_ERR_UNSUPPORTED, "SwiGLU epilogue needs N = 2 F with F %% 64 == 0 (got N = %lld)", (long long)b->proto.N);
    if (workspace_bytes < b200q_bank_workspace_bytes(b, n_slots)) return fail(B200Q_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, b200q_bank_workspace_bytes(b, n_slots));
    CUDA_TRY(launch_matvec_grouped(b, sel_dev, n_slots, (const uint8_t*)xq, x_rows, x_slot_div, nullptr, B200Q_F32, b->proto.N, (uint8_t*)workspace,
                                   (cudaStream_t)stream, xq_out));
    return B200Q_OK;
}

int32_t b200q_matmul_path(const b200q_weight* w, int32_t path, const void* x, int32_t x_dtype, int64_t M, int64_t ldx, void* y,
                          int32_t y_dtype, int64_t ldy, void* workspace, size_t workspace_bytes, void* stream) {
    if (!w || !x || !y || !workspace) return fail(B200Q_ERR_INVALID_ARG, "null argument");
    if (M <= 0) return fail(B200Q_ERR_INVALID_ARG, "M must be positive");
    if (ldx < w->K || ldy < w->N) return fail(B200Q_ERR_INVALID_ARG, "ldx/ldy smaller than K/N");
    if (x_dtype < 0 || x_dtype > 2 || y_dtype < 0 || y_dtype > 2) return fail(B200Q_ERR_INVALID_ARG, "bad dtype");
    if (((uintptr_t)workspace & 255) != 0) return fail(B200Q_ERR_WORKSPACE, "workspace must be 256-byte aligned");
    if (path == 0) path = (M <= 4) ? 1 : 2;
    cudaStream_t st = (cudaStream_t)stream;
    if (path == 1) {
        if (M > 4) return fail(B200Q_ERR_UNSUPPORTED, "dp4a matvec path handles M <= 4");
        size_t mv = align256(matvec_ws_bytes(w, M));
        size_t need = mv + align256(b200q_act_bytes(w->K, M));
        if (workspace_bytes < need) return fail(B200Q_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, need);
        uint8_t* xq = (uint8_t*)workspace + mv;
        CUDA_TRY(launch_act_quant(x, x_dtype, M, w->K, w->K_pad, ldx, w->perm, xq, st));
        CUDA_TRY(launch_matvec(w, xq, M, y, y_dtype, ldy, (uint8_t*)workspace, st));
        return B200Q_OK;
    }
    if (path == 2) {
        size_t need = align256(gemm_ws_bytes(w, M));
        if (workspace_bytes < need) return fail(B200Q_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, need);
        cudaError_t e = launch_gemm_tc(w, x, x_dtype, M, ldx, y, y_dtype, ldy, (uint8_t*)workspace, workspace_bytes, st);
        if (e == cudaErrorNotSupported) return fail(B200Q_ERR_UNSUPPORTED, "tcgen05 GEMM path not available for this weight/shape");
        if (e != cudaSuccess) return cuda_fail(e, "launch_gemm_tc");
        return B200Q_OK;
    }
    return fail(B200Q_ERR_INVALID_ARG, "unknown path %d", path);
}

int32_t b200q_matmul(const b200q_weight* w, const void* x, int32_t x_dtype, int64_t M, int64_t ldx, void* y, int32_t y_dtype, int64_t ldy,
                     void* workspace, size_t workspace_bytes, void* stream) {
    return b200q_matmul_path(w, 0, x, x_dtype, M, ldx, y, y_dtype, ldy, workspace, workspace_bytes, stream);
}

int32_t b200q_dequantize(const b200q_weight* w, void* out, int32_t dtype, void* stream) {
    if (!w || !out || dtype < 0 || dtype > 2) return fail(B200Q_ERR_INVALID_ARG, "bad dequantize arguments");
    CUDA_TRY(launch_dequantize(w, out, dtype, (cudaStream_t)stream));
    return B200Q_OK;
}

int32_t b200q_act_unpack(const void* xq, int64_t M, int64_t K, int8_t* q, float* d, int32_t* bsum16, void* stream) {
    if (!xq || !q || !d || !bsum16 || M <= 0 || K <= 0) return fail(B200Q_ERR_INVALID_ARG, "bad act_unpack arguments");
    int64_t K_pad = (K + CHUNK_K - 1) / CHUNK_K * CHUNK_K;
    CUDA_TRY(launch_act_unpack((const uint8_t*)xq, M, K_pad, q, d, bsum16, (cudaStream_t)stream));
    return B200Q_OK;
}

int32_t b200q_int_partials(const b200q_weight* w, const void* xq, int64_t M, int32_t* partials, void* stream) {
    if (!w || !xq || !partials || M <= 0 || M > 65535) return fail(B200Q_ERR_INVALID_ARG, "bad int_partials arguments");
    CUDA_TRY(launch_int_partials(w, (const uint8_t*)xq, M, partials, (cudaStream_t)stream));
    return B200Q_OK;
}

static int32_t fused_common(const b200q_weight* w, int64_t M, void* y, int32_t y_dtype, int64_t ldy, void* workspace, size_t workspace_bytes) {
    if (!w || !y || !workspace) return fail(B200Q_ERR_INVALID_ARG, "null argument");
    if (M < 1 || M > 4) return fail(B200Q_ERR_UNSUPPORTED, "fused decode matmul handles M in [1,4] (got %lld)", (long long)M);
    if (ldy < w->N || y_dtype < 0 || y_dtype > 2) return fail(B200Q_ERR_INVALID_ARG, "bad ldy / y_dtype");
    if (w->perm) return fail(B200Q_ERR_UNSUPPORTED, "act-order (permuted K) weights need the split quantize_act + matmul_q8 path");
    if (w->K != w->K_pad) return fail(B200Q_ERR_UNSUPPORTED, "fused prologues need K %% 256 == 0");
    if (workspace_bytes < align256(matvec_ws_bytes(w, M))) return fail(B200Q_ERR_WORKSPACE, "workspace too small");
    return B200Q_OK;
}

int32_t b200q_matmul_norm(const b200q_weight* w, const float* h_in, const float* delta, float* h_out, const float* norm_w, float eps, int64_t M,
                          void* y, int32_t y_dtype, int64_t ldy, void* workspace, size_t workspace_bytes, void* stream) {
    int32_t rc = fused_common(w, M, y, y_dtype, ldy, workspace, workspace_bytes);
    if (rc) return rc;
    if (!h_in || !norm_w) return fail(B200Q_ERR_INVALID_ARG, "null h_in / norm_w");
    {
        const int64_t ept = w->K / 512;  // elements per consumer thread: the lane-parallel prologue needs a power of two <= 16
        if (w->K % 512 || ept > 16 || (ept & (ept - 1))) return fail(B200Q_ERR_UNSUPPORTED, "fused norm prologue supports K in {512, 1024, 2048, 4096, 8192} (got %lld)", (long long)w->K);
    }
    if (delta && h_out == h_in) return fail(B200Q_ERR_INVALID_ARG, "h_out must not alias h_in when delta is given");
    FusedPrologue fp{1, h_in, delta, h_out, norm_w, eps, nullptr};
    CUDA_TRY(launch_matvec(w, nullptr, M, y, y_dtype, ldy, (uint8_t*)workspace, (cudaStream_t)stream, &fp));
    return B200Q_OK;
}

/* ---- fused SwiGLU epilogue: w = gate|up with rows interleaved per 128-row tile (b200q_gate_up_row); writes the quantised
 * activation records of the following down projection instead of y ---- */
static int32_t swiglu_weight_ok(const b200q_weight* w) {
    if (w->N % 128) return fail(B200Q_ERR_UNSUPPORTED, "SwiGLU epilogue needs N = 2 F with F %% 64 == 0 (got N = %lld)", (long long)w->N);
    return B200Q_OK;
}
int64_t b200q_gate_up_row(int64_t F, int64_t r) {
    /* source row, in the concatenated [gate (F rows); up (F rows)] matrix, of row r of the interleaved weight */
    const int64_t t = r / 128, rr = r % 128, w_ = rr / 8, s_ = (rr % 8) / 4, g_ = rr % 4;
    return (s_ ? F : 0) + 64 * t + 4 * w_ + g_;
}
int32_t b200q_matmul_q8_swiglu(const b200q_weight* w, const void* xq, int64_t M, void* xq_out, void* workspace, size_t workspace_bytes, void* stream) {
    if (!w || !xq || !xq_out || !workspace) return fail(B200Q_ERR_INVALID_ARG, "null argument");
    if (M < 1 || M > 4) return fail(B200Q_ERR_UNSUPPORTED, "matmul_q8_swiglu handles M in [1,4] (got %lld)", (long long)M);
    if (int32_t rc = swiglu_weight_ok(w)) return rc;
    if (workspace_bytes < align256(matvec_ws_bytes(w, M))) return fail(B200Q_ERR_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, align256(matvec_ws_bytes(w, M)));
    CUDA_TRY(launch_matvec(w, (const uint8_t*)xq, M, nullptr, B200Q_F32, w->N, (uint8_t*)workspace, (cudaStream_t)stream, nullptr, nullptr, xq_out));
    return B200Q_OK;
}
int32_t b200q_matmul_norm_swiglu(const b200q_weight* w, const float* h_in, const float* delta, float* h_out, const float* norm_w, float eps, int64_t M,
                                 void* xq_out, void* workspace, size_t workspace_bytes, void* stream) {
    if (!xq_out) return fail(B200Q_ERR_INVALID_ARG, "null xq_out");
    float dummy;
    int32_t rc = fused_common(w, M, &dummy, B200Q_F32, w ? w->N : 0, workspace, workspace_bytes);
    if (rc) return rc;
    if ((rc = swiglu_weight_ok(w))) return rc;
    if (!h_in || !norm_w) return fail(B200Q_ERR_INVALID_ARG, "null h_in / norm_w");
    {
        const int64_t ept = w->K / 512;
        if (w->K % 512 || ept > 16 || (ept & (ept - 1))) return fail(B200Q_ERR_UNSUPPORTED, "fused norm prologue supports K in {512, 1024, 2048, 4096, 8192} (got %lld)", (long long)w->K);
    }
    if (delta && h_out == h_in) return fail(B200Q_ERR_INVALID_ARG, "h_out must not alias h_in when delta is given");
    FusedPrologue fp{1, h_in, delta, h_out, norm_w, eps, nullptr};
    CUDA_TRY(launch_matvec(w, nullptr, M, nullptr, B200Q_F32, w->N, (uint8_t*)workspace, (cudaStream_t)stream, &fp, nullptr, xq_out));
    return B200Q_OK;
}

int32_t b200q_matmul_swiglu(const b200q_weight* w, const float* gate_up, int64_t M, void* y, int32_t y_dtype, int64_t ldy, void* workspace,
                            size_t workspace_bytes, void* stream) {
    int32_t rc = fused_common(w, M, y, y_dtype, ldy, workspace, workspace_bytes);
    if (rc) return rc;
    if (!gate_up) return fail(B200Q_ERR_INVALID_ARG, "null gate_up");
    FusedPrologue fp{2, nullptr, nullptr, nullptr, nullptr, 0.0f, gate_up};
    CUDA_TRY(launch_matvec(w, nullptr, M, y, y_dtype, ldy, (uint8_t*)workspace, (cudaStream_t)stream, &fp));
    return B200Q_OK;
}

/* debug only (not in b200q.h): per-CTA globaltimer trace of the matvec kernel */
int32_t b200q_debug_set_matvec_trace(void* dev_buf) {
    set_matvec_trace((long long*)dev_buf);
    return B200Q_OK;
}

}  // extern "C"
