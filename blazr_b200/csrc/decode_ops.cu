// decode_ops.cu -- the small operators that sit between the quantized matvecs of one decode step
// (SURVEY.md section 8f rows 2-4: norm -> activation-quant, RoPE + KV append + decode attention, SwiGLU,
// residual, lm_head argmax).  They are NOT the graded hot path; they exist so that a whole decode step can
// be captured in one CUDA graph and timed as tokens/s, and each one emits the int8 activation records the
// next matvec consumes (so no separate quantise pass runs).  Every kernel is PDL-aware: it lets its
// dependents launch immediately (the following matvec prefetches weights meanwhile) and waits for its own
// producers before touching global memory.
#include <cooperative_groups.h>
#include <cstdlib>
#include <type_traits>

#include "comm_dev.cuh"
#include "common.cuh"
#include "internal.h"

namespace b200q {

// sticky per-device error word raised by kernels that detect an argument they cannot honour without corrupting
// memory (they write nothing and return); read and cleared by b200q_decode_error()
__device__ int g_decode_error = 0;

// TRACE builds only (make TRACE=1; tools/trace_step.py): globaltimer stamps of the glue kernels in launch order --
// record = {kind, entry, after griddepcontrol.wait, exit, 4 phase marks} written by thread 0 of block (0, 0)
#ifdef B200Q_MV_TRACE
__device__ long long* g_glue_trace = nullptr;
__device__ unsigned int g_glue_n = 0;
__device__ unsigned int g_glue_cap = 0;
struct GlueTrace {
    long long* rec;
    __device__ __forceinline__ GlueTrace(int kind) : rec(nullptr) {
        if (threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0 && g_glue_trace) {
            const unsigned int i = atomicAdd(&g_glue_n, 1u);
            if (i < g_glue_cap) { rec = g_glue_trace + 8 * (size_t)i; rec[0] = kind; rec[1] = globaltimer_ns(); }
        }
    }
    __device__ __forceinline__ void waited() { if (rec) rec[2] = globaltimer_ns(); }
    __device__ __forceinline__ void done() { if (rec) rec[3] = globaltimer_ns(); }
    __device__ __forceinline__ void mark(int j) { if (rec) rec[4 + j] = globaltimer_ns(); }   // j < 4: kernel-internal phases
};
#else
struct GlueTrace {
    __device__ __forceinline__ GlueTrace(int) {}
    __device__ __forceinline__ void waited() {}
    __device__ __forceinline__ void done() {}
    __device__ __forceinline__ void mark(int) {}
};
#endif
constexpr int B200Q_DECODE_ERR_POSITION = 1;  // attention: pos[m] outside [0, max_ctx)

// ---- shared: quantise 256 values held one per thread (thread t <-> k = kc*256 + t) into a record ----
__device__ __forceinline__ void quant_store_record(float v, uint8_t* rec, int t) {
    const int wid = t >> 5, lane = t & 31;
    float amax = fabsf(v);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    const float d = __fdiv_rn(amax, 127.0f);
    const float id = (d != 0.0f) ? __fdiv_rn(1.0f, d) : 0.0f;
    const int q = (int)roundf(__fmul_rn(v, id));
    int s = q;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const int s_hi = __shfl_sync(0xffffffffu, s, 16);
    rec[t] = (uint8_t)(int8_t)q;
    if (lane == 0) {
        reinterpret_cast<float*>(rec + 256)[wid] = d;
        reinterpret_cast<uint32_t*>(rec + 288)[wid] = ((uint32_t)s & 0xFFFFu) | ((uint32_t)s_hi << 16);
    }
}

template <typename... Args>
static cudaError_t launch_pdl(void (*kern)(Args...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args...);
    count_launch();
    return e;
}

// ------------------------------------------------------------------------------------------------
// h_out = h_in (+ delta) ; xq = quant(rmsnorm(h_out) * w)
// One CTA of NORM_NT threads per (256-k chunk, token row): every CTA recomputes the row's sum of squares (the row
// is 8-32 KB and L2 resident) and then normalises / quantises / writes only its own chunk, so the operator
// runs H/256 CTAs wide instead of one.  h_in and h_out must be different buffers when delta != null.
// ------------------------------------------------------------------------------------------------
constexpr int NORM_NT = 1024;  // one float4 of the row per thread for H = 4096: the whole row is one load round trip
__global__ void __launch_bounds__(NORM_NT) add_rmsnorm_quant_kernel(const float* __restrict__ h_in, const float* __restrict__ delta,
                                                                     float* __restrict__ h_out, const float* __restrict__ w, float eps, int H, int M,
                                                                     uint8_t* __restrict__ xq, float* __restrict__ xnorm) {
    GlueTrace gt(3);
    pdl_launch_dependents();
    const int kc = blockIdx.x, m = blockIdx.y, t = threadIdx.x;
    const float* hr = h_in + (size_t)m * H;
    const float* dr = delta ? delta + (size_t)m * H : nullptr;
    __shared__ double red[NORM_NT / 32];
    const float wk = (t < CHUNK_K) ? w[kc * CHUNK_K + t] : 0.0f;  // static weights: fetched before the dependency wait
    pdl_wait();
    gt.waited();
    // f64: exact squares, order-independent sum -> bit-reproducible against the oracle (4 independent chains)
    float mine = 0.0f;
    if (t < CHUNK_K) {
        mine = hr[kc * CHUNK_K + t];
        if (dr) mine = __fadd_rn(mine, dr[kc * CHUNK_K + t]);
    }
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll 2
    for (int k4 = t; k4 < H / 4; k4 += NORM_NT) {
        float4 v = reinterpret_cast<const float4*>(hr)[k4];
        if (dr) {
            const float4 d4 = reinterpret_cast<const float4*>(dr)[k4];
            v.x = __fadd_rn(v.x, d4.x); v.y = __fadd_rn(v.y, d4.y); v.z = __fadd_rn(v.z, d4.z); v.w = __fadd_rn(v.w, d4.w);
        }
        s0 = fma((double)v.x, (double)v.x, s0); s1 = fma((double)v.y, (double)v.y, s1);
        s2 = fma((double)v.z, (double)v.z, s2); s3 = fma((double)v.w, (double)v.w, s3);
    }
    double ss = (s0 + s1) + (s2 + s3);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if ((t & 31) == 0) red[t >> 5] = ss;
    __syncthreads();
    if (t >= CHUNK_K) return;
    double tot = 0.0;
#pragma unroll
    for (int i = 0; i < NORM_NT / 32; i++) tot += red[i];
    const float inv = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(__fdiv_rn((float)tot, (float)H), eps)));
    const int k = kc * CHUNK_K + t;
    h_out[(size_t)m * H + k] = mine;
    const float v = __fmul_rn(__fmul_rn(mine, inv), wk);
    if (xnorm) xnorm[(size_t)m * H + k] = v;
    if (xq) quant_store_record(v, xq + ((size_t)kc * M + m) * ACT_REC_BYTES, t);
    gt.done();
}

// ------------------------------------------------------------------------------------------------
// Cluster form of the same operator, and the CONSUMER of the fused tensor-parallel exchange (comm_dev.cuh):
//     delta = f32( sum over ranks, in rank order, of the f64 partial row sums the row-parallel matvec pushed )   [TP]
//     h_out = h_in (+ delta) ; xq = quant(rmsnorm(h_out) * w)
// One thread-block CLUSTER per token row, one column per thread (1024 columns per CTA, up to 8 CTAs = H <= 8192): the row
// is read once (instead of once per 256-column CTA), the sum of squares is combined through distributed shared memory
// in CTA order (f64: order-independent up to 1e-16, same bits as the oracle), and each warp quantises its own 32-block.
// TP: the kernel first polls the `world` epoch flags in its own memory; the reduced delta never exists in HBM.
// ------------------------------------------------------------------------------------------------
constexpr int NORMC_NT = 1024;
__global__ void __launch_bounds__(NORMC_NT) add_rmsnorm_quant_cluster_kernel(const CommDev c, const float* __restrict__ h_in, const float* __restrict__ delta,
                                                                             float* __restrict__ h_out, const float* __restrict__ w, float eps, int H, int M,
                                                                             uint8_t* __restrict__ xq, float* __restrict__ xnorm) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    GlueTrace gt(2);
    pdl_launch_dependents();
    const int cta = blockIdx.x, ncta = gridDim.x, m = blockIdx.y, t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int k = cta * NORMC_NT + t;
    const bool active = k < H;
    __shared__ double red[NORMC_NT / 32];
    __shared__ double cta_part;   // this CTA's share of the sum of squares (read by every CTA of the cluster)
    __shared__ float s_inv;
    const float wk = active ? w[k] : 0.0f;  // static weights: fetched before the dependency wait
    pdl_wait();
    gt.waited();
    float v = 0.0f;
    double* zslot = nullptr;   // TP: this thread's element of the rank-0 slot of the consumed parity (emptied after the cluster barrier)
    if (c.world > 0 && active) {   // (threads beyond the row take no part: they must never poll an element another thread empties)
        // The producing matvec of THIS rank completed before the wait returned (its epoch is published); peers may lag: every
        // thread waits for the `world` partial sums of its own column -- the slots are their own ready flags (comm_dev.cuh).
        // ONE L2 round trip: the epoch and this column's slot elements of BOTH parities are requested together; the parity
        // that is not being exchanged is empty or stale and simply ignored.
        uint8_t* mine = c.peers[c.rank];
        const size_t idx = (size_t)m * H + (size_t)k;
        double sv[2][COMM_MAX_WORLD];
        const unsigned int epoch = __ldcg(reinterpret_cast<const unsigned int*>(mine + COMM_OFF_AR_EPOCH));
#pragma unroll
        for (int pr = 0; pr < 2; pr++)
#pragma unroll
            for (int r = 0; r < COMM_MAX_WORLD; r++)
                if (r < c.world) sv[pr][r] = ld_volatile_f64(reinterpret_cast<const double*>(mine + comm_ar_slot_off(c, pr, r)) + idx);
        const float hv = h_in[(size_t)m * H + k];
        const int par = (int)(epoch & 1u);
        double s = 0.0;
#pragma unroll
        for (int r = 0; r < COMM_MAX_WORLD; r++)
            if (r < c.world) {
                double x = par ? sv[1][r] : sv[0][r];
                const double* q = reinterpret_cast<const double*>(mine + comm_ar_slot_off(c, par, r)) + idx;
                for (int spin = 0; __double_as_longlong(x) == 0ll && spin < COMM_SPIN_LIMIT; spin++) x = ld_volatile_f64(q);   // bounded: a lost peer must not hang the GPU
                s += x;   // rank order, from +0.0 (an exact zero travels as -0.0)
            }
        zslot = reinterpret_cast<double*>(mine + comm_ar_slot_off(c, par, 0)) + idx;
        v = __fadd_rn(hv, (float)s);
    } else if (c.world <= 0 && active) {
        v = h_in[(size_t)m * H + k];
        if (delta) v = __fadd_rn(v, delta[(size_t)m * H + k]);
    }
    gt.mark(0);   // inputs (all ranks' partial sums) are in registers
    double ss = (double)v * (double)v;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if (lane == 0) red[warp] = ss;
    __syncthreads();
    if (warp == 0) {
        double p = red[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) p += __shfl_xor_sync(0xffffffffu, p, o);
        if (lane == 0) cta_part = p;
    }
    gt.mark(1);
    cluster.sync();
    gt.mark(2);
    if (warp == 0) {
        // lane r fetches CTA r's share (ONE distributed-shared-memory latency instead of ncta dependent ones: measured 1.4 us
        // between the cluster barrier and the stores in round 2), then the shares are summed in CTA order: identical on every CTA
        double mine_part = 0.0;
        if (lane < ncta) mine_part = *cluster.map_shared_rank(&cta_part, lane);
        double tot = 0.0;
        for (int r = 0; r < ncta; r++) tot += __shfl_sync(0xffffffffu, mine_part, r);
        if (lane == 0) s_inv = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(__fdiv_rn((float)tot, (float)H), eps)));
    }
    // a CTA's shared memory must stay alive until its peers have read cta_part: arrive now, wait only before exiting.
    // .relaxed: this barrier orders execution only (no data is handed over), so it does not wait for the global stores below
    asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
    if (zslot) {   // the consumed slots are free for the exchange after next (issued here: off the barrier's release path)
        for (int r = 0; r < c.world; r++) zslot[(size_t)r * (size_t)c.slot_elems] = 0.0;
    }
    __syncthreads();  // s_inv
    if (active) {
        h_out[(size_t)m * H + k] = v;
        const float x = __fmul_rn(__fmul_rn(v, s_inv), wk);
        if (xnorm) xnorm[(size_t)m * H + k] = x;
        if (xq) quant_store_record(x, xq + ((size_t)(k / CHUNK_K) * M + m) * ACT_REC_BYTES, k % CHUNK_K);
    }
    gt.mark(3);   // outputs stored
    asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
    gt.done();
}

// ------------------------------------------------------------------------------------------------
// act = silu(gate) * up ; xq = quant(act)       gate_up: [M, 2*F] (gate first), F % 32 == 0; the records are
// zero-padded up to the next multiple of 256 (DeepSeek-V2-Lite experts: F = 1408 = 5.5 chunks)
// ------------------------------------------------------------------------------------------------
// il != 0: gate_up columns are in the SwiGLU-epilogue row order of the weight (b200q_gate_up_row): tile t of 128 columns holds
// the pairs (gate j, up j), j = 64 t .. 64 t + 63, at columns 128 t + 8 (j%64 / 4) + (j % 4) and + 4.
__global__ void __launch_bounds__(256) swiglu_quant_kernel(const float* __restrict__ gu, int F, int M, uint8_t* __restrict__ xq, float* __restrict__ act, int il) {
    pdl_launch_dependents();
    pdl_wait();
    const int kc = blockIdx.x, m = blockIdx.y, t = threadIdx.x;
    const int k = kc * CHUNK_K + t;
    float v = 0.0f;
    if (k < F) {
        const int j = k & 63;
        const size_t cg = il ? (size_t)(k >> 6) * 128 + 8 * (j >> 2) + (j & 3) : (size_t)k;
        const size_t cu = il ? cg + 4 : (size_t)F + k;
        const float g = gu[(size_t)m * 2 * F + cg], u = gu[(size_t)m * 2 * F + cu];
        v = __fmul_rn(__fdiv_rn(g, __fadd_rn(1.0f, det_expf(-g))), u);
        if (act) act[(size_t)m * F + k] = v;
    }
    if (xq) quant_store_record(v, xq + ((size_t)kc * M + m) * ACT_REC_BYTES, t);
}

// ------------------------------------------------------------------------------------------------
// RoPE (adjacent pairs, cos/sin from a host-built table) + KV append + single-query attention + output quant.
// Two passes with f64 reductions and the deterministic exp, so the result is bit-reproducible against the
// oracle:  s_j = f32(sum_e q_e k_je) * scale;  p_j = det_exp(s_j - max);  o_e = f32(sum_j p_j v_je) / f32(sum_j p_j).
// qkv: [M, (nh + 2 nkv) * hd] f32; cache_k/v: [M seqs][max_ctx][nkv][hd] f32; pos[m] = position of the new
// token; rope: [max_ctx][hd/2][2] (cos, sin).  One CTA of ATT_NT threads per (head, m); dynamic smem = max_ctx f32.
// ------------------------------------------------------------------------------------------------
constexpr int ATT_NT = 512;  // threads per (head, m): 128 positions per score sweep, so a short context is one round trip
constexpr int ATTN_SINGLE_MAX_CTX = 160 * 1024 / 4;   // the single-CTA kernel's score buffer: 160 KB of dynamic shared memory
constexpr int ATTN_SPLIT_MIN = 256;   // split-context kernels: fewest positions per split (short contexts use fewer CTAs)
constexpr int ATTN_SPLIT_CAP = 128;   // ... and most splits per (kv head, sequence); longer contexts get longer splits
// PAGED (reference src/engine/batch_decode.rs:77-147, forward_with_paged_kv_cache): cache_k / cache_v are block POOLS
// [num_blocks][block_size][nkv][hd]; position j of sequence m lives in block block_table[m][j / block_size] at offset
// j % block_size; the new token goes to slot_mapping[m] (= block * block_size + offset; derived from the block table when
// slot_mapping is null).  max_ctx = max_blocks * block_size bounds the positions.  Same arithmetic, same bits.
struct PagedKv {
    const int* block_table;   // [M][max_blocks]
    const int* slot_mapping;  // [M] or null
    int block_size, max_blocks;
};

// KV cache element type T: float, or __half (kv_f16_rn on append).  Every cached value widens exactly to f32 on load, so all
// arithmetic after the load is the same for both.  kv_line_t is one 16-byte load (4 f32 / 8 f16 elements), kv_quad_t one load
// of 4 elements (16 / 8 bytes).
template <typename T> using kv_line_t = std::conditional_t<std::is_same_v<T, float>, float4, uint4>;
template <typename T> using kv_quad_t = std::conditional_t<std::is_same_v<T, float>, float4, uint2>;
template <typename T> constexpr int KV_LINE = 16 / (int)sizeof(T);
template <typename T> __device__ __forceinline__ kv_line_t<T> kv_ld_line(const T* p) { return *reinterpret_cast<const kv_line_t<T>*>(p); }
template <typename T> __device__ __forceinline__ kv_quad_t<T> kv_ld_quad(const T* p) { return *reinterpret_cast<const kv_quad_t<T>*>(p); }
template <typename T> __device__ __forceinline__ T kv_store_val(float x) {
    if constexpr (std::is_same_v<T, float>) return x;
    else return kv_f16_rn(x);
}
__device__ __forceinline__ float4 kv_widen(const float4& v) { return v; }
__device__ __forceinline__ float4 kv_widen(const uint2& v) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
    return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void kv_widen(const uint4& v, float* o) {
    const float4 a = kv_widen(make_uint2(v.x, v.y)), b = kv_widen(make_uint2(v.z, v.w));
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
}
// 4 consecutive elements, widened
template <typename T> __device__ __forceinline__ float4 kv_ld4(const T* p) { return kv_widen(kv_ld_quad(p)); }

// f16: one CTA per SM in the bound (ptxas otherwise caps it at 64 registers and spills at head_dim 128); f32 as it always was
template <int HD, bool PAGED, typename T>
__global__ void __launch_bounds__(ATT_NT, std::is_same_v<T, float> ? 0 : 1) attn_decode_kernel(const float* __restrict__ qkv, const int* __restrict__ pos, T* __restrict__ cache_k,
                                                           T* __restrict__ cache_v, const float* __restrict__ rope, int nh, int nkv,
                                                           int max_ctx, int M, uint8_t* __restrict__ xq, float* __restrict__ attn_out, const PagedKv pg) {
    GlueTrace gt(1);
    pdl_launch_dependents();
    extern __shared__ float s_sc[];  // scores, then probabilities, for positions 0..p
    const int head = blockIdx.x, m = blockIdx.y, t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int kvh = head / (nh / nkv);
    // a position outside the cache (host bookkeeping bug, or a graph replayed past max_ctx) must never index the
    // RoPE table, the KV cache or the score buffer: loads ahead of the wait use a clamped position, and after the
    // wait the CTA raises the sticky device error flag (b200q_decode_error) and writes nothing
    const int p_raw = pos[m];
    bool bad_pos = p_raw < 0 || p_raw >= max_ctx;
    if constexpr (PAGED) {
        if (pg.slot_mapping && pg.slot_mapping[m] < 0) bad_pos = true;   // -1 = the block table was too short (batch_decode.rs:88)
    }
    const int p = bad_pos ? 0 : p_raw;
    const int row = (nh + 2 * nkv) * HD;
    const float* qsrc = qkv + (size_t)m * row + (size_t)head * HD;
    const float* ksrc = qkv + (size_t)m * row + (size_t)(nh + kvh) * HD;
    const float* vsrc = qkv + (size_t)m * row + (size_t)(nh + nkv + kvh) * HD;
    const size_t pstride = (size_t)nkv * HD;
    // row of position j in the K / V cache of this (sequence, kv head): contiguous [max_ctx] rows, or through the block table
    const int* bt = PAGED ? pg.block_table + (size_t)m * pg.max_blocks : nullptr;
    auto row_of = [&](int j) -> size_t {
        if constexpr (PAGED) return ((size_t)bt[j / pg.block_size] * pg.block_size + (size_t)(j % pg.block_size)) * pstride + (size_t)kvh * HD;
        else return ((size_t)m * max_ctx + (size_t)j) * pstride + (size_t)kvh * HD;
    };
    T* ck = cache_k;
    T* cv = cache_v;
    const float* rt = rope + (size_t)p * HD;  // [hd/2][2]

    // sk / sv: the new token's k / v as the cache stores them (the f16 cache scores its own row from the rounded values)
    __shared__ __align__(16) float sq[HD];
    __shared__ __align__(16) T sk[HD], sv[HD];
    constexpr int NW = ATT_NT / 32;
    __shared__ float s_redf[NW];
    __shared__ double s_redd[NW];
    // ---- before griddepcontrol.wait: everything that does not depend on the qkv matvec running just ahead of this
    // kernel -- pos (advanced by the previous step's argmax; stable here because embed_kernel, the first kernel of
    // every step, releases its dependents only after that argmax completed), the RoPE row and the cached K / V rows
    // j < p (written by earlier steps) -- is pulled into registers, so only the new q/k/v load remains on the
    // critical path after it.
    constexpr int QE = HD / 4;          // score pass: elements per thread (4 threads per position)
    constexpr int EG = HD / 4;          // output pass: element groups of 4
    constexpr int JG = ATT_NT / EG;     // output pass: position groups (16 for hd 128, 32 for hd 64)
    constexpr int VPF = 8;              // prefetched output-pass iterations (positions < VPF * JG)
    constexpr int KL = KV_LINE<T>;      // score pass: elements per 16-byte load
    const int part = t & 3;
    const int eg = t % EG, jg = t / EG;
    kv_line_t<T> kpre[QE / KL];
    kv_quad_t<T> vpre[VPF];
    float rc = 0.0f, rs = 0.0f;
    {
        const int j = t >> 2;
        if (j < p) {
#pragma unroll
            for (int e = 0; e < QE / KL; e++) kpre[e] = kv_ld_line(ck + row_of(j) + part * QE + KL * e);
        }
#pragma unroll
        for (int it = 0; it < VPF; it++) {
            const int jv = jg + it * JG;
            if (jv < p) vpre[it] = kv_ld_quad(cv + row_of(jv) + 4 * eg);
        }
        if (t < HD / 2) { rc = rt[2 * t]; rs = rt[2 * t + 1]; }
    }
    pdl_wait();
    gt.waited();
    if (bad_pos) {
        if (t == 0) atomicOr(&g_decode_error, B200Q_DECODE_ERR_POSITION);
        return;
    }
    if (t < HD / 2) {
        const float c = rc, sn = rs;
        const float q0 = qsrc[2 * t], q1 = qsrc[2 * t + 1];
        sq[2 * t] = __fsub_rn(__fmul_rn(q0, c), __fmul_rn(q1, sn));
        sq[2 * t + 1] = __fadd_rn(__fmul_rn(q0, sn), __fmul_rn(q1, c));
        const float k0 = ksrc[2 * t], k1 = ksrc[2 * t + 1];
        const T r0 = kv_store_val<T>(__fsub_rn(__fmul_rn(k0, c), __fmul_rn(k1, sn))), r1 = kv_store_val<T>(__fadd_rn(__fmul_rn(k0, sn), __fmul_rn(k1, c)));
        sk[2 * t] = r0; sk[2 * t + 1] = r1;
        sv[2 * t] = kv_store_val<T>(vsrc[2 * t]); sv[2 * t + 1] = kv_store_val<T>(vsrc[2 * t + 1]);
        if (head % (nh / nkv) == 0) {  // one head of each kv group appends the new k, v
            size_t wrow = row_of(p);
            if constexpr (PAGED) {
                if (pg.slot_mapping) wrow = (size_t)pg.slot_mapping[m] * pstride + (size_t)kvh * HD;   // the scheduler's slot (batch_decode.rs:84-90)
            }
            ck[wrow + 2 * t] = r0; ck[wrow + 2 * t + 1] = r1;
            cv[wrow + 2 * t] = kv_store_val<T>(vsrc[2 * t]); cv[wrow + 2 * t + 1] = kv_store_val<T>(vsrc[2 * t + 1]);
        }
    }
    __syncthreads();
    // ---- pass 1: scores; 4 threads per position (a quarter of the head each), 32 positions per sweep ----
    const float scale = __fdiv_rn(1.0f, __fsqrt_rn((float)HD));
    float lmax = -INFINITY;
    {
        for (int j0 = 0; j0 <= p; j0 += ATT_NT / 4) {
            const int j = j0 + (t >> 2);
            double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
            if (j <= p) {
                const T* kr = (j < p) ? ck + row_of(j) + part * QE : sk + part * QE;  // the new key comes from smem
                const float* qq = sq + part * QE;
                if constexpr (std::is_same_v<T, float>) {
#pragma unroll
                    for (int e = 0; e < QE; e += 4) {
                        const float4 kk = (j0 == 0 && j < p) ? kpre[e / 4] : *reinterpret_cast<const float4*>(kr + e);
                        d0 = fma((double)qq[e + 0], (double)kk.x, d0); d1 = fma((double)qq[e + 1], (double)kk.y, d1);
                        d2 = fma((double)qq[e + 2], (double)kk.z, d2); d3 = fma((double)qq[e + 3], (double)kk.w, d3);
                    }
                } else {   // 8 halves per 16-byte load, the same 4 fma chains over e mod 4
#pragma unroll
                    for (int e = 0; e < QE; e += KL) {
                        float kk[KL];
                        kv_widen((j0 == 0 && j < p) ? kpre[e / KL] : kv_ld_line(kr + e), kk);
#pragma unroll
                        for (int i = 0; i < KL; i += 4) {
                            d0 = fma((double)qq[e + i + 0], (double)kk[i + 0], d0); d1 = fma((double)qq[e + i + 1], (double)kk[i + 1], d1);
                            d2 = fma((double)qq[e + i + 2], (double)kk[i + 2], d2); d3 = fma((double)qq[e + i + 3], (double)kk[i + 3], d3);
                        }
                    }
                }
            }
            double d = (d0 + d1) + (d2 + d3);
            d += __shfl_xor_sync(0xffffffffu, d, 1);
            d += __shfl_xor_sync(0xffffffffu, d, 2);
            if (j <= p) {
                const float sc = __fmul_rn((float)d, scale);
                if (part == 0) s_sc[j] = sc;
                lmax = fmaxf(lmax, sc);
            }
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, off));
    if (lane == 0) s_redf[warp] = lmax;
    __syncthreads();
    float gmax = s_redf[0];
#pragma unroll
    for (int i = 1; i < NW; i++) gmax = fmaxf(gmax, s_redf[i]);
    double lsum = 0.0;
    for (int j = t; j <= p; j += ATT_NT) {
        const float pj = det_expf(__fsub_rn(s_sc[j], gmax));
        s_sc[j] = pj;
        lsum += (double)pj;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, off);
    if (lane == 0) s_redd[warp] = lsum;
    __syncthreads();
    double dsum = 0.0;
#pragma unroll
    for (int i = 0; i < NW; i++) dsum += s_redd[i];
    const float den = (float)dsum;
    // ---- pass 2: thread (eg, jg) accumulates 4 output elements over every 4th position; combine through smem ----
    __shared__ double s_o[JG][HD];
    {
        double o0 = 0.0, o1 = 0.0, o2 = 0.0, o3 = 0.0;
#pragma unroll
        for (int it = 0; it < VPF; it++) {  // prefetched rows (and the new token's row when it falls in this range)
            const int j = jg + it * JG;
            if (j <= p) {
                const float pj = s_sc[j];
                const float4 vv = (j < p) ? kv_widen(vpre[it]) : kv_ld4(sv + 4 * eg);
                o0 = fma((double)pj, (double)vv.x, o0); o1 = fma((double)pj, (double)vv.y, o1);
                o2 = fma((double)pj, (double)vv.z, o2); o3 = fma((double)pj, (double)vv.w, o3);
            }
        }
        for (int j = jg + VPF * JG; j <= p; j += JG) {
            const float pj = s_sc[j];
            const float4 vv = (j < p) ? kv_ld4(cv + row_of(j) + 4 * eg) : kv_ld4(sv + 4 * eg);
            o0 = fma((double)pj, (double)vv.x, o0); o1 = fma((double)pj, (double)vv.y, o1);
            o2 = fma((double)pj, (double)vv.z, o2); o3 = fma((double)pj, (double)vv.w, o3);
        }
        s_o[jg][4 * eg + 0] = o0; s_o[jg][4 * eg + 1] = o1; s_o[jg][4 * eg + 2] = o2; s_o[jg][4 * eg + 3] = o3;
        __syncthreads();
    }
    float outv = 0.0f;
    if (t < HD) {
        double o = 0.0;
#pragma unroll
        for (int i = 0; i < JG; i++) o += s_o[i][t];
        outv = __fdiv_rn((float)o, den);
        if (attn_out) attn_out[(size_t)m * nh * HD + (size_t)head * HD + t] = outv;
        // quantise this head's HD outputs into the o_proj activation records (32-blocks never straddle heads)
        if (!xq) return;  // batched decode: the projection takes attn_out (f32)
        const int kglob = head * HD + t;
        const int kc = kglob / CHUNK_K, tin = kglob % CHUNK_K;
        uint8_t* rec = xq + ((size_t)kc * M + m) * ACT_REC_BYTES;
        float amax = fabsf(outv);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, off));
        const float d = __fdiv_rn(amax, 127.0f);
        const float id = (d != 0.0f) ? __fdiv_rn(1.0f, d) : 0.0f;
        const int q = (int)roundf(__fmul_rn(outv, id));
        int s = q;
#pragma unroll
        for (int off = 8; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        const int s_hi = __shfl_sync(0xffffffffu, s, 16);
        rec[tin] = (uint8_t)(int8_t)q;
        if (lane == 0) {
            reinterpret_cast<float*>(rec + 256)[tin >> 5] = d;
            reinterpret_cast<uint32_t*>(rec + 288)[tin >> 5] = ((uint32_t)s & 0xFFFFu) | ((uint32_t)s_hi << 16);
        }
        gt.done();
    }
}

// ------------------------------------------------------------------------------------------------
// Split-context decode attention: the same definition as attn_decode_kernel for any max_ctx (the single-CTA kernel keeps
// every score of a (head, m) in shared memory, so it stops at ATTN_SINGLE_MAX_CTX positions).  Three PDL-chained kernels
// over a caller-provided workspace:
//   A  attn_split_scores_kernel  grid (nkv, M, S_max): split s of the positions [0, p] of sequence m; ONE CTA serves all
//      G = nh / nkv query heads of its kv head (every K row is read once and dotted with G rotated queries).  Writes the
//      f32 scores [M][nh][max_ctx] and each split's maximum [M][nh][S_max].  The CTA owning position p appends the new row.
//   B  attn_split_pv_kernel      same grid: global maximum = max of the split maxima, p_j = det_exp(s_j - max), f64
//      partials sum_j p_j and sum_j p_j v_j of the split -> [M][nh][S_max] and [M][nh][S_max][hd].
//   C  attn_split_combine_kernel grid (nh, M): partials summed in split order, one division, attn_out / xq records.
// Scores are bit-identical to the single-CTA kernel's (same f64 operation order of each dot product, same f32 rounding and
// scale); only the order of the f64 sums of pass 2 differs (DESIGN section 2 contract 3: invisible up to 1e-16).  Split
// boundaries are a function of p only (attn_split_range), so results are deterministic; the launch shape depends only on
// max_ctx (graph-capturable).  No reader ever reads row p from the cache (the new k / v come from qkv), so the append in
// kernel A cannot race with the other CTAs.
// ------------------------------------------------------------------------------------------------
constexpr int ATT_SPLIT_NT = 256;       // threads per split CTA (kernels A and B)
constexpr int ATT_SPLIT_GC = 8;         // query heads per pass over a split's rows (G > 8 makes ceil(G / 8) passes)
constexpr int ATT_SPLIT_TILE = 64;      // kernel B: positions whose probabilities are staged in shared memory at a time

__host__ __device__ __forceinline__ int attn_split_max(int max_ctx) {
    const int s = (int)(((int64_t)max_ctx + ATTN_SPLIT_MIN - 1) / ATTN_SPLIT_MIN);
    return s < ATTN_SPLIT_CAP ? s : ATTN_SPLIT_CAP;
}
// split s of the positions [0, p]: S_eff = min(S_max, ceil((p + 1) / ATTN_SPLIT_MIN)) balanced ranges [j0, j1); s >= S_eff -> empty
__device__ __forceinline__ void attn_split_range(int p, int s_max, int s, int& j0, int& j1, int& s_eff) {
    const int64_t n = (int64_t)p + 1;
    const int64_t want = (n + ATTN_SPLIT_MIN - 1) / ATTN_SPLIT_MIN;
    s_eff = (int)(want < s_max ? want : s_max);
    if (s >= s_eff) { j0 = j1 = 0; return; }
    j0 = (int)((int64_t)s * n / s_eff);
    j1 = (int)((int64_t)(s + 1) * n / s_eff);
}

struct AttnSplitWs {
    float* scores;    // [M][nh][max_ctx]
    float* smax;      // [M][nh][S_max]
    double* psum;     // [M][nh][S_max]
    double* pv;       // [M][nh][S_max][hd]
};

// the position checks of attn_decode_kernel: the same clamped position ahead of the wait, and the same verdict in all three kernels
template <bool PAGED>
__device__ __forceinline__ int attn_checked_pos(const int* pos, int m, int max_ctx, const PagedKv& pg, bool& bad_pos) {
    const int p_raw = pos[m];
    bad_pos = p_raw < 0 || p_raw >= max_ctx;
    if constexpr (PAGED) {
        if (pg.slot_mapping && pg.slot_mapping[m] < 0) bad_pos = true;
    }
    return bad_pos ? 0 : p_raw;
}

template <int HD, bool PAGED, typename T>
__global__ void __launch_bounds__(ATT_SPLIT_NT) attn_split_scores_kernel(const float* __restrict__ qkv, const int* __restrict__ pos, T* __restrict__ cache_k,
                                                                       T* __restrict__ cache_v, const float* __restrict__ rope, int nh, int nkv, int max_ctx,
                                                                       const PagedKv pg, const AttnSplitWs ws) {
    pdl_launch_dependents();
    const int kvh = blockIdx.x, m = blockIdx.y, s = blockIdx.z, t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int G = nh / nkv, s_max = gridDim.z;
    constexpr int QE = HD / 4;          // elements per thread: 4 threads per position, a quarter of the head each
    constexpr int QP = QE + 2;          // padded quarter (doubles): the 4 quarters of a query fall in different banks
    constexpr int NW = ATT_SPLIT_NT / 32;
    bool bad_pos;
    const int p = attn_checked_pos<PAGED>(pos, m, max_ctx, pg, bad_pos);
    int j0, j1, s_eff;
    attn_split_range(p, s_max, s, j0, j1, s_eff);
    const int row = (nh + 2 * nkv) * HD;
    const float* ksrc = qkv + (size_t)m * row + (size_t)(nh + kvh) * HD;
    const float* vsrc = qkv + (size_t)m * row + (size_t)(nh + nkv + kvh) * HD;
    const size_t pstride = (size_t)nkv * HD;
    const int* bt = PAGED ? pg.block_table + (size_t)m * pg.max_blocks : nullptr;
    auto row_of = [&](int j) -> size_t {
        if constexpr (PAGED) return ((size_t)bt[j / pg.block_size] * pg.block_size + (size_t)(j % pg.block_size)) * pstride + (size_t)kvh * HD;
        else return ((size_t)m * max_ctx + (size_t)j) * pstride + (size_t)kvh * HD;
    };
    const float* rt = rope + (size_t)p * HD;
    constexpr int KL = KV_LINE<T>;      // elements per 16-byte load
    __shared__ __align__(16) double sq[ATT_SPLIT_GC][4][QP];
    __shared__ __align__(16) T sk[HD];  // the new key as the cache stores it
    __shared__ float s_red[NW][ATT_SPLIT_GC];
    pdl_wait();
    if (bad_pos) {
        if (t == 0 && s == 0 && kvh == 0) atomicOr(&g_decode_error, B200Q_DECODE_ERR_POSITION);
        return;
    }
    if (s >= s_eff) return;
    const bool owns_p = j1 == p + 1;
    if (t < HD / 2) {   // the new key, rotated exactly as attn_decode_kernel does (it is scored from here, never from the cache)
        const float c = rt[2 * t], sn = rt[2 * t + 1];
        const float k0 = ksrc[2 * t], k1 = ksrc[2 * t + 1];
        const T r0 = kv_store_val<T>(__fsub_rn(__fmul_rn(k0, c), __fmul_rn(k1, sn))), r1 = kv_store_val<T>(__fadd_rn(__fmul_rn(k0, sn), __fmul_rn(k1, c)));
        sk[2 * t] = r0; sk[2 * t + 1] = r1;
        if (owns_p) {
            size_t wrow = row_of(p);
            if constexpr (PAGED) {
                if (pg.slot_mapping) wrow = (size_t)pg.slot_mapping[m] * pstride + (size_t)kvh * HD;
            }
            cache_k[wrow + 2 * t] = r0; cache_k[wrow + 2 * t + 1] = r1;
            cache_v[wrow + 2 * t] = kv_store_val<T>(vsrc[2 * t]); cache_v[wrow + 2 * t + 1] = kv_store_val<T>(vsrc[2 * t + 1]);
        }
    }
    const float scale = __fdiv_rn(1.0f, __fsqrt_rn((float)HD));
    const int part = t & 3;
    for (int g0 = 0; g0 < G; g0 += ATT_SPLIT_GC) {
        const int gc = min(ATT_SPLIT_GC, G - g0);
        __syncthreads();   // sk is written / the previous pass is done with sq and s_red
        for (int i = t; i < gc * (HD / 2); i += ATT_SPLIT_NT) {
            const int g = i / (HD / 2), e2 = 2 * (i % (HD / 2));
            const float* qsrc = qkv + (size_t)m * row + (size_t)(kvh * G + g0 + g) * HD;
            const float c = rt[e2], sn = rt[e2 + 1];
            const float q0 = qsrc[e2], q1 = qsrc[e2 + 1];
            sq[g][e2 / QE][e2 % QE] = (double)__fsub_rn(__fmul_rn(q0, c), __fmul_rn(q1, sn));
            sq[g][e2 / QE][e2 % QE + 1] = (double)__fadd_rn(__fmul_rn(q0, sn), __fmul_rn(q1, c));
        }
        __syncthreads();
        float lmax[ATT_SPLIT_GC];
#pragma unroll
        for (int g = 0; g < ATT_SPLIT_GC; g++) lmax[g] = -INFINITY;
        float* sc_out = ws.scores + ((size_t)m * nh + (size_t)kvh * G + g0) * (size_t)max_ctx;
        // 4 threads per position; a warp's 8 positions are processed together (the shuffles need the whole warp)
        for (int jb = j0; jb < j1; jb += ATT_SPLIT_NT / 4) {
            const int j = jb + (t >> 2);
            const bool live = j < j1;
            double kd[QE];
            if (live) {
                const T* kr = (j < p) ? cache_k + row_of(j) + part * QE : sk + part * QE;
                if constexpr (std::is_same_v<T, float>) {
#pragma unroll
                    for (int e = 0; e < QE; e += 4) {
                        const float4 kk = *reinterpret_cast<const float4*>(kr + e);
                        kd[e] = (double)kk.x; kd[e + 1] = (double)kk.y; kd[e + 2] = (double)kk.z; kd[e + 3] = (double)kk.w;
                    }
                } else {   // 8 halves per 16-byte load
#pragma unroll
                    for (int e = 0; e < QE; e += KL) {
                        float kk[KL];
                        kv_widen(kv_ld_line(kr + e), kk);
#pragma unroll
                        for (int i = 0; i < KL; i++) kd[e + i] = (double)kk[i];
                    }
                }
            } else {
#pragma unroll
                for (int e = 0; e < QE; e++) kd[e] = 0.0;
            }
#pragma unroll
            for (int g = 0; g < ATT_SPLIT_GC; g++) {
                if (g < gc) {
                    // attn_decode_kernel's operation order: 4 fma chains over e mod 4, (d0+d1)+(d2+d3), then (P0+P1)+(P2+P3)
                    const double* qq = sq[g][part];
                    double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
#pragma unroll
                    for (int e = 0; e < QE; e += 4) {
                        d0 = fma(qq[e + 0], kd[e + 0], d0); d1 = fma(qq[e + 1], kd[e + 1], d1);
                        d2 = fma(qq[e + 2], kd[e + 2], d2); d3 = fma(qq[e + 3], kd[e + 3], d3);
                    }
                    double d = (d0 + d1) + (d2 + d3);
                    d += __shfl_xor_sync(0xffffffffu, d, 1);
                    d += __shfl_xor_sync(0xffffffffu, d, 2);
                    if (live) {
                        const float sc = __fmul_rn((float)d, scale);
                        if (part == (g & 3)) sc_out[(size_t)g * max_ctx + j] = sc;
                        lmax[g] = fmaxf(lmax[g], sc);
                    }
                }
            }
        }
#pragma unroll
        for (int g = 0; g < ATT_SPLIT_GC; g++) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) lmax[g] = fmaxf(lmax[g], __shfl_xor_sync(0xffffffffu, lmax[g], off));
            if (lane == 0) s_red[warp][g] = lmax[g];
        }
        __syncthreads();
        if (t < gc) {
            float mx = s_red[0][t];
#pragma unroll
            for (int w = 1; w < NW; w++) mx = fmaxf(mx, s_red[w][t]);
            ws.smax[((size_t)m * nh + (size_t)kvh * G + g0 + t) * s_max + s] = mx;
        }
    }
}

template <int HD, bool PAGED, typename T>
__global__ void __launch_bounds__(ATT_SPLIT_NT) attn_split_pv_kernel(const float* __restrict__ qkv, const int* __restrict__ pos, const T* __restrict__ cache_v,
                                                                   int nh, int nkv, int max_ctx, const PagedKv pg, const AttnSplitWs ws) {
    pdl_launch_dependents();
    const int kvh = blockIdx.x, m = blockIdx.y, s = blockIdx.z, t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int G = nh / nkv, s_max = gridDim.z;
    constexpr int EG = HD / 4;                 // element groups of 4 (one float4 of a V row)
    constexpr int JG = ATT_SPLIT_NT / EG;      // position lanes: 8 for hd 128, 16 for hd 64 (adjacent lanes of a warp)
    constexpr int NW = ATT_SPLIT_NT / 32;
    const int jg = t % JG, eg = t / JG;
    bool bad_pos;
    const int p = attn_checked_pos<PAGED>(pos, m, max_ctx, pg, bad_pos);
    int j0, j1, s_eff;
    attn_split_range(p, s_max, s, j0, j1, s_eff);
    const int row = (nh + 2 * nkv) * HD;
    const float* vsrc = qkv + (size_t)m * row + (size_t)(nh + nkv + kvh) * HD;
    const size_t pstride = (size_t)nkv * HD;
    const int* bt = PAGED ? pg.block_table + (size_t)m * pg.max_blocks : nullptr;
    auto row_of = [&](int j) -> size_t {
        if constexpr (PAGED) return ((size_t)bt[j / pg.block_size] * pg.block_size + (size_t)(j % pg.block_size)) * pstride + (size_t)kvh * HD;
        else return ((size_t)m * max_ctx + (size_t)j) * pstride + (size_t)kvh * HD;
    };
    __shared__ float sp[ATT_SPLIT_GC][ATT_SPLIT_TILE];
    __shared__ float gmax[ATT_SPLIT_GC];
    __shared__ __align__(16) T sv[HD];   // the new value as the cache stores it
    __shared__ double s_red[2][NW];
    pdl_wait();
    if (bad_pos || s >= s_eff) return;
    for (int i = t; i < HD; i += ATT_SPLIT_NT) sv[i] = kv_store_val<T>(vsrc[i]);
    for (int g0 = 0; g0 < G; g0 += ATT_SPLIT_GC) {
        const int gc = min(ATT_SPLIT_GC, G - g0);
        const size_t hrow = (size_t)m * nh + (size_t)kvh * G + g0;   // first (m, head) row of this pass
        __syncthreads();
        if (t < gc) {
            const float* sm = ws.smax + (hrow + t) * s_max;
            float mx = sm[0];
            for (int i = 1; i < s_eff; i++) mx = fmaxf(mx, sm[i]);
            gmax[t] = mx;
        }
        double o[ATT_SPLIT_GC][4];
#pragma unroll
        for (int g = 0; g < ATT_SPLIT_GC; g++) o[g][0] = o[g][1] = o[g][2] = o[g][3] = 0.0;
        double ls0 = 0.0, ls1 = 0.0;   // sum of p of heads t / 64 and 4 + t / 64
        for (int jt = j0; jt < j1; jt += ATT_SPLIT_TILE) {
            __syncthreads();   // gmax ready / the previous tile's probabilities are consumed
            {
                const int jj = t % ATT_SPLIT_TILE, g = t / ATT_SPLIT_TILE, j = jt + jj;
                static_assert(ATT_SPLIT_NT == 4 * ATT_SPLIT_TILE && ATT_SPLIT_GC == 8, "two probabilities per thread");
                float pa = 0.0f, pb = 0.0f;
                if (j < j1) {
                    if (g < gc) pa = det_expf(__fsub_rn(ws.scores[(hrow + g) * max_ctx + j], gmax[g]));
                    if (g + 4 < gc) pb = det_expf(__fsub_rn(ws.scores[(hrow + g + 4) * max_ctx + j], gmax[g + 4]));
                }
                sp[g][jj] = pa; sp[g + 4][jj] = pb;
                ls0 += (double)pa; ls1 += (double)pb;
            }
            __syncthreads();
            const int jn = min(ATT_SPLIT_TILE, j1 - jt);
            for (int jj = jg; jj < jn; jj += JG) {
                const int j = jt + jj;
                const float4 vv = (j < p) ? kv_ld4(cache_v + row_of(j) + 4 * eg) : kv_ld4(sv + 4 * eg);
#pragma unroll
                for (int g = 0; g < ATT_SPLIT_GC; g++) {
                    const double pj = (double)sp[g][jj];
                    o[g][0] = fma(pj, (double)vv.x, o[g][0]); o[g][1] = fma(pj, (double)vv.y, o[g][1]);
                    o[g][2] = fma(pj, (double)vv.z, o[g][2]); o[g][3] = fma(pj, (double)vv.w, o[g][3]);
                }
            }
        }
        // the JG position lanes of an element group are adjacent lanes of one warp
#pragma unroll
        for (int g = 0; g < ATT_SPLIT_GC; g++)
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int off = 1; off < JG; off <<= 1) o[g][i] += __shfl_xor_sync(0xffffffffu, o[g][i], off);
        if (jg == 0) {
#pragma unroll
            for (int g = 0; g < ATT_SPLIT_GC; g++)
                if (g < gc) {
                    double* dst = ws.pv + ((hrow + g) * s_max + s) * HD + 4 * eg;
                    dst[0] = o[g][0]; dst[1] = o[g][1]; dst[2] = o[g][2]; dst[3] = o[g][3];
                }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            ls0 += __shfl_xor_sync(0xffffffffu, ls0, off);
            ls1 += __shfl_xor_sync(0xffffffffu, ls1, off);
        }
        if (lane == 0) { s_red[0][warp] = ls0; s_red[1][warp] = ls1; }
        __syncthreads();
        if (t < gc) {   // warps 2 h and 2 h + 1 hold head h (h < 4) in s_red[0] and head h + 4 in s_red[1]
            const int hb = t & 3, k = t >> 2;
            ws.psum[(hrow + t) * s_max + s] = s_red[k][2 * hb] + s_red[k][2 * hb + 1];
        }
    }
}

template <int HD, bool PAGED>
__global__ void __launch_bounds__(HD) attn_split_combine_kernel(const int* __restrict__ pos, int nh, int max_ctx, int s_max, int M, const PagedKv pg,
                                                               const AttnSplitWs ws, uint8_t* __restrict__ xq, float* __restrict__ attn_out) {
    pdl_launch_dependents();
    const int head = blockIdx.x, m = blockIdx.y, t = threadIdx.x, lane = t & 31;
    bool bad_pos;
    const int p = attn_checked_pos<PAGED>(pos, m, max_ctx, pg, bad_pos);
    int j0, j1, s_eff;
    attn_split_range(p, s_max, 0, j0, j1, s_eff);
    pdl_wait();
    if (bad_pos) return;
    const size_t hrow = (size_t)m * nh + head;
    double o = 0.0, dsum = 0.0;
    const double* pv = ws.pv + hrow * s_max * HD + t;
    const double* ps = ws.psum + hrow * s_max;
#pragma unroll 8
    for (int i = 0; i < s_eff; i++) {   // split order
        o += pv[(size_t)i * HD];
        dsum += ps[i];
    }
    const float outv = __fdiv_rn((float)o, (float)dsum);
    if (attn_out) attn_out[(size_t)m * nh * HD + (size_t)head * HD + t] = outv;
    if (!xq) return;
    // the o_proj activation records, quantised as attn_decode_kernel does (32-blocks never straddle heads)
    const int kglob = head * HD + t;
    const int kc = kglob / CHUNK_K, tin = kglob % CHUNK_K;
    uint8_t* rec = xq + ((size_t)kc * M + m) * ACT_REC_BYTES;
    float amax = fabsf(outv);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, off));
    const float d = __fdiv_rn(amax, 127.0f);
    const float id = (d != 0.0f) ? __fdiv_rn(1.0f, d) : 0.0f;
    const int q = (int)roundf(__fmul_rn(outv, id));
    int sm = q;
#pragma unroll
    for (int off = 8; off > 0; off >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, off);
    const int s_hi = __shfl_sync(0xffffffffu, sm, 16);
    rec[tin] = (uint8_t)(int8_t)q;
    if (lane == 0) {
        reinterpret_cast<float*>(rec + 256)[tin >> 5] = d;
        reinterpret_cast<uint32_t*>(rec + 288)[tin >> 5] = ((uint32_t)sm & 0xFFFFu) | ((uint32_t)s_hi << 16);
    }
}

// workspace regions, each 256-byte aligned; returns the total (0 for arguments no split kernel accepts)
static size_t attn_split_layout(int64_t nh, int64_t hd, int64_t max_ctx, int64_t M, uint8_t* base, AttnSplitWs* ws) {
    if (nh <= 0 || max_ctx <= 0 || M <= 0 || (hd != 64 && hd != 128)) return 0;
    const size_t smax = (size_t)attn_split_max((int)max_ctx);
    const size_t rows = (size_t)M * (size_t)nh;
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t b_sc = al(rows * (size_t)max_ctx * 4), b_mx = al(rows * smax * 4), b_ps = al(rows * smax * 8), b_pv = al(rows * smax * (size_t)hd * 8);
    if (ws) {
        ws->scores = reinterpret_cast<float*>(base);
        ws->smax = reinterpret_cast<float*>(base + b_sc);
        ws->psum = reinterpret_cast<double*>(base + b_sc + b_mx);
        ws->pv = reinterpret_cast<double*>(base + b_sc + b_mx + b_ps);
    }
    return b_sc + b_mx + b_ps + b_pv;
}

template <int HD, bool PAGED, typename T>
static cudaError_t launch_attn_split(const float* qkv, const int* pos, T* ck, T* cv, const float* rope, int nh, int nkv, int max_ctx, int M,
                                     uint8_t* xq, float* attn_out, const PagedKv& pg, const AttnSplitWs& ws, cudaStream_t st) {
    const int s_max = attn_split_max(max_ctx);
    const dim3 grid((unsigned)nkv, (unsigned)M, (unsigned)s_max);
    cudaError_t e = launch_pdl(attn_split_scores_kernel<HD, PAGED, T>, grid, dim3(ATT_SPLIT_NT), 0, st, qkv, pos, ck, cv, rope, nh, nkv, max_ctx, pg, ws);
    if (e == cudaSuccess)
        e = launch_pdl(attn_split_pv_kernel<HD, PAGED, T>, grid, dim3(ATT_SPLIT_NT), 0, st, qkv, pos, (const T*)cv, nh, nkv, max_ctx, pg, ws);
    if (e == cudaSuccess)
        e = launch_pdl(attn_split_combine_kernel<HD, PAGED>, dim3((unsigned)nh, (unsigned)M), dim3(HD), 0, st, pos, nh, max_ctx, s_max, M, pg, ws, xq, attn_out);
    return e;
}

template <int HD, bool PAGED, typename T>
static cudaError_t launch_attn_single(const float* qkv, const int* pos, T* ck, T* cv, const float* rope, int nh, int nkv, int max_ctx, int M,
                                      uint8_t* xq, float* attn_out, const PagedKv& pg, cudaStream_t st) {
    const size_t smem = (size_t)max_ctx * sizeof(float);
    if (smem > 48 * 1024) cudaFuncSetAttribute(attn_decode_kernel<HD, PAGED, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    return launch_pdl(attn_decode_kernel<HD, PAGED, T>, dim3((unsigned)nh, (unsigned)M), dim3(ATT_NT), smem, st, qkv, pos, ck, cv, rope, nh, nkv, max_ctx, M,
                      xq, attn_out, pg);
}

template <typename T>
static cudaError_t launch_attn_split_hd(int32_t hd, const float* qkv, const int32_t* pos, T* ck, T* cv, const float* rope, int32_t nh, int32_t nkv,
                                        int max_ctx, int M, uint8_t* xq, float* attn_out, const PagedKv& pg, const AttnSplitWs& ws, cudaStream_t st) {
    const bool paged = pg.block_table != nullptr;
    if (hd == 128)
        return paged ? launch_attn_split<128, true>(qkv, pos, ck, cv, rope, nh, nkv, max_ctx, M, xq, attn_out, pg, ws, st)
                     : launch_attn_split<128, false>(qkv, pos, ck, cv, rope, nh, nkv, max_ctx, M, xq, attn_out, pg, ws, st);
    return paged ? launch_attn_split<64, true>(qkv, pos, ck, cv, rope, nh, nkv, max_ctx, M, xq, attn_out, pg, ws, st)
                 : launch_attn_split<64, false>(qkv, pos, ck, cv, rope, nh, nkv, max_ctx, M, xq, attn_out, pg, ws, st);
}

// ------------------------------------------------------------------------------------------------
// greedy sampling: argmax over the vocabulary, lowest index wins ties.  One CTA of 1024 threads per row.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) argmax_kernel(const float* __restrict__ logits, int V, int64_t* __restrict__ out, int* __restrict__ pos_inc) {
    pdl_launch_dependents();
    pdl_wait();
    const int m = blockIdx.x, t = threadIdx.x;
    const float* row = logits + (size_t)m * V;
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = t; i < V; i += 1024) {
        const float v = row[i];
        if (v > best || (v == best && i < bi)) { best = v; bi = i; }
    }
    __shared__ float sv[32];
    __shared__ int si[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    if ((t & 31) == 0) { sv[t >> 5] = best; si[t >> 5] = bi; }
    __syncthreads();
    if (t < 32) {
        best = sv[t]; bi = si[t];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if (t == 0) {
            out[m] = bi;
            if (pos_inc) pos_inc[m] += 1;  // advance the sequence position for the next graph replay
        }
    }
}

// Consumer of the fused lm_head all-gather (comm_dev.cuh): rank r's logits for row m live at gather[r][m * vs + j] and are
// vocabulary id r * vs + j (columns no rank wrote stay -inf).  Waits for every rank's flag, then the same arg-max.
__global__ void __launch_bounds__(1024) argmax_gathered_kernel(const CommDev c, int vs, int M, int64_t* __restrict__ out, int* __restrict__ pos_inc) {
    pdl_launch_dependents();
    pdl_wait();
    const int m = blockIdx.x, t = threadIdx.x;
    const uint8_t* mine = c.peers[c.rank];
    const unsigned int epoch = __ldcg(reinterpret_cast<const unsigned int*>(mine + COMM_OFF_AG_EPOCH));
    comm_wait_flags(c, COMM_OFF_AG_FLAGS, 0, epoch, t);
    __syncthreads();
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int r = 0; r < c.world; r++) {
        const float* row = reinterpret_cast<const float*>(mine + comm_ag_off(c, r)) + (size_t)m * vs;
        for (int j = t; j < vs; j += 1024) {
            const float v = __ldcg(row + j);
            const int i = r * vs + j;
            if (v > best || (v == best && i < bi)) { best = v; bi = i; }
        }
    }
    __shared__ float sv[32];
    __shared__ int si[32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    if ((t & 31) == 0) { sv[t >> 5] = best; si[t >> 5] = bi; }
    __syncthreads();
    if (t < 32) {
        best = sv[t]; bi = si[t];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if (t == 0) {
            out[m] = bi;
            if (pos_inc) pos_inc[m] += 1;
        }
    }
}

// MoE combine: out[t, h] = sum_j gate_w[t, j] * y[t * top_k + j, h], j ascending, separate f32 multiply and add (no FMA): the
// order is part of the contract so the expert-parallel partial sums of different ranks are reproducible.
__global__ void __launch_bounds__(256) moe_combine_kernel(const float* __restrict__ y, const float* __restrict__ gate_w, int top_k, int H, float* __restrict__ out) {
    pdl_launch_dependents();
    pdl_wait();
    const int t = blockIdx.y;
    const int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= H) return;
    float acc = 0.0f;
    for (int j = 0; j < top_k; j++) acc = __fadd_rn(acc, __fmul_rn(gate_w[(size_t)t * top_k + j], y[((size_t)t * top_k + j) * H + h]));
    out[(size_t)t * H + h] = acc;
}

// embedding gather: h[m, :] = table[ids[m], :] (f16 table -> f32)
// First kernel of a decode step: it releases its dependents only AFTER its own dependency wait, which breaks the
// programmatic chain at the step boundary -- nothing of step s+1 (in particular the attention prologue, which reads
// pos[] ahead of its wait) can start before step s's argmax has advanced pos[] and written the token ids.
__global__ void embed_kernel(const __half* __restrict__ table, const int64_t* __restrict__ ids, int H, float* __restrict__ h) {
    pdl_wait();
    pdl_launch_dependents();
    const int m = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < H) h[(size_t)m * H + k] = __half2float(table[(size_t)ids[m] * H + k]);
}

}  // namespace b200q

using namespace b200q;

extern "C" {

static cudaError_t launch_norm_cluster(const CommDev& c, const float* h_in, const float* delta, float* h_out, const float* w, float eps, int64_t H, int64_t M,
                                       void* xq, float* xnorm, cudaStream_t st) {
    const unsigned ncta = (unsigned)((H + NORMC_NT - 1) / NORMC_NT);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(ncta, (unsigned)M);
    cfg.blockDim = dim3(NORMC_NT);
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = ncta;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    cudaError_t e = cudaLaunchKernelEx(&cfg, add_rmsnorm_quant_cluster_kernel, (const CommDev)c, h_in, delta, h_out, w, eps, (int)H, (int)M, (uint8_t*)xq, xnorm);
    count_launch();
    return e;
}

int32_t b200q_add_rmsnorm_quant(const float* h_in, const float* delta, float* h_out, const float* w, float eps, int64_t H, int64_t M, void* xq,
                                float* xnorm, void* stream) {
    if (!h_in || !h_out || !w || (!xq && !xnorm) || H <= 0 || H % CHUNK_K || M <= 0) return B200Q_ERR_INVALID_ARG;
    if (delta && h_in == h_out) return B200Q_ERR_INVALID_ARG;  // CTAs re-read the whole input row: no in-place update
    // measured (round 2, Mistral-7B / Llama-3.2-1B steps): without an exchange to consume, the H/256-CTA kernel (every CTA
    // re-reads the L2-resident row) beats the cluster form by ~1.3 us per call -- two cluster barriers cost more than the
    // redundant reads.  The cluster kernel is the tensor-parallel consumer (reading `world` slots per CTA would not scale);
    // B200Q_NORM_CLUSTER=1 forces it here for A/B runs.
    static const bool use_cluster = [] { const char* e_ = getenv("B200Q_NORM_CLUSTER"); return e_ && atoi(e_) != 0; }();
    if (H <= 8 * NORMC_NT && use_cluster) {
        cudaError_t e = launch_norm_cluster(CommDev{}, h_in, delta, h_out, w, eps, H, M, xq, xnorm, (cudaStream_t)stream);
        return e == cudaSuccess ? B200Q_OK : B200Q_ERR_CUDA;
    }
    cudaError_t e = launch_pdl(add_rmsnorm_quant_kernel, dim3((unsigned)(H / CHUNK_K), (unsigned)M), dim3(NORM_NT), 0, (cudaStream_t)stream, h_in, delta,
                               h_out, w, eps, (int)H, (int)M, (uint8_t*)xq, xnorm);
    return e == cudaSuccess ? B200Q_OK : B200Q_ERR_CUDA;
}

/* Consumer of b200q_matmul_q8_rowpar: h_out = h_in + allreduce(partials); xq = quant(rmsnorm(h_out) * w); the reduced
 * delta is summed in rank order from the communicator's slots (identical bits on every rank, equal to the 1-GPU sum). */
int32_t b200q_allreduce_add_rmsnorm_quant(b200q_comm* comm, const float* h_in, float* h_out, const float* w, float eps, int64_t H, int64_t M, void* xq,
                                          float* xnorm, void* stream) {
    if (!comm || !h_in || !h_out || !w || (!xq && !xnorm) || H <= 0 || H % CHUNK_K || M <= 0) return set_error(B200Q_ERR_INVALID_ARG, "allreduce_add_rmsnorm_quant: bad arguments");
    if (H > 8 * NORMC_NT) return set_error(B200Q_ERR_UNSUPPORTED, "allreduce_add_rmsnorm_quant: H = %lld > %d", (long long)H, 8 * NORMC_NT);
    if (M * H > comm_slot_elems(comm)) return set_error(B200Q_ERR_INVALID_ARG, "allreduce_add_rmsnorm_quant: M * H = %lld exceeds the communicator's slot capacity %lld", (long long)(M * H), (long long)comm_slot_elems(comm));
    CommDev c;
    if (!comm_dev(comm, &c)) return set_error(B200Q_ERR_INVALID_ARG, "allreduce_add_rmsnorm_quant: communicator not connected");
    cudaError_t e = launch_norm_cluster(c, h_in, nullptr, h_out, w, eps, H, M, xq, xnorm, (cudaStream_t)stream);
    return e == cudaSuccess ? B200Q_OK : set_error(B200Q_ERR_CUDA, "allreduce_add_rmsnorm_quant launch: %s", cudaGetErrorString(e));
}

/* Consumer of b200q_matmul_q8_gather: greedy token over the gathered [world][M][vs] logits */
int32_t b200q_argmax_gathered(b200q_comm* comm, int64_t vs, int64_t M, int64_t* out_ids, int32_t* pos_inc, void* stream) {
    if (!comm || !out_ids || vs <= 0 || M <= 0 || M * vs > comm_gather_elems(comm)) return set_error(B200Q_ERR_INVALID_ARG, "argmax_gathered: bad arguments");
    CommDev c;
    if (!comm_dev(comm, &c)) return set_error(B200Q_ERR_INVALID_ARG, "argmax_gathered: communicator not connected");
    cudaError_t e = launch_pdl(argmax_gathered_kernel, dim3((unsigned)M), dim3(1024), 0, (cudaStream_t)stream, (const CommDev)c, (int)vs, (int)M, out_ids, (int*)pos_inc);
    return e == cudaSuccess ? B200Q_OK : set_error(B200Q_ERR_CUDA, "argmax_gathered launch: %s", cudaGetErrorString(e));
}

int32_t b200q_swiglu_quant(const float* gate_up, int64_t F, int64_t M, void* xq, void* stream) {
    if (!gate_up || !xq || F <= 0 || F % 32 || M <= 0 || M > 65535) return B200Q_ERR_INVALID_ARG;
    cudaError_t e = launch_pdl(swiglu_quant_kernel, dim3((unsigned)((F + CHUNK_K - 1) / CHUNK_K), (unsigned)M), dim3(256), 0, (cudaStream_t)stream, gate_up, (int)F,
                               (int)M, (uint8_t*)xq, (float*)nullptr, 0);
    return e == cudaSuccess ? B200Q_OK : B200Q_ERR_CUDA;
}

/* batched decode (M > 4: the projections run on the tcgen05 path and take f32 activations): act[M, F] = silu(gate) * up */
int32_t b200q_swiglu_f32(const float* gate_up, int64_t F, int64_t M, float* act, void* stream) {
    if (!gate_up || !act || F <= 0 || F % 32 || M <= 0 || M > 65535) return B200Q_ERR_INVALID_ARG;
    cudaError_t e = launch_pdl(swiglu_quant_kernel, dim3((unsigned)((F + CHUNK_K - 1) / CHUNK_K), (unsigned)M), dim3(256), 0, (cudaStream_t)stream, gate_up, (int)F,
                               (int)M, (uint8_t*)nullptr, act, 0);
    return e == cudaSuccess ? B200Q_OK : B200Q_ERR_CUDA;
}

/* same for a gate|up output whose columns are in the SwiGLU-epilogue row order of the weight (b200q_gate_up_row): the M > 4
 * paths (prefill, batched decode) of a model whose gate|up weight is uploaded interleaved for the fused decode epilogue */
int32_t b200q_swiglu_f32_interleaved(const float* gate_up, int64_t F, int64_t M, float* act, void* stream) {
    if (!gate_up || !act || F <= 0 || F % 64 || M <= 0 || M > 65535) return B200Q_ERR_INVALID_ARG;
    cudaError_t e = launch_pdl(swiglu_quant_kernel, dim3((unsigned)((F + CHUNK_K - 1) / CHUNK_K), (unsigned)M), dim3(256), 0, (cudaStream_t)stream, gate_up, (int)F,
                               (int)M, (uint8_t*)nullptr, act, 1);
    return e == cudaSuccess ? B200Q_OK : B200Q_ERR_CUDA;
}

// KV cache element type and alignment: every attention form vector-loads 16 bytes of a cache row (the row starts are 16-byte
// aligned for head_dim 64 / 128 in both dtypes, so the base pointers must be too)
static int32_t attn_kv_check(const void* ck, const void* cv, int32_t kv_dtype, const char* who) {
    if (kv_dtype != B200Q_F32 && kv_dtype != B200Q_F16) return set_error(B200Q_ERR_UNSUPPORTED, "%s: kv_dtype %d (B200Q_F32 or B200Q_F16)", who, (int)kv_dtype);
    if (((uintptr_t)ck | (uintptr_t)cv) & 15) return set_error(B200Q_ERR_INVALID_ARG, "%s: KV cache pointers must be 16-byte aligned", who);
    return B200Q_OK;
}

static int32_t attn_single_dispatch(const float* qkv, const int32_t* pos, void* ck, void* cv, int32_t kv_dtype, const float* rope, int32_t nh, int32_t nkv,
                                    int32_t hd, int64_t max_ctx, int64_t M, void* xq, float* attn_out, const PagedKv& pg, void* stream, const char* who) {
    if (max_ctx > ATTN_SINGLE_MAX_CTX) return set_error(B200Q_ERR_UNSUPPORTED, "%s: max_ctx %lld > %d (use the split form)", who, (long long)max_ctx, ATTN_SINGLE_MAX_CTX);
    if (hd != 64 && hd != 128) return set_error(B200Q_ERR_UNSUPPORTED, "%s: head_dim %d (64 or 128)", who, (int)hd);
    const int32_t rc = attn_kv_check(ck, cv, kv_dtype, who);
    if (rc != B200Q_OK) return rc;
    const cudaStream_t st = (cudaStream_t)stream;
    const bool paged = pg.block_table != nullptr;
    const int mc = (int)max_ctx, m = (int)M;
    uint8_t* x = (uint8_t*)xq;
    cudaError_t e;
    if (kv_dtype == B200Q_F16) {
        __half* k = (__half*)ck;
        __half* v = (__half*)cv;
        if (hd == 128)
            e = paged ? launch_attn_single<128, true>(qkv, pos, k, v, rope, nh, nkv, mc, m, x, attn_out, pg, st)
                      : launch_attn_single<128, false>(qkv, pos, k, v, rope, nh, nkv, mc, m, x, attn_out, pg, st);
        else
            e = paged ? launch_attn_single<64, true>(qkv, pos, k, v, rope, nh, nkv, mc, m, x, attn_out, pg, st)
                      : launch_attn_single<64, false>(qkv, pos, k, v, rope, nh, nkv, mc, m, x, attn_out, pg, st);
    } else {
        float* k = (float*)ck;
        float* v = (float*)cv;
        if (hd == 128)
            e = paged ? launch_attn_single<128, true>(qkv, pos, k, v, rope, nh, nkv, mc, m, x, attn_out, pg, st)
                      : launch_attn_single<128, false>(qkv, pos, k, v, rope, nh, nkv, mc, m, x, attn_out, pg, st);
        else
            e = paged ? launch_attn_single<64, true>(qkv, pos, k, v, rope, nh, nkv, mc, m, x, attn_out, pg, st)
                      : launch_attn_single<64, false>(qkv, pos, k, v, rope, nh, nkv, mc, m, x, attn_out, pg, st);
    }
    return e == cudaSuccess ? B200Q_OK : set_error(B200Q_ERR_CUDA, "%s launch: %s", who, cudaGetErrorString(e));
}

int32_t b200q_attn_decode_kv(const float* qkv, const int32_t* pos, void* cache_k, void* cache_v, int32_t kv_dtype, const float* rope_table, int32_t n_heads,
                             int32_t n_kv_heads, int32_t head_dim, int32_t max_ctx, int64_t M, void* xq, float* attn_out, void* stream) {
    if (!qkv || !pos || !cache_k || !cache_v || !rope_table || (!xq && !attn_out) || n_heads <= 0 || n_kv_heads <= 0 || n_heads % n_kv_heads || M <= 0 || max_ctx <= 0)
        return set_error(B200Q_ERR_INVALID_ARG, "attn_decode: bad arguments");
    if (((int64_t)n_heads * head_dim) % CHUNK_K) return set_error(B200Q_ERR_INVALID_ARG, "attn_decode: n_heads * head_dim not a multiple of %d", CHUNK_K);
    const PagedKv none{nullptr, nullptr, 0, 0};
    return attn_single_dispatch(qkv, pos, cache_k, cache_v, kv_dtype, rope_table, n_heads, n_kv_heads, head_dim, max_ctx, M, xq, attn_out, none, stream,
                                "attn_decode");
}

int32_t b200q_attn_decode(const float* qkv, const int32_t* pos, float* cache_k, float* cache_v, const float* rope_table, int32_t n_heads,
                          int32_t n_kv_heads, int32_t head_dim, int32_t max_ctx, int64_t M, void* xq, float* attn_out, void* stream) {
    return b200q_attn_decode_kv(qkv, pos, cache_k, cache_v, B200Q_F32, rope_table, n_heads, n_kv_heads, head_dim, max_ctx, M, xq, attn_out, stream);
}

/* Paged form (reference forward_with_paged_kv_cache, src/engine/batch_decode.rs:115-147): k_pool / v_pool are
 * [num_blocks][block_size][nkv][hd] pools shared by all sequences, block_table int32 [M][max_blocks] (padding entries are
 * never read: only blocks below pos[m] / block_size are), slot_mapping int32 [M] = block * block_size + offset of the NEW
 * token (nullable: derived from block_table and pos).  pos[m] = sequence length - 1.  A slot of -1 or a position >=
 * max_blocks * block_size writes nothing and raises the sticky device error (b200q_decode_error). */
int32_t b200q_attn_decode_paged_kv(const float* qkv, const int32_t* pos, void* k_pool, void* v_pool, int32_t kv_dtype, const int32_t* block_table,
                                   const int32_t* slot_mapping, int32_t block_size, int32_t max_blocks, const float* rope_table, int32_t n_heads,
                                   int32_t n_kv_heads, int32_t head_dim, int64_t M, void* xq, float* attn_out, void* stream) {
    if (!qkv || !pos || !k_pool || !v_pool || !block_table || !rope_table || (!xq && !attn_out) || n_heads <= 0 || n_kv_heads <= 0 || n_heads % n_kv_heads || M <= 0 ||
        block_size <= 0 || max_blocks <= 0)
        return set_error(B200Q_ERR_INVALID_ARG, "attn_decode_paged: bad arguments");
    if (((int64_t)n_heads * head_dim) % CHUNK_K) return set_error(B200Q_ERR_INVALID_ARG, "attn_decode_paged: n_heads * head_dim not a multiple of %d", CHUNK_K);
    const PagedKv pg{block_table, slot_mapping, block_size, max_blocks};
    return attn_single_dispatch(qkv, pos, k_pool, v_pool, kv_dtype, rope_table, n_heads, n_kv_heads, head_dim, (int64_t)block_size * max_blocks, M, xq,
                                attn_out, pg, stream, "attn_decode_paged");
}

int32_t b200q_attn_decode_paged(const float* qkv, const int32_t* pos, float* k_pool, float* v_pool, const int32_t* block_table, const int32_t* slot_mapping,
                                int32_t block_size, int32_t max_blocks, const float* rope_table, int32_t n_heads, int32_t n_kv_heads, int32_t head_dim,
                                int64_t M, void* xq, float* attn_out, void* stream) {
    return b200q_attn_decode_paged_kv(qkv, pos, k_pool, v_pool, B200Q_F32, block_table, slot_mapping, block_size, max_blocks, rope_table, n_heads, n_kv_heads,
                                      head_dim, M, xq, attn_out, stream);
}

int32_t b200q_attn_decode_max_ctx(void) { return ATTN_SINGLE_MAX_CTX; }

size_t b200q_attn_split_workspace_bytes(int32_t n_heads, int32_t n_kv_heads, int32_t head_dim, int32_t max_ctx, int64_t M) {
    if (n_kv_heads <= 0 || n_heads % n_kv_heads) return 0;
    return attn_split_layout(n_heads, head_dim, max_ctx, M, nullptr, nullptr);
}

static int32_t attn_split_dispatch(const float* qkv, const int32_t* pos, void* ck, void* cv, int32_t kv_dtype, const float* rope, int32_t nh, int32_t nkv,
                                   int32_t hd, int64_t max_ctx, int64_t M, void* xq, float* attn_out, const PagedKv& pg, void* workspace,
                                   size_t workspace_bytes, void* stream, const char* who) {
    if (hd != 64 && hd != 128) return set_error(B200Q_ERR_UNSUPPORTED, "%s: head_dim %d (64 or 128)", who, (int)hd);
    if (max_ctx > INT32_MAX || M > 65535) return set_error(B200Q_ERR_INVALID_ARG, "%s: max_ctx %lld / M %lld out of range", who, (long long)max_ctx, (long long)M);
    const int32_t rc = attn_kv_check(ck, cv, kv_dtype, who);
    if (rc != B200Q_OK) return rc;
    AttnSplitWs ws;
    const size_t need = attn_split_layout(nh, hd, max_ctx, M, (uint8_t*)workspace, &ws);
    if (!workspace || workspace_bytes < need)
        return set_error(B200Q_ERR_WORKSPACE, "%s: workspace of %zu bytes, %zu needed (b200q_attn_split_workspace_bytes)", who, workspace_bytes, need);
    const cudaStream_t st = (cudaStream_t)stream;
    const cudaError_t e =
        kv_dtype == B200Q_F16
            ? launch_attn_split_hd(hd, qkv, pos, (__half*)ck, (__half*)cv, rope, nh, nkv, (int)max_ctx, (int)M, (uint8_t*)xq, attn_out, pg, ws, st)
            : launch_attn_split_hd(hd, qkv, pos, (float*)ck, (float*)cv, rope, nh, nkv, (int)max_ctx, (int)M, (uint8_t*)xq, attn_out, pg, ws, st);
    return e == cudaSuccess ? B200Q_OK : set_error(B200Q_ERR_CUDA, "%s launch: %s", who, cudaGetErrorString(e));
}

/* Split-context form of b200q_attn_decode_kv for any max_ctx >= 1 (same arguments, same results up to the order of the f64 sums). */
int32_t b200q_attn_decode_split_kv(const float* qkv, const int32_t* pos, void* cache_k, void* cache_v, int32_t kv_dtype, const float* rope_table,
                                   int32_t n_heads, int32_t n_kv_heads, int32_t head_dim, int32_t max_ctx, int64_t M, void* xq, float* attn_out,
                                   void* workspace, size_t workspace_bytes, void* stream) {
    if (!qkv || !pos || !cache_k || !cache_v || !rope_table || (!xq && !attn_out) || n_heads <= 0 || n_kv_heads <= 0 || n_heads % n_kv_heads || M <= 0 || max_ctx <= 0)
        return set_error(B200Q_ERR_INVALID_ARG, "attn_decode_split: bad arguments");
    if (((int64_t)n_heads * head_dim) % CHUNK_K) return set_error(B200Q_ERR_INVALID_ARG, "attn_decode_split: n_heads * head_dim not a multiple of %d", CHUNK_K);
    const PagedKv none{nullptr, nullptr, 0, 0};
    return attn_split_dispatch(qkv, pos, cache_k, cache_v, kv_dtype, rope_table, n_heads, n_kv_heads, head_dim, max_ctx, M, xq, attn_out, none, workspace,
                               workspace_bytes, stream, "attn_decode_split");
}

int32_t b200q_attn_decode_split(const float* qkv, const int32_t* pos, float* cache_k, float* cache_v, const float* rope_table, int32_t n_heads,
                                int32_t n_kv_heads, int32_t head_dim, int32_t max_ctx, int64_t M, void* xq, float* attn_out, void* workspace,
                                size_t workspace_bytes, void* stream) {
    return b200q_attn_decode_split_kv(qkv, pos, cache_k, cache_v, B200Q_F32, rope_table, n_heads, n_kv_heads, head_dim, max_ctx, M, xq, attn_out, workspace,
                                      workspace_bytes, stream);
}

/* Split-context form of b200q_attn_decode_paged_kv; max_ctx = block_size * max_blocks sizes the workspace. */
int32_t b200q_attn_decode_paged_split_kv(const float* qkv, const int32_t* pos, void* k_pool, void* v_pool, int32_t kv_dtype, const int32_t* block_table,
                                         const int32_t* slot_mapping, int32_t block_size, int32_t max_blocks, const float* rope_table, int32_t n_heads,
                                         int32_t n_kv_heads, int32_t head_dim, int64_t M, void* xq, float* attn_out, void* workspace, size_t workspace_bytes,
                                         void* stream) {
    if (!qkv || !pos || !k_pool || !v_pool || !block_table || !rope_table || (!xq && !attn_out) || n_heads <= 0 || n_kv_heads <= 0 || n_heads % n_kv_heads || M <= 0 ||
        block_size <= 0 || max_blocks <= 0)
        return set_error(B200Q_ERR_INVALID_ARG, "attn_decode_paged_split: bad arguments");
    if (((int64_t)n_heads * head_dim) % CHUNK_K) return set_error(B200Q_ERR_INVALID_ARG, "attn_decode_paged_split: n_heads * head_dim not a multiple of %d", CHUNK_K);
    const PagedKv pg{block_table, slot_mapping, block_size, max_blocks};
    return attn_split_dispatch(qkv, pos, k_pool, v_pool, kv_dtype, rope_table, n_heads, n_kv_heads, head_dim, (int64_t)block_size * max_blocks, M, xq, attn_out,
                               pg, workspace, workspace_bytes, stream, "attn_decode_paged_split");
}

int32_t b200q_attn_decode_paged_split(const float* qkv, const int32_t* pos, float* k_pool, float* v_pool, const int32_t* block_table, const int32_t* slot_mapping,
                                      int32_t block_size, int32_t max_blocks, const float* rope_table, int32_t n_heads, int32_t n_kv_heads, int32_t head_dim,
                                      int64_t M, void* xq, float* attn_out, void* workspace, size_t workspace_bytes, void* stream) {
    return b200q_attn_decode_paged_split_kv(qkv, pos, k_pool, v_pool, B200Q_F32, block_table, slot_mapping, block_size, max_blocks, rope_table, n_heads,
                                            n_kv_heads, head_dim, M, xq, attn_out, workspace, workspace_bytes, stream);
}

/* Reads and clears the sticky device error word of the CURRENT device (synchronises the device: call it outside
 * graph capture, e.g. once per generate()).  0 = no error; bit 0 = a decode-attention position was outside [0, max_ctx). */
int32_t b200q_decode_error(int32_t* out_flags) {
    if (!out_flags) return B200Q_ERR_INVALID_ARG;
    int v = 0;
    if (cudaMemcpyFromSymbol(&v, g_decode_error, sizeof(int)) != cudaSuccess) return B200Q_ERR_CUDA;
    if (v != 0) {
        const int zero = 0;
        if (cudaMemcpyToSymbol(g_decode_error, &zero, sizeof(int)) != cudaSuccess) return B200Q_ERR_CUDA;
    }
    *out_flags = v;
    return B200Q_OK;
}

/* TRACE builds (make TRACE=1) only: dev_buf receives {kind, entry, after-wait, exit, 4 phase marks} globaltimer records (8 x int64 each) of
 * the glue kernels in launch order, up to `cap` records; null stops the trace.  kind: 1 attention, 2 cluster add+norm, 3 add+norm */
int32_t b200q_debug_set_glue_trace(void* dev_buf, int32_t cap) {
#ifdef B200Q_MV_TRACE
    long long* p = (long long*)dev_buf;
    unsigned int zero = 0, c = dev_buf ? (unsigned int)cap : 0u;
    if (cudaMemcpyToSymbol(g_glue_trace, &p, sizeof(p)) != cudaSuccess) return B200Q_ERR_CUDA;
    if (cudaMemcpyToSymbol(g_glue_n, &zero, sizeof(zero)) != cudaSuccess) return B200Q_ERR_CUDA;
    if (cudaMemcpyToSymbol(g_glue_cap, &c, sizeof(c)) != cudaSuccess) return B200Q_ERR_CUDA;
    return B200Q_OK;
#else
    (void)dev_buf; (void)cap;
    return B200Q_ERR_UNSUPPORTED;
#endif
}

int32_t b200q_argmax(const float* logits, int64_t V, int64_t M, int64_t* out_ids, int32_t* pos_inc, void* stream) {
    if (!logits || !out_ids || V <= 0 || M <= 0) return B200Q_ERR_INVALID_ARG;
    cudaError_t e = launch_pdl(argmax_kernel, dim3((unsigned)M), dim3(1024), 0, (cudaStream_t)stream, logits, (int)V, out_ids, (int*)pos_inc);
    return e == cudaSuccess ? B200Q_OK : B200Q_ERR_CUDA;
}

/* MoE decode combine (after the grouped down projection): out[T, H] = sum over the top_k slots of gate_w[t, j] * y[t * top_k + j, :] */
int32_t b200q_moe_combine(const float* y, const float* gate_w, int64_t T, int64_t top_k, int64_t H, float* out, void* stream) {
    if (!y || !gate_w || !out || T <= 0 || T > 65535 || top_k <= 0 || H <= 0) return B200Q_ERR_INVALID_ARG;
    cudaError_t e = launch_pdl(moe_combine_kernel, dim3((unsigned)((H + 255) / 256), (unsigned)T), dim3(256), 0, (cudaStream_t)stream, y, gate_w, (int)top_k, (int)H, out);
    return e == cudaSuccess ? B200Q_OK : B200Q_ERR_CUDA;
}

int32_t b200q_embed(const void* table_f16, const int64_t* ids, int64_t H, int64_t M, float* h, void* stream) {
    if (!table_f16 || !ids || !h || H <= 0 || M <= 0) return B200Q_ERR_INVALID_ARG;
    cudaError_t e = launch_pdl(embed_kernel, dim3((unsigned)((H + 255) / 256), (unsigned)M), dim3(256), 0, (cudaStream_t)stream,
                               (const __half*)table_f16, ids, (int)H, h);
    return e == cudaSuccess ? B200Q_OK : B200Q_ERR_CUDA;
}

}  // extern "C"
