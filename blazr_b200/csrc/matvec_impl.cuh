// matvec.cu -- decode-time dequant-matvec (M = 1..4): the HBM-bound hot kernel.
//
// Design (DESIGN.md "Kernel 1"):
//   * stream-K over the tile-major chunk array: CTA g owns the contiguous chunk range
//     [g*C/G, (g+1)*C/G)  -> every SM streams one contiguous region of HBM, perfect balance for any N,K;
//   * one producer thread feeds a ring of shared-memory stages with cp.async.bulk (TMA engine, 1-D,
//     mbarrier complete_tx): 1 copy of the 18-35 KB weight chunk + 1 copy of the M x 320 B quantised
//     activation record per stage, so ~100 KB per SM are in flight independent of occupancy;
//   * 16 consumer warps: warp w owns rows 8w..8w+7 of the tile, 8 lanes x 16 B walk one row's
//     256-k chunk (unit i = 32 consecutive k), 4 rows per step; activations stay in registers for the
//     8 rows; integer dot products with dp4a, per-sub-block scales applied in f32;
//   * at tile end an 8-lane shuffle reduction; tiles split between CTAs are combined DETERMINISTICALLY
//     through per-CTA partial slots in the workspace that double as their own ready flags (+0.0 bits = empty):
//     two contributors -> the first one's fix-up warp polls and sums beside the consumers; three or more ->
//     all 16 consumer warps of contributor gf + 1 poll one contributor each (MV_WIDE_MIN); always CTA order,
//     no float atomics;
//   * compile-time variants: norm prologue (PRO), SwiGLU epilogue / fused tensor-parallel exchange (OUT),
//     grouped expert-bank launch (GRP), dual-format launch (F2 != F: two weights of different formats, one grid).
#pragma once
#include <atomic>
#include <type_traits>
#include "matvec_common.cuh"

namespace b200q {

// ------------------------------------------------------------------------------------------------
// Fused activation producers.  Executed by the 16 consumer warps after griddepcontrol.wait, while the first
// ring-full of weight chunks (requested before the wait) is still in flight, so the separate norm / SwiGLU
// kernels of a decode step (and their launch + drain gaps) disappear.  Arithmetic is identical to
// decode_ops.cu (f64 sum of squares, explicit f32 ops, deterministic exp) => same bits as the oracle.
// Records: xhat[(kc*M + m)*320] = { int8 q[256]; float d[8]; (int16 bsum16[2])[8] }.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void quant_block_to_record(float v, uint8_t* rec, int blk_in_chunk, int lane) {
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
    rec[blk_in_chunk * 32 + lane] = (uint8_t)(int8_t)q;
    if (lane == 0) {
        reinterpret_cast<float*>(rec + 256)[blk_in_chunk] = d;
        reinterpret_cast<uint32_t*>(rec + 288)[blk_in_chunk] = ((uint32_t)s & 0xFFFFu) | ((uint32_t)s_hi << 16);
    }
}

// static norm weights of this thread's elements (plain loads: never written during the step), fetched ahead of the wait
template <int EPT>
__device__ __forceinline__ void load_nw(const float* __restrict__ w, int tid, float (&nw)[EPT]) {
    if constexpr (EPT >= 4) {
#pragma unroll
        for (int q = 0; q < EPT / 4; q++) {
            const float4 f = reinterpret_cast<const float4*>(w + EPT * tid)[q];
            nw[4 * q] = f.x; nw[4 * q + 1] = f.y; nw[4 * q + 2] = f.z; nw[4 * q + 3] = f.w;
        }
    } else {
#pragma unroll
        for (int j = 0; j < EPT; j++) nw[j] = w[EPT * tid + j];
    }
}
__device__ __forceinline__ void pdl_wait_again() { pdl_wait(); }  // PRO kernels: the consumers' dependency wait, after their static loads

// ---- norm prologue, lane-parallel form: thread t of the 512 consumer threads owns the EPT = K / 512 consecutive elements
// [EPT t, EPT t + EPT); a 32-block is 32 / EPT adjacent lanes, so every lane belongs to exactly ONE block: the two IEEE
// divides of the quantiser run once per lane (not once per block per warp), the block maximum / sums are 1-5 shuffles.
// Everything that does not depend on the preceding kernel (norm weights) is loaded by the caller ahead of
// griddepcontrol.wait.  One L2 round trip (h_in, delta) + one 512-thread barrier for the sum of squares.
template <int EPT>
__device__ __forceinline__ void load_ept(const float* __restrict__ p, float (&v)[EPT]) {
    if constexpr (EPT >= 4) {
#pragma unroll
        for (int q = 0; q < EPT / 4; q++) {
            const float4 f = __ldcg(reinterpret_cast<const float4*>(p) + q);  // written by the kernel ahead: L2
            v[4 * q] = f.x; v[4 * q + 1] = f.y; v[4 * q + 2] = f.z; v[4 * q + 3] = f.w;
        }
    } else if constexpr (EPT == 2) {
        const float2 f = __ldcg(reinterpret_cast<const float2*>(p));
        v[0] = f.x; v[1] = f.y;
    } else {
        v[0] = __ldcg(p);
    }
}
template <int EPT>
__device__ __forceinline__ void store_ept(float* __restrict__ p, const float (&v)[EPT]) {
    if constexpr (EPT >= 4) {
#pragma unroll
        for (int q = 0; q < EPT / 4; q++) reinterpret_cast<float4*>(p)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    } else if constexpr (EPT == 2) {
        *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
    } else {
        p[0] = v[0];
    }
}

template <int MB, int EPT>
__device__ __forceinline__ void norm_prologue(const MatvecParams& p, uint8_t* xhat, const float (&nw)[EPT], int tid, int warp, int lane, bool writer,
                                              double* red /*[16]*/) {
    constexpr int NT = MV_CONSUMER_WARPS * 32;
    constexpr int LPB = 32 / EPT;  // lanes per 32-block
    const int K = EPT * NT;
    const int e0 = EPT * tid;
    for (int m = 0; m < p.M; m++) {
        float v[EPT];
        load_ept<EPT>(p.h_in + (size_t)m * K + e0, v);
        if (p.delta) {
            float dl[EPT];
            load_ept<EPT>(p.delta + (size_t)m * K + e0, dl);
#pragma unroll
            for (int j = 0; j < EPT; j++) v[j] = __fadd_rn(v[j], dl[j]);
        }
        if (writer && p.h_out) store_ept<EPT>(p.h_out + (size_t)m * K + e0, v);
        double ss = 0.0;
#pragma unroll
        for (int j = 0; j < EPT; j++) ss = fma((double)v[j], (double)v[j], ss);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if (lane == 0) red[warp] = ss;
        named_bar_sync(4, NT);
        double tot = 0.0;
#pragma unroll
        for (int i = 0; i < MV_CONSUMER_WARPS; i++) tot += red[i];
        const float inv = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(__fdiv_rn((float)tot, (float)K), p.eps)));
        float x[EPT];
        float amax = 0.0f;
#pragma unroll
        for (int j = 0; j < EPT; j++) {
            x[j] = __fmul_rn(__fmul_rn(v[j], inv), nw[j]);
            amax = fmaxf(amax, fabsf(x[j]));
        }
#pragma unroll
        for (int o = LPB / 2; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
        const float d = __fdiv_rn(amax, 127.0f);
        const float id = (d != 0.0f) ? __fdiv_rn(1.0f, d) : 0.0f;
        int s = 0;
        uint8_t* rec = xhat + ((size_t)(e0 / CHUNK_K) * p.M + m) * ACT_REC_BYTES;
        const int off = e0 % CHUNK_K;
        if constexpr (EPT >= 4) {
#pragma unroll
            for (int q4 = 0; q4 < EPT / 4; q4++) {
                uint32_t wv = 0;
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const int q = (int)roundf(__fmul_rn(x[4 * q4 + c], id));
                    s += q;
                    wv |= ((uint32_t)q & 0xFFu) << (8 * c);
                }
                *reinterpret_cast<uint32_t*>(rec + off + 4 * q4) = wv;
            }
        } else {
#pragma unroll
            for (int j = 0; j < EPT; j++) {
                const int q = (int)roundf(__fmul_rn(x[j], id));
                s += q;
                rec[off + j] = (uint8_t)(int8_t)q;
            }
        }
        // sums of the two 16-element halves of the block: lanes [0, LPB/2) of the block hold the first half
        if constexpr (LPB >= 4) {
#pragma unroll
            for (int o = LPB / 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        }
        int s_lo, s_hi;
        if constexpr (LPB >= 2) {
            const int other = __shfl_xor_sync(0xffffffffu, s, LPB / 2);
            s_lo = s; s_hi = other;  // valid on the block's first lane
        } else {  // EPT == 32 is not instantiated
            s_lo = s; s_hi = 0;
        }
        if ((lane % LPB) == 0) {
            const int blk = off / 32;
            reinterpret_cast<float*>(rec + 256)[blk] = d;
            reinterpret_cast<uint32_t*>(rec + 288)[blk] = ((uint32_t)s_lo & 0xFFFFu) | ((uint32_t)s_hi << 16);
        }
        if (m + 1 < p.M) named_bar_sync(4, NT);  // red[] is reused by the next row
    }
    named_bar_sync(4, NT);  // records visible to every consumer warp
}

template <int MB>
__device__ __forceinline__ void fused_prologue(const MatvecParams& p, uint8_t* xhat, int tid, int warp, int lane, bool writer) {
    constexpr int NT = MV_CONSUMER_WARPS * 32;
    const int K = (int)p.KC * CHUNK_K;
    const int nblk = K / 32;
    {
        // ---- xhat = quant(silu(gate) * up), gate_up[M, 2K] ----
        for (int m = 0; m < p.M; m++) {
            const float* gr = p.gate_up + (size_t)m * 2 * K;
            for (int b = warp; b < nblk; b += MV_CONSUMER_WARPS) {
                const int k = b * 32 + lane;
                const float gv = gr[k], uv = gr[K + k];
                const float v = __fmul_rn(__fdiv_rn(gv, __fadd_rn(1.0f, det_expf(-gv))), uv);
                quant_block_to_record(v, xhat + ((size_t)(b >> 3) * p.M + m) * ACT_REC_BYTES, b & 7, lane);
            }
        }
    }
    named_bar_sync(4, NT);  // records visible to every consumer warp
}

// int32 -> f64.  -DB200Q_MV_MAGIC_I2D: without the conversion unit -- the double with high word 0x43300000 and low word
// (s ^ 0x80000000) is 2^52 + 2^31 + s exactly, one DADD (FP64 pipe) removes the bias -- instead of I2F.F64 (XU pipe, 8 issue
// cycles per warp instruction, 3-4 per chunk).  Measured in round 2: NEUTRAL (Q4_K gate|up 15.69 vs 15.59 us, 70B step 108.7 vs
// 109.7 tok/s): the XU pipe (24-26 % busy) is not what paces the consumer loop.  Kept as a compile-time experiment.
#ifdef B200Q_MV_MAGIC_I2D
__device__ __forceinline__ double i2d(int s) { return __hiloint2double(0x43300000, (int)((unsigned)s ^ 0x80000000u)) - 4503601774854144.0; }
#else
__device__ __forceinline__ double i2d(int s) { return (double)s; }
#endif

// Per-CTA globaltimer trace and the "skip the math" debug flag cost ~6 instructions per chunk in the consumer loop: they are
// compiled in only with -DB200Q_MV_TRACE (make TRACE=1; tools/trace_matvec.py, tools/trace_step.py need that build).
#ifdef B200Q_MV_TRACE
#define MV_TRACE_ON(p) ((p).trace != nullptr)
#define MV_DEBUG_SKIP(p) (((p).debug_flags & 1) != 0)
#else
#define MV_TRACE_ON(p) false
#define MV_DEBUG_SKIP(p) false
#endif

// ---- output of one finished row sum: local y, or (fused TP exchange) the same element of every rank's slot ----
struct RpState {
    unsigned int epoch;  // epoch of this exchange (previous + 1)
    size_t off;          // byte offset of this rank's slot / gather region inside every rank's buffer
};
__device__ __forceinline__ RpState rp_begin(const MatvecParams& p) {
    RpState r{0u, 0};
    if (p.rp_mode == RP_NONE) return r;
    const uint8_t* mine = p.comm.peers[p.comm.rank];
    const bool ar = p.rp_mode == RP_ALLREDUCE;
    // written by the last CTA of the previous exchange of this kind; that launch completed before griddepcontrol.wait returned
    r.epoch = __ldcg(reinterpret_cast<const unsigned int*>(mine + (ar ? COMM_OFF_AR_EPOCH : COMM_OFF_AG_EPOCH))) + 1u;
    r.off = ar ? comm_ar_slot_off(p.comm, (int)(r.epoch & 1u), p.comm.rank) : comm_ag_off(p.comm, p.comm.rank);
    return r;
}
template <bool RP>
__device__ __forceinline__ void mv_store(const MatvecParams& p, const RpState& rp, int64_t idx, double v) {
    if constexpr (!RP) {
        store_out_d(p.y, p.y_dtype, idx, v);
    } else if (p.rp_mode == RP_ALLREDUCE) {
        const double e = ar_encode(v);   // the slot element is its own ready flag (comm_dev.cuh)
        for (int r = 0; r < p.comm.world; r++) reinterpret_cast<double*>(p.comm.peers[r] + rp.off)[idx] = e;
    } else {
        const float f = (float)v;
        for (int r = 0; r < p.comm.world; r++) reinterpret_cast<float*>(p.comm.peers[r] + rp.off)[idx] = f;
    }
}
// row-parallel shards each add their partial sum: the bias must enter the total once (rank 0)
template <bool RP>
__device__ __forceinline__ bool mv_use_bias(const MatvecParams& p) { return p.bias && (!RP || p.rp_mode != RP_ALLREDUCE || p.comm.rank == 0); }
constexpr int MV_BAR_DONE = 5;  // consumers + fix-up warp: every output store of this CTA is issued
constexpr int MV_BAR_EPI_FULL = 6;   // (+ buffer 0/1) consumers -> fix-up warp: a finished tile sits in s_y[buffer]
constexpr int MV_BAR_EPI_FREE = 8;   // (+ buffer 0/1) fix-up warp -> consumers: s_y[buffer] may be overwritten

// where finished row sums go (compile time, like GRP: the plain matvec carries none of the other forms)
enum { OUT_PLAIN = 0, OUT_REMOTE = 1 /* fused tensor-parallel exchange */, OUT_SWIGLU = 2 /* fused SwiGLU + quantise epilogue */ };

// ---- OUT_SWIGLU: one finished 128-row tile (64 gate / 64 up rows interleaved, f32 in shared memory) -> 64 activations
// silu(gate) * up -> two quantised 32-blocks of the next matvec's records.  Executed by the fix-up warp; arithmetic identical
// to swiglu_quant_kernel (decode_ops.cu), so the records carry the same bits as the separate operator. ----
__device__ __forceinline__ void swiglu_tile_epilogue(const MatvecParams& p, const float* sy /*[TILE_ROWS]*/, int64_t tile_in_weight, int rec_row, int lane) {
#pragma unroll
    for (int b = 0; b < 2; b++) {
        const int j = 32 * b + lane, w_ = j >> 2, g_ = j & 3;
        const float gv = sy[8 * w_ + g_], uv = sy[8 * w_ + 4 + g_];
        const float v = __fmul_rn(__fdiv_rn(gv, __fadd_rn(1.0f, det_expf(-gv))), uv);
        const int64_t f = 64 * tile_in_weight + 32 * b;  // first ffn index of this block (F % 64 == 0: blocks are all-valid or absent)
        if (f < p.epi_F) quant_block_to_record(v, p.xq_out + ((size_t)(f / CHUNK_K) * p.epi_rows + rec_row) * ACT_REC_BYTES, (int)((f % CHUNK_K) / 32), lane);
    }
}


// contributors of tile tq under the stream-K split: CTAs gf..gl; sgf = workspace slot (0 head / 1 tail) the first one uses
__device__ __forceinline__ void sk_tile_span(const MatvecParams& p, int64_t tq, int64_t G, int& gf, int& gl, int& sgf) {
    if (p.plan32) {
        gf = (int)((((uint32_t)(tq * p.KC) + 1u) * (uint32_t)G - 1u) / (uint32_t)p.C);
        gl = (int)((((uint32_t)((tq + 1) * p.KC - 1) + 1u) * (uint32_t)G - 1u) / (uint32_t)p.C);
        sgf = ((int64_t)sk_begin32((uint32_t)gf, (uint32_t)p.C, (uint32_t)G) == tq * p.KC) ? 0 : 1;
    } else {
        gf = (int)sk_owner(tq * p.KC, p.C, G);
        gl = (int)sk_owner((tq + 1) * p.KC - 1, p.C, G);
        sgf = (sk_begin(gf, p.C, G) == tq * p.KC) ? 0 : 1;
    }
}
// a split tile with >= MV_WIDE_MIN contributors is reduced by ALL consumer warps of contributor gf + 1 (whose whole chunk range
// lies inside the tile, so the reduction is the last thing that CTA does): warp w polls contributor gf + w, one L2 round trip
// for up to 16 contributors instead of one per 4 in the single fix-up warp (measured 4.6 us of tail on 17-way split tiles)
constexpr int MV_WIDE_MIN = 3;

template <class F, int MB, bool PRO, bool GRP, int OUT, class F2 = F>
__global__ void __launch_bounds__(MV_THREADS, 1) matvec_kernel(const MatvecParams p) {
    constexpr bool RP = OUT == OUT_REMOTE;
    constexpr bool EPI = OUT == OUT_SWIGLU;
    constexpr bool DUAL = !std::is_same<F, F2>::value;   // two weights of different formats in one grid (MatvecParams::w2)
    // M = 1: two chunks per trip of the consumer loop (one counter test and branch per pair); the M = 2 / 4 loops would spill
    constexpr int MV_CHUNK_UNROLL = MB == 1 ? 2 : 1;
    static_assert(!DUAL || (!GRP && OUT == OUT_PLAIN), "the dual-format launch is a plain matvec");
    __shared__ float s_y[EPI ? 2 : 1][EPI ? MB : 1][EPI ? TILE_ROWS : 1];   // finished full tiles (double-buffered)
    __shared__ float s_yfix[EPI ? MB : 1][EPI ? TILE_ROWS : 1];             // finished split tile (fix-up warp only)
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* full = reinterpret_cast<uint64_t*>(smem);
    uint64_t* empty = full + MV_MAX_STAGES;
    uint8_t* xhat = smem + MV_HDR_BYTES;                  // fused prologue: quantised activation records [kc][m][320]
    uint8_t* stages = smem + MV_HDR_BYTES + (PRO ? p.xhat_bytes : 0);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t G = gridDim.x, g = blockIdx.x;
    if (MV_TRACE_ON(p) && tid == 0) {
        p.trace[g * 8 + 0] = globaltimer_ns();
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        p.trace[g * 8 + 2] = smid;
    }
    int64_t c0, c1;
    if (p.plan32) {  // the usual case: no 64-bit division on the prologue's critical path
        c0 = sk_begin32((uint32_t)g, (uint32_t)p.C, (uint32_t)G);
        c1 = sk_begin32((uint32_t)g + 1u, (uint32_t)p.C, (uint32_t)G);
    } else {
        c0 = sk_begin(g, p.C, G);
        c1 = sk_begin(g + 1, p.C, G);
    }
    const int n_chunks = (int)(c1 - c0);
    const int KC = (int)p.KC;
    const int nst = p.nstages;
    SkPlan& sp = *reinterpret_cast<SkPlan*>(smem + 2 * MV_MAX_STAGES * 8);       // shared plan (computed once)
    pdl_launch_dependents();  // let the next kernel of the stream start its own weight prefetch

    // The producer lane initialises the barriers and requests the first ring-full of weights BEFORE the CTA-wide barrier:
    // the TMA stream starts a few hundred cycles after the CTA lands on the SM, while thread 0 publishes the plan.
    const bool is_producer = warp == MV_CONSUMER_WARPS && lane == 0;
    SkPlan spp;  // the producer's private copy of the plan
    if (is_producer) {
        spp = p.plan32 ? sk_plan32((uint32_t)c0, (uint32_t)c1, (uint32_t)p.KC) : sk_plan(c0, c1, p.KC);
        for (int s = 0; s < nst; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], MV_CONSUMER_WARPS);
        }
        fence_mbar_init();
        fence_proxy_async();
        if (!GRP) {
            const uint64_t pol0 = policy_evict_first();
            const uint32_t xbytes0 = PRO ? 0u : (uint32_t)p.M * ACT_REC_BYTES;
            const int pre0 = n_chunks < nst ? n_chunks : nst;
            for (int j = 0; j < pre0; j++) {
                const int64_t vc0 = sk_chunk_at(spp, c0, j);
                const uint8_t* src0 = p.w + vc0 * (int64_t)p.cb1;
                uint32_t wb0 = (uint32_t)p.cb1;
                if (DUAL && vc0 >= (int64_t)p.T1 * p.KC) { src0 = p.w2 + (vc0 - (int64_t)p.T1 * p.KC) * (int64_t)p.cb2; wb0 = (uint32_t)p.cb2; }
                mbar_arrive_expect_tx(&full[j], wb0 + xbytes0);
                bulk_g2s_hint(stages + (size_t)j * p.stage_bytes, src0, wb0, &full[j], pol0);
            }
        }
    }
    if (tid == 0) sp = p.plan32 ? sk_plan32((uint32_t)c0, (uint32_t)c1, (uint32_t)p.KC) : sk_plan(c0, c1, p.KC);
    __syncthreads();

    if (warp == MV_CONSUMER_WARPS) {
        // ===================== producer: one thread drives the TMA engine =====================
        if (lane == 0) {
            const uint64_t pol = policy_evict_first();
            const uint32_t xbytes = PRO ? 0u : (uint32_t)p.M * ACT_REC_BYTES;
            const uint32_t wbytes = (uint32_t)p.cb1;              // bytes of one chunk of w (dual: chunks of w2 have cb2, see chunk_src)
            const uint32_t xoff_in_stage = (uint32_t)p.chunk_bytes;  // offset of the activation records inside a stage
            constexpr bool grouped = GRP;  // expert-bank launch (compile-time: the plain matvec carries none of it)
            const int64_t cpw = (int64_t)p.tpw * p.KC;  // grouped: chunks per weight
            if (grouped) pdl_wait();                      // the expert selection is produced by the preceding kernel
            // j-th processed chunk -> (weight address, activation record address)
            auto chunk_vc = [&](int j) -> int64_t {      // chunk index in the (concatenated) chunk array
                if (j < sp.nH) return c0 + j;
                if (j < sp.nH + sp.nT) return c0 + sp.nH + sp.nF + (j - sp.nH);
                return c0 + sp.nH + (j - sp.nH - sp.nT);
            };
            auto chunk_src = [&](int j) -> const uint8_t* {
                const int64_t vc = chunk_vc(j);
                if (DUAL && vc >= (int64_t)p.T1 * p.KC) return p.w2 + (vc - (int64_t)p.T1 * p.KC) * (int64_t)p.cb2;
                if (!grouped) return p.w + vc * (int64_t)wbytes;
                const int64_t slot = vc / cpw;
                const int e = p.sel[slot];
                return (e < 0 || e >= p.n_experts) ? nullptr : p.w_table[e] + (vc - slot * cpw) * (int64_t)wbytes;   // never index past the bank
            };
            auto chunk_x = [&](int j) -> const uint8_t* {
                int kc;
                if (j < sp.nH) kc = sp.kcH + j;
                else if (j < sp.nH + sp.nT) kc = j - sp.nH;
                else kc = (j - sp.nH - sp.nT) % KC;
                if (!grouped) return p.xq + (size_t)kc * xbytes;
                const int64_t slot = chunk_vc(j) / cpw;
                return p.xq + ((size_t)kc * p.x_rows + (size_t)(slot / p.x_slot_div)) * ACT_REC_BYTES;
            };
            // Phase 1 (before griddepcontrol.wait): weights do not depend on the preceding kernels.  Fill the
            // shared-memory ring and ask the TMA engine to pull the rest of this CTA's range into L2, so HBM
            // keeps streaming across the kernel boundary while the predecessor drains.
            const int pre = n_chunks < nst ? n_chunks : nst;
            // grouped mode: a slot whose selection is negative (expert not hosted by this rank) is skipped -- no weight
            // copy, a flag behind the stage's activation record tells the consumers to leave the accumulators at zero
            auto issue_w = [&](int j, uint8_t* st, uint64_t* bar) {
                const uint8_t* src = chunk_src(j);
                const uint32_t wb = (DUAL && chunk_vc(j) >= (int64_t)p.T1 * p.KC) ? (uint32_t)p.cb2 : wbytes;
                if (grouped) {
                    const bool skip = src == nullptr;
                    *reinterpret_cast<volatile int*>(st + wbytes + xbytes) = skip ? 1 : 0;
                    mbar_arrive_expect_tx(bar, (skip ? 0u : wbytes) + xbytes);
                    if (skip) return;
                } else {
                    mbar_arrive_expect_tx(bar, wb + xbytes);
                }
                bulk_g2s_hint(st, src, wb, bar, pol);
            };
            if (GRP)  // (the plain forms requested their first ring-full ahead of the CTA barrier)
                for (int j = 0; j < pre; j++) issue_w(j, stages + (size_t)j * p.stage_bytes, &full[j]);
            int npf = n_chunks - pre;
            if (npf > p.l2_prefetch_chunks) npf = p.l2_prefetch_chunks;
            for (int j = pre; j < pre + npf; j++)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(chunk_src(j)), "r"(wbytes) : "memory");
            pdl_wait();  // activations (written by the preceding kernel) are visible from here on
            if (MV_TRACE_ON(p)) p.trace[g * 8 + 4] = globaltimer_ns();
            if (!PRO)
                for (int j = 0; j < pre; j++)
                    bulk_g2s(stages + (size_t)j * p.stage_bytes + xoff_in_stage, chunk_x(j), xbytes, &full[j]);
            int s = 0;
            uint32_t ph = 0;  // second use of each stage waits for the consumers' first release (phase 0)
            for (int j = pre; j < n_chunks; j++) {
                mbar_wait(&empty[s], ph);
                uint8_t* st = stages + (size_t)s * p.stage_bytes;
                issue_w(j, st, &full[s]);
                if (!PRO) bulk_g2s(st + xoff_in_stage, chunk_x(j), xbytes, &full[s]);
                if (++s == nst) { s = 0; ph ^= 1u; }
            }
            // every chunk of this launch is requested: keep HBM busy with the successor's first chunks (L2 prefetch)
            if (!GRP && p.next_pf > 0) {
                for (int64_t ng = g; ng < p.next_G; ng += G) {
                    const int64_t a0 = sk_begin(ng, p.next_C, p.next_G), a1 = sk_begin(ng + 1, p.next_C, p.next_G);
                    const SkPlan np_ = sk_plan(a0, a1, p.next_KC);
                    const int n = (int)(a1 - a0) < p.next_pf ? (int)(a1 - a0) : p.next_pf;
                    for (int j = 0; j < n; j++)
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p.next_w + sk_chunk_at(np_, a0, j) * (int64_t)p.next_chunk_bytes),
                                     "r"(p.next_chunk_bytes)
                                     : "memory");
                }
            }
        }
        return;
    }
    if (warp == MV_CONSUMER_WARPS + 1) {
        // ===================== fix-up warp: arrival atomics + ordered reduction of split tiles =====================
        // Runs beside the consumers (they only bar.arrive), so neither the math nor the TMA stream ever waits
        // for an atomic round trip.  Split tiles are processed first, so this finishes long before the CTA does.
        constexpr bool rp_on = RP;
        if (sp.nH == 0 && sp.nT == 0 && !EPI) {
            if (rp_on) named_bar_sync(MV_BAR_DONE, MV_CONSUMER_WARPS * 32 + 32);
            return;
        }
        pdl_wait();
        RpState rp{0u, 0};
        if constexpr (RP) rp = rp_begin(p);
        // Split tiles: every contributor leaves its 128 x MB partial sums in its own workspace slot and moves on; ONE designated
        // contributor per tile -- a CTA whose share of the tile is the last thing it computes -- polls the slots until every
        // value has landed, sums them in CTA order (deterministic) and writes y.  The slots double as their own ready flags:
        // the workspace is zero-filled, contributors store -0.0 for an exact zero, so +0.0 bits mean "not written yet", and
        // the reducer restores +0.0 after reading.  One L2 visibility latency after the last partial store, instead of a
        // release fence + atomic round trip + load round trip behind it (measured 2-3.8 us of tail per launch in round 2).
        int64_t tqs[2] = {sp.tH, sp.tT};
#pragma unroll
        for (int seg = 0; seg < 2; seg++) {
            if ((seg == 0 ? sp.nH : sp.nT) == 0) continue;
            const int64_t tq = tqs[seg];
            int gf, gl, sgf;
            sk_tile_span(p, tq, G, gf, gl, sgf);
            const int nc = gl - gf + 1;
            if (nc >= MV_WIDE_MIN) continue;              // reduced by the consumer warps of contributor gf + 1 (wide reducer)
            if ((int)g != gf) continue;                   // two contributors: the first one's fix-up warp reduces
            if (MV_TRACE_ON(p) && lane == 0) p.trace[g * 8 + 5] = globaltimer_ns();
            const int64_t tql = GRP ? tq % p.tpw : tq;                      // tile index inside its weight
            const int64_t ybase = GRP ? (tq / p.tpw) * p.y_slot_stride : 0;  // grouped: output of slot tq / tpw
            constexpr int PASSES = 2 * MB;                       // 64 doubles (one double2 per lane) per pass
            double2 sum[PASSES];
#pragma unroll
            for (int v = 0; v < PASSES; v++) sum[v] = make_double2(0.0, 0.0);
            constexpr int NB = MB == 1 ? 4 : (MB == 2 ? 2 : 1);  // contributors polled together (one L2 round trip per batch when ready); 32 registers
            for (int g0 = gf; g0 <= gl; g0 += NB) {
                double2 tb[NB][PASSES];
                for (int spin = 0; spin < (1 << 22); spin++) {  // bounded: a lost contributor must not hang the GPU
                    bool ready = true;
#pragma unroll
                    for (int u = 0; u < NB; u++) {
                        const int gg = g0 + u;
                        const double* src = p.ws_part + ((size_t)gg * 2 + (gg == gf ? sgf : 0)) * (TILE_ROWS * MB) + lane * 2;
#pragma unroll
                        for (int v = 0; v < PASSES; v++) {
                            if (gg <= gl) {
                                asm volatile("ld.volatile.global.v2.f64 {%0,%1}, [%2];" : "=d"(tb[u][v].x), "=d"(tb[u][v].y) : "l"(src + v * 64));
                            } else {
                                tb[u][v] = make_double2(-0.0, -0.0);
                            }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < NB; u++)
#pragma unroll
                        for (int v = 0; v < PASSES; v++) ready = ready && __double_as_longlong(tb[u][v].x) != 0ll && __double_as_longlong(tb[u][v].y) != 0ll;
                    if (__all_sync(0xffffffffu, ready)) break;
                }
#pragma unroll
                for (int u = 0; u < NB; u++) {
                    const int gg = g0 + u;
                    double* src = p.ws_part + ((size_t)gg * 2 + (gg == gf ? sgf : 0)) * (TILE_ROWS * MB) + lane * 2;
#pragma unroll
                    for (int v = 0; v < PASSES; v++) {
                        sum[v].x += tb[u][v].x;
                        sum[v].y += tb[u][v].y;
                        if (gg <= gl) *reinterpret_cast<double2*>(src + v * 64) = make_double2(0.0, 0.0);   // slot free for the next launch
                    }
                }
            }
#pragma unroll
            for (int v = 0; v < PASSES; v++) {
                const int idx = (v * 32 + lane) * 2;
                // an exact zero was published as -0.0; the sum of zeros is +0.0 (as the oracle's accumulation from +0.0)
                const double sv[2] = {sum[v].x == 0.0 ? 0.0 : sum[v].x, sum[v].y == 0.0 ? 0.0 : sum[v].y};
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const int rr = (idx + e) / MB, m = (idx + e) % MB;
                    const int64_t n = tql * TILE_ROWS + rr;
                    if constexpr (EPI) {
                        if (m < p.M) s_yfix[m][rr] = (float)(sv[e] + ((p.bias && n < p.N) ? (double)p.bias[n] : 0.0));
                    } else {
                        if (n < p.N && m < p.M) mv_store<RP>(p, rp, ybase + (int64_t)m * p.ldy + n, sv[e] + (mv_use_bias<RP>(p) ? (double)p.bias[n] : 0.0));
                    }
                }
            }
            if constexpr (EPI) {
                __syncwarp();
                for (int m = 0; m < p.M; m++) swiglu_tile_epilogue(p, s_yfix[m], tql, GRP ? (int)(tq / p.tpw) : m, lane);
                __syncwarp();
            }
            if (MV_TRACE_ON(p) && lane == 0) p.trace[g * 8 + 7] = globaltimer_ns();
        }
        if constexpr (EPI) {
            // full tiles of this CTA, in the consumers' order: wait for the tile, activate + quantise it, hand the buffer back
            const int n_full = sp.nF / KC;
            for (int ft = 0; ft < n_full; ft++) {
                const int buf = ft & 1;
                const int64_t tq = (int64_t)sp.tF + ft;
                named_bar_sync(MV_BAR_EPI_FULL + buf, MV_CONSUMER_WARPS * 32 + 32);
                for (int m = 0; m < p.M; m++) swiglu_tile_epilogue(p, s_y[buf][m], GRP ? tq % p.tpw : tq, GRP ? (int)(tq / p.tpw) : m, lane);
                __syncwarp();
                asm volatile("bar.arrive %0, %1;" ::"r"(MV_BAR_EPI_FREE + buf), "r"(MV_CONSUMER_WARPS * 32 + 32) : "memory");
            }
        }
        if (rp_on) named_bar_sync(MV_BAR_DONE, MV_CONSUMER_WARPS * 32 + 32);
        return;
    }

    // ===================== consumers =====================
    if constexpr (!PRO) pdl_wait();  // y, the workspace and the bias may still be in use by the preceding kernel before this point
    RpState rp{0u, 0};
    if constexpr (RP) rp = rp_begin(p);
    const int g4 = lane >> 3, i = lane & 7;
    const FmtMeta meta{p.gpc};
    // f64 accumulators: every term is an exact product of an f32 scale and an integer partial, so the sum is
    // independent of the summation order up to 1e-16 -> the result is bit-reproducible against the oracle for any
    // grid size / stream-K split (oracle orc_matmul_q8).
    double acc[MV_STEPS][MB];
#pragma unroll
    for (int s4 = 0; s4 < MV_STEPS; s4++)
#pragma unroll
        for (int m = 0; m < MB; m++) acc[s4][m] = 0.0;

    if constexpr (PRO) {
        if (p.pro == 1) {
            // norm prologue: K = EPT * 512 with EPT in {1, 2, 4, 8, 16} (checked by the host)
            __shared__ double s_red[MV_CONSUMER_WARPS];
            switch ((int)p.KC * CHUNK_K / (MV_CONSUMER_WARPS * 32)) {
                case 16: { float nw[16]; load_nw<16>(p.norm_w, tid, nw); pdl_wait_again(); norm_prologue<MB, 16>(p, xhat, nw, tid, warp, lane, g == 0, s_red); break; }
                case 8: { float nw[8]; load_nw<8>(p.norm_w, tid, nw); pdl_wait_again(); norm_prologue<MB, 8>(p, xhat, nw, tid, warp, lane, g == 0, s_red); break; }
                case 4: { float nw[4]; load_nw<4>(p.norm_w, tid, nw); pdl_wait_again(); norm_prologue<MB, 4>(p, xhat, nw, tid, warp, lane, g == 0, s_red); break; }
                case 2: { float nw[2]; load_nw<2>(p.norm_w, tid, nw); pdl_wait_again(); norm_prologue<MB, 2>(p, xhat, nw, tid, warp, lane, g == 0, s_red); break; }
                default: { float nw[1]; load_nw<1>(p.norm_w, tid, nw); pdl_wait_again(); norm_prologue<MB, 1>(p, xhat, nw, tid, warp, lane, g == 0, s_red); break; }
            }
        } else {
            pdl_wait_again();
            fused_prologue<MB>(p, xhat, tid, warp, lane, g == 0);
        }
    }

    // am I the wide reducer of my head tile?  (then that segment is my whole range: see MV_WIDE_MIN)
    bool wide_reducer = false;
    int wide_gf = 0, wide_gl = 0, wide_sgf = 0;
    if (sp.nH > 0) {
        sk_tile_span(p, sp.tH, G, wide_gf, wide_gl, wide_sgf);
        wide_reducer = (wide_gl - wide_gf + 1) >= MV_WIDE_MIN && (int)g == wide_gf + 1;
    }
    // segment walk: 0 = head (partial, slot 0), 1 = tail (partial, slot 1), 2 = full tiles
    int kcur = sp.nH > 0 ? sp.kcH : 0;  // k-chunk index of the chunk being processed (fused prologue addressing)
    int seg = sp.nH > 0 ? 0 : (sp.nT > 0 ? 1 : 2);
    int seg_left = seg == 0 ? sp.nH : (seg == 1 ? sp.nT : KC);  // chunks until the next flush
    int t = seg == 0 ? sp.tH : (seg == 1 ? sp.tT : sp.tF);
    uint32_t ph = 0;
    int n_full_done = 0;  // OUT_SWIGLU: full tiles flushed so far (selects the s_y buffer)
    // Everything the hot loop addresses is a 32-bit shared-window address built from values computed ONCE here: the ring /
    // barrier bases and, per lane, the byte offsets of its (row, unit) inside a chunk and of its unit inside an activation
    // record.  (Left to the compiler, these were re-derived from threadIdx every chunk: ~25 of ~120 instructions per chunk.)
    constexpr int NOFF = FmtNoff<F>::value;
    const uint32_t stages_sa = smem_u32(stages), full_sa = keep_in_reg(smem_u32(full)), xhat_sa = smem_u32(xhat);
    constexpr uint32_t EMPTY_OFF = MV_MAX_STAGES * 8;                     // empty[] follows full[]
    const uint32_t ring_bytes = keep_in_reg((uint32_t)nst * (uint32_t)p.stage_bytes);
    uint32_t st_off = 0;                                                   // byte offset of stage s inside the ring
    uint32_t bar_sa = full_sa;                                             // full[s]; empty[s] = + EMPTY_OFF
    uint32_t uoff[NOFF > 0 ? NOFF : 1];
    if constexpr (NOFF > 0) {
        F::unit_offsets(MV_ROWS_PER_WARP * warp + g4, i, meta, uoff);
#pragma unroll
        for (int q = 0; q < NOFF; q++) uoff[q] = keep_in_reg(uoff[q] + stages_sa);
    }
    constexpr int NOFF2 = DUAL ? FmtNoff<F2>::value : 0;   // dual-format launch: the second weight's lane offsets
    const FmtMeta meta2{p.gpc2};
    uint32_t uoff2[NOFF2 > 0 ? NOFF2 : 1];
    if constexpr (NOFF2 > 0) {
        F2::unit_offsets(MV_ROWS_PER_WARP * warp + g4, i, meta2, uoff2);
#pragma unroll
        for (int q = 0; q < NOFF2; q++) uoff2[q] = keep_in_reg(uoff2[q] + stages_sa);
    }
    const uint32_t xq_off = keep_in_reg((PRO ? xhat_sa : stages_sa + (uint32_t)p.chunk_bytes) + 32u * (uint32_t)i);      // int8 activations of unit i
    const uint32_t xs_off = keep_in_reg((PRO ? xhat_sa : stages_sa + (uint32_t)p.chunk_bytes) + 256u + 4u * (uint32_t)i); // its scale; + 32: block sums
    const uint32_t xrec_step = keep_in_reg((uint32_t)p.M * ACT_REC_BYTES);
    const uint32_t stage_bytes = keep_in_reg((uint32_t)p.stage_bytes);
    uint32_t xk_off = PRO ? (uint32_t)kcur * xrec_step : 0u;               // PRO: record of k-chunk kcur inside xhat
    // one trip of the outer loop per segment; a segment never crosses a tile boundary, so kcur does not wrap inside it
    for (int j = 0; j < n_chunks;) {
#pragma unroll(MV_CHUNK_UNROLL)
        for (int c = seg_left; c > 0; c--) {
            mbar_wait_sa(bar_sa, ph);
            if (MV_TRACE_ON(p) && tid == 0 && j == 0 && c == seg_left) p.trace[g * 8 + 1] = globaltimer_ns();
            const uint8_t* wc = stages + st_off;
            const uint32_t xbase = PRO ? xk_off : st_off;
            if (PRO) xk_off += xrec_step;

            uint4 xa[MB], xb[MB];
            float dx[MB];
            int bsA[MB], bsB[MB];
#pragma unroll
            for (int m = 0; m < MB; m++) {
                xa[m] = lds128_sa(xq_off + xbase + m * ACT_REC_BYTES);
                xb[m] = lds128_sa(xq_off + xbase + m * ACT_REC_BYTES + 16);
                dx[m] = __uint_as_float(lds32_sa(xs_off + xbase + m * ACT_REC_BYTES));
                const uint32_t bs = lds32_sa(xs_off + xbase + m * ACT_REC_BYTES + 32);
                bsA[m] = (int)(int16_t)(bs & 0xFFFFu);
                bsB[m] = (int)(int16_t)(bs >> 16);
            }
            const bool skip_chunk = GRP && *reinterpret_cast<const volatile int*>(wc + p.chunk_bytes + p.M * ACT_REC_BYTES) != 0;
            // the units of this chunk: rows 8 warp + 4 s4 + g4, unit i -- format FF (dual-format launches pick it per tile)
            auto chunk_math = [&](auto tag, const auto& uo, const FmtMeta& mt) {
                using FF = decltype(tag);
                constexpr int NO = FmtNoff<FF>::value;
#pragma unroll
                for (int s4 = 0; s4 < MV_STEPS; s4++) {
                    Unit u;
                    if constexpr (NO > 0) {
                        if (s4 == 0) FF::template load_unit_at<0>(st_off, uo, i, u, mt);
                        else FF::template load_unit_at<1>(st_off, uo, i, u, mt);
                    } else {
                        const int r = MV_ROWS_PER_WARP * warp + 4 * s4 + g4;
                        FF::template load_unit<true, FF::NIB>(wc, r, i, u, mt);
                    }
#pragma unroll
                    for (int m = 0; m < MB; m++) {
                        const float dxm = FmtAbScale<FF>::value ? __fmul_rn(dx[m], FmtAbScale<FF>::inv) : dx[m];
                        int sA = 0, sB = 0;
                        sA = __dp4a((int)u.v[0], (int)xa[m].x, sA); sA = __dp4a((int)u.v[1], (int)xa[m].y, sA);
                        sA = __dp4a((int)u.v[2], (int)xa[m].z, sA); sA = __dp4a((int)u.v[3], (int)xa[m].w, sA);
                        if constexpr (FF::NIB) {  // bytes hold 16 x q (unsigned): exact u8 x s8 dot, one arithmetic shift back
                            sB = dp4a_us(u.v[4], xb[m].x, sB); sB = dp4a_us(u.v[5], xb[m].y, sB);
                            sB = dp4a_us(u.v[6], xb[m].z, sB); sB = dp4a_us(u.v[7], xb[m].w, sB);
                            sB >>= 4;
                        } else {
                            sB = __dp4a((int)u.v[4], (int)xb[m].x, sB); sB = __dp4a((int)u.v[5], (int)xb[m].y, sB);
                            sB = __dp4a((int)u.v[6], (int)xb[m].z, sB); sB = __dp4a((int)u.v[7], (int)xb[m].w, sB);
                        }
                        sA -= u.off[0] * bsA[m];
                        sB -= u.off[1] * bsB[m];
                        double a_ = acc[s4][m];
                        if (FF::SUB == 32) {  // one scale per 32 weights
                            a_ = fma((double)__fmul_rn(u.a[0], dxm), i2d(sA + sB), a_);
                            if (FF::HAS_MIN) a_ = fma(-(double)__fmul_rn(u.b[0], dxm), i2d(bsA[m] + bsB[m]), a_);
                        } else {             // two 16-wide sub-blocks with their own scales
                            a_ = fma((double)__fmul_rn(u.a[0], dxm), i2d(sA), a_);
                            if (FF::HAS_MIN) a_ = fma(-(double)__fmul_rn(u.b[0], dxm), i2d(bsA[m]), a_);
                            a_ = fma((double)__fmul_rn(u.a[1], dxm), i2d(sB), a_);
                            if (FF::HAS_MIN) a_ = fma(-(double)__fmul_rn(u.b[1], dxm), i2d(bsB[m]), a_);
                        }
                        acc[s4][m] = a_;
                    }
                }
            };
            if (!MV_DEBUG_SKIP(p) && !skip_chunk) {
                if constexpr (DUAL) {
                    if (t >= p.T1) chunk_math(F2{}, uoff2, meta2);   // warp-uniform: a tile belongs to one weight
                    else chunk_math(F{}, uoff, meta);
                } else {
                    chunk_math(F{}, uoff, meta);
                }
            }
            // release the stage: the warp is converged here, so every lane's loads of it were issued before lane 0's arrive (no
            // __syncwarp and its divergence check), and the producer's refill lands a whole HBM round trip after the arrive
            if (lane == 0) mbar_arrive_sa(bar_sa + EMPTY_OFF);
            st_off += stage_bytes;
            bar_sa += 8u;
            if (st_off == ring_bytes) { ph ^= 1u; st_off = 0u; bar_sa = full_sa; }
        }

        // ---- segment / tile boundary: reduce the 8 lanes of each row and flush ----
#pragma unroll
        for (int s4 = 0; s4 < MV_STEPS; s4++)
#pragma unroll
            for (int m = 0; m < MB; m++) {
                double v = acc[s4][m];
                v += __shfl_xor_sync(0xffffffffu, v, 1);
                v += __shfl_xor_sync(0xffffffffu, v, 2);
                v += __shfl_xor_sync(0xffffffffu, v, 4);
                acc[s4][m] = v;
            }
        if (EPI && seg == 2) {
            // finished full tile -> shared memory (f32, as the unfused path stores it) -> the fix-up warp's SwiGLU epilogue
            const int buf = n_full_done & 1;
            if (n_full_done >= 2) named_bar_sync(MV_BAR_EPI_FREE + buf, MV_CONSUMER_WARPS * 32 + 32);  // tile n-2 has been consumed
            if (i == 0) {
                const int64_t tl = GRP ? t % p.tpw : t;
#pragma unroll
                for (int s4 = 0; s4 < MV_STEPS; s4++) {
                    const int rr = MV_ROWS_PER_WARP * warp + 4 * s4 + g4;
                    const int64_t n = tl * TILE_ROWS + rr;
                    const double bv = (p.bias && n < p.N) ? (double)p.bias[n] : 0.0;
#pragma unroll
                    for (int m = 0; m < MB; m++) s_y[buf][m][rr] = (float)(acc[s4][m] + bv);
                }
                __threadfence_block();
            }
            __syncwarp();
            asm volatile("bar.arrive %0, %1;" ::"r"(MV_BAR_EPI_FULL + buf), "r"(MV_CONSUMER_WARPS * 32 + 32) : "memory");
            n_full_done++;
        } else if (seg == 2) {
            if (i == 0) {
#pragma unroll
                const int64_t tl = GRP ? t % p.tpw : t;
                const int64_t ybase = GRP ? (int64_t)(t / p.tpw) * p.y_slot_stride : 0;
                for (int s4 = 0; s4 < MV_STEPS; s4++) {
                    const int64_t n = tl * TILE_ROWS + MV_ROWS_PER_WARP * warp + 4 * s4 + g4;
                    if (n < p.N) {
                        const double bv = mv_use_bias<RP>(p) ? (double)p.bias[n] : 0.0;
#pragma unroll
                        for (int m = 0; m < MB; m++)
                            if (m < p.M) mv_store<RP>(p, rp, ybase + (int64_t)m * p.ldy + n, acc[s4][m] + bv);
                    }
                }
            }
        } else {
            // partial tile: publish my share in my workspace slot (the slot doubles as its own ready flag)
            double* part = p.ws_part + ((size_t)g * 2 + seg) * (TILE_ROWS * MB);
            if (i == 0) {
#pragma unroll
                for (int s4 = 0; s4 < MV_STEPS; s4++) {
                    const int rr = MV_ROWS_PER_WARP * warp + 4 * s4 + g4;
#pragma unroll
                    for (int m = 0; m < MB; m++) {
                        const double v = acc[s4][m];
                        // +0.0 bits mean "slot not written yet" to the tile's reducer: publish an exact zero as -0.0
                        asm volatile("st.volatile.global.f64 [%0], %1;" ::"l"(part + rr * MB + m), "d"(v == 0.0 ? -0.0 : v) : "memory");
                    }
                }
            }
            if (seg == 0 && wide_reducer) {
                // ---- wide reducer: this CTA's whole range was the head segment; every consumer warp polls one contributor ----
                constexpr int NT = MV_CONSUMER_WARPS * 32;
                constexpr int PASSES = 2 * MB;                                  // 64 doubles (one double2 per lane) per pass
                named_bar_sync(4, NT);                                          // every warp is done with the ring: reuse it
                if (MV_TRACE_ON(p) && tid == 0) p.trace[g * 8 + 5] = globaltimer_ns();
                double* red = reinterpret_cast<double*>(stages);                // [wpr][TILE_ROWS * MB]
                int wpr = (int)(ring_bytes / (uint32_t)(TILE_ROWS * MB * 8));   // contributors per round (ring >= 2 stages >= 36 KB)
                if (wpr > MV_CONSUMER_WARPS) wpr = MV_CONSUMER_WARPS;
                double sum = 0.0;
                for (int base = wide_gf; base <= wide_gl; base += wpr) {
                    const int gg = base + warp;
                    if (warp < wpr && gg <= wide_gl) {
                        double* src = p.ws_part + ((size_t)gg * 2 + (gg == wide_gf ? wide_sgf : 0)) * (TILE_ROWS * MB) + lane * 2;
                        double2 tb[PASSES];
                        for (int spin = 0; spin < (1 << 22); spin++) {          // bounded: a lost contributor must not hang the GPU
                            bool ready = true;
#pragma unroll
                            for (int v = 0; v < PASSES; v++) {
                                asm volatile("ld.volatile.global.v2.f64 {%0,%1}, [%2];" : "=d"(tb[v].x), "=d"(tb[v].y) : "l"(src + v * 64));
                                ready = ready && __double_as_longlong(tb[v].x) != 0ll && __double_as_longlong(tb[v].y) != 0ll;
                            }
                            if (__all_sync(0xffffffffu, ready)) break;
                        }
#pragma unroll
                        for (int v = 0; v < PASSES; v++) {
                            *reinterpret_cast<double2*>(src + v * 64) = make_double2(0.0, 0.0);   // slot free for the next launch
                            *reinterpret_cast<double2*>(red + (size_t)warp * (TILE_ROWS * MB) + v * 64 + lane * 2) = tb[v];
                        }
                    }
                    named_bar_sync(4, NT);
                    if (tid < TILE_ROWS * MB) {
                        const int n_here = (wide_gl - base + 1) < wpr ? (wide_gl - base + 1) : wpr;
                        for (int w_ = 0; w_ < n_here; w_++) sum += red[(size_t)w_ * (TILE_ROWS * MB) + tid];   // CTA order: deterministic
                    }
                    if (base + wpr <= wide_gl) named_bar_sync(4, NT);            // the next round overwrites red[]
                }
                const int64_t tql = GRP ? (int64_t)t % p.tpw : (int64_t)t;      // tile index inside its weight
                const int64_t ybase = GRP ? ((int64_t)t / p.tpw) * p.y_slot_stride : 0;
                if (tid < TILE_ROWS * MB) {
                    const double sv = sum == 0.0 ? 0.0 : sum;                   // an exact zero was published as -0.0
                    const int rr = tid / MB, m = tid % MB;
                    const int64_t n = tql * TILE_ROWS + rr;
                    if constexpr (EPI) {
                        if (m < p.M) s_yfix[m][rr] = (float)(sv + ((p.bias && n < p.N) ? (double)p.bias[n] : 0.0));
                    } else {
                        if (n < p.N && m < p.M) mv_store<RP>(p, rp, ybase + (int64_t)m * p.ldy + n, sv + (mv_use_bias<RP>(p) ? (double)p.bias[n] : 0.0));
                    }
                }
                if constexpr (EPI) {
                    named_bar_sync(4, NT);
                    if (warp == 0)
                        for (int m = 0; m < p.M; m++) swiglu_tile_epilogue(p, s_yfix[m], tql, GRP ? (int)(t / p.tpw) : m, lane);
                }
                if (MV_TRACE_ON(p) && tid == 0) p.trace[g * 8 + 7] = globaltimer_ns();
            }
        }
#pragma unroll
        for (int s4 = 0; s4 < MV_STEPS; s4++)
#pragma unroll
            for (int m = 0; m < MB; m++) acc[s4][m] = 0.0;

        // ---- next segment / tile ----
        j += seg_left;
        xk_off = 0u;
        if (seg == 0 && sp.nT > 0) { seg = 1; seg_left = sp.nT; t = sp.tT; }
        else if (seg != 2) { seg = 2; seg_left = KC; t = sp.tF; }
        else { seg_left = KC; t++; }

    }
    if constexpr (RP) {
        // ---- fused exchange, producer side: this CTA's peer stores are all issued; the last CTA of the launch publishes ----
        named_bar_sync(MV_BAR_DONE, MV_CONSUMER_WARPS * 32 + 32);
        if (tid == 0) {
            uint8_t* mine = p.comm.peers[p.comm.rank];
            if (p.rp_mode == RP_ALLREDUCE) {
                // self-validating slots: no fence, no flag -- only the local epoch bookkeeping (last CTA advances it)
                ar_epoch_arrive(mine, rp.epoch, (unsigned int)G);
            } else {
                unsigned int* done = reinterpret_cast<unsigned int*>(mine + COMM_OFF_AG_DONE);
                asm volatile("fence.acq_rel.sys;" ::: "memory");  // the CTA's peer stores (ordered before this thread by the barrier) are performed system-wide
                unsigned int old;
                asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(done) : "memory");
                if (old == (unsigned int)(G - 1)) {
                    *done = 0u;  // next launch (ordered after this one by the stream)
                    comm_raise_flags(p.comm, COMM_OFF_AG_FLAGS, 0, rp.epoch);
                    *reinterpret_cast<unsigned int*>(mine + COMM_OFF_AG_EPOCH) = rp.epoch;
                }
            }
        }
    }
    if (MV_TRACE_ON(p) && tid == 0) p.trace[g * 8 + 3] = globaltimer_ns();
}

template <class F, int MB, bool PRO, bool GRP, int OUT = OUT_PLAIN, class F2 = F>
static cudaError_t launch_t(const MatvecParams& p, int grid, int smem, cudaStream_t st) {
    static std::atomic<bool> configured[16];   // per device; racing first calls both set the attribute (idempotent): re-entrant
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 16 || !configured[dev].load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(matvec_kernel<F, MB, PRO, GRP, OUT, F2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024);  // + static shared memory (epilogue tiles, reductions) <= 227 KB
        if (e != cudaSuccess) return e;
        if (dev < 16) configured[dev].store(true, std::memory_order_release);
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(MV_THREADS);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // PDL: overlap with the predecessor's tail
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t le = cudaLaunchKernelEx(&cfg, matvec_kernel<F, MB, PRO, GRP, OUT, F2>, p);
    if (le != cudaSuccess) return le;
    count_launch();
    return cudaGetLastError();
}

// dual-format launch (MatvecParams::w2): plain output, optional norm prologue
template <class F, class F2>
static cudaError_t launch_dual(const MatvecParams& p, int mb, int grid, int smem, cudaStream_t st) {
    if (p.w_table || p.rp_mode != RP_NONE || p.xq_out || !p.w2) return cudaErrorInvalidValue;
    switch (mb) {
        case 1: return p.pro ? launch_t<F, 1, true, false, OUT_PLAIN, F2>(p, grid, smem, st) : launch_t<F, 1, false, false, OUT_PLAIN, F2>(p, grid, smem, st);
        case 2: return p.pro ? launch_t<F, 2, true, false, OUT_PLAIN, F2>(p, grid, smem, st) : launch_t<F, 2, false, false, OUT_PLAIN, F2>(p, grid, smem, st);
        case 4: return p.pro ? launch_t<F, 4, true, false, OUT_PLAIN, F2>(p, grid, smem, st) : launch_t<F, 4, false, false, OUT_PLAIN, F2>(p, grid, smem, st);
        default: return cudaErrorInvalidValue;
    }
}

template <class F>
static cudaError_t launch_f(const MatvecParams& p, int mb, int grid, int smem, cudaStream_t st) {
    if (p.w_table) {
        if (mb != 1 || p.pro || p.rp_mode) return cudaErrorInvalidValue;
        return p.xq_out ? launch_t<F, 1, false, true, OUT_SWIGLU>(p, grid, smem, st) : launch_t<F, 1, false, true>(p, grid, smem, st);
    }
    if (p.rp_mode != RP_NONE) {  // fused tensor-parallel exchange (row-parallel o / down, vocabulary-parallel lm_head)
        if (p.pro || p.xq_out) return cudaErrorInvalidValue;
        switch (mb) {
            case 1: return launch_t<F, 1, false, false, OUT_REMOTE>(p, grid, smem, st);
            case 2: return launch_t<F, 2, false, false, OUT_REMOTE>(p, grid, smem, st);
            case 4: return launch_t<F, 4, false, false, OUT_REMOTE>(p, grid, smem, st);
            default: return cudaErrorInvalidValue;
        }
    }
    if (p.xq_out) {  // fused SwiGLU + quantise epilogue (interleaved gate|up weight)
        switch (mb) {
            case 1: return p.pro ? launch_t<F, 1, true, false, OUT_SWIGLU>(p, grid, smem, st) : launch_t<F, 1, false, false, OUT_SWIGLU>(p, grid, smem, st);
            case 2: return p.pro ? launch_t<F, 2, true, false, OUT_SWIGLU>(p, grid, smem, st) : launch_t<F, 2, false, false, OUT_SWIGLU>(p, grid, smem, st);
            case 4: return p.pro ? launch_t<F, 4, true, false, OUT_SWIGLU>(p, grid, smem, st) : launch_t<F, 4, false, false, OUT_SWIGLU>(p, grid, smem, st);
            default: return cudaErrorInvalidValue;
        }
    }
    switch (mb) {
        case 1: return p.pro ? launch_t<F, 1, true, false>(p, grid, smem, st) : launch_t<F, 1, false, false>(p, grid, smem, st);
        case 2: return p.pro ? launch_t<F, 2, true, false>(p, grid, smem, st) : launch_t<F, 2, false, false>(p, grid, smem, st);
        case 4: return p.pro ? launch_t<F, 4, true, false>(p, grid, smem, st) : launch_t<F, 4, false, false>(p, grid, smem, st);
        default: return cudaErrorInvalidValue;
    }
}


}  // namespace b200q
