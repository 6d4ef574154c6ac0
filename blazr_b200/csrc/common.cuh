// common.cuh -- PTX wrappers (mbarrier, bulk async copy, PDL, dp4a) and small helpers for sm_100a.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace b200q {

constexpr int TILE_ROWS = 128;  // weight rows per tile (= UMMA M)
constexpr int CHUNK_K = 256;    // k elements per chunk (one K-quant super-block)
constexpr int ACT_REC_BYTES = 320;  // per (k-chunk, m): 256 x int8 | 8 x f32 d | 8 x (2 x int16 bsum16)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ---- mbarrier ----
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// raw 32-bit shared-window addresses (computed once outside hot loops: no per-iteration cvta)
__device__ __forceinline__ void mbar_arrive_sa(uint32_t bar_sa) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar_sa) : "memory");
}
// the retry loop stays inside one asm statement: no compiler-built loop (and convergence region) around a per-lane flag
__device__ __forceinline__ void mbar_wait_sa(uint32_t bar_sa, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n"
        "MBAR_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra MBAR_WAIT;\n\t}" ::"r"(bar_sa),
        "r"(parity)
        : "memory");
}

// ---- bulk async copy global -> shared (TMA engine, 1-D), completion on an mbarrier ----
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// same with an L2 evict-first policy for streamed-once weights
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
        : "memory");
}

__device__ __forceinline__ long long globaltimer_ns() {
    long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// Deterministic expf: only IEEE add/mul/fma in a fixed order, mirrored line by line by oracle/quant_oracle.c
// orc_det_expf, so activations downstream of softmax / SiLU are bit-reproducible against the CPU oracle.
__device__ __forceinline__ float det_expf(float x) {
    x = fminf(fmaxf(x, -87.0f), 88.0f);
    const float n = rintf(__fmul_rn(x, 1.44269504f));
    float r = fmaf(n, -0.693145752f, x);
    r = fmaf(n, -1.42860677e-6f, r);
    float p = 1.0f / 720.0f;
    p = fmaf(p, r, 1.0f / 120.0f);
    p = fmaf(p, r, 1.0f / 24.0f);
    p = fmaf(p, r, 1.0f / 6.0f);
    p = fmaf(p, r, 0.5f);
    p = fmaf(p, r, 1.0f);
    p = fmaf(p, r, 1.0f);
    return __fmul_rn(p, __int_as_float(((int)n + 127) << 23));
}

// Element rule of an f16 KV cache (decode attention): f16_rn(clamp(x, +-65504)).  Finite inputs stay finite; fmaxf maps NaN
// to -65504.  Restated by blazr_b200/decode.py kv_round (prefill writes) and tests/kv16_ref.py kv_round_np (the oracle).
__device__ __forceinline__ __half kv_f16_rn(float x) { return __float2half_rn(fminf(fmaxf(x, -65504.0f), 65504.0f)); }

// one elected lane of a converged warp (the compiler then emits tcgen05 / TMA instructions of the guarded region
// without per-instruction uniformity loops)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// ---- programmatic dependent launch ----
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- named barrier over a subset of the CTA ----
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// unsigned-byte x signed-byte dot product accumulate (dp4a.u32.s32)
__device__ __forceinline__ int dp4a_us(uint32_t a_u8x4, uint32_t b_s8x4, int c) {
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a_u8x4), "r"(b_s8x4), "r"(c));
    return d;
}

// ---- shared memory loads ----
__device__ __forceinline__ uint4 lds128(const void* p) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem_u32(p)));
    return v;
}
__device__ __forceinline__ uint2 lds64(const void* p) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(smem_u32(p)));
    return v;
}

__device__ __forceinline__ uint4 lds128_sa(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint2 lds64_sa(uint32_t a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds32_sa(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds16_sa(uint32_t a) {
    uint32_t v;
    asm volatile("{\n\t.reg .u16 t;\n\tld.shared.u16 t, [%1];\n\tcvt.u32.u16 %0, t;\n\t}" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds8_sa(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
// a lane-constant value the compiler must keep in a register instead of re-deriving it from threadIdx inside a hot loop
__device__ __forceinline__ uint32_t keep_in_reg(uint32_t v) {
    asm volatile("" : "+r"(v));
    return v;
}

__device__ __forceinline__ float half_bits_to_float(uint16_t h) { return __half2float(__ushort_as_half(h)); }
// (f16 in the low or high half of hw) x (f16 in the low half of q), one rounding to f32 (sm_100 FHFMA); with q = an integer
// n < 1024 as f16 bits (the subnormal n * 2^-24) the result is h * n * 2^-24, exact whenever h * n has <= 24 significant bits
template <int HALF>
__device__ __forceinline__ float fma_f16_f32(uint32_t hw, uint32_t q) {
    uint16_t lo, hi;
    asm("mov.b32 {%0,%1}, %2;" : "=h"(lo), "=h"(hi) : "r"(hw));
    float r;
    asm("fma.rn.f32.f16 %0, %1, %2, %3;" : "=f"(r) : "h"(HALF ? hi : lo), "h"((uint16_t)q), "f"(-0.0f));
    return r;
}

// dtype codes mirror b200q_dtype
template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

__device__ __forceinline__ void store_out(void* y, int dtype, int64_t idx, float v) {
    if (dtype == 0) reinterpret_cast<float*>(y)[idx] = v;
    else if (dtype == 1) reinterpret_cast<__half*>(y)[idx] = __float2half_rn(v);
    else reinterpret_cast<__nv_bfloat16*>(y)[idx] = __float2bfloat16_rn(v);
}
// matvec epilogue: the exact f64 sum is rounded once to the output type, or kept (dtype 3) for the TP all-reduce
__device__ __forceinline__ void store_out_d(void* y, int dtype, int64_t idx, double v) {
    if (dtype == 3) reinterpret_cast<double*>(y)[idx] = v;
    else store_out(y, dtype, idx, (float)v);
}
__device__ __forceinline__ float load_in(const void* x, int dtype, int64_t idx) {
    if (dtype == 0) return reinterpret_cast<const float*>(x)[idx];
    if (dtype == 1) return __half2float(reinterpret_cast<const __half*>(x)[idx]);
    return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(x)[idx]);
}

}  // namespace b200q
