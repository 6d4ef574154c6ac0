"""Shared builders for the GPU parity tests: one synthetic weight -> (device handle, oracle views), the f16 weight the
tcgen05 GEMM multiplies, a Python restatement of its launch plan and the per-element error bound it is held to."""
from __future__ import annotations

import math

import numpy as np

import oracle
from blazr_b200 import ops, synth

GGML_GPU = ["Q4_K", "Q6_K", "Q8_0", "Q4_0", "Q5_0", "IQ4_NL"]  # the last three run as exact re-encodings (formats.cuh adaptors)
INT4 = ["AWQ", "GPTQ", "GPTQ_ACT", "GPTQ_Z0", "AWQ_G64"]
ALL = GGML_GPU + INT4
# the remaining K / IQ / TQ formats (tests/test_zz_gpu_new_formats.py)
NEW = ["Q5_K", "Q4_1", "Q5_1", "Q2_K", "Q3_K", "IQ4_XS", "TQ2_0", "TQ1_0", "IQ2_XXS", "IQ2_XS", "IQ3_XXS", "IQ2_S", "IQ3_S", "IQ1_S", "IQ1_M"]

# integer-exact data (Case(exact=True)): every scale is a small power of two, so every f16 weight is a multiple of 2^-8
EXACT_GGML_SCALE = 2.0 ** -8
EXACT_GROUP_SCALES = (2.0 ** -8, 2.0 ** -7, 2.0 ** -6)
EXACT_BIAS_UNIT = 2.0 ** -10   # = smallest weight scale x activation unit 2^-2: bias adds exactly to the accumulator


def _exact_ggml(t: int, blocks: np.ndarray) -> np.ndarray:
    """overwrite every f16 d and min field of random blocks with 2^-8"""
    N = blocks.shape[0]
    bb = synth.GGML_SIZES[t][1]
    blk = blocks.reshape(-1, bb).copy()
    d_off, m_off, _, _ = synth._FIELDS[t]
    one = np.full(blk.shape[0], EXACT_GGML_SCALE, dtype=np.float16)
    for o in list(d_off) + list(m_off):
        blk[:, o:o + 2] = one.view(np.uint8).reshape(-1, 2)
    if t == synth.GGML["IQ1_M"]:
        synth.set_iq1m_d(blk, one)
    return blk.reshape(N, -1)


class Case:
    """Holds the device weight and everything the oracle needs for the same weight.  client None: oracle views only.
    exact: integer-exact data (scales 2^-8 / from {2^-8, 2^-7, 2^-6}, integer zeros, bias a multiple of 2^-10)."""

    def __init__(self, client, fmt: str, N: int, K: int, seed: int = 0, bias: bool = False, exact: bool = False):
        self.fmt, self.N, self.K = fmt, N, K
        self.perm = None
        self.bias = None
        self.w = None
        rng = np.random.Generator(np.random.PCG64(seed + 977))
        if fmt in synth.GGML:
            t = synth.GGML[fmt]
            self.blocks = synth.random_ggml(t, N, K, seed=seed)
            if exact:
                self.blocks = _exact_ggml(t, self.blocks)
            self.t = t
            if client is not None:
                self.w = client.weight_from_ggml(t, self.blocks, N, K)
            self.qi, self.a, self.b, self.sub = oracle.decompose_ggml(t, self.blocks, N, K)
            self.deq = oracle.dequant_ggml(t, self.blocks, N, K)
        elif fmt.startswith("AWQ"):
            gs = 64 if fmt == "AWQ_G64" else 128
            qw, sc, zr = synth.random_awq(N, K, gs, seed=seed)
            if exact:
                sc = rng.choice(EXACT_GROUP_SCALES, size=sc.shape).astype(np.float32)
            self.src = (qw, sc, zr, gs)
            dq = ops.DecomposedQuantTensor(qw, sc, zr, None, ops.DecomposedQuantMethod("awq", gs), (N, K))
            if client is not None:
                self.w = client.weight_from_decomposed(dq)
            self.qi, self.a, self.b, self.sub = oracle.awq_decompose(qw, sc, zr, gs)
            self.deq = oracle.awq_dequant(qw, sc, zr, gs)
        elif fmt.startswith("GPTQ"):
            gs = 128
            act = fmt == "GPTQ_ACT"
            zpo = 0 if fmt == "GPTQ_Z0" else 1
            qw, sc, qz, gi, bs = synth.random_gptq(N, K, gs, seed=seed, act_order=act, bias=bias)
            if exact:
                sc = rng.choice(EXACT_GROUP_SCALES, size=sc.shape).astype(np.float32)
                if bias:
                    bs = (rng.integers(-512, 513, size=N) * EXACT_BIAS_UNIT).astype(np.float32)
            self.bias = bs
            dq = ops.DecomposedQuantTensor(qw, sc, qz, gi, ops.DecomposedQuantMethod("gptq", gs), (N, K), bias=bs, zero_plus_one=zpo)
            if client is not None:
                self.w = client.weight_from_decomposed(dq)
            self.qi, self.a, self.b, self.sub, self.perm = oracle.gptq_decompose(qw, sc, qz, gi if act else None, gs, zpo)
            self.deq = oracle.gptq_dequant(qw, sc, qz, gi, gs, zpo)
        else:
            raise ValueError(fmt)

    def x_perm(self, x: np.ndarray) -> np.ndarray:
        """activations in the K order the decomposition uses (GPTQ act-order permutes K)"""
        return x if self.perm is None else np.ascontiguousarray(x[:, self.perm])

    def oracle_a(self, x: np.ndarray) -> np.ndarray:
        return oracle.matmul_dense(self.deq, x, self.bias)

    def oracle_b(self, x: np.ndarray) -> np.ndarray:
        return oracle.matmul_q8(self.qi, self.a, self.b, self.sub, self.x_perm(x), self.bias)

    def w16(self) -> np.ndarray:
        """f16 [N, K] weight the tcgen05 GEMM multiplies, in decomposition (x_perm) order: unit_to_f16 (gemm_impl.cuh) rounds
        a and b to f16 and forms a16 * q - b16 with ONE rounding (HFMA2).  The exact value is formed in f64 and numpy's
        f64 -> f16 conversion rounds once (torch's goes through f32 and can round twice)."""
        a16 = np.repeat(self.a.astype(np.float16).astype(np.float64), self.sub, axis=1)
        b16 = np.repeat(self.b.astype(np.float16).astype(np.float64), self.sub, axis=1)
        return (self.qi.astype(np.float64) * a16 - b16).astype(np.float16)


def stage_x16(x: np.ndarray) -> np.ndarray:
    """the activation staging of the GEMM (gemm_tc.cu stage_x_kernel): f16_rn(clamp(x, +-65504))"""
    x = np.asarray(x, dtype=np.float32)
    return np.clip(x, np.float32(-65504.0), np.float32(65504.0)).astype(np.float16)


# ---- restatement of the GEMM launch plan (gemm_tc.cu pick_mt / pick_splits / gemm_ws_bytes / launch_gemm_tc), without the
# opt-in tail-split and multicast experiments and the B200Q_GEMM_* tuning variables ----
TILE_ROWS, CHUNK_K = 128, 256
SMEM_LIMIT, GT_HDR, GT_NX, GT_MAX_NW = 227 * 1024, 1024, 16, 4


def _align256(n: int) -> int:
    return (n + 255) // 256 * 256


def gemm_plan(N: int, K_pad: int, chunk_bytes: int, device_bytes: int, M: int, sms: int) -> dict:
    T, KC = -(-N // TILE_ROWS), K_pad // CHUNK_K
    MT = -(-M // 256)
    per = -(-M // MT)
    Mt = -(-per // 32) * 32
    tiles = T * MT
    smax = max(1, min(8, KC // 2))
    if M > 128:
        S = max(1, min(smax, sms // tiles))
    else:
        S, best = 1, 0.0
        for s in range(1, smax + 1):
            items = tiles * s
            waves = -(-items // sms)
            eff = items / (waves * sms)
            extra = s * M * N * 8.0 / device_bytes if s > 1 else 0.0
            eff = eff / (1.0 + extra) - 0.01 * (s - 1)
            if eff > best:
                best, S = eff, s
    xsub = 4 if Mt <= 64 else 1
    x_stage = Mt * 128 * xsub
    nx = max(4, min(GT_NX, (128 * 1024) // x_stage))
    if xsub == 4:
        nx = 4 if Mt <= 32 else 3
    w_stage = (chunk_bytes + 127) // 128 * 128
    nw = min(GT_MAX_NW, (SMEM_LIMIT - GT_HDR - nx * x_stage) // w_stage)
    items = tiles * S
    grid = min(items, sms)
    xs = _align256(MT * Mt * K_pad * 2)
    ws = _align256(xs + (S * M * N * 4 if S > 1 else 0))
    per_cta = [len(range(b, items, grid)) for b in range(grid)]
    return dict(M=M, N=N, K_pad=K_pad, T=T, KC=KC, Mt=Mt, MT=MT, S=S, xsub=xsub, nx=nx, nw=nw, nslots=2 if Mt > 64 else 3,
                dq_warps=16 if Mt <= 128 else 8, items=items, grid=grid, max_items=max(per_cta),
                odd_multi=any(c >= 3 and c % 2 for c in per_cta), ws_bytes=ws)


def plan_for(w, M: int, sms: int) -> dict:
    i = w.info
    return gemm_plan(int(i.N), int(i.K_pad), int(i.chunk_bytes), int(i.device_bytes), M, sms)


def elementwise_bound(x16: np.ndarray, w16: np.ndarray, K_pad: int, S: int, bias=None):
    """(ref64, tol) of the tcgen05 GEMM on arbitrary data: ref64 = x16 . w16^T (+ bias) in f64, and
    |y - ref64| <= (ceil(K_pad / 16) + S + 2) * 2^-23 * (|x16| . |w16|^T + |bias|): one truncating f32 rounding per 16-k MMA
    step, one per split-K partial add, the bias add and the output rounding.  x16 in the weight's K order."""
    xa, wa = x16.astype(np.float64), w16.astype(np.float64)
    ref = xa @ wa.T
    mag = np.abs(xa) @ np.abs(wa).T
    if bias is not None:
        ref = ref + bias.astype(np.float64)
        mag = mag + np.abs(bias.astype(np.float64))
    return ref, (math.ceil(K_pad / 16) + S + 2) * 2.0 ** -23 * mag


def elementwise_violations(y: np.ndarray, ref: np.ndarray, tol: np.ndarray) -> int:
    return int((np.abs(y.astype(np.float64) - ref) > tol).sum())
