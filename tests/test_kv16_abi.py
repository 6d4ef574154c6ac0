"""CPU: host surface of the f16 KV cache -- the *_kv attention entry points, their refusals before any launch, the split
workspace (independent of the cache type), and the element rule f16_rn(clamp(x, +-65504)) as the oracle helper and the
Decoder's prefill write restate it."""
import ctypes as C

import numpy as np
import torch

from blazr_b200 import decode, ops
from kv16_ref import Kv16Rows, kv_round_np

KV_FNS = ("b200q_attn_decode_kv", "b200q_attn_decode_paged_kv", "b200q_attn_decode_split_kv", "b200q_attn_decode_paged_split_kv")


def test_kv_entry_points_are_exported():
    L = ops.lib()
    for name in KV_FNS:
        assert name in ops.EXPORTS
        getattr(L, name)
    assert decode.KV_DTYPES["f32"][1] == 0 and decode.KV_DTYPES["f16"][1] == 1   # B200Q_F32, B200Q_F16


def _call(name, ck, kv_dtype, ws_bytes):
    """every other argument is valid; dummy device pointers are never dereferenced: each call below fails on the host"""
    L = ops.lib()
    d = C.c_void_p(16)
    nh, nkv, hd, max_ctx, M = 8, 2, 64, 65536, 1
    ws = (d, C.c_size_t(ws_bytes))
    if name == "b200q_attn_decode_kv":
        return L.b200q_attn_decode_kv(d, d, ck, d, kv_dtype, d, nh, nkv, hd, 4096, C.c_int64(M), d, None, None)
    if name == "b200q_attn_decode_paged_kv":
        return L.b200q_attn_decode_paged_kv(d, d, ck, d, kv_dtype, d, None, 16, 256, d, nh, nkv, hd, C.c_int64(M), d, None, None)
    if name == "b200q_attn_decode_split_kv":
        return L.b200q_attn_decode_split_kv(d, d, ck, d, kv_dtype, d, nh, nkv, hd, max_ctx, C.c_int64(M), d, None, *ws, None)
    return L.b200q_attn_decode_paged_split_kv(d, d, ck, d, kv_dtype, d, None, 16, max_ctx // 16, d, nh, nkv, hd, C.c_int64(M), d, None, *ws, None)


def test_bad_kv_dtype_and_misaligned_cache_are_refused_before_launch():
    L = ops.lib()
    need = int(L.b200q_attn_split_workspace_bytes(8, 2, 64, 65536, 1))
    for name in KV_FNS:
        short = need - 256   # a short workspace too: the cache checks come first
        for bad in (2, 3, -1, 7):   # B200Q_BF16, B200Q_F64, and values no enum has
            assert _call(name, C.c_void_p(16), bad, short) == -2, (name, bad)
            assert b"kv_dtype" in L.b200q_last_error()
        for kv_dtype in (0, 1):
            for addr in (8, 18, 20, 4104):
                assert _call(name, C.c_void_p(addr), kv_dtype, short) == -1, (name, kv_dtype, addr)
                assert b"aligned" in L.b200q_last_error()
        if "split" in name:   # with an aligned cache the next check is the workspace
            assert _call(name, C.c_void_p(16), 1, short) == -4


def test_split_workspace_does_not_depend_on_the_cache_type():
    # the workspace holds f32 scores and f64 partial sums only; the f16 and f32 forms take the same size
    L = ops.lib()
    for nh, nkv, hd, max_ctx, M in ((32, 8, 64, 131072, 1), (64, 8, 128, 131072, 4), (8, 8, 128, 1, 1)):
        n = int(L.b200q_attn_split_workspace_bytes(nh, nkv, hd, max_ctx, M))
        assert n > 0
        assert all(_ws_accepted(L, nh, nkv, hd, max_ctx, M, n, t) for t in (0, 1))


def _ws_accepted(L, nh, nkv, hd, max_ctx, M, n, kv_dtype):
    """a workspace one byte short is refused (-4) for either cache type; the exact size passes every host check (so the call is
    not made: it would launch)"""
    d = C.c_void_p(16)
    return L.b200q_attn_decode_split_kv(d, d, d, d, kv_dtype, d, nh, nkv, hd, max_ctx, C.c_int64(M), d, None, d, C.c_size_t(n - 1), None) == -4


EDGE = np.array([0.0, -0.0, 1.0, -1.0, 65504.0, -65504.0, 65519.9, -65519.9, 65520.0, 1e6, -1e6, np.inf, -np.inf,
                 2.0 ** -24, -(2.0 ** -24), 2.0 ** -25, 1.5 * 2.0 ** -25, 2.0 ** -14, 3.0 * 2.0 ** -16, 0.1, 1.0 / 3.0, 2049.0, 2051.0],
                dtype=np.float32)


def test_element_rule_on_edge_values():
    got = kv_round_np(EDGE)
    assert got.dtype == np.float16
    want = {65504.0: 65504.0, -65504.0: -65504.0, 65519.9: 65504.0, -65519.9: -65504.0, 65520.0: 65504.0, 1e6: 65504.0,
            -1e6: -65504.0, np.inf: 65504.0, -np.inf: -65504.0, 2.0 ** -24: 2.0 ** -24, 2.0 ** -25: 0.0, 1.5 * 2.0 ** -25: 2.0 ** -24,
            2049.0: 2048.0, 2051.0: 2052.0}
    for x, y in want.items():
        assert float(got[EDGE == np.float32(x)][0]) == y, x
    # ties go to even: 2^-25 (half the smallest subnormal) rounds to +0; negative tiny values keep their sign
    assert got[EDGE == np.float32(2.0 ** -25)].view(np.uint16)[0] == 0
    assert got[EDGE == np.float32(-(2.0 ** -24))].view(np.uint16)[0] == 0x8001
    assert np.isfinite(got).all()
    # NaN -> -65504 (fmaxf(NaN, -65504) = -65504 in the kernels)
    nan = kv_round_np(np.array([np.nan, -np.nan], dtype=np.float32))
    assert (nan == np.float16(-65504.0)).all()
    # agrees with torch's clamp-and-convert for finite values, and with the Decoder's write helper everywhere
    t = torch.from_numpy(EDGE)
    fin = torch.isfinite(t)
    ref = torch.clamp(t[fin], -65504.0, 65504.0).to(torch.float16).numpy()
    assert np.array_equal(got[fin.numpy()].view(np.uint16), ref.view(np.uint16))
    assert np.array_equal(decode.kv_round(t).numpy().view(np.uint16), got.view(np.uint16))
    assert float(decode.kv_round(torch.tensor([float("nan")]))[0]) == -65504.0


def test_element_rule_matches_torch_on_random_f32():
    rng = np.random.Generator(np.random.PCG64(16))
    x = np.concatenate([rng.standard_normal(100000) * s for s in (1e-6, 1e-3, 1.0, 1e3, 1e5)]).astype(np.float32)
    ref = torch.clamp(torch.from_numpy(x), -65504.0, 65504.0).to(torch.float16).numpy()
    assert np.array_equal(kv_round_np(x).view(np.uint16), ref.view(np.uint16))


def test_oracle_rows_are_stored_rounded():
    rows = Kv16Rows(np.array([[1e5, 0.1]], dtype=np.float32))
    rows.append(np.array([np.nan, -7.0], dtype=np.float32))
    assert all(r.dtype == np.float16 for r in rows)
    st = np.stack(rows).astype(np.float64)
    assert st.tolist() == [[65504.0, float(np.float16(0.1))], [-65504.0, -7.0]]
