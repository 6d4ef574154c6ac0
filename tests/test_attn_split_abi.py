"""CPU: host-side surface of the split-context decode attention -- the single-CTA limit, the workspace size rule, and the
argument / workspace checks that return before anything is launched."""
import ctypes as C

import numpy as np

from blazr_b200 import ops


def _expected_ws(nh, hd, max_ctx, M):
    al = lambda b: (b + 255) // 256 * 256
    s_max = min(-(-max_ctx // 256), 128)
    rows = M * nh
    return al(rows * max_ctx * 4) + al(rows * s_max * 4) + al(rows * s_max * 8) + al(rows * s_max * hd * 8)


def test_single_cta_limit_and_workspace_bytes():
    L = ops.lib()
    assert L.b200q_attn_decode_max_ctx() == 40960
    for nh, nkv, hd, max_ctx, M in ((32, 8, 64, 131072, 1), (64, 8, 128, 131072, 4), (8, 8, 128, 1, 1), (32, 8, 128, 40960, 256)):
        assert L.b200q_attn_split_workspace_bytes(nh, nkv, hd, max_ctx, M) == _expected_ws(nh, hd, max_ctx, M)
    # score offsets of M = 256 at 128k positions pass 2^31: the size is computed in 64 bits
    assert L.b200q_attn_split_workspace_bytes(32, 8, 128, 131072, 256) > 2 ** 32
    for bad in ((32, 8, 96, 4096, 1), (32, 7, 64, 4096, 1), (32, 8, 64, 0, 1), (32, 8, 64, 4096, 0), (32, 0, 64, 4096, 1)):
        assert L.b200q_attn_split_workspace_bytes(*bad) == 0


def test_short_workspace_and_bad_arguments_are_refused_before_launch():
    L = ops.lib()
    nh, nkv, hd, max_ctx, M = 8, 2, 64, 65536, 1
    need = int(L.b200q_attn_split_workspace_bytes(nh, nkv, hd, max_ctx, M))
    dummy = C.c_void_p(16)   # never dereferenced: every check below fails on the host
    rc = L.b200q_attn_decode_split(dummy, dummy, dummy, dummy, dummy, nh, nkv, hd, max_ctx, C.c_int64(M), dummy, None, dummy,
                                   C.c_size_t(need - 256), None)
    assert rc == -4 and b"workspace" in L.b200q_last_error()
    rc = L.b200q_attn_decode_paged_split(dummy, dummy, dummy, dummy, dummy, None, 16, max_ctx // 16, dummy, nh, nkv, hd, C.c_int64(M), dummy,
                                         None, dummy, C.c_size_t(need - 256), None)
    assert rc == -4
    rc = L.b200q_attn_decode_split(dummy, dummy, dummy, dummy, dummy, nh, nkv, 96, max_ctx, C.c_int64(M), dummy, None, dummy,
                                   C.c_size_t(need), None)
    assert rc == -2   # head_dim 96: no kernel
    rc = L.b200q_attn_decode_split(dummy, dummy, dummy, dummy, dummy, nh, 3, hd, max_ctx, C.c_int64(M), dummy, None, dummy, C.c_size_t(need), None)
    assert rc == -1
    rc = L.b200q_attn_decode_split(dummy, dummy, dummy, dummy, dummy, nh, nkv, hd, max_ctx, C.c_int64(M), None, None, dummy, C.c_size_t(need), None)
    assert rc == -1   # neither xq nor attn_out
    # the single-CTA entry point keeps its limit
    rc = L.b200q_attn_decode(dummy, dummy, dummy, dummy, dummy, nh, nkv, hd, 40961, C.c_int64(M), dummy, None, None)
    assert rc == -2
