"""GPU parity of the remaining K / IQ / TQ formats: Q5_K, Q4_1, Q5_1, Q2_K, Q3_K, IQ4_XS, TQ2_0, TQ1_0, IQ2_XXS, IQ2_XS, IQ3_XXS,
IQ2_S, IQ3_S, IQ1_S, IQ1_M -- the same contracts as the headline formats (#1 dequantized weights, #2 integer partials, #3 matvec,
GEMM tolerance).  Round 1 shipped them xfail(strict=False) because they had never run on a B200; round 2's first GPU call ran all
of them green (gpurun_out/r2_pytest_gpu_1.log: 271 xpassed), so the marks are gone: a failure now turns the suite red.
"""
import pytest

import test_gpu_gemm as tg
import test_gpu_quant as tq
from qcases import NEW

pytestmark = [pytest.mark.gpu]


@pytest.mark.parametrize("name", NEW)
def test_dequant_golden_fixture_bit_exact(client, name):
    tq.test_dequant_golden_fixture_bit_exact(client, name)


@pytest.mark.parametrize("fmt", NEW)
@pytest.mark.parametrize("shape", [(128, 256), (200, 768), (8, 2048)])
def test_dequant_bit_exact_vs_oracle(client, fmt, shape):
    tq.test_dequant_bit_exact_vs_oracle(client, fmt, shape)


@pytest.mark.parametrize("fmt", NEW)
def test_int_partials_bit_exact(client, fmt):
    tq.test_int_partials_bit_exact(client, fmt)


@pytest.mark.parametrize("fmt", NEW)
@pytest.mark.parametrize("shape", tq.SHAPES)
def test_matvec_m1_vs_oracle(client, fmt, shape):
    tq.test_matvec_m1_vs_oracle(client, fmt, shape)


@pytest.mark.parametrize("fmt", NEW)
@pytest.mark.parametrize("M", [2, 4])
def test_matvec_small_batch(client, fmt, M):
    tq.test_matvec_small_batch(client, fmt, M)


@pytest.mark.parametrize("fmt", NEW)
@pytest.mark.parametrize("NKM", [(128, 256, 32), (200, 768, 100), (384, 4096, 256), (256, 14336, 64)])
def test_gemm_vs_oracle(client, fmt, NKM):
    tg.test_gemm_vs_oracle(client, fmt, NKM)


def test_moe_layer_from_gguf_file(client, tmp_path):
    """GGUF stacked expert tensors -> expert banks -> MoE decode; equals the per-expert oracle (same status: Python glue over
    verified kernels)"""
    import gguf
    import numpy as np
    import torch
    import oracle
    from blazr_b200 import gguf_loader, synth
    E, hidden, ffn, top_k = 4, 512, 256, 2
    tq4, tq8 = synth.GGML["Q4_K"], synth.GGML["Q8_0"]
    gate = [synth.random_ggml(tq4, ffn, hidden, seed=10 + e) for e in range(E)]
    up = [synth.random_ggml(tq4, ffn, hidden, seed=20 + e) for e in range(E)]
    down = [synth.random_ggml(tq8, hidden, ffn, seed=30 + e) for e in range(E)]
    path = str(tmp_path / "moe.gguf")
    w = gguf.GGUFWriter(path, "llama")
    w.add_block_count(1)
    QT = gguf.GGMLQuantizationType
    for name, mats, qt in (("ffn_gate_exps", gate, QT.Q4_K), ("ffn_up_exps", up, QT.Q4_K), ("ffn_down_exps", down, QT.Q8_0)):
        st = np.ascontiguousarray(np.stack(mats, axis=0))
        w.add_tensor(f"blk.0.{name}.weight", st, raw_shape=st.shape, raw_dtype=qt)
    w.write_header_to_file(); w.write_kv_data_to_file(); w.write_tensors_to_file(); w.close()
    moe = gguf_loader.moe_mlp_from_gguf(client, gguf_loader.Gguf.open(path), 0)
    x = synth.random_act(1, hidden, seed=3)
    sel = np.array([[2, 0]], dtype=np.int32)
    gw = np.array([[0.7, 0.3]], dtype=np.float32)
    out = moe.forward_decode(torch.from_numpy(x).cuda(), torch.from_numpy(sel).cuda(), torch.from_numpy(gw).cuda()).cpu().numpy()
    ref = np.zeros((1, hidden), dtype=np.float32)
    for j in range(top_k):
        e = int(sel[0, j])
        gu = oracle.matmul_q8(*oracle.decompose_ggml(tq4, np.concatenate([gate[e], up[e]], axis=0), 2 * ffn, hidden), x)
        g_, u_ = gu[:, :ffn], gu[:, ffn:]
        act = ((g_ / (np.float32(1.0) + oracle.det_exp(-g_))).astype(np.float32) * u_).astype(np.float32)
        ref += gw[0, j] * oracle.matmul_q8(*oracle.decompose_ggml(tq8, down[e], hidden, ffn), act)
    assert float(np.abs(out - ref).max() / np.abs(ref).max()) < 1e-6
