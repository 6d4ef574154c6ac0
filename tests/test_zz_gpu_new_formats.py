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


# ---- EXPERIMENTAL persistent op-list kernel (csrc/dstep_impl.cuh): green on hardware in round 2 (8 passed) and measured SLOWER
# than the PDL-chained launches (407 vs 560 tok/s on Mistral-7B Q6_K), so it stays opt-in.  A persistent kernel with grid barriers
# can hang if it is ever broken, and a hung kernel cannot be interrupted by pytest: the test only runs when asked for
# (B200Q_TEST_EXPERIMENTAL=1, under `timeout`), never in the default -m gpu suite.
@pytest.mark.skipif(__import__("os").environ.get("B200Q_TEST_EXPERIMENTAL", "0") == "0", reason="experimental persistent kernel: opt-in (B200Q_TEST_EXPERIMENTAL=1)")
@pytest.mark.parametrize("mode", ["1", "2"])
@pytest.mark.parametrize("scheme", ["Q6_K", "Q4_K_M", "Q8_0", "AWQ"])
def test_dstep_programs_reproduce_the_launch_per_op_step(client, scheme, mode, monkeypatch):
    """B200Q_DSTEP=1: 3 launches per layer (program, attention, program); B200Q_DSTEP=2: the whole step in ONE launch.
    Both must give the same logits, bit for bit, as the 8 separate launches per layer (identical arithmetic), over several
    dependent steps; then under CUDA-graph replay"""
    import numpy as np
    import torch
    from blazr_b200 import decode
    cfg = decode.PRESETS["tiny"]
    hm = decode.build_host_model(cfg, scheme, seed=31)
    ref = decode.Decoder(client, cfg, scheme, batch=1, max_ctx=64, host=hm)
    monkeypatch.setenv("B200Q_DSTEP", mode)
    exp = decode.Decoder(client, cfg, scheme, batch=1, max_ctx=64, host=hm)
    assert (exp.programs is not None) if mode == "1" else (exp.step_program is not None)
    for d in (ref, exp):
        d.reset([3])
    for _ in range(6):
        ref.step()
        exp.step()
        torch.cuda.synchronize()
        a, b = ref.logits.cpu().numpy(), exp.logits.cpu().numpy()
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    prompt = np.asarray([[3, 1, 4, 1, 5]])
    assert np.array_equal(ref.generate(prompt, 16, use_graph=True), exp.generate(prompt, 16, use_graph=True))


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
