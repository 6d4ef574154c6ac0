"""GPU parity tests for the tcgen05/TMEM dequant-GEMM path (M >= 5: batched decode and prefill) against
the CPU oracle's f32 flavour A (dequantized weights x f32 activations, double accumulation).

Tolerance (north_star): max-abs error / max-abs reference <= 1e-2.  The kernel rounds weights and
activations to f16 (2^-11 relative each) and accumulates in f32, so the observed error is ~1e-3.  On top of that contract,
every element is held to the error bound of its own arithmetic (qcases.elementwise_bound: the f16 weight of unit_to_f16, the
f16 staging of the activations, one f32 rounding per 16-k MMA step and per split-K add), which the 1e-2 metric cannot see.
tests/test_gpu_gemm_exact.py pins the same kernel bit for bit on exactly representable data.
"""
import numpy as np
import pytest
import torch

from blazr_b200 import ops, synth
from qcases import ALL, Case, elementwise_bound, elementwise_violations, plan_for, stage_x16

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(120)]
TOL = 1e-2


def rel_err(y, ref):
    return float(np.abs(y.astype(np.float64) - ref.astype(np.float64)).max() / max(np.abs(ref).max(), 1e-30))


def assert_elementwise(c: Case, x: np.ndarray, y: np.ndarray, M: int):
    """every element within the bound of the GEMM's own arithmetic (split factor from the plan of an M-row call)"""
    S = plan_for(c.w, M, torch.cuda.get_device_properties(0).multi_processor_count)["S"]
    ref, tol = elementwise_bound(stage_x16(c.x_perm(x)), c.w16(), c.w.K_pad, S, c.bias)
    bad = elementwise_violations(y, ref, tol)
    assert bad == 0, f"{c.fmt} [{c.N}x{c.K}] M={M} S={S}: {bad} elements outside the per-element bound, worst " \
                     f"{float((np.abs(y.astype(np.float64) - ref) / np.maximum(tol, 1e-300)).max()):.3g} x tol"


@pytest.mark.parametrize("fmt", ALL)
@pytest.mark.parametrize("NKM", [(128, 256, 32), (256, 1024, 5), (200, 768, 100), (1408, 2048, 32), (384, 4096, 256), (256, 14336, 64)])
def test_gemm_vs_oracle(client, fmt, NKM):
    N, K, M = NKM
    c = Case(client, fmt, N, K, seed=N + K + M)
    x = synth.random_act(M, K, seed=M)
    y = client.quant_matmul(torch.from_numpy(x).cuda(), c.w, path=ops.PATH_GEMM).cpu().numpy()
    assert y.shape == (M, N)
    assert np.isfinite(y).all()
    assert rel_err(y, c.oracle_a(x)) < TOL
    assert_elementwise(c, x, y, M)


@pytest.mark.parametrize("fmt", ["Q4_K", "Q6_K", "Q8_0", "AWQ"])
def test_gemm_multiple_m_tiles_and_ragged_m(client, fmt):
    N, K, M = 640, 1024, 300  # two m-tiles of 160 rows (last one ragged) x 5 n-tiles: persistent loop
    c = Case(client, fmt, N, K, seed=4)
    x = synth.random_act(M, K, seed=2)
    y = client.quant_matmul(torch.from_numpy(x).cuda(), c.w).cpu().numpy()  # auto dispatch -> GEMM
    assert rel_err(y, c.oracle_a(x)) < TOL


def test_gemm_many_tiles_persistent(client):
    """more tiles than SMs: each CTA walks several (n-tile, m-tile) pairs and re-uses its TMEM"""
    N, K, M = 128 * 40, 512, 1024  # 40 x 4 = 160 tiles
    c = Case(client, "Q4_K", N, K, seed=6)
    x = synth.random_act(M, K, seed=3)
    y = client.quant_matmul(torch.from_numpy(x).cuda(), c.w).cpu().numpy()
    assert rel_err(y, c.oracle_a(x)) < TOL


def test_gemm_matches_matvec_path(client):
    """M = 4 through both kernels: int8-activation dp4a path and f16 tensor path agree within tolerance"""
    N, K, M = 512, 2048, 4
    c = Case(client, "Q6_K", N, K, seed=8)
    x = torch.from_numpy(synth.random_act(M, K)).cuda()
    y1 = client.quant_matmul(x, c.w, path=ops.PATH_MATVEC).cpu().numpy()
    y2 = client.quant_matmul(x, c.w, path=ops.PATH_GEMM).cpu().numpy()
    assert rel_err(y2, y1) < TOL


def test_gemm_half_io_bias_and_strides(client):
    N, K, M = 256, 1024, 48
    c = Case(client, "GPTQ", N, K, seed=9, bias=True)
    xbig = torch.from_numpy(synth.random_act(M, K + 8)).cuda().half()
    x = xbig[:, :K]
    ybig = torch.zeros((M, N + 16), device="cuda", dtype=torch.float16)
    client.quant_matmul(x, c.w, out=ybig[:, :N])
    ref = c.oracle_a(x.float().cpu().numpy())
    assert rel_err(ybig[:, :N].float().cpu().numpy(), ref) < TOL
    assert float(ybig[:, N:].abs().max()) == 0.0


def test_gemm_act_order_permutation(client):
    N, K, M = 256, 1024, 64
    c = Case(client, "GPTQ_ACT", N, K, seed=10)
    x = synth.random_act(M, K, seed=1)
    y = client.quant_matmul(torch.from_numpy(x).cuda(), c.w).cpu().numpy()
    assert rel_err(y, c.oracle_a(x)) < TOL


def test_gemm_prefill_shape_property(client):
    """BASELINE config shape (Mistral-7B q_proj, S = 2048): check sampled rows against the oracle and
    linearity in the activations (scaling x by 2 is exact in f16/f32)"""
    N, K, M = 4096, 4096, 2048
    c = Case(client, "Q6_K", N, K, seed=42)
    x = torch.from_numpy(synth.random_act(M, K, seed=4)).cuda()
    y = client.quant_matmul(x, c.w)
    y2 = client.quant_matmul(2.0 * x, c.w)
    assert torch.allclose(y2, 2.0 * y, rtol=1e-3, atol=1e-3)  # f16 staging: subnormal inputs round differently
    rows = [0, 1, 777, 2047]
    ref = c.oracle_a(x[rows].cpu().numpy())
    assert rel_err(y[rows].cpu().numpy(), ref) < TOL
    assert_elementwise(c, x[rows].cpu().numpy(), y[rows].cpu().numpy(), M)


@pytest.mark.parametrize("fmt,bias", [("Q6_K", False), ("Q4_K", False), ("GPTQ", True)])
def test_gemm_tail_split_k_wave_quantisation(client, fmt, bias, monkeypatch):
    """(opt-in path, B200Q_GEMM_TAIL=1 -- the switch is read once per process, so the driver's default suite exercises the plain
    persistent loop on this shape and `B200Q_GEMM_TAIL=1 pytest -k tail_split` the split form; both were run green in round 2)
    wide-M launch whose tile count is not a multiple of the SM count: the tiles of the last, partial wave are split along K
    (tail split-K: 19 x 8 = 152 tiles on 148 SMs -> 4 tail tiles x 4 splits), partial accumulators reduced by a second kernel;
    ragged M so the last activation tile is partly empty"""
    N, K, M = 128 * 19, 2048, 2000
    c = Case(client, fmt, N, K, seed=12, bias=bias) if bias else Case(client, fmt, N, K, seed=12)
    x = synth.random_act(M, K, seed=5)
    y = client.quant_matmul(torch.from_numpy(x).cuda(), c.w).cpu().numpy()
    assert rel_err(y, c.oracle_a(x)) < TOL
