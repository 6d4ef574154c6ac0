"""The tcgen05 dequant-GEMM, bit for bit.

Its arithmetic is fully defined: the weight is W16 = f16(a16 * q - b16) with one rounding (unit_to_f16, Case.w16), the
activations are staged as f16_rn(clamp(x, +-65504)), f16 x f16 products are exact in f32 and the accumulation is f32.
So on data where every partial sum is exactly representable, the output does not depend on the accumulation order, the
tile plan or the split-K factor, and must equal the f64 reference exactly:

  * the identity probe: x = c * I gives c * W16^T (+ bias), per format (dequant arithmetic, chunk -> tile -> row mapping,
    unit order and the [0,2,1,3] pair permutation shared by unit_to_f16 and the staging kernel);
  * the plan sweep: integer-exact data over shapes found by searching a Python restatement of the launch plan
    (qcases.gemm_plan), which covers every m-tile class, dequant-warp layout, weight-ring depth and split factor, and asserts
    that it did.

The CPU tests at the end check the references themselves and record what the per-element bound of tests/test_gpu_gemm.py
sees that the old 1e-2 metric did not.
"""
import os

import numpy as np
import pytest
import torch

from blazr_b200 import ops, synth
from qcases import ALL, NEW, Case, elementwise_bound, elementwise_violations, gemm_plan, plan_for, stage_x16
from test_gpu_gemm import TOL, rel_err

TORCH_DT = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
BLOCK32 = {"Q8_0", "Q4_0", "Q5_0", "IQ4_NL", "Q4_1", "Q5_1", "AWQ", "AWQ_G64", "GPTQ", "GPTQ_ACT", "GPTQ_Z0"}


def _sms() -> int:
    return torch.cuda.get_device_properties(0).multi_processor_count


def _w16_k_order(c: Case) -> np.ndarray:
    """W16 with its columns in the activations' K order (GPTQ act-order decomposes in permuted order)"""
    w16 = c.w16()
    return w16 if c.perm is None else np.ascontiguousarray(w16[:, np.argsort(c.perm)])


def _unit(v: np.ndarray) -> float:
    """largest power of two that divides every element"""
    v = np.abs(np.asarray(v, dtype=np.float64))
    v = v[v != 0]
    if v.size == 0:
        return 1.0
    m, e = np.frexp(v)
    im = (m * 2.0 ** 53).astype(np.int64)
    tz = np.log2((im & -im).astype(np.float64)).astype(np.int64)
    return 2.0 ** int((e - 53 + tz).min())


# ================================================================================================================================
# 1. identity probe
# ================================================================================================================================
PROBE = [(f, K) for f in ALL + NEW for K in ((256, 1408, 4096) if f in BLOCK32 else (256, 4096))]


@pytest.mark.gpu
@pytest.mark.timeout(300)
@pytest.mark.parametrize("fmt,K", PROBE)
def test_gemm_identity_is_the_f16_weight(client, fmt, K):
    """quant_matmul(c * I_K, w) == c * W16^T (+ bias, rounded once in f32), bit for bit: each output is one exact product.
    The Q4_K / Q6_K weights include f16-subnormal W16 values (~0.3 %): the probe shows tcgen05 keeps subnormal f16 operands."""
    c_ = 0.5
    eye = torch.eye(K, device="cuda") * c_
    xs = {"f32": eye, "bf16": eye.bfloat16()}
    fails, nsubn = [], 0
    for N in (8, 200, 1408):
        c = Case(client, fmt, N, K, seed=N + K, bias=fmt == "GPTQ")
        w16 = _w16_k_order(c)
        ref = c_ * w16.astype(np.float64).T
        if c.bias is not None:
            ref = ref + c.bias.astype(np.float64)
        ref32 = torch.from_numpy(ref.astype(np.float32)).cuda()
        w16t = torch.from_numpy(np.ascontiguousarray(w16.T)).cuda()
        subn = (w16t != 0) & (w16t.float().abs() < 2.0 ** -14)
        nsubn += int(subn.sum())
        for xd in ("f32", "bf16"):
            for yd in ("f32", "f16"):
                y = client.quant_matmul(xs[xd], c.w, out_dtype=TORCH_DT[yd], path=ops.PATH_GEMM)
                bad = y != ref32.to(TORCH_DT[yd])
                nbad = int(bad.sum())
                if nbad:
                    nsub = int((bad & subn).sum())
                    zero = int((bad & subn & (y == 0)).sum())
                    k, n = [int(i) for i in bad.nonzero()[0]]
                    fails.append(f"N={N} x {xd} y {yd}: {nbad} of {y.numel()} differ ({nsub} at f16-subnormal weights, {zero} of those "
                                 f"read 0; W16 has {int(subn.sum())} subnormals); first k={k} n={n}: {float(y[k, n])!r} vs "
                                 f"{float(ref32[k, n])!r}")
        c.w.free()
    assert not fails, f"{fmt} K={K}:\n" + "\n".join(fails)
    if fmt in ("Q4_K", "Q6_K"):
        assert nsubn > 0, "the probe data has no f16-subnormal weight"


# ================================================================================================================================
# 2. integer-exact sweep of the launch plan
# ================================================================================================================================
# candidate formats: one per distinct chunk size, plus the GPTQ variants the plan features name
SWEEP_FMTS = {  # name -> (Case format, bias, device chunk bytes)
    "Q4_K": ("Q4_K", False, 128 * 144), "Q6_K": ("Q6_K", False, 128 * 210), "Q8_0": ("Q8_0", False, 128 * 272),
    "AWQ": ("AWQ", False, 128 * 128 + 128 * 2 * 3), "GPTQ": ("GPTQ", False, 128 * 128 + 128 * 2 * 3),
    "GPTQ+bias": ("GPTQ", True, 128 * 128 + 128 * 2 * 3), "GPTQ_ACT": ("GPTQ_ACT", False, 128 * 128 + 128 * 2 * 3),
}
SWEEP_N = [8, 72, 200, 640, 1408, 2432, 4864, 5504, 38016]
SWEEP_K = [256, 512, 768, 1408, 1792, 2304, 3584, 4096]   # <= 4096 keeps the Q6_K column sums under 2^24 units
SWEEP_M = [1, 2, 3, 4, 5, 8, 24, 32, 33, 48, 64, 65, 96, 100, 128, 129, 160, 192, 200, 224, 256, 300, 384, 512, 1024, 2048]


def _k_ok(fmt: str, K: int) -> bool:
    return K % 256 == 0 if fmt in ("Q4_K", "Q6_K") else K % (32 if fmt == "Q8_0" else 128) == 0


# plan features the sweep must reach: name -> predicate over a candidate (fmt, N, K, M, plan)
FEATURES = {}
for _v in range(32, 257, 32):
    FEATURES[f"m-tile Mt={_v}"] = (lambda v: lambda c: c["plan"]["Mt"] == v)(_v)
FEATURES.update({
    "X stage xsub=4": lambda c: c["plan"]["xsub"] == 4,
    "X stage xsub=1": lambda c: c["plan"]["xsub"] == 1,
    "16 dequant warps + epilogue warps": lambda c: c["plan"]["dq_warps"] == 16,
    "8 dequant warps": lambda c: c["plan"]["dq_warps"] == 8,
    "weight ring nw=2": lambda c: c["plan"]["nw"] == 2,
    "weight ring nw=3": lambda c: c["plan"]["nw"] == 3,
    "weight ring nw=4": lambda c: c["plan"]["nw"] == 4,
})
for _s in range(1, 9):
    FEATURES[f"M<=128, S={_s}"] = (lambda s: lambda c: c["M"] <= 128 and c["plan"]["S"] == s)(_s)
FEATURES.update({
    "M>128, S>1, MT>=2": lambda c: c["M"] > 128 and c["plan"]["S"] > 1 and c["plan"]["MT"] >= 2,
    "odd KC, S>1": lambda c: c["plan"]["KC"] % 2 == 1 and c["plan"]["S"] > 1,
    "KC % S != 0": lambda c: c["plan"]["KC"] % c["plan"]["S"] != 0,
    "a CTA with >= 3 items": lambda c: c["plan"]["max_items"] >= 3,
    "odd item count >= 3 per CTA, epilogue warps": lambda c: c["plan"]["dq_warps"] == 16 and c["plan"]["odd_multi"],
    "N < 128": lambda c: c["N"] < 128,
    "N > 128, N % 128 != 0": lambda c: c["N"] > 128 and c["N"] % 128 != 0,
    "ragged last m-tile, MT>=2": lambda c: c["plan"]["MT"] >= 2 and c["M"] % c["plan"]["Mt"] != 0,
    "M=1": lambda c: c["M"] == 1, "M=2": lambda c: c["M"] == 2, "M=3": lambda c: c["M"] == 3, "M=4": lambda c: c["M"] == 4,
    "K % 256 != 0": lambda c: c["K"] % 256 != 0,
    "GPTQ bias, S>1": lambda c: c["fmt"] == "GPTQ+bias" and c["plan"]["S"] > 1,
    "GPTQ bias, S=1": lambda c: c["fmt"] == "GPTQ+bias" and c["plan"]["S"] == 1,
    "GPTQ act-order, S>1": lambda c: c["fmt"] == "GPTQ_ACT" and c["plan"]["S"] > 1,
    "a CTA with >= 3 items, 8 dequant warps": lambda c: c["plan"]["dq_warps"] == 8 and c["plan"]["max_items"] >= 3,
})
for _f in ("Q4_K", "Q6_K", "Q8_0", "AWQ"):   # every chunk size on both dequant-warp layouts, split
    FEATURES[f"{_f}, S>1"] = (lambda f: lambda c: c["fmt"] == f and c["plan"]["S"] > 1)(_f)
    FEATURES[f"{_f}, 8 dequant warps, MT>=2"] = (lambda f: lambda c: c["fmt"] == f and c["plan"]["dq_warps"] == 8 and c["plan"]["MT"] >= 2)(_f)
# features of the call rather than of the plan: assigned round-robin over the chosen cases
CALL_FEATURES = ["x f32", "x f16", "x bf16", "y f32", "y f16", "y bf16", "ldx > K, ldy > N, guards untouched",
                 "workspace reuse", "graph replay"]
TUNING = sorted(k for k in os.environ if k.startswith("B200Q_GEMM_"))


def _candidates(sms: int):
    for fmt, (_, _, chunk) in SWEEP_FMTS.items():
        for N in SWEEP_N:
            for K in SWEEP_K:
                if not _k_ok(fmt, K) or N * K > 2.5e7:
                    continue
                K_pad = -(-K // 256) * 256
                dev_bytes = -(-N // 128) * (K_pad // 256) * chunk
                for M in SWEEP_M:
                    if M * N * K > 2.5e10:
                        continue
                    yield dict(fmt=fmt, N=N, K=K, M=M, cost=M * N * K + 64 * N * K + 2e6,
                               plan=gemm_plan(N, K_pad, chunk, dev_bytes, M, sms))


def _search(sms: int):
    """for every feature in turn, the cheapest candidate that has it, unless an already chosen case has it"""
    cands = sorted(_candidates(sms), key=lambda c: c["cost"])
    chosen, missing = [], []
    for name, pred in FEATURES.items():
        if any(pred(c) for c in chosen):
            continue
        hit = next((c for c in cands if pred(c)), None)
        if hit is None:
            missing.append(name)
        else:
            chosen.append(hit)
    return chosen, missing


def _exact_x(M: int, K: int, seed: int) -> np.ndarray:
    """integers in [-3, 3] * 2^-2, about a quarter of them zero: exact in f16 and bf16"""
    rng = np.random.Generator(np.random.PCG64(seed))
    v = rng.integers(1, 4, size=(M, K)) * rng.choice(np.array([-1, 1]), size=(M, K))
    v[rng.random((M, K)) < 0.25] = 0
    return (v * 0.25).astype(np.float32)


def _exact_ref(c: Case, x: np.ndarray, u_w: float):
    """f64 reference of integer-exact data, after asserting that every partial sum is exact in f32"""
    X = torch.from_numpy(c.x_perm(x)).cuda().double()
    W = torch.from_numpy(c.w16()).cuda().double()
    ref, mag = X @ W.T, X.abs() @ W.abs().T
    if c.bias is not None:
        b = torch.from_numpy(c.bias).cuda().double()
        ref, mag = ref + b, mag + b.abs()
    u_x = _unit(x)
    if c.bias is not None:
        assert _unit(c.bias) >= u_w * u_x
    assert float(mag.max()) < 2.0 ** 24 * u_w * u_x, "precondition: the column sums are not exact in f32"
    return ref


def _assert_exact(y: torch.Tensor, ref: torch.Tensor, yd: str, what: str):
    want = ref if yd == "f32" else ref.float().to(TORCH_DT[yd])
    got = y.double() if yd == "f32" else y
    bad = got != want
    if bool(bad.any()):
        m, n = [int(i) for i in bad.nonzero()[0]]
        raise AssertionError(f"{what}: {int(bad.sum())} of {y.numel()} outputs differ; first m={m} n={n}: {float(y[m, n])!r} vs "
                             f"{float(ref[m, n])!r}")


def _run_case(client, i: int, cand: dict, sms: int, feats: dict):
    fmt, N, K, M = cand["fmt"], cand["N"], cand["K"], cand["M"]
    cfmt, bias, chunk = SWEEP_FMTS[fmt]
    c = Case(client, cfmt, N, K, seed=1000 + i, bias=bias, exact=True)
    plan = plan_for(c.w, M, sms)
    assert int(c.w.info.chunk_bytes) == chunk and plan == cand["plan"], (fmt, N, K, M)
    xd, yd = ("f32", "f16", "bf16")[i % 3], ("f32", "f16", "bf16")[(i // 3) % 3]
    strided = i % 2 == 1
    what = f"case {i}: {fmt} N={N} K={K} M={M} Mt={plan['Mt']} MT={plan['MT']} S={plan['S']} x {xd} y {yd}"
    u_w = _unit(c.w16())
    px, py = (8, 16) if strided else (0, 0)
    xbuf = torch.full((M, K + px), 1024.0, dtype=TORCH_DT[xd], device="cuda")   # guard columns: large, must not be read
    ybuf = torch.full((M, N + py), -3.0, dtype=TORCH_DT[yd], device="cuda")     # guard columns: must stay -3
    x, y = xbuf[:, :K], ybuf[:, :N]
    if TUNING:
        ws = c.w.workspace(M)
    else:   # the workspace the restated plan needs is exactly the library's requirement
        ws = torch.zeros(plan["ws_bytes"], dtype=torch.uint8, device="cuda")
        with pytest.raises(ops.B200QError) as ei:
            client.quant_matmul(x, c.w, out=y, path=ops.PATH_GEMM, workspace=ws[:-256])
        assert ei.value.code == -4, what

    def run(seed, tag):
        xv = _exact_x(M, K, seed)
        x.copy_(torch.from_numpy(xv))
        client.quant_matmul(x, c.w, out=y, path=ops.PATH_GEMM, workspace=ws)
        _assert_exact(y, _exact_ref(c, xv, u_w), yd, f"{what} ({tag})")

    run(2 * i, "first call")
    run(2 * i + 1, "second call on the same workspace")   # the split partials / staged tiles of the first call are stale
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        client.quant_matmul(x, c.w, out=y, path=ops.PATH_GEMM, workspace=ws)
    xv = _exact_x(M, K, 7919 + i)
    x.copy_(torch.from_numpy(xv))
    g.replay()
    torch.cuda.synchronize()
    _assert_exact(y, _exact_ref(c, xv, u_w), yd, f"{what} (graph replay)")
    if strided:
        assert bool((xbuf[:, K:] == 1024.0).all()) and bool((ybuf[:, N:] == -3.0).all()), f"{what}: guard columns changed"
    del g
    c.w.free()
    for f in (f"x {xd}", f"y {yd}", "workspace reuse", "graph replay") + (("ldx > K, ldy > N, guards untouched",) if strided else ()):
        feats[f].append(i)
    return plan


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_gemm_exact_plan_sweep(client):
    """integer-exact data over the launch plan: every output equals the f64 reference (f16 / bf16: one rounding of it)"""
    sms = _sms()
    chosen, missing = _search(sms)
    feats = {name: [] for name in list(FEATURES) + CALL_FEATURES}
    rows = []
    for i, cand in enumerate(chosen):
        plan = _run_case(client, i, cand, sms, feats)
        for name, pred in FEATURES.items():
            if pred(dict(cand, plan=plan)):
                feats[name].append(i)
        rows.append(f"{i:3d} {cand['fmt']:9s} N={cand['N']:6d} K={cand['K']:5d} M={cand['M']:5d} Mt={plan['Mt']:3d} MT={plan['MT']:2d} "
                    f"S={plan['S']} KC={plan['KC']:2d} xsub={plan['xsub']} nw={plan['nw']} nslots={plan['nslots']} dq={plan['dq_warps']:2d} "
                    f"items={plan['items']:4d} grid={plan['grid']:3d} max/CTA={plan['max_items']}")
    print(f"\nexact GEMM sweep on {sms} SMs: {len(chosen)} cases\n" + "\n".join(rows))
    print("plan coverage:\n" + "\n".join(f"  {name:45s} cases {v[:8]}" for name, v in feats.items()))
    if TUNING:
        pytest.skip(f"all {len(chosen)} cases exact; coverage not asserted: tuning variables {TUNING} change the plan")
    assert not missing, f"no candidate shape reaches {missing}"
    uncovered = [name for name, v in feats.items() if not v]
    assert not uncovered, f"plan features not covered: {uncovered}"


# ================================================================================================================================
# 4. staging range
# ================================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("xd", ["f32", "bf16"])
def test_gemm_staging_saturates_and_keeps_subnormals(client, xd):
    """stage_x_kernel clamps to +-65504 before the f16 conversion (+-1e5 and +-inf give the +-65504 result) and keeps
    f16-subnormal activations (~1e-6).  (NaN is not pinned: both paths currently turn it into finite values.)"""
    N, K, M = 256, 1024, 8
    c = Case(client, "Q4_K", N, K, seed=5)
    rng = np.random.Generator(np.random.PCG64(6))
    sign = rng.choice(np.array([-1.0, 1.0], dtype=np.float32), size=(M, K))
    x = rng.standard_normal((M, K)).astype(np.float32)
    x[0] = 1e5 * sign[0]
    x[1] = np.inf * sign[1]
    x[2] = 1e-6 * sign[2] * rng.uniform(0.5, 1.5, size=K).astype(np.float32)
    x[3, ::7] = 1e5 * sign[3, ::7]
    x[3, 3::7] = np.inf * sign[3, 3::7]
    x[4, ::2] = 3e-7 * sign[4, ::2]
    x[5] = np.inf
    x[6] = -1e5
    xt = torch.from_numpy(x).to(TORCH_DT[xd]).cuda()
    x_in = xt.float().cpu().numpy()   # what the kernel reads (bf16 rounds 1e5 and 1e-6)
    y = client.quant_matmul(xt, c.w, out_dtype=torch.float32, path=ops.PATH_GEMM).cpu().numpy()
    assert np.isfinite(y).all()
    x16 = stage_x16(x_in)
    assert (np.abs(x16[[0, 1, 5, 6]].astype(np.float32)) == 65504.0).all()
    assert ((x16[2] != 0) & (np.abs(x16[2].astype(np.float32)) < 2.0 ** -14)).all()
    ref, tol = elementwise_bound(x16, c.w16(), c.w.K_pad, plan_for(c.w, M, _sms())["S"])
    bad = elementwise_violations(y, ref, tol)
    assert bad == 0, f"{bad} outputs outside the bound; per-row worst {(np.abs(y - ref) / tol).max(axis=1)}"


# ================================================================================================================================
# CPU self-checks of the references
# ================================================================================================================================
def test_numpy_f64_to_f16_rounds_once():
    """Case.w16 relies on it: 1 + 2^-11 + 2^-40 is above the midpoint, so one rounding gives 1 + 2^-10 (a conversion through
    f32 first lands on the midpoint 1 + 2^-11 and rounds to even, 1.0)"""
    v = 1.0 + 2.0 ** -11 + 2.0 ** -40
    assert float(np.float64(v).astype(np.float16)) == 1.0 + 2.0 ** -10
    assert float(np.array([v, -v]).astype(np.float16)[1]) == -(1.0 + 2.0 ** -10)
    assert float(np.float32(v).astype(np.float16)) == 1.0


@pytest.mark.parametrize("fmt", ALL + NEW)
def test_w16_is_the_f16_oracle_weight_where_scales_are_f16(fmt):
    """where a and b are exact in f16, the HFMA2 weight is the f16 of the oracle's f32 dequantized weight"""
    c = Case(None, fmt, 64, 512, seed=3)
    ok = (c.a.astype(np.float16).astype(np.float32) == c.a) & (c.b.astype(np.float16).astype(np.float32) == c.b)
    mask = np.repeat(ok, c.sub, axis=1)
    assert mask.any()
    w16, deq16 = c.w16(), c.x_perm(c.deq).astype(np.float16)
    assert np.array_equal(w16[mask], deq16[mask])


def _rz_f32(v: np.ndarray) -> np.ndarray:
    r = v.astype(np.float32)
    up = np.abs(r.astype(np.float64)) > np.abs(v)
    r[up] = np.nextafter(r[up], np.float32(0))
    return r


def test_elementwise_bound_rejects_what_rel_err_accepts():
    """the per-element bound of tests/test_gpu_gemm.py against two subtly wrong kernels the 1e-2 metric lets through, and
    against a model of the right one (f32 accumulation truncated once per 16-k step), at the loosest split factor S = 8"""
    # x staged with round-toward-zero instead of round-to-nearest
    N, K, M = 128, 256, 16
    c = Case(None, "Q4_K", N, K, seed=21)
    x = synth.random_act(M, K, seed=22)
    x16 = stage_x16(x)
    w16 = c.w16().astype(np.float64)
    ref, tol = elementwise_bound(x16, c.w16(), K, 8)
    x_rz = x16.copy()
    up = np.abs(x16.astype(np.float32)) > np.abs(x)
    x_rz[up] = np.nextafter(x16[up], np.float16(0))
    y_rz = (x_rz.astype(np.float64) @ w16.T).astype(np.float32)
    assert rel_err(y_rz, c.oracle_a(x)) < TOL
    assert elementwise_violations(y_rz, ref, tol) > 0
    acc = np.zeros((M, N), dtype=np.float32)
    for k0 in range(0, K, 16):
        acc = _rz_f32(acc.astype(np.float64) + x16[:, k0:k0 + 16].astype(np.float64) @ w16[:, k0:k0 + 16].T)
    assert elementwise_violations(acc, ref, tol) == 0
    assert rel_err(acc, c.oracle_a(x)) < TOL
    # one 16-k sub-block missing from one output element (a typical one: the median contribution of that element)
    N, K, M = 128, 14336, 16
    c = Case(None, "Q4_K", N, K, seed=23)
    x = synth.random_act(M, K, seed=24)
    x16 = stage_x16(x)
    ref, tol = elementwise_bound(x16, c.w16(), K, 8)
    contrib = (x16[0].astype(np.float64) * c.w16()[5].astype(np.float64)).reshape(-1, 16).sum(axis=1)
    j = int(np.argsort(np.abs(contrib))[len(contrib) // 2])
    y = ref.astype(np.float32)
    y[0, 5] = np.float32(ref[0, 5] - contrib[j])
    assert elementwise_violations(ref.astype(np.float32), ref, tol) == 0
    assert rel_err(y, c.oracle_a(x)) < TOL
    assert elementwise_violations(y, ref, tol) == 1
