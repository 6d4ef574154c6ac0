"""GPU: the f16 KV cache of decode attention (b200q_attn_decode_kv and its paged / split forms, Decoder(kv_dtype="f16")).

- every form appends f16_rn(clamp(x, +-65504)) of the rotated k and the raw v;
- f16 single-CTA and f16 split agree as the f32 kernels do (scores bit-identical, outputs within 1 f32 ulp on <= 0.1 %),
  and paged equals contiguous bit for bit;
- the split kernels equal an f64 restatement over the widened f16 cache up to 131 071 positions;
- large k / v clamp to +-65504, bad positions and slot -1 write nothing;
- a Decoder with an f16 cache matches the CPU oracle with the same cache rule (tests/kv16_ref.py): logits, greedy streams,
  batch 2, paged with scheduler slots, 50 000 positions on the split path, the M = 8 GEMM path, prefill;
- what f16 costs against f32 on the small-1b shape, and tensor parallel with an f16 cache."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle
from blazr_b200 import decode, ops
from kv16_ref import Kv16Rows, kv_round_np, oracle_model
from rope_ref import oracle_with_table
from test_gpu_attn_long import BS, P_, Case, _rot, decode_error, split_bounds

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

F16 = 1   # B200Q_F16
NEAR_TIE = 1e-4


def rel_err(y, ref):
    return float(np.abs(y.astype(np.float64) - ref.astype(np.float64)).max() / max(np.abs(ref).max(), 1e-30))


def run16(cs, split, ck, cv, xq=None, ao=None, ws=None):
    """one call of the _kv entry point of this case's layout with f16 caches"""
    L = ops.lib()
    st = ops._stream_ptr(torch.device("cuda"))
    M, nh, nkv, hd = C.c_int64(cs.M), cs.nh, cs.nkv, cs.hd
    if split:
        if ws is None:
            ws = torch.zeros(int(L.b200q_attn_split_workspace_bytes(nh, nkv, hd, cs.max_ctx, cs.M)), dtype=torch.uint8, device="cuda")
        extra = (P_(ws), C.c_size_t(ws.numel()), st)
    else:
        extra = (st,)
    if cs.layout == "contig":
        fn = L.b200q_attn_decode_split_kv if split else L.b200q_attn_decode_kv
        return fn(P_(cs.qkv), P_(cs.pos), P_(ck), P_(cv), F16, P_(cs.rope), nh, nkv, hd, cs.max_ctx, M, P_(xq), P_(ao), *extra)
    fn = L.b200q_attn_decode_paged_split_kv if split else L.b200q_attn_decode_paged_kv
    return fn(P_(cs.qkv), P_(cs.pos), P_(ck), P_(cv), F16, P_(cs.bt), P_(cs.slot), BS, cs.nblk, P_(cs.rope), nh, nkv, hd, M, P_(xq), P_(ao), *extra)


def f16_cache(cs):
    return decode.kv_round(cs.ck), decode.kv_round(cs.cv)


def new_rows(cs, m, p):
    """the f32 k (rotated) and v the kernels append for sequence m at position p"""
    nh, nkv, hd = cs.nh, cs.nkv, cs.hd
    qkv = cs.qkv[m]
    return _rot(qkv[nh * hd:(nh + nkv) * hd].reshape(nkv, hd), cs.rope[p]), qkv[(nh + nkv) * hd:].reshape(nkv, hd)


P_SET = [0, 1, 127, 128, 1000, 4095, 40959]


@pytest.mark.parametrize("layout", ["contig", "paged_slot", "paged"])
@pytest.mark.parametrize("G", [1, 4, 8])
@pytest.mark.parametrize("hd", [64, 128])
def test_f16_forms_append_the_rounded_row_and_agree(client, hd, G, layout):
    nh = 8
    nkv = nh // G
    max_ctx = ops.lib().b200q_attn_decode_max_ctx()
    total_diff = 0
    for M, pos_sets, use_xq in ((1, [[p] for p in P_SET], True), (3, [[0, 40959, 1000], [127, 128, 4095], [1, 40959, 40959]], True),
                                (8, [P_SET + [20000]], False)):
        cs = Case(nh, nkv, hd, max_ctx, M, layout, seed=2000 * hd + 10 * G + M, q_std=3.0)
        ck0, cv0 = f16_cache(cs)
        for pos in pos_sets:
            cs.set_pos(pos)
            ck1, cv1, ck2, cv2 = ck0.clone(), cv0.clone(), ck0.clone(), cv0.clone()
            xq1, ao1 = cs.outputs(use_xq)
            xq2, ao2 = cs.outputs(use_xq)
            ops._check(run16(cs, False, ck1, cv1, xq1, ao1))
            ops._check(run16(cs, True, ck2, cv2, xq2, ao2))
            torch.cuda.synchronize()
            assert decode_error() == 0
            assert torch.equal(ck1, ck2) and torch.equal(cv1, cv2), ("appended rows differ", pos)
            for m, p in enumerate(pos):   # the appended row is the element rule applied to the rotated k and the raw v
                r = cs.row_index(m, p)
                k, v = new_rows(cs, m, p)
                assert torch.equal(ck1[r].view(torch.int16), decode.kv_round(k).view(torch.int16)), (pos, m)
                assert torch.equal(cv1[r].view(torch.int16), decode.kv_round(v).view(torch.int16)), (pos, m)
            a, b = ao1.cpu().numpy().view(np.int32), ao2.cpu().numpy().view(np.int32)
            assert np.isfinite(ao1.cpu().numpy()).all()
            diff = a != b
            n = int(diff.sum())
            total_diff += n
            assert n <= 0.001 * a.size, (pos, n)
            assert int(np.abs(a.astype(np.int64) - b.astype(np.int64)).max()) <= 1, pos
            if use_xq:
                K = nh * hd
                q1, d1, s1 = client.act_unpack(xq1, M, K)
                q2, d2, s2 = client.act_unpack(xq2, M, K)
                same_head = ~diff.reshape(M, nh, hd).any(axis=2)
                for m in range(M):
                    for h in range(nh):
                        if same_head[m, h]:
                            sl = slice(h * hd, (h + 1) * hd)
                            assert torch.equal(q1[m, sl], q2[m, sl]), (pos, m, h)
                            assert torch.equal(d1[m, h * hd // 32:(h + 1) * hd // 32], d2[m, h * hd // 32:(h + 1) * hd // 32])
                            assert torch.equal(s1[m, h * hd // 16:(h + 1) * hd // 16], s2[m, h * hd // 16:(h + 1) * hd // 16])
            if layout != "contig":   # paged equals contiguous bit for bit (same rows, laid out contiguously)
                cc = Case(nh, nkv, hd, max_ctx, M, "contig", seed=2000 * hd + 10 * G + M, q_std=3.0)
                cc.set_pos(pos)
                idx = torch.cat([cs.row_index(m, torch.arange(max_ctx, device="cuda")) for m in range(M)])
                ckc, cvc = ck0[idx].clone(), cv0[idx].clone()
                xq3, ao3 = cc.outputs(use_xq)
                ops._check(run16(cc, False, ckc, cvc, xq3, ao3))
                torch.cuda.synchronize()
                assert torch.equal(ao3.view(torch.int32), ao1.view(torch.int32)), pos
                assert torch.equal(ckc, ck1[idx]) and torch.equal(cvc, cv1[idx])
    print(f"f16 hd {hd} G {G} {layout}: attn_out elements differing between the split and single-CTA kernels: {total_diff}")


@pytest.mark.parametrize("layout", ["contig", "paged_slot"])
@pytest.mark.parametrize("hd", [64, 128])
def test_f16_split_matches_f64_restatement_to_128k(client, hd, layout):
    nh, nkv, M, max_ctx = 8, 2, 4, 131072
    G = nh // nkv
    pos = [40959, 40960, 100000, 131071]
    cs = Case(nh, nkv, hd, max_ctx, M, layout, seed=91 + hd, q_std=3.0)
    cs.set_pos(pos)
    scale = np.float32(1.0) / np.sqrt(np.float32(hd))
    rng = np.random.Generator(np.random.PCG64(hd + 5))
    dominant = {}
    for m, p in enumerate(pos):   # needles as in test_gpu_attn_long: ~12 at every split boundary, one dominant (~45) row for head 0
        q_rot = _rot(cs.qkv[m][:nh * hd].reshape(nh, hd), cs.rope[p])
        bounds = split_bounds(p, max_ctx)
        needles = {0, 40959, 40960} | {b + d for b in bounds[1:-1] for d in (-1, 0)}
        needles |= {16 * int(k) + d for k in rng.integers(1, p // 16, 6) for d in (-1, 0)}
        needles = sorted(j for j in needles if 0 <= j < p)
        for kvh in range(nkv):
            qh = q_rot[kvh * G].double()
            unit = (qh / qh.dot(qh)).float()
            for j in needles:
                cs.ck[cs.row_index(m, j), kvh] = unit * float(12.0 / scale)
        jd = [0, bounds[1], needles[len(needles) // 2], 40960][m]
        qh = q_rot[0].double()
        cs.ck[cs.row_index(m, jd), 0] = (qh / qh.dot(qh)).float() * float(45.0 / scale)
        dominant[m] = jd
    ck, cv = f16_cache(cs)
    xq, ao = cs.outputs(True)
    ops._check(run16(cs, True, ck, cv, xq, ao))
    torch.cuda.synchronize()
    assert decode_error() == 0
    got = ao.cpu().numpy().reshape(M, nh, hd)
    ref = np.empty_like(got)
    for m, p in enumerate(pos):
        q_rot = _rot(cs.qkv[m][:nh * hd].reshape(nh, hd), cs.rope[p])
        k_new, v_new = new_rows(cs, m, p)
        idx = cs.row_index(m, torch.arange(p + 1, device="cuda"))
        assert torch.equal(ck[idx[-1]], decode.kv_round(k_new)) and torch.equal(cv[idx[-1]], decode.kv_round(v_new)), "appended row"
        K, V = ck[idx].double(), cv[idx].double()   # the widened f16 cache, row p included
        for h in range(nh):
            kvh = h // G
            sc = (K[:, kvh, :] @ q_rot[h].double()).float().cpu().numpy() * scale
            pj = oracle.det_exp((sc - sc.max()).astype(np.float32))
            pd = torch.from_numpy(pj.astype(np.float64)).cuda()
            num = (pd[:, None] * V[:, kvh, :]).sum(0).float().cpu().numpy()
            ref[m, h] = num / np.float32(pj.astype(np.float64).sum())
        vrow = V[dominant[m], 0].float().cpu().numpy()   # the dominant needle's f16 V row
        err = np.abs(got[m, 0] - vrow).max() / np.abs(vrow).max()
        assert err < 1e-5, ("dominant needle", m, dominant[m], err)
    err = float(np.abs(got.astype(np.float64) - ref).max() / np.abs(ref).max())
    same = float((got.view(np.uint32) == ref.view(np.uint32)).mean())
    print(f"f16 hd {hd} {layout}: rel err vs f64 restatement over the widened f16 cache {err:.2e}, identical bits {same:.4f}")
    assert err < 1e-5 and same >= 0.99


@pytest.mark.parametrize("split", [False, True])
def test_f16_clamp_and_bad_positions(client, split):
    nh, nkv, hd, M = 8, 2, 128, 2
    max_ctx = 40960 if not split else 65536
    for layout in ("contig", "paged_slot", "paged"):
        cs = Case(nh, nkv, hd, max_ctx, M, layout, seed=31)
        # k / v elements of +-1e5: the appended rows hold +-65504 and the outputs stay finite
        big = torch.where(torch.rand(2 * nkv * hd, device="cuda", generator=cs.g) < 0.5, -1e5, 1e5)
        cs.qkv[:, nh * hd:] = big
        cs.set_pos([7, 300])
        ck, cv = f16_cache(cs)
        xq, ao = cs.outputs(True)
        ops._check(run16(cs, split, ck, cv, xq, ao))
        torch.cuda.synchronize()
        assert decode_error() == 0
        assert torch.isfinite(ao).all()
        for m, p in enumerate([7, 300]):
            r = cs.row_index(m, p)
            assert torch.equal(cv[r].abs().float(), torch.full_like(cv[r].float(), 65504.0))
            k, _ = new_rows(cs, m, p)
            assert torch.equal(ck[r], decode.kv_round(k)) and ck[r].abs().max().item() == 65504.0
        # bad positions / slot -1 write nothing and raise the device error
        cs = Case(nh, nkv, hd, max_ctx, M, layout, seed=9)
        decode_error()
        for pos, kill_slot in (([max_ctx, 100], False), ([5, -1], False), ([70, 80], True)):
            if kill_slot and layout != "paged_slot":
                continue
            cs.set_pos(pos)
            if kill_slot:
                cs.slot[1] = -1
            ck0, cv0 = f16_cache(cs)
            ck, cv = ck0.clone(), cv0.clone()
            xq, ao = cs.outputs(True)
            ops._check(run16(cs, split, ck, cv, xq, ao))
            torch.cuda.synchronize()
            assert decode_error() & 1, pos
            bad = 0 if pos[0] >= max_ctx else 1
            good = 1 - bad
            assert torch.isnan(ao[bad]).all() and torch.isfinite(ao[good]).all()
            changed = ((ck != ck0).any(dim=(1, 2)) | (cv != cv0).any(dim=(1, 2))).nonzero().flatten().tolist()
            assert changed == [int(cs.row_index(good, pos[good]))], (layout, pos, changed)
    # a Decoder whose device position runs past its f16 cache reports the flag as an error
    dec = decode.Decoder(client, decode.PRESETS["tiny"], "Q8_0", batch=1, max_ctx=16 if not split else 40960 + 16, kv_dtype="f16",
                         host=decode.build_host_model(decode.PRESETS["tiny"], "Q8_0", seed=1))
    assert dec.attn_split == split
    dec.reset([1])
    dec.pos.fill_(dec.max_ctx)
    dec.step()
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match="position"):
        dec.check_device_errors()


def _teacher_forced(client, cfg, scheme, hm, toks, **kw):
    om = oracle_model(hm, kv_dtype="f16")
    dec = decode.Decoder(client, cfg, scheme, batch=1, max_ctx=64, host=hm, kv_dtype="f16", **kw)
    dec.reset([toks[0]])
    for i, t in enumerate(toks):
        dec.ids.fill_(t)
        dec.step()
        torch.cuda.synchronize()
        ref = om.step(t)
        got = dec.logits[0].cpu().numpy()
        assert rel_err(got, ref) < 1e-5, (scheme, i)
        assert (got.view(np.uint32) == ref.view(np.uint32)).mean() > 0.99, (scheme, i)
    return dec


@pytest.mark.parametrize("scheme", ["Q4_K_M", "Q8_0"])
def test_decoder_f16_matches_oracle(client, scheme):
    cfg = decode.PRESETS["tiny"]
    hm = decode.build_host_model(cfg, scheme, seed=3)
    toks = [5, 17, 900, 33, 1200, 7, 7, 2047]
    dec = _teacher_forced(client, cfg, scheme, hm, toks)
    assert dec.layers[0]["ck"].dtype == torch.float16
    assert dec.kv_cache_bytes == 2 * cfg.n_layers * 64 * cfg.n_kv_heads * cfg.head_dim * 2
    k, v = dec.kv_rows(dec.layers[0], 0, len(toks))
    assert k.dtype == torch.float16 and v.dtype == torch.float16
    # graph-replayed steps give the same logits as the oracle
    om = oracle_model(hm, kv_dtype="f16")
    dec = decode.Decoder(client, cfg, scheme, batch=1, max_ctx=64, host=hm, kv_dtype="f16")
    dec.reset([toks[0]])
    dec.capture()
    for i, t in enumerate(toks):
        dec.ids.fill_(t)
        dec.replay()
        torch.cuda.synchronize()
        ref = om.step(t)
        got = dec.logits[0].cpu().numpy()
        assert rel_err(got, ref) < 1e-5 and (got.view(np.uint32) == ref.view(np.uint32)).mean() > 0.99, ("replay", i)
    # greedy streams, seeds 1-3, 128 tokens
    prompt = [1, 5, 9, 2]
    for seed in range(1, 4):
        hm = decode.build_host_model(cfg, scheme, seed=seed)
        ref, gaps = oracle_model(hm, kv_dtype="f16").generate(prompt, 128)
        got = decode.Decoder(client, cfg, scheme, batch=1, max_ctx=160, host=hm, kv_dtype="f16").generate(np.asarray(prompt)[None, :], 128)[0]
        if not np.array_equal(got, ref):
            j = int(np.nonzero(got != ref)[0][0])
            assert gaps[j] < NEAR_TIE, f"seed {seed}: streams diverge at step {j} where the oracle's top-2 gap is {gaps[j]:.3e}"


def test_decoder_f16_batch_and_scheduler_paged(client):
    from blazr_b200 import batch as bb
    cfg = decode.PRESETS["tiny"]
    hm = decode.build_host_model(cfg, "Q6_K", seed=11)
    p0, p1 = [3, 1, 4, 1, 5], [9, 2, 6, 5, 3]
    dec = decode.Decoder(client, cfg, "Q6_K", batch=2, max_ctx=64, host=hm, kv_dtype="f16")
    got = dec.generate(np.asarray([p0, p1]), 12, use_graph=True)
    for m, p in enumerate((p0, p1)):
        toks, gaps = oracle_model(hm, kv_dtype="f16").generate(p, 12)
        if not np.array_equal(got[m], toks):
            j = int(np.nonzero(got[m] != toks)[0][0])
            assert gaps[j] < NEAR_TIE
    # paged with block_table / slot_mapping from the scheduler mirror equals the contiguous f16 cache bit for bit
    batch, bs = 2, 4
    rng = np.random.Generator(np.random.PCG64(4))
    prompts = rng.integers(0, cfg.vocab, size=(batch, 6))
    ref = decode.Decoder(client, cfg, "Q6_K", batch=batch, max_ctx=32, host=hm, kv_dtype="f16")
    pg = decode.Decoder(client, cfg, "Q6_K", batch=batch, max_ctx=32, host=hm, paged=True, block_size=bs, kv_dtype="f16")
    ref.reset(prompts[:, 0]); pg.reset(prompts[:, 0])
    hist = {m: [] for m in range(batch)}
    tables = {m: [] for m in range(batch)}
    next_block = 0
    pg.slot_mapping = torch.zeros(batch, dtype=torch.int32, device="cuda")
    toks = prompts[:, 0].copy()
    for step in range(14):
        for m in range(batch):
            hist[m].append(int(toks[m]))
            if len(hist[m]) > len(tables[m]) * bs:
                tables[m].append(next_block); next_block += 1
        db = bb.build_decode_batch(list(range(batch)), hist, tables, bs)
        bt = np.zeros((batch, pg.max_blocks), dtype=np.int32)
        bt[:, :db.block_table.shape[1]] = db.block_table
        pg.block_table.copy_(torch.from_numpy(bt))
        pg.slot_mapping.copy_(torch.from_numpy(db.slot_mapping))
        for d in (ref, pg):
            d.ids.copy_(torch.from_numpy(db.input_ids[:, 0]))
            d.step()
        torch.cuda.synchronize()
        assert np.array_equal(ref.full_logits().cpu().numpy().view(np.uint32), pg.full_logits().cpu().numpy().view(np.uint32)), step
        toks = ref.ids.cpu().numpy()
    pg.check_device_errors()
    for m in range(batch):   # the same f16 rows, whatever the layout
        S = len(hist[m])
        ka, va = ref.kv_rows(ref.layers[1], m, S)
        kb, vb = pg.kv_rows(pg.layers[1], m, S)
        assert torch.equal(ka, kb) and torch.equal(va, vb)


LONG_CFGS = {64: decode.ModelConfig("long-hd64", 512, 2, 8, 2, 64, 1024, 2048, 500000.0),
             128: decode.ModelConfig("long-hd128", 1024, 2, 8, 2, 128, 1024, 2048, 500000.0)}


@pytest.mark.parametrize("paged", [False, True])
@pytest.mark.parametrize("hd", [64, 128])
def test_decoder_f16_at_50k_positions_matches_oracle(client, hd, paged):
    cfg = LONG_CFGS[hd]
    P, max_ctx = 50000, 65536 + 64
    hm = decode.build_host_model(cfg, "Q8_0", seed=hd)
    dec = decode.Decoder(client, cfg, "Q8_0", batch=1, max_ctx=max_ctx, host=hm, paged=paged, kv_dtype="f16")
    assert dec.attn_split
    om = oracle_with_table(oracle_model(hm, kv_dtype="f16"), max_ctx)
    rng = np.random.Generator(np.random.PCG64(200 + hd))
    kv = []
    for lay in dec.layers:
        k = (rng.standard_normal((P, cfg.n_kv_heads, hd)) * 0.5).astype(np.float32)
        v = rng.standard_normal((P, cfg.n_kv_heads, hd)).astype(np.float32)
        dec._kv_write(lay, 0, torch.from_numpy(k).cuda(), torch.from_numpy(v).cuda())
        kv.append((k, v))
    ks, vs = dec.kv_rows(dec.layers[0], 0, P)
    assert np.array_equal(ks.cpu().numpy().view(np.uint16), kv_round_np(kv[0][0]).view(np.uint16))
    toks = [5, 900, 17, 1200]
    for mode in ("eager", "replay"):
        for li, (k, v) in enumerate(kv):
            om.k_cache[li] = Kv16Rows(k)
            om.v_cache[li] = Kv16Rows(v)
        om.pos = P
        dec.pos.fill_(P)
        dec._host_pos = P
        dec.ids.fill_(toks[0])
        if mode == "replay":
            dec.capture()
        for i, t in enumerate(toks):
            dec.ids.fill_(t)
            dec.replay() if mode == "replay" else dec.step()
            torch.cuda.synchronize()
            ref = om.step(t)
            got = dec.logits[0].cpu().numpy()
            assert rel_err(got, ref) < 1e-5, (mode, i)
            assert (got.view(np.uint32) == ref.view(np.uint32)).mean() > 0.99, (mode, i)
    dec.check_device_errors()


@pytest.mark.parametrize("scheme", ["Q4_K_M", "Q8_0"])
def test_f16_wide_path_and_prefill(client, scheme):
    cfg = decode.PRESETS["tiny"]
    hm = decode.build_host_model(cfg, scheme, seed=13)
    # M = 8: the tcgen05 GEMM path against the f32 CPU path (flavour A) with the f16 cache rule, tolerance 1e-2
    rng = np.random.Generator(np.random.PCG64(8))
    prompts = rng.integers(0, cfg.vocab, size=(8, 4))
    dec = decode.Decoder(client, cfg, scheme, batch=8, max_ctx=64, host=hm, kv_dtype="f16")
    assert dec.wide
    dec.reset(prompts[:, 0])
    oms = [oracle_model(hm, flavour="A", kv_dtype="f16") for _ in range(8)]
    for i in range(prompts.shape[1]):
        dec.ids.copy_(torch.from_numpy(prompts[:, i]).cuda())
        dec.step()
        torch.cuda.synchronize()
        got = dec.full_logits().cpu().numpy()
        for m in range(8):
            assert rel_err(got[m], oms[m].step(int(prompts[m, i]))) < 1e-2, (i, m)
    # prefill into an f16 cache, then decode steps (tolerances of the f32 prefill test)
    hm = decode.build_host_model(cfg, scheme, seed=9)
    prompt = np.random.Generator(np.random.PCG64(3)).integers(0, cfg.vocab, size=48)
    oa = oracle_model(hm, flavour="A", kv_dtype="f16")
    ref = None
    for t in prompt:
        ref = oa.step(int(t))
    dec = decode.Decoder(client, cfg, scheme, batch=1, max_ctx=96, host=hm, kv_dtype="f16")
    logits = dec.prefill(prompt).cpu().numpy()
    assert rel_err(logits, ref) < 1e-2
    dec2 = decode.Decoder(client, cfg, scheme, batch=1, max_ctx=96, host=hm, kv_dtype="f16")
    dec2.reset([int(prompt[0])])
    for t in prompt:
        dec2.ids.fill_(int(t))
        dec2.step()
    torch.cuda.synchronize()
    S = len(prompt)
    for la, lb in zip(dec.layers, dec2.layers):
        assert la["ck"].dtype == torch.float16
        ka, kb = la["ck"][0, :S].float().cpu().numpy(), lb["ck"][0, :S].float().cpu().numpy()
        va, vb = la["cv"][0, :S].float().cpu().numpy(), lb["cv"][0, :S].float().cpu().numpy()
        assert rel_err(ka, kb) < 2e-2 and rel_err(va, vb) < 2e-2
    nxt = int(dec.ids[0])
    dec.step()
    dec2.ids.fill_(nxt)
    dec2.step()
    torch.cuda.synchronize()
    ref2 = oa.step(nxt)
    assert rel_err(dec.logits[0].cpu().numpy(), dec2.logits[0].cpu().numpy()) < 3e-2
    assert rel_err(dec.logits[0].cpu().numpy(), ref2) < 5e-2


# The largest relative deviation of f16-cache logits from f32-cache logits over the 32 teacher-forced steps below: 2.28e-2 in
# the CPU oracle (f32 vs f16 cache rule), the same on a B200 (DESIGN section 2).  The ceiling leaves a factor of about 2.
F16_VS_F32_CEILING = 5e-2


def test_cost_of_f16_kv_on_small_1b(client):
    cfg = decode.PRESETS["small-1b"]
    hm = decode.build_host_model(cfg, "Q4_K_M", seed=5)
    d32 = decode.Decoder(client, cfg, "Q4_K_M", batch=1, max_ctx=64, host=hm)
    d16 = decode.Decoder(client, cfg, "Q4_K_M", batch=1, max_ctx=64, host=hm, kv_dtype="f16")
    assert d16.kv_cache_bytes * 2 == d32.kv_cache_bytes
    toks = np.random.Generator(np.random.PCG64(32)).integers(0, cfg.vocab, size=32)
    d32.reset([int(toks[0])]); d16.reset([int(toks[0])])
    worst, same_argmax = 0.0, 0
    for t in toks:   # teacher-forced: both decoders see the same tokens
        for d in (d32, d16):
            d.ids.fill_(int(t))
            d.step()
        torch.cuda.synchronize()
        a, b = d32.logits[0].cpu().numpy(), d16.logits[0].cpu().numpy()
        worst = max(worst, rel_err(b, a))
        same_argmax += int(np.argmax(a) == np.argmax(b))
    print(f"small-1b Q4_K_M, 32 steps: f16 KV vs f32 KV logits max rel deviation {worst:.3e}, same argmax at {same_argmax}/32 steps")
    assert 0.0 < worst < F16_VS_F32_CEILING


@pytest.mark.parametrize("world", [2, 4, 8])
def test_tensor_parallel_f16_kv_matches_one_gpu(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                        "--master-port", str(29700 + world), os.path.join(root, "tools", "tp_check.py"), "--kv-dtype", "f16"],
                       capture_output=True, text=True, timeout=600)
    tail = "\n".join(l for l in (r.stdout + r.stderr).splitlines() if l.startswith("tp") or "TP_CHECK" in l or "Error" in l)
    print(tail)   # the "logits differing in any bit" line: a rank's attention touches only its own kv heads
    assert "TP_CHECK PASS" in r.stdout, tail
