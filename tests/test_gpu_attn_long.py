"""GPU: split-context decode attention (b200q_attn_decode_split / _paged_split) and Llama 3.1 / 3.2 RoPE factors.

- where both kernels run (max_ctx = 40960) the split kernels append the same cache rows and give the same outputs as the
  single-CTA kernel (scores are bit-identical; only the order of the f64 sums of the weighted sum differs);
- up to p = 131071 they match an f64 restatement of the attention, including planted needle rows at every split boundary;
- a 2-layer Decoder at 50 000 positions matches the CPU oracle, eager and graph-replayed, contiguous and paged;
- bad positions write nothing; a short workspace is refused;
- a Llama-3.1-style GGUF file with rope_freqs.weight decodes the oracle's greedy stream."""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

import oracle
from blazr_b200 import decode, ops
from oracle.model import OracleModel
from rope_ref import llama3_rope_factors, oracle_with_table

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

SPLIT_MIN, SPLIT_CAP = 256, 128   # decode_ops.cu ATTN_SPLIT_MIN / ATTN_SPLIT_CAP
BS = 16                           # paged block size
P_ = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None


def split_bounds(p, max_ctx):
    """the split boundaries the kernels use for position p (decode_ops.cu attn_split_range)"""
    n = p + 1
    s_eff = min(min(-(-max_ctx // SPLIT_MIN), SPLIT_CAP), -(-n // SPLIT_MIN))
    return [s * n // s_eff for s in range(s_eff + 1)]


class Case:
    """qkv / caches / rope of one attention call, contiguous or paged (with or without slot_mapping)"""

    def __init__(self, nh, nkv, hd, max_ctx, M, layout, seed, k_std=1.0, v_std=1.0, q_std=1.0):
        self.nh, self.nkv, self.hd, self.max_ctx, self.M, self.layout = nh, nkv, hd, max_ctx, M, layout
        g = torch.Generator(device="cuda")
        g.manual_seed(seed)
        self.g = g
        rows = M * max_ctx
        self.ck = torch.randn((rows, nkv, hd), device="cuda", generator=g) * k_std
        self.cv = torch.randn((rows, nkv, hd), device="cuda", generator=g) * v_std
        self.qkv = torch.randn((M, (nh + 2 * nkv) * hd), device="cuda", generator=g)
        self.qkv[:, :nh * hd] *= q_std
        self.rope = torch.from_numpy(decode.rope_table(max_ctx, hd, 500000.0)).cuda()
        self.nblk = max_ctx // BS
        if layout != "contig":
            perm = np.random.Generator(np.random.PCG64(seed)).permutation(M * self.nblk).astype(np.int32)
            self.bt = torch.from_numpy(perm.reshape(M, self.nblk)).cuda()
        self.slot = None

    def row_index(self, m, j):
        """flat cache row of position(s) j of sequence m"""
        j = torch.as_tensor(j, device="cuda", dtype=torch.int64)
        if self.layout == "contig":
            return m * self.max_ctx + j
        return self.bt[m, j // BS].long() * BS + j % BS

    def set_pos(self, pos):
        self.pos = torch.tensor(pos, dtype=torch.int32, device="cuda")
        if self.layout == "paged_slot":
            # (a position outside the cache keeps a valid slot: the position alone must make the kernels refuse the sequence)
            self.slot = torch.stack([self.row_index(m, min(max(p, 0), self.max_ctx - 1)) for m, p in enumerate(pos)]).to(torch.int32)

    def run(self, split, ck, cv, xq=None, ao=None, ws=None, ws_bytes=None):
        L = ops.lib()
        st = ops._stream_ptr(torch.device("cuda"))
        M, nh, nkv, hd = C.c_int64(self.M), self.nh, self.nkv, self.hd
        if split:
            if ws is None:
                ws = torch.zeros(int(L.b200q_attn_split_workspace_bytes(nh, nkv, hd, self.max_ctx, self.M)), dtype=torch.uint8, device="cuda")
            extra = (P_(ws), C.c_size_t(ws.numel() if ws_bytes is None else ws_bytes), st)
        else:
            extra = (st,)
        if self.layout == "contig":
            fn = L.b200q_attn_decode_split if split else L.b200q_attn_decode
            return fn(P_(self.qkv), P_(self.pos), P_(ck), P_(cv), P_(self.rope), nh, nkv, hd, self.max_ctx, M, P_(xq), P_(ao), *extra)
        fn = L.b200q_attn_decode_paged_split if split else L.b200q_attn_decode_paged
        return fn(P_(self.qkv), P_(self.pos), P_(ck), P_(cv), P_(self.bt), P_(self.slot), BS, self.nblk, P_(self.rope), nh, nkv, hd, M,
                  P_(xq), P_(ao), *extra)

    def outputs(self, use_xq):
        xq = torch.full((int(ops.lib().b200q_act_bytes(C.c_int64(self.nh * self.hd), C.c_int64(self.M))),), 0x5A, dtype=torch.uint8, device="cuda") if use_xq else None
        ao = torch.full((self.M, self.nh * self.hd), float("nan"), device="cuda")
        return xq, ao


def decode_error():
    f = C.c_int32(0)
    ops._check(ops.lib().b200q_decode_error(C.byref(f)))
    return f.value


P_SET = [0, 1, 127, 128, 1000, 4095, 40959]


@pytest.mark.parametrize("layout", ["contig", "paged_slot", "paged"])
@pytest.mark.parametrize("G", [1, 4, 8])
@pytest.mark.parametrize("hd", [64, 128])
def test_split_matches_single_cta(client, hd, G, layout):
    nh = 8
    nkv = nh // G
    max_ctx = ops.lib().b200q_attn_decode_max_ctx()
    assert max_ctx == 40960
    total_diff = 0
    for M, pos_sets, use_xq in ((1, [[p] for p in P_SET], True), (3, [[0, 40959, 1000], [127, 128, 4095], [1, 40959, 40959]], True),
                                (8, [P_SET + [20000]], False)):
        # scores spread wide enough (std ~3) that a few hundred positions carry the weight
        cs = Case(nh, nkv, hd, max_ctx, M, layout, seed=1000 * hd + 10 * G + M, q_std=3.0)
        for pos in pos_sets:
            cs.set_pos(pos)
            ck1, cv1, ck2, cv2 = cs.ck.clone(), cs.cv.clone(), cs.ck.clone(), cs.cv.clone()
            xq1, ao1 = cs.outputs(use_xq)
            xq2, ao2 = cs.outputs(use_xq)
            ops._check(cs.run(False, ck1, cv1, xq1, ao1))
            ops._check(cs.run(True, ck2, cv2, xq2, ao2))
            torch.cuda.synchronize()
            assert decode_error() == 0
            assert torch.equal(ck1, ck2) and torch.equal(cv1, cv2), ("appended rows differ", pos)
            for m, p in enumerate(pos):   # the new row was appended (rotated k, raw v)
                r = cs.row_index(m, p)
                assert not torch.equal(ck1[r], cs.ck[r])
            a, b = ao1.cpu().numpy().view(np.int32), ao2.cpu().numpy().view(np.int32)
            assert np.isfinite(ao1.cpu().numpy()).all()
            diff = a != b
            n = int(diff.sum())
            total_diff += n
            assert n <= 0.001 * a.size, (pos, n)
            assert int(np.abs(a.astype(np.int64) - b.astype(np.int64)).max()) <= 1, pos   # at most 1 f32 ulp (same sign)
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
    print(f"hd {hd} G {G} {layout}: attn_out elements differing between the split and single-CTA kernels: {total_diff}")


def _rot(x, cs):
    """adjacent-pair RoPE with separate f32 multiplies and adds (the kernels' operation sequence); x [..., hd], cs [hd/2, 2]"""
    x0, x1 = x[..., 0::2], x[..., 1::2]
    c, s = cs[:, 0], cs[:, 1]
    out = torch.empty_like(x)
    out[..., 0::2] = (x0 * c) - (x1 * s)
    out[..., 1::2] = (x0 * s) + (x1 * c)
    return out


@pytest.mark.parametrize("layout", ["contig", "paged_slot"])
@pytest.mark.parametrize("hd", [64, 128])
def test_split_matches_f64_restatement_to_128k(client, hd, layout):
    nh, nkv, M, max_ctx = 8, 2, 4, 131072
    G = nh // nkv
    pos = [40959, 40960, 100000, 131071]
    cs = Case(nh, nkv, hd, max_ctx, M, layout, seed=77 + hd, q_std=3.0)
    cs.set_pos(pos)
    scale = np.float32(1.0) / np.sqrt(np.float32(hd))
    rng = np.random.Generator(np.random.PCG64(hd))
    dominant = {}
    for m, p in enumerate(pos):
        qkv = cs.qkv[m]
        q = qkv[:nh * hd].reshape(nh, hd)
        q_rot = _rot(q, cs.rope[p])
        bounds = split_bounds(p, max_ctx)
        needles = {0, 40959, 40960} | {b + d for b in bounds[1:-1] for d in (-1, 0)}
        needles |= {16 * int(k) + d for k in rng.integers(1, p // 16, 6) for d in (-1, 0)}
        needles = sorted(j for j in needles if 0 <= j < p)
        # needle rows of every kv group score ~12 against the group's first query head (random rows: std 3)
        for kvh in range(nkv):
            qh = q_rot[kvh * G].double()
            unit = (qh / qh.dot(qh)).float()
            for j in needles:
                cs.ck[cs.row_index(m, j), kvh] = unit * float(12.0 / scale)
        # one needle per sequence dominates head 0 (score ~45): the output must be that needle's V row
        jd = [0, bounds[1], needles[len(needles) // 2], 40960][m]
        qh = q_rot[0].double()
        cs.ck[cs.row_index(m, jd), 0] = (qh / qh.dot(qh)).float() * float(45.0 / scale)
        dominant[m] = jd
    ck, cv = cs.ck.clone(), cs.cv.clone()
    xq, ao = cs.outputs(True)
    ops._check(cs.run(True, ck, cv, xq, ao))
    torch.cuda.synchronize()
    assert decode_error() == 0
    got = ao.cpu().numpy().reshape(M, nh, hd)
    ref = np.empty_like(got)
    for m, p in enumerate(pos):
        qkv = cs.qkv[m]
        q_rot = _rot(qkv[:nh * hd].reshape(nh, hd), cs.rope[p])
        k_new = _rot(qkv[nh * hd:(nh + nkv) * hd].reshape(nkv, hd), cs.rope[p])
        v_new = qkv[(nh + nkv) * hd:].reshape(nkv, hd)
        idx = cs.row_index(m, torch.arange(p + 1, device="cuda"))
        assert torch.equal(ck[idx[-1]], k_new) and torch.equal(cv[idx[-1]], v_new), "appended row"
        K, V = ck[idx].double(), cv[idx].double()                   # [p+1, nkv, hd]
        for h in range(nh):
            kvh = h // G
            sc = (K[:, kvh, :] @ q_rot[h].double()).float().cpu().numpy() * scale    # f64 dot, one rounding, f32 scale
            pj = oracle.det_exp((sc - sc.max()).astype(np.float32))
            pd = torch.from_numpy(pj.astype(np.float64)).cuda()
            num = (pd[:, None] * V[:, kvh, :]).sum(0).float().cpu().numpy()
            ref[m, h] = num / np.float32(pj.astype(np.float64).sum())
        vrow = V[dominant[m], 0].float().cpu().numpy()   # only head 0's query was aimed at the dominant needle
        err = np.abs(got[m, 0] - vrow).max() / np.abs(vrow).max()
        assert err < 1e-5, ("dominant needle", m, dominant[m], err)
    err = float(np.abs(got.astype(np.float64) - ref).max() / np.abs(ref).max())
    same = float((got.view(np.uint32) == ref.view(np.uint32)).mean())
    print(f"hd {hd} {layout}: rel err vs f64 restatement {err:.2e}, identical bits {same:.4f}")
    assert err < 1e-5 and same >= 0.99


@pytest.mark.parametrize("layout", ["contig", "paged_slot", "paged"])
def test_bad_position_writes_nothing_and_workspace_size(client, layout):
    nh, nkv, hd, M, max_ctx = 8, 2, 128, 2, 65536
    cs = Case(nh, nkv, hd, max_ctx, M, layout, seed=9)
    decode_error()
    for pos, kill_slot in (([max_ctx, 100], False), ([5, -1], False), ([70, 80], True)):
        if kill_slot and layout != "paged_slot":
            continue
        cs.set_pos(pos)
        if kill_slot:
            cs.slot[1] = -1
        ck, cv = cs.ck.clone(), cs.cv.clone()
        xq, ao = cs.outputs(True)
        xq0 = xq.clone()
        ops._check(cs.run(True, ck, cv, xq, ao))
        torch.cuda.synchronize()
        assert decode_error() & 1, pos
        bad = 0 if pos[0] >= max_ctx else 1
        good = 1 - bad
        # the bad sequence wrote nothing: no cache row, no attn_out, no record byte of its row
        assert torch.isnan(ao[bad]).all()
        K = nh * hd
        q0, d0, s0 = client.act_unpack(xq0, M, K)
        q1, d1, s1 = client.act_unpack(xq, M, K)
        assert torch.equal(q0[bad], q1[bad]) and torch.equal(d0[bad].view(torch.int32), d1[bad].view(torch.int32))
        assert torch.isfinite(ao[good]).all()
        changed = (ck != cs.ck).any(dim=(1, 2)).nonzero().flatten().tolist()
        assert changed == [int(cs.row_index(good, pos[good]))], changed
    # exact workspace size succeeds, 256 bytes less is refused
    cs.set_pos([3, 4])
    need = int(ops.lib().b200q_attn_split_workspace_bytes(nh, nkv, hd, max_ctx, M))
    ws = torch.zeros(need, dtype=torch.uint8, device="cuda")
    xq, ao = cs.outputs(True)
    assert cs.run(True, cs.ck.clone(), cs.cv.clone(), xq, ao, ws=ws, ws_bytes=need) == 0
    assert cs.run(True, cs.ck.clone(), cs.cv.clone(), xq, ao, ws=ws, ws_bytes=need - 256) == -4
    torch.cuda.synchronize()
    assert decode_error() == 0 and torch.isfinite(ao).all()


def rel_err(y, ref):
    return float(np.abs(y.astype(np.float64) - ref.astype(np.float64)).max() / max(np.abs(ref).max(), 1e-30))


LONG_CFGS = {64: decode.ModelConfig("long-hd64", 512, 2, 8, 2, 64, 1024, 2048, 500000.0),
             128: decode.ModelConfig("long-hd128", 1024, 2, 8, 2, 128, 1024, 2048, 500000.0)}


@pytest.mark.parametrize("paged", [False, True])
@pytest.mark.parametrize("hd", [64, 128])
def test_decoder_at_50k_positions_matches_oracle(client, hd, paged):
    cfg = LONG_CFGS[hd]
    P, max_ctx = 50000, 65536 + 64
    hm = decode.build_host_model(cfg, "Q8_0", seed=hd)
    dec = decode.Decoder(client, cfg, "Q8_0", batch=1, max_ctx=max_ctx, host=hm, paged=paged)
    assert dec.attn_split
    om = oracle_with_table(OracleModel(hm), max_ctx)
    rng = np.random.Generator(np.random.PCG64(100 + hd))
    kv = []
    for li, lay in enumerate(dec.layers):
        k = (rng.standard_normal((P, cfg.n_kv_heads, hd)) * 0.5).astype(np.float32)
        v = rng.standard_normal((P, cfg.n_kv_heads, hd)).astype(np.float32)
        dec._kv_write(lay, 0, torch.from_numpy(k).cuda(), torch.from_numpy(v).cuda())
        kv.append((k, v))
    toks = [5, 900, 17, 1200]

    def oracle_at_P():
        for li, (k, v) in enumerate(kv):
            om.k_cache[li] = list(k)
            om.v_cache[li] = list(v)
        om.pos = P

    oracle_at_P()
    dec.reset([toks[0]])
    dec.pos.fill_(P)
    dec._host_pos = P
    for i, t in enumerate(toks):   # eager, teacher-forced
        dec.ids.fill_(t)
        dec.step()
        torch.cuda.synchronize()
        ref = om.step(t)
        got = dec.logits[0].cpu().numpy()
        assert rel_err(got, ref) < 1e-5, ("eager", i)
        assert (got.view(np.uint32) == ref.view(np.uint32)).mean() > 0.99, ("eager", i)
    oracle_at_P()
    dec.pos.fill_(P)
    dec._host_pos = P
    dec.ids.fill_(toks[0])
    dec.capture()
    for i, t in enumerate(toks):   # graph-replayed
        dec.ids.fill_(t)
        dec.replay()
        torch.cuda.synchronize()
        ref = om.step(t)
        got = dec.logits[0].cpu().numpy()
        assert rel_err(got, ref) < 1e-5, ("replay", i)
        assert (got.view(np.uint32) == ref.view(np.uint32)).mean() > 0.99, ("replay", i)
        assert int(dec.pos[0]) == P + i + 1
    dec.check_device_errors()


def test_llama31_gguf_with_rope_freqs_end_to_end(client, tmp_path):
    from blazr_b200 import gguf_loader
    from gguf_util import write_gguf
    hm = decode.build_host_model(decode.PRESETS["tiny"], "Q4_K_M", seed=21)
    f = llama3_rope_factors(hm.cfg.head_dim, hm.cfg.rope_theta, factor=8.0, low_freq_factor=1.0, high_freq_factor=4.0, original_context=64)
    assert f.min() == 1.0 and f.max() == 8.0 and np.any((f > 1) & (f < 8))
    path = str(tmp_path / "l31.gguf")
    write_gguf(path, hm, extra_tensors={"rope_freqs.weight": f})
    dec, cfg = gguf_loader.load_gguf(client, path, max_ctx=64)
    assert cfg.rope_freq_factors == tuple(float(x) for x in f)
    prompt = np.asarray([[5, 3, 8, 1]])
    got = dec.generate(prompt, 24, use_graph=True)[0]
    hm_f = dataclasses.replace(hm, cfg=dataclasses.replace(hm.cfg, rope_freq_factors=cfg.rope_freq_factors))
    toks, gaps = oracle_with_table(OracleModel(hm_f), 4096, cfg.rope_freq_factors).generate(prompt[0], 24)
    if not np.array_equal(got, toks):
        j = int(np.nonzero(got != toks)[0][0])
        assert gaps[j] < 1e-4
    # the factors are applied: a decoder without them computes different logits from the second position on
    plain = decode.Decoder(client, hm.cfg, hm.scheme, batch=1, max_ctx=64, host=hm)
    for d in (dec, plain):
        d.reset([5])
        for t in (5, 3, 8):
            d.ids.fill_(t)
            d.step()
    torch.cuda.synchronize()
    assert not torch.equal(dec.logits, plain.logits)
