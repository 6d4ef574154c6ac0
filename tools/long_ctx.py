"""Long-context decode measurements: the split-context attention kernels against the single-CTA kernel, and whole captured
decode steps at positions up to 120k.  Needs a GPU (no fallback); writes DIR/long_ctx.json and prints a markdown table.

    python tools/long_ctx.py --out DIR [--quick] [--kv-dtype f32|f16|both]

Operator: Llama-3.2-1B (32/8/64), Llama-3.1-8B (32/8/128) and 70B (64/8/128) attention at M = 1, CUDA events around calls
that cycle through one KV cache per layer, enough caches that the K+V working set exceeds the 126 MB L2 several times.  Both
kernels run at positions <= 40959 (same caches, max_ctx 40960), the split kernels alone at 65535 / 131071 (max_ctx 131072).
Reported: us per call, K+V bytes, GB/s, share of the HBM bound and of the f64 bound (the data-sheet rates below), and how many
outputs differ between the two kernels.  An f16 cache holds the same seeded data rounded to f16 (bytes counted at 2 per element).
Whole step: random-weight Q4_K_M decoders with the Llama 3.1 RoPE factors, caches filled from a seed up to P, pos = P, graph
replays timed with CUDA events; with f16, one capacity row f32 cannot hold: the 8B shape at batch 8 and max_ctx 131072."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from blazr_b200 import decode, ops  # noqa: E402

HBM_BPS = 7.7e12        # NVIDIA HGX B200 data sheet, one GPU
F64_FLOPS = 37e12       # same data sheet: FP64 per GPU (one DFMA = 2 flops)
L2_BYTES = 126 << 20
SHAPES = {"llama-3.2-1b": (32, 8, 64), "llama-3.1-8b": (32, 8, 128), "llama-3-70b": (64, 8, 128)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def llama31_factors(hd, theta=500000.0, factor=8.0, low=1.0, high=4.0, orig=8192):
    import math
    out = []
    for f in 1.0 / (theta ** (np.arange(0, hd, 2, dtype=np.float32) / hd)):
        wl = 2 * math.pi / f
        if wl < orig / high:
            out.append(1.0)
        elif wl > orig / low:
            out.append(factor)
        else:
            s = (orig / wl - low) / (high - low)
            out.append(1 / ((1 - s) / factor + s))
    return tuple(float(x) for x in np.asarray(out, dtype=np.float32))


def time_calls(fn, n_caches, min_ms=200.0):
    for i in range(n_caches):   # warm-up: every cache once
        fn(i)
    torch.cuda.synchronize()
    reps = 1
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for r in range(reps):
            for i in range(n_caches):
                fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= min_ms or reps >= 64:
            return 1000.0 * ms / (reps * n_caches)
        reps *= 2


KV_CODE = {"f32": 0, "f16": 1}   # B200Q_F32 / B200Q_F16


def operator_rows(quick, dtypes):
    L = ops.lib()
    st = ops._stream_ptr(torch.device("cuda"))
    P = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    rows = []
    positions = [1023, 4095, 16383, 40959, 65535, 131071] if not quick else [1023, 40959, 65535]
    for name, (nh, nkv, hd) in SHAPES.items():
        for p, dt in [(p, dt) for p in positions for dt in dtypes]:
            max_ctx = 40960 if p < 40960 else 131072
            esize = 4 if dt == "f32" else 2
            kvt = C.c_int32(KV_CODE[dt])
            kv_bytes = 2 * (p + 1) * nkv * hd * esize
            n_caches = int(min(256, max(2, -(-4 * L2_BYTES // kv_bytes))))
            g = torch.Generator(device="cuda")
            g.manual_seed(p)
            # M = 1: the kernels touch rows 0..p of the cache only, so each cache holds p + 1 rows.  f16: the same seeded data, rounded
            conv = (lambda t: t) if dt == "f32" else decode.kv_round
            caches = [(conv(torch.randn((p + 1, nkv, hd), device="cuda", generator=g)), conv(torch.randn((p + 1, nkv, hd), device="cuda", generator=g)))
                      for _ in range(n_caches)]
            qkv = torch.randn((1, (nh + 2 * nkv) * hd), device="cuda", generator=g) * 2.0
            pos = torch.tensor([p], dtype=torch.int32, device="cuda")
            rope = torch.from_numpy(decode.rope_table(max_ctx, hd, 500000.0)).cuda()
            ws = torch.zeros(int(L.b200q_attn_split_workspace_bytes(nh, nkv, hd, max_ctx, 1)), dtype=torch.uint8, device="cuda")
            out_s = torch.empty((1, nh * hd), device="cuda")
            out_1 = torch.empty((1, nh * hd), device="cuda")

            def split(i, out=out_s):
                ops._check(L.b200q_attn_decode_split_kv(P(qkv), P(pos), P(caches[i][0]), P(caches[i][1]), kvt, P(rope), nh, nkv, hd, max_ctx,
                                                        C.c_int64(1), None, P(out), P(ws), C.c_size_t(ws.numel()), st))

            def single(i, out=out_1):
                ops._check(L.b200q_attn_decode_kv(P(qkv), P(pos), P(caches[i][0]), P(caches[i][1]), kvt, P(rope), nh, nkv, hd, max_ctx,
                                                  C.c_int64(1), None, P(out), st))

            flops = 4.0 * nh * hd * (p + 1)      # scores and weighted sum: one DFMA per (query head, element, position) each
            t_hbm, t_f64 = kv_bytes / HBM_BPS * 1e6, flops / F64_FLOPS * 1e6
            row = dict(shape=name, kv_dtype=dt, nh=nh, nkv=nkv, hd=hd, pos=p, max_ctx=max_ctx, kv_bytes=kv_bytes, caches=n_caches,
                       hbm_bound_us=round(t_hbm, 2), f64_bound_us=round(t_f64, 2))
            us = time_calls(split, n_caches)
            row.update(split_us=round(us, 2), split_gbps=round(kv_bytes / us / 1e3, 1), split_hbm_share=round(t_hbm / us, 3),
                       split_f64_share=round(t_f64 / us, 3))
            if max_ctx == 40960:
                us1 = time_calls(single, n_caches)
                row.update(single_us=round(us1, 2), single_gbps=round(kv_bytes / us1 / 1e3, 1), single_hbm_share=round(t_hbm / us1, 3),
                           single_f64_share=round(t_f64 / us1, 3))
                split(0)
                single(0)
                torch.cuda.synchronize()
                a, b = out_s.cpu().numpy().view(np.uint32), out_1.cpu().numpy().view(np.uint32)
                row["outputs_differing"] = int((a != b).sum())
                row["outputs"] = int(a.size)
            else:
                row.update(single_us=None, outputs_differing=None)
            print(json.dumps(row), flush=True)
            rows.append(row)
            del caches, ws
            torch.cuda.empty_cache()
    return rows


def fill_caches(dec, P, seed):
    g = torch.Generator(device=dec.dev)
    g.manual_seed(seed)
    for lay in dec.layers:
        for key in ("ck", "cv"):
            c = lay[key]
            for m in range(dec.M):
                for j0 in range(0, P, 8192):   # in slices: no P-sized temporary (an f16 cache stores the rounded values)
                    j1 = min(P, j0 + 8192)
                    x = torch.randn(c[m, j0:j1].shape, device=dec.dev, generator=g) * 0.5
                    c[m, j0:j1].copy_(x if c.dtype == torch.float32 else decode.kv_round(x))


def step_rows(quick, dtypes):
    client = ops.B200Client(0)
    rows = []
    runs = []   # (model, position, max_ctx, batch, kv dtype)
    for model in ("llama-3-8b", "llama-3.2-1b"):
        for dt in dtypes:
            for P in ((1024, 32768, 65536, 122880) if not quick else (1024, 65536)):
                runs.append((model, P, 131072, 1, dt))
            runs.append((model, 32768, 40960, 1, dt))
    for dt in dtypes:
        runs.append(("llama-3-70b", 65536, 65536 + 512, 1, dt))
        if not quick:
            runs.append(("llama-3-70b", 122880, 122880 + 512, 1, dt))
    if "f16" in dtypes and not quick:
        runs.append(("llama-3-8b", 122880, 131072, 8, "f16"))   # capacity: 128 GiB of f16 cache (256 GiB in f32)
    for model, P, max_ctx, batch, dt in runs:
        base = decode.PRESETS[model]
        cfg = decode.ModelConfig(*[getattr(base, f) for f in ("name", "hidden", "n_layers", "n_heads", "n_kv_heads", "head_dim", "ffn", "vocab",
                                                             "rope_theta", "eps")], rope_freq_factors=llama31_factors(base.head_dim))
        kv = 2 * cfg.n_layers * batch * max_ctx * cfg.n_kv_heads * cfg.head_dim * (4 if dt == "f32" else 2)
        wbytes = 4.9 / 8 * cfg.n_layers * (cfg.hidden * (cfg.n_heads + 2 * cfg.n_kv_heads) * cfg.head_dim + cfg.hidden * cfg.n_heads * cfg.head_dim
                                           + 3 * cfg.hidden * cfg.ffn) + 2.5 * cfg.vocab * cfg.hidden
        free, _ = torch.cuda.mem_get_info()
        row = dict(model=model, kv_dtype=dt, batch=batch, pos=P, max_ctx=max_ctx, kv_cache_bytes=kv, est_weight_bytes=int(wbytes), free_bytes=int(free))
        if kv + wbytes + (4 << 30) > free:
            row.update(skipped=f"needs ~{(kv + wbytes) / 2**30:.0f} GiB, {free / 2**30:.0f} GiB free")
            print(json.dumps(row), flush=True)
            rows.append(row)
            continue
        t0 = time.time()
        dec = decode.Decoder(client, cfg, "Q4_K_M", batch=batch, max_ctx=max_ctx, kv_dtype=dt)
        assert dec.kv_cache_bytes == kv
        fill_caches(dec, P, seed=P)
        dec.reset([1] * batch)
        dec.pos.fill_(P)
        dec._host_pos = P
        dec.capture()
        for _ in range(3):
            dec.replay()
        torch.cuda.synchronize()
        steps = 32
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            dec.replay()
        e1.record()
        torch.cuda.synchronize()
        dec.check_device_errors()
        ms = e0.elapsed_time(e1) / steps
        row.update(path="split" if dec.attn_split else "single-CTA", ms_per_step=round(ms, 3), tok_s=round(1000.0 * batch / ms, 1),
                   setup_s=round(time.time() - t0, 1))
        print(json.dumps(row), flush=True)
        rows.append(row)
        del dec
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--quick", action="store_true", help="fewer positions (a rehearsal)")
    ap.add_argument("--skip-steps", action="store_true")
    ap.add_argument("--kv-dtype", choices=["f32", "f16", "both"], default="f32", help="KV cache element type(s) to measure")
    a = ap.parse_args()
    dtypes = ["f32", "f16"] if a.kv_dtype == "both" else [a.kv_dtype]
    if not torch.cuda.is_available():
        raise SystemExit("long_ctx.py measures on a GPU: none is present")
    os.makedirs(a.out, exist_ok=True)
    res = dict(info=gpu_info(), hbm_bps_datasheet=HBM_BPS, f64_flops_datasheet=F64_FLOPS)
    print(json.dumps(res["info"]), flush=True)
    res["operator"] = operator_rows(a.quick, dtypes)
    with open(os.path.join(a.out, "long_ctx.json"), "w") as f:
        json.dump(res, f, indent=1)
    if not a.skip_steps:
        res["step"] = step_rows(a.quick, dtypes)
    with open(os.path.join(a.out, "long_ctx.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
