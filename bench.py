#!/usr/bin/env python
"""bench.py -- decode tokens/s of the quantized linear-layer hot path on B200 (BASELINE.json metric).

A *step* is one decode token of the named random-init model: every quantized projection of the model
(4 fused matvec launches per layer + lm_head; 7L+1 projections) plus the glue operators, replayed from one
CUDA graph (the caller pattern of reference src/engine/cuda_graphs.rs:166-189).

    python bench.py --gpus 1 --steps 128 --warmup 16                 # Llama-3-70B GGUF Q4_K_M, batch-1 decode
    torchrun ... bench.py --gpus N ...                               # same model, tensor-parallel over N GPUs (fused NVLink exchange)
    python bench.py --workload mistral-7b:Q6_K                       # any other preset:scheme (also reported in extra.configs)
    python bench.py --impl reference ...                             # the CPU path (oracle port) on host cores

JSON line (one, from rank 0): value = tokens/s with inputs resident in HBM (graph replay, device timed);
e2e = tokens/s through the public step API with the token id coming from / going to pinned host memory every
step (what blazr's decode loop does: one upload, one 8-byte D2H per token, executor_generate.rs:362-405);
roofline = the dominant kernel (gate|up matvec) against MEASURED_PEAKS.json; cpu_baseline = the oracle's
packed-block int8 path on the host cores (reported only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="llama-3-70b:Q4_K_M", help="<model preset>:<scheme>  e.g. mistral-7b:Q6_K, llama-3-8b:AWQ (default: the config "
                    "BASELINE.json's target sentence names; it fits one B200 at 42 GB and runs tensor-parallel at --gpus N)")
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--prompt", type=int, default=32, help="prompt tokens fed before the timed region (reference bench.rs:24)")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary measurements (prefill GEMM, batch-32)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (logits, next token ids) as DIR/<name>.npy, "
                    "so that two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200: the reference arm times a sample of matvecs, not whole decode steps")
    return args


DUMP_LIMIT = 64_000_000  # bytes on disk, all files of one dump together


def write_outputs(out_dir: str, arrays: dict, limit: int = DUMP_LIMIT):
    """Each array goes to out_dir/<name>.npy as float32 (float64 for 64-bit inputs such as token ids, which it holds exactly).
    An array larger than its share of `limit` bytes is replaced by a fixed sample of its flattened elements (seeded, so the
    same elements for the same shape on every run and every build) and the sample's flat indices go to <name>_index.npy."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    share = limit // len(arrays) - 256  # room for the .npy headers of an array and its index
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64 if a.dtype.itemsize == 8 else np.float32)
        if a.nbytes > share:
            rng = np.random.Generator(np.random.PCG64(a.size))
            idx = np.sort(rng.choice(a.size, share // (a.itemsize + 8), replace=False))
            np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)"""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle's packed-block int8 path (the only place bench.py executes oracle/)
# ------------------------------------------------------------------------------------------------
def cpu_tokens_per_s(model: str, scheme: str, batch: int, budget_s: float = 12.0):
    """Times the CPU port on a bounded sample of the workload: whole layers (all 7 projections, M = batch)
    until ~budget_s of work, then scales to 7L+1 projections.  Returns (tok/s, cores, sample text)."""
    import numpy as np

    import oracle
    from blazr_b200 import decode, synth

    cfg = decode.PRESETS[model]
    cores = os.cpu_count() or 1
    try:  # torchrun exports OMP_NUM_THREADS=1 to its workers: the CPU arm uses every host core regardless
        import ctypes
        oracle.lib()
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(int(cores))
    except Exception:
        pass
    fm = decode.layer_formats(cfg, scheme, cfg.n_layers // 2)
    qd, kvd = cfg.n_heads * cfg.head_dim, cfg.n_kv_heads * cfg.head_dim
    shapes = dict(q=(qd, cfg.hidden), k=(kvd, cfg.hidden), v=(kvd, cfg.hidden), o=(cfg.hidden, qd), gate=(cfg.ffn, cfg.hidden),
                  up=(cfg.ffn, cfg.hidden), down=(cfg.hidden, cfg.ffn))
    ggml_like = {p: (f if f in synth.GGML else "Q4_K") for p, f in fm.items()}  # INT4 group formats: timed as the 4-bit block format with a tuned kernel
    lin = []
    for p, (N, K) in shapes.items():
        t = synth.GGML[ggml_like[p]]
        lin.append((t, N, K, synth.random_ggml(t, N, K, seed=1)))
    xs = {K: oracle.quantize_act(synth.random_act(batch, K)) for K in {s[1] for s in shapes.values()}}
    params_layer = sum(N * K for _, N, K, _ in lin)
    # warm-up + timed repetitions of one layer
    for t, N, K, blk in lin[:2]:
        oracle.matvec_ggml_q8_fast(t, blk, N, K, *xs[K])
    reps, t0 = 0, time.perf_counter()
    while True:
        for t, N, K, blk in lin:
            oracle.matvec_ggml_q8_fast(t, blk, N, K, *xs[K])
        reps += 1
        if time.perf_counter() - t0 > budget_s:
            break
    t_layer = (time.perf_counter() - t0) / reps
    params_total = params_layer * cfg.n_layers + cfg.vocab * cfg.hidden
    t_token = t_layer * params_total / params_layer
    sample = (f"{reps} x one layer ({params_layer / 1e6:.0f}M weights, 7 projections, M={batch}) of {model} {scheme} through the CPU port's "
              f"AVX2 packed-block int8 matvec (oracle/cpu_fast.c), OpenMP over rows; scaled by weights to 7L+1 projections")
    return batch / t_token, cores, sample


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model, scheme = args.workload.split(":")
    toks, cores, sample = cpu_tokens_per_s(model, scheme, args.batch, budget_s=20.0)
    out = {
        "metric": "decode_tokens_per_s", "value": toks, "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * args.batch / toks, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int8 x int4/6/8 -> f32",
        "data": "synthetic", "impl": "reference",
        "config": {"workload": f"{model} GGUF {scheme} random-init, batch-{args.batch} greedy decode, {args.prompt}-token prompt then {args.steps} tokens",
                   "parallelism": f"cpu x{cores} threads", "l2": "n/a (CPU path: weights streamed from host DRAM)",
                   "note": "each step is a bounded sample: whole layers through the CPU port, scaled by weights to 7L+1 projections"},
        "cpu_baseline": {"value": toks, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": toks, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def arm_watchdog(seconds: float, what: str):
    """A multi-rank run that deadlocks (a collective with mismatched counts, a peer that died) must not hold the box:
    after `seconds` rank 0 prints an error line in the bench's JSON shape and every rank leaves."""
    def fire():
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"metric": "decode_tokens_per_s", "value": None, "unit": "tokens/s", "impl": "b200",
                              "error": f"watchdog: {what} did not finish within {seconds:.0f} s"}), flush=True)
        os._exit(3)
    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()
    return t


def run_b200(args):
    import numpy as np
    import torch

    from blazr_b200 import decode, ops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    model, scheme = args.workload.split(":")
    cfg = decode.PRESETS[model]
    watchdog = arm_watchdog(float(os.environ.get("B200Q_BENCH_WATCHDOG_S", "900")), f"bench.py --gpus {args.gpus} ({args.workload})")
    client = ops.B200Client(local)
    M = args.batch
    max_ctx = args.prompt + args.warmup + 2 * args.steps + 64
    launches0 = ops.launch_count()
    emu = int(os.environ.get("B200Q_EMULATE_TP", "0"))   # profiling aid: rank 0's shard of a TP-emu model alone on this GPU (world-1 exchange)
    if emu > 1 and world == 1:
        dec = decode.Decoder(client, cfg, scheme, batch=M, max_ctx=max_ctx, tp_rank=0, tp_world=emu, emulate_shard=True)
    else:
        dec = decode.Decoder(client, cfg, scheme, batch=M, max_ctx=max_ctx, tp_rank=rank, tp_world=world)
    if world > 1:
        dist.barrier()
    dec.capture()
    g = dec.graph
    dev = client.device

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    rng = np.random.Generator(np.random.PCG64(11))
    prompt = rng.integers(0, cfg.vocab, size=(M, args.prompt))
    dec.reset(prompt[:, 0])
    for s in range(args.prompt - 1):  # feed the prompt through decode steps (keeps the KV cache realistic)
        dec.replay()
        dec.ids.copy_(torch.from_numpy(prompt[:, s + 1]).to(dev))
    for _ in range(max(3, args.warmup)):
        dec.replay()

    # ---- device-resident throughput: K graph replays between events ----
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        dec.replay()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    outputs = None
    if args.dump_outputs and rank == 0:  # taken now: the end-to-end loop below decodes further tokens into the same buffers
        logits = dec.logits_local if emu > 1 and world == 1 else dec.full_logits()
        outputs = {"logits": logits.cpu().numpy(), "next_ids": dec.ids.cpu().numpy()}

    # ---- end to end through the step API with host buffers ----
    pin_in = torch.zeros(M, dtype=torch.int64).pin_memory()
    pin_out = torch.zeros(M, dtype=torch.int64).pin_memory()
    pin_in.copy_(dec.ids.cpu())
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        dec.ids.copy_(pin_in, non_blocking=True)   # H2D: this step's input token ids
        dec.replay()
        pin_out.copy_(dec.ids, non_blocking=True)  # D2H: the sampled token ids
        torch.cuda.current_stream().synchronize()  # the host needs the token before it can issue the next step
        pin_in.copy_(pin_out)
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)

    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])

    # ---- roofline of the dominant kernel: the fused gate|up matvec, timed alone over all layers ----
    pk, pk_kind = peaks()
    gu = [lay["gu"][0] for lay in dec.layers]
    reps = 20
    import ctypes as C
    L_ = ops.lib()
    P_ = lambda t_: C.c_void_p(t_.data_ptr())
    epi = bool(dec.layers[0]["swiglu_epi"])
    gu_variant = ("norm prologue + " if (dec.fused and epi) else "") + ("SwiGLU epilogue" if epi else "plain")

    def run_gu():  # the same entry point (kernel variant) the decode step launches for gate|up, over every layer's weight
        st_ = ops._stream_ptr(dev)  # the CURRENT stream (the capturing one inside torch.cuda.graph)
        for lay, ln in zip(dec.layers, gu):
            if epi and dec.fused:
                ops._check(L_.b200q_matmul_norm_swiglu(ln.w.handle, P_(dec.h), None, P_(dec.h2), P_(lay["mlp_norm"]), C.c_float(cfg.eps), C.c_int64(M),
                                                       P_(dec.xq_ff), P_(ln.ws), C.c_size_t(ln.ws.numel()), st_))
            elif epi:
                ops._check(L_.b200q_matmul_q8_swiglu(ln.w.handle, P_(dec.xq_h), C.c_int64(M), P_(dec.xq_ff), P_(ln.ws), C.c_size_t(ln.ws.numel()), st_))
            else:
                dec._matvec([ln], dec.xq_h, dec.gu)

    run_gu()
    torch.cuda.synchronize(dev)
    g2 = torch.cuda.CUDAGraph()
    s2 = torch.cuda.Stream(dev)
    s2.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s2):
        with torch.cuda.graph(g2, stream=s2):
            run_gu()
        for _ in range(3):
            g2.replay()
        s2.synchronize()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record(s2)
        for _ in range(reps):
            g2.replay()
        k1.record(s2)
        s2.synchronize()
    us_gu = k0.elapsed_time(k1) * 1e3 / (reps * len(gu))
    w0 = gu[0].w
    bytes_gu = w0.canonical_bytes + M * w0.K * 1.25 + M * w0.N * 4  # canonical packed weights + int8 activation records + f32 outputs
    achieved = bytes_gu / (us_gu * 1e-6) / 1e9
    # whole-step view: all matvec weight bytes over the step time
    step_bytes = dec.weight_bytes
    # DRAM bytes per launch of this kernel from the committed `ncu --set full` capture (profiles/, tools/ncu_summary.py)
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        tk = tj.get(f"{decode.layer_formats(cfg, scheme, 0)['gate']}:{w0.N}x{w0.K}:M{M}")
        if tk:
            traffic = tk["dram_bytes_read"] + tk["dram_bytes_write"]
    except Exception:
        traffic = None
    roof = {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"], "traffic": traffic,
            "kernel": f"matvec_kernel<{decode.layer_formats(cfg, scheme, 0)['gate']}, MB={M}> gate|up N={w0.N} K={w0.K} ({gu_variant})", "us_per_launch": us_gu,
            "algorithmic_bytes_per_launch": bytes_gu, "peak_kind": pk_kind + " burst (kernel timed alone)",
            "step_weight_bytes": step_bytes, "step_GBs": step_bytes / (ms / args.steps * 1e-3) / 1e9,
            "step_frac": step_bytes / (ms / args.steps * 1e-3) / 1e9 / pk["hbm_gbs"]}

    launches_per_step = dec.launches_per_step()
    extra = {}
    if not args.no_extra and rank == 0 and world == 1:
        try:
            # the headline model (42 GB for the default) is released first: the extras build their own models
            del g2, g, gu
            dec.graph = None
            del dec
            torch.cuda.empty_cache()
            extra = extras(client, cfg, scheme, pk, args)
        except Exception as ex:  # secondary measurements must never take the headline line down
            extra = {"error": repr(ex)[:300]}

    if rank == 0:
        toks = M * args.steps / (ms * 1e-3)
        toks_e2e = M * args.steps / (ms_e2e * 1e-3)
        cpu_v, cores, sample = cpu_tokens_per_s(model, scheme, M, budget_s=12.0) if world == 1 else (None, None, None)
        out = {
            "metric": "decode_tokens_per_s", "value": toks, "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int8 activations x int4/6/8 weights, f64-exact accumulate -> f32", "data": "synthetic",
            "config": {"workload": f"{model} GGUF {scheme} random-init, batch-{M} greedy decode, {args.prompt}-token prompt then {args.steps} tokens",
                       "parallelism": f"tp{world}" + (" (fused NVLink exchange: row-parallel matvec pushes, norm / arg-max consume)" if world > 1 else ""), "l2": f"weights {step_bytes * world / 1e9:.1f} GB streamed once per token (>> 126 MB L2)",
                       "launches_per_step": launches_per_step},
            "clocks": clocks,
            "e2e": {"value": toks_e2e, "unit": "tokens/s", "h2d_bytes_per_step": 8 * M, "d2h_bytes_per_step": 8 * M},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": roof,
            "impl": "b200",
        }
        if cpu_v is not None:
            out["cpu_baseline"] = {"value": cpu_v, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample}
        if extra:
            out["extra"] = extra
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(out), flush=True)
    watchdog.cancel()
    if world > 1:
        # NCCL kernels are baked into the captured graphs: drop the graphs, then leave without the collective
        # teardown (destroy_process_group can block on communicators that captured graphs still reference)
        dist.barrier()
        torch.cuda.synchronize(dev)
        sys.stdout.flush()
        os._exit(0)


def time_decode(dec, steps: int, warmup: int = 6, prompt: int = 16):
    """tokens/s of a captured decode step (graph replay, device timed), after `prompt` context tokens"""
    import torch

    dec.capture()
    dec.reset([1] * dec.M)
    for _ in range(prompt + warmup):
        dec.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        dec.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return dec.M / (ms * 1e-3), ms


def matvec_shape_table(client, pk):
    """kernel GB/s of the decode matvec for every projection shape of the 7B/8B configs x the north_star's lead formats:
    one launch per rotating weight copy (copies > 2x L2), graph replay, CUDA events (tools/kbench.py method)."""
    import torch

    from blazr_b200 import decode, ops, synth

    shapes = [("qkv", 6144, 4096), ("o", 4096, 4096), ("gate|up", 28672, 4096), ("down", 4096, 14336), ("lm_head", 32000, 4096)]
    rows = []
    dev = client.device
    for fmt in ("Q4_K", "Q6_K", "Q8_0", "AWQ"):
        for name, N, K in shapes:
            def mk(i):
                if fmt in synth.GGML:
                    return client.weight_from_ggml(synth.GGML[fmt], decode.random_ggml_device(fmt, N, K, 300 + i, dev), N, K)
                qw, sc, z = decode.random_int4_device(fmt, N, K, 128, 300 + i, dev)
                return client.weight_from_decomposed(ops.DecomposedQuantTensor(qw, sc, z, None, ops.DecomposedQuantMethod("awq", 128), (N, K)))
            w0 = mk(0)
            copies = int(min(48, max(2, -(-300e6 // w0.canonical_bytes))))
            ws = [w0] + [mk(i) for i in range(1, copies)]
            xq = client.quantize_act(torch.randn((1, K), device=dev))
            y = torch.empty((1, N), device=dev)
            wss = [w.workspace(1) for w in ws]

            def run_all():
                for w, s_ in zip(ws, wss):
                    client.matmul_q8(xq, 1, w, out=y, workspace=s_)

            run_all()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            st = torch.cuda.Stream()
            st.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(st):
                with torch.cuda.graph(g, stream=st):
                    run_all()
                for _ in range(3):
                    g.replay()
                st.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                reps = 10
                for _ in range(reps):
                    g.replay()
                e1.record(st)
                st.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / (reps * copies)
            b = w0.canonical_bytes + K * 1.25 + N * 4
            rows.append({"fmt": fmt, "proj": name, "N": N, "K": K, "us": round(us, 2), "GBs": round(b / (us * 1e-6) / 1e9, 1),
                         "frac_hbm": round(b / (us * 1e-6) / 1e9 / pk["hbm_gbs"], 3)})
            del g
            for w in ws:
                w.free()
    return rows


def extras(client, cfg, scheme, pk, args):
    """secondary numbers of the north_star, all driver-run with the default command: (1) batch-1 decode tok/s of the other named
    configs, (2) the per-shape matvec table, (3) prefill dequant-GEMM TFLOP/s + prefill pass tokens/s, (4) batch-32 decode,
    (5) a DeepSeek-V2-Lite-shaped MoE layer."""
    import time

    import torch

    from blazr_b200 import decode, ops, synth

    out = {}
    t_start = time.perf_counter()
    budget_s = float(os.environ.get("B200Q_BENCH_EXTRA_S", "170"))   # the default run must end within minutes
    # (1) the other BASELINE configs, batch-1 greedy decode, whole step from one CUDA graph
    cfgs = []
    for wl in ("llama-3.2-1b:Q4_K_M", "mistral-7b:Q6_K", "mistral-7b:Q8_0", "mistral-7b:Q4_K", "llama-3-8b:AWQ", "llama-3-8b:GPTQ", "llama-3-70b:Q4_K_M"):
        if wl == args.workload or time.perf_counter() - t_start > budget_s:
            continue
        m_, s_ = wl.split(":")
        try:
            d_ = decode.Decoder(client, decode.PRESETS[m_], s_, batch=1, max_ctx=160)
            toks, ms = time_decode(d_, 48)
            cfgs.append({"workload": wl, "tokens_per_s": round(toks, 1), "ms_per_step": round(ms, 4), "launches_per_step": d_.launches_per_step(),
                         "step_frac_hbm": round(d_.weight_bytes / (ms * 1e-3) / 1e9 / pk["hbm_gbs"], 3)})
            del d_
        except Exception as ex:
            cfgs.append({"workload": wl, "error": repr(ex)[:200]})
        torch.cuda.empty_cache()
    out["configs"] = cfgs
    # (1b) prefill pass: the whole prompt at M = S through all 7L+1 projections on the tcgen05 dequant-GEMM (+ torch SDPA attention)
    pf = []
    for wl, S in (("mistral-7b:Q6_K", 2048), ("llama-3-8b:AWQ", 4096)):
        if time.perf_counter() - t_start > budget_s:
            break
        m_, s_ = wl.split(":")
        try:
            c_ = decode.PRESETS[m_]
            d_ = decode.Decoder(client, c_, s_, batch=1, max_ctx=S + 16)
            prompt = torch.randint(0, c_.vocab, (S,)).numpy()
            d_.prefill(prompt)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 2
            e0.record()
            for _ in range(reps):
                d_.prefill(prompt)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            lin_flops = 2.0 * S * sum(ln.w.N * ln.w.K for lay in d_.layers for key in ("qkv", "o", "gu", "down") for ln in lay[key])
            pf.append({"workload": wl, "prompt_tokens": S, "ms": round(ms, 2), "prefill_tokens_per_s": round(S / (ms * 1e-3), 1),
                       "linear_TFLOPs": round(lin_flops / (ms * 1e-3) / 1e12, 1), "frac_bf16_burst_incl_attention_and_glue": round(lin_flops / (ms * 1e-3) / 1e12 / pk["bf16_tflops"], 3)})
            del d_
        except Exception as ex:
            pf.append({"workload": wl, "error": repr(ex)[:200]})
        torch.cuda.empty_cache()
    out["prefill_pass"] = pf
    # (2) per-shape kernel table
    if time.perf_counter() - t_start < budget_s:
        try:
            out["matvec_shapes"] = matvec_shape_table(client, pk)
        except Exception as ex:
            out["matvec_shapes"] = {"error": repr(ex)[:200]}
    # (3)-(5) on the Mistral-7B shapes (BASELINE config 2) whatever the headline workload is
    cfg = decode.PRESETS["mistral-7b"]
    scheme = "Q6_K"
    # prefill dequant-GEMM (tcgen05/TMEM) on the gate projection shape: Mistral-7B Q6_K / Q8_0 at S = 2048 (config 2),
    # Llama-3-8B AWQ at S = 4096 (config 3); skinny M = 32 (batched decode) on the same weight
    N, K = cfg.ffn, cfg.hidden
    dev = client.device

    def mk_weight(fmt, i):
        if fmt in synth.GGML:
            return client.weight_from_ggml(synth.GGML[fmt], decode.random_ggml_device(fmt, N, K, 100 + i, dev), N, K)
        qw, sc, z = decode.random_int4_device(fmt, N, K, 128, 100 + i, dev)
        return client.weight_from_decomposed(ops.DecomposedQuantTensor(qw, sc, z, None, ops.DecomposedQuantMethod("awq", 128), (N, K)))

    for name, fmt, Mx in (("prefill_2048", "Q6_K", 2048), ("prefill_2048_q8_0", "Q8_0", 2048), ("prefill_4096_awq", "AWQ", 4096), ("decode_batch32", "Q6_K", 32)):
        if time.perf_counter() - t_start > budget_s:
            break
        try:
            copies = 4
            ws = [mk_weight(fmt, i) for i in range(copies)]
            x = torch.randn((Mx, K), device=dev)
            if fmt == "AWQ":
                x = x.half()   # AWQ / GPTQ activations are f16 in blazr (awq.rs:69-71)
            y = torch.empty((Mx, N), device=dev, dtype=x.dtype)
            wss = [w.workspace(Mx) for w in ws]
            for w, s_ in zip(ws, wss):
                client.quant_matmul(x, w, out=y, workspace=s_)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 5
            e0.record()
            for _ in range(reps):
                for w, s_ in zip(ws, wss):
                    client.quant_matmul(x, w, out=y, workspace=s_)
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / (reps * copies)
            tf = 2.0 * Mx * N * K / (us * 1e-6) / 1e12
            out[name] = {"shape": f"{fmt} N={N} K={K} M={Mx}", "us": us, "TFLOPs": tf, "frac_bf16_burst": tf / pk["bf16_tflops"],
                         "frac_bf16_sustained": tf / pk.get("bf16_tflops_sustained", pk["bf16_tflops"]),
                         "GBs": ws[0].canonical_bytes / (us * 1e-6) / 1e9, "includes": "f16 activation staging kernel + tcgen05 GEMM"}
            for w in ws:
                w.free()
        except Exception as ex:
            out[name] = {"error": repr(ex)[:200]}
    # whole-step batched decode (BASELINE metric: "decode tok/s at batch 1 and batch 32"): 32 sequences, every
    # projection on the tcgen05 path, replayed from one CUDA graph
    try:
        B = 32
        decb = decode.Decoder(client, cfg, scheme, batch=B, max_ctx=96)
        decb.capture()
        decb.reset([1] * B)
        for _ in range(8):
            decb.graph.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        steps = 24
        e0.record()
        for _ in range(steps):
            decb.graph.replay()
        e1.record()
        torch.cuda.synchronize()
        msb = e0.elapsed_time(e1) / steps
        out["decode_batch32_step"] = {"tokens_per_s": B / (msb * 1e-3), "ms_per_step": msb, "launches_per_step": decb.launches_per_step(),
                                      "step_frac_hbm": decb.weight_bytes / (msb * 1e-3) / 1e9 / pk["hbm_gbs"],
                                      "what": f"{cfg.name} {scheme} batch-32 greedy decode, whole step (graph replay), context 9..32"}
        del decb
    except Exception as ex:  # secondary number: never take the headline down with it
        out["decode_batch32_step"] = {"error": repr(ex)[:200]}
    # MoE decode (BASELINE config 5 shapes: DeepSeek-V2-Lite, 64 routed experts + 2 shared halves, top-6; gate|up Q4_K
    # [2816 x 2048] in the SwiGLU-epilogue row order, down Q8_0 [2048 x 1408] because K = 1408 is not a multiple of 256): one token
    # through the expert MLP = quantise, grouped gate|up + SwiGLU epilogue, grouped down, combine -- 4 PDL-chained launches,
    # 16 different routings captured in ONE CUDA graph (every expert weight is touched, > L2)
    try:
        E, top_k, hidden, ffn = 66, 8, 2048, 1408
        tg, td = synth.GGML["Q4_K"], synth.GGML["Q8_0"]
        gu = [client.weight_from_ggml(tg, decode.random_ggml_device("Q4_K", 2 * ffn, hidden, 500 + e, client.device), 2 * ffn, hidden) for e in range(E)]
        dn = [client.weight_from_ggml(td, decode.random_ggml_device("Q8_0", hidden, ffn, 700 + e, client.device), hidden, ffn) for e in range(E)]
        moe = ops.MoeMlp(client, [ops.ExpertWeights(g, d, interleaved=True) for g, d in zip(gu, dn)], ffn, hidden)
        x = torch.randn((1, hidden), device=client.device)
        gen = torch.Generator(device="cpu"); gen.manual_seed(3)
        nsel = 16
        sels = [torch.cat([torch.randperm(64, generator=gen)[:6], torch.tensor([64, 65])]).to(torch.int32).reshape(1, top_k).to(client.device) for _ in range(nsel)]
        gw = torch.full((1, top_k), 1.0 / top_k, device=client.device)
        n0 = ops.launch_count()
        moe.forward_decode(x, sels[0], gw)
        per_call = ops.launch_count() - n0
        torch.cuda.synchronize()
        gm = torch.cuda.CUDAGraph()
        sm = torch.cuda.Stream()
        sm.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(sm):
            with torch.cuda.graph(gm, stream=sm):
                for sl in sels:
                    moe.forward_decode(x, sl, gw)
            for _ in range(3):
                gm.replay()
            sm.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 10
            e0.record(sm)
            for _ in range(reps):
                gm.replay()
            e1.record(sm)
            sm.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / (reps * nsel)
        wbytes = top_k * (gu[0].canonical_bytes + dn[0].canonical_bytes)
        out["moe_decode_layer"] = {"us": us, "GBs": wbytes / (us * 1e-6) / 1e9, "frac_hbm": wbytes / (us * 1e-6) / 1e9 / pk["hbm_gbs"],
                                   "weight_bytes_per_token": wbytes, "launches_per_layer": per_call,
                                   "what": "DeepSeek-V2-Lite expert MLP, 1 token: 6 routed of 64 + 2 shared halves, Q4_K gate|up + Q8_0 down; quantise, grouped "
                                           "gate|up with fused SwiGLU epilogue, grouped down, combine; graph replay over 16 routings"}
    except Exception as ex:
        out["moe_decode_layer"] = {"error": repr(ex)[:200]}
    return out


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
