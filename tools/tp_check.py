"""torchrun script: tensor-parallel decode over N GPUs equals the 1-GPU decode (logits within 1e-5, same greedy
stream).  Rank 0 also runs the 1-GPU model for reference.  --kv-dtype f16 runs both with an f16 KV cache (default f32)."""
import argparse, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from blazr_b200 import decode, ops

ap = argparse.ArgumentParser()
ap.add_argument("--kv-dtype", choices=sorted(decode.KV_DTYPES), default="f32")
kv_dtype = ap.parse_args().kv_dtype

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
cfg = decode.PRESETS["tiny" if world <= 2 else "small-1b"]   # tiny has 2 kv heads; small-1b (32 heads / 8 kv) shards up to TP8
ok = True
for scheme in (("Q4_K_M", "Q8_0", "AWQ") if world <= 2 else ("Q4_K_M",)):
    hm = decode.build_host_model(cfg, scheme, seed=2)
    client = ops.B200Client(local)
    dec = decode.Decoder(client, cfg, scheme, batch=1, max_ctx=96, host=hm, tp_rank=rank, tp_world=world, kv_dtype=kv_dtype)
    prompt = np.asarray([[3, 1, 4, 1, 5, 9, 2, 6]])
    got = dec.generate(prompt, 48, use_graph=True)[0]
    logits_tp = dec.full_logits()[0].cpu().numpy()
    if rank == 0:
        ref_dec = decode.Decoder(client, cfg, scheme, batch=1, max_ctx=96, host=hm, kv_dtype=kv_dtype)
        ref = ref_dec.generate(prompt, 48, use_graph=True)[0]
        lref = ref_dec.logits[0].cpu().numpy()
        same = bool(np.array_equal(got, ref))
        err = float(np.abs(logits_tp - lref).max() / np.abs(lref).max())
        bits = float((logits_tp.view(np.uint32) != lref.view(np.uint32)).mean())
        print(f"tp{world} {scheme} kv {kv_dtype}: exchange={'fused peer-memory (matvec push -> norm / arg-max consumer)' if dec.comm is not None else 'NCCL'} logits differing in any bit: {bits:.2e}", flush=True)
        print(f"tp{world} {scheme} kv {kv_dtype}: greedy stream equal={same} first mismatch={int(np.nonzero(got != ref)[0][0]) if not same else -1} last-step logits rel err={err:.2e}", flush=True)
        ok = ok and (same or err < 1e-4)
    dist.barrier()
if rank == 0:
    print("TP_CHECK", "PASS" if ok else "FAIL", flush=True)
torch.cuda.synchronize()
sys.stdout.flush()
os._exit(0)
