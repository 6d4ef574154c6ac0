"""Random-init Llama-family decode harness: drives the quantized matvec kernels through one whole decode
step (the caller pattern of reference src/engine/executor_generate.rs:362-405 and the captured step of
src/engine/cuda_graphs.rs:101-189), so kernel GB/s turns into tokens/s.

Per layer (batch-1..4 decode, everything enqueued on one stream, PDL-chained, graph-capturable):
    add+rmsnorm+quant -> [q|k|v] matvec(s) -> RoPE+KV-append+attention+quant -> o matvec
    add+rmsnorm+quant -> [gate|up] matvec(s) -> SwiGLU+quant -> down matvec
then add+rmsnorm+quant -> lm_head matvec -> argmax (greedy, the configs' sampling mode).

Projections of equal format are fused at upload (q,k,v / gate,up share one weight handle, i.e. one launch);
the GGUF "Q4_K_M" mix keeps attn_v / ffn_down of the "more bits" layers in Q6_K (SURVEY.md Appendix B).
Tensor parallel (reference src/engine/tensor_parallel.rs, Megatron split): column-split q/k/v/gate/up by
heads / rows, row-split o/down along K at block granularity, all-reduce after o and down, vocab-split
lm_head + all-gather.

PyTorch is plumbing only (buffers, streams, NCCL); all math runs in libb200q kernels.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import ops, synth, tp


@dataclass
class ModelConfig:
    name: str
    hidden: int
    n_layers: int
    n_heads: int
    n_kv_heads: int
    head_dim: int
    ffn: int
    vocab: int
    rope_theta: float = 10000.0
    eps: float = 1e-5
    # Llama 3.1 / 3.2 ("llama3" rope scaling): per-frequency divisors of the RoPE frequencies, head_dim / 2 values
    # (llama.cpp stores them as the rope_freqs.weight tensor); None = unscaled
    rope_freq_factors: Optional[Tuple[float, ...]] = None


PRESETS: Dict[str, ModelConfig] = {
    "llama-3.2-1b": ModelConfig("llama-3.2-1b", 2048, 16, 32, 8, 64, 8192, 128256, 500000.0),
    "mistral-7b": ModelConfig("mistral-7b", 4096, 32, 32, 8, 128, 14336, 32000, 10000.0),
    "llama-3-8b": ModelConfig("llama-3-8b", 4096, 32, 32, 8, 128, 14336, 128256, 500000.0),
    "llama-3-70b": ModelConfig("llama-3-70b", 8192, 80, 64, 8, 128, 28672, 128256, 500000.0),
    # reduced shapes for tests (same structure, seconds on the CPU oracle)
    "tiny": ModelConfig("tiny", 512, 2, 8, 2, 64, 1024, 2048, 10000.0),
    "small-1b": ModelConfig("small-1b", 2048, 4, 32, 8, 64, 8192, 16384, 500000.0),
}


# Decoder(kv_dtype=...): torch element type of the KV cache and the b200q_dtype the *_kv attention entry points take
KV_DTYPES = {"f32": (torch.float32, 0), "f16": (torch.float16, 1)}


def kv_round(x: torch.Tensor) -> torch.Tensor:
    """The f16 KV cache element rule of the attention kernels: f16_rn(clamp(x, +-65504)), NaN -> -65504 (torch's conversion
    rounds to nearest even, as __float2half_rn does)"""
    return x.nan_to_num(nan=-65504.0).clamp(-65504.0, 65504.0).to(torch.float16)


def rope_table(max_ctx: int, head_dim: int, theta: float, factors=None) -> np.ndarray:
    """[max_ctx, hd/2, 2] f32 (cos, sin) of pos * theta^(-2i/hd) / factors[i], computed in f64 and rounded once.  The same
    formula is restated in oracle/model.py (unscaled) and tests/rope_ref.py (with factors); a table (instead of device
    powf/sincos) keeps RoPE bit-reproducible.
    factors: the Llama 3.1 / 3.2 frequency divisors (ggml divides theta by them); None leaves the frequencies unscaled."""
    i = np.arange(head_dim // 2, dtype=np.float64)
    freq = np.power(float(theta), -2.0 * i / head_dim)
    if factors is not None:
        freq = freq / np.asarray(factors, dtype=np.float64).reshape(head_dim // 2)
    ang = np.arange(max_ctx, dtype=np.float64)[:, None] * freq[None, :]
    return np.stack([np.cos(ang), np.sin(ang)], axis=-1).astype(np.float32)


def use_more_bits(i: int, n: int) -> bool:
    """llama.cpp's layer rule for the *_M mixes (public convention, SURVEY.md Appendix B)"""
    return i < n // 8 or i >= 7 * n // 8 or (i - n // 8) % 3 == 2


def layer_formats(cfg: ModelConfig, scheme: str, i: int) -> Dict[str, str]:
    """format of each projection of layer i under a quantisation scheme"""
    if scheme == "Q4_K_M":
        hi = "Q6_K" if use_more_bits(i, cfg.n_layers) else "Q4_K"
        return dict(q="Q4_K", k="Q4_K", v=hi, o="Q4_K", gate="Q4_K", up="Q4_K", down=hi)
    return {p: scheme for p in ("q", "k", "v", "o", "gate", "up", "down")}


def head_format(scheme: str) -> str:
    return "Q6_K" if scheme == "Q4_K_M" else scheme


# ------------------------------------------------------------------------------------------------
# host-side random weights (numpy; the oracle consumes the very same arrays)
# ------------------------------------------------------------------------------------------------
@dataclass
class HostLinear:
    fmt: str
    N: int
    K: int
    data: object  # ggml: uint8 [N, row_bytes]; AWQ: (qweight, scales, zeros, gs); GPTQ: (qweight, scales, qzeros, g_idx, gs)


@dataclass
class HostModel:
    cfg: ModelConfig
    scheme: str
    embed: np.ndarray                 # f16 [V, H]
    layers: List[Dict[str, object]] = field(default_factory=list)  # per layer: HostLinear per projection + norms
    final_norm: Optional[np.ndarray] = None
    lm_head: Optional[HostLinear] = None


def _host_linear(fmt: str, N: int, K: int, seed: int) -> HostLinear:
    if fmt in synth.GGML:
        return HostLinear(fmt, N, K, synth.random_ggml(synth.GGML[fmt], N, K, seed=seed))
    if fmt == "AWQ":
        return HostLinear(fmt, N, K, synth.random_awq(N, K, 128, seed=seed) + (128,))
    if fmt == "GPTQ":
        qw, sc, qz, gi, _ = synth.random_gptq(N, K, 128, seed=seed)
        return HostLinear(fmt, N, K, (qw, sc, qz, gi, 128))
    raise ValueError(fmt)


def build_host_model(cfg: ModelConfig, scheme: str, seed: int = 0xB200) -> HostModel:
    rng = np.random.Generator(np.random.PCG64(seed))
    hm = HostModel(cfg, scheme, embed=rng.standard_normal((cfg.vocab, cfg.hidden)).astype(np.float16))
    qd, kvd = cfg.n_heads * cfg.head_dim, cfg.n_kv_heads * cfg.head_dim
    shapes = dict(q=(qd, cfg.hidden), k=(kvd, cfg.hidden), v=(kvd, cfg.hidden), o=(cfg.hidden, qd), gate=(cfg.ffn, cfg.hidden),
                  up=(cfg.ffn, cfg.hidden), down=(cfg.hidden, cfg.ffn))
    for i in range(cfg.n_layers):
        fm = layer_formats(cfg, scheme, i)
        lay: Dict[str, object] = {}
        for j, (p, (N, K)) in enumerate(shapes.items()):
            lay[p] = _host_linear(fm[p], N, K, seed + 1000 * (i + 1) + j)
        lay["attn_norm"] = (1.0 + 0.1 * rng.standard_normal(cfg.hidden)).astype(np.float32)
        lay["mlp_norm"] = (1.0 + 0.1 * rng.standard_normal(cfg.hidden)).astype(np.float32)
        hm.layers.append(lay)
    hm.final_norm = (1.0 + 0.1 * rng.standard_normal(cfg.hidden)).astype(np.float32)
    hm.lm_head = _host_linear(head_format(scheme), cfg.vocab, cfg.hidden, seed + 999)
    return hm


# ------------------------------------------------------------------------------------------------
# device-side random ggml blocks (bench: 6-39 GB of weights are generated directly in HBM)
# ------------------------------------------------------------------------------------------------
def random_ggml_device(fmt: str, N: int, K: int, seed: int, device) -> torch.Tensor:
    t = synth.GGML[fmt]
    be, bb = synth.GGML_SIZES[t]
    nb = N * (K // be)
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    blk = torch.randint(0, 256, (nb, bb), dtype=torch.uint8, device=device, generator=g)
    d_off, m_off, ratio, std1 = synth._FIELDS[t]
    sigma = 1.0 / (std1 * float(np.sqrt(K)))
    d = ((torch.rand(nb, device=device, generator=g) + 0.5) * sigma).to(torch.float16)
    if t == 29:
        raise NotImplementedError("IQ1_M keeps d in scattered nibbles: use synth.random_ggml (host) for it")
    for o in d_off:
        blk[:, o:o + 2] = d.view(torch.uint8).reshape(nb, 2)
    if m_off:
        mm = (d.float() * ratio).to(torch.float16)
        for o in m_off:
            blk[:, o:o + 2] = mm.view(torch.uint8).reshape(nb, 2)
    return blk.reshape(N, K // be * bb)


def random_int4_device(kind: str, N: int, K: int, gs: int, seed: int, device):
    """AWQ / GPTQ tensors of blazr's loader layouts generated directly in HBM (bench: no host round trip).
    AWQ : qweight u32 [K, N/8], scales f32 [K/gs, N] (f16-representable), zeros f32 [K/gs, N] integers 0..15
    GPTQ: qweight u32 [K/8, N], scales f32 [G, N], qzeros u32 [G, N/8] packed (no act-order)"""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    G = K // gs
    u32 = lambda *shape: torch.randint(-2 ** 31, 2 ** 31, shape, dtype=torch.int32, device=device, generator=g)
    scales = ((torch.rand((G, N), device=device, generator=g) + 0.5) / (4.6 * float(np.sqrt(K)))).to(torch.float16).to(torch.float32)
    if kind == "AWQ":
        zeros = torch.randint(0, 16, (G, N), device=device, generator=g).to(torch.float32)
        return u32(K, N // 8), scales, zeros
    return u32(K // 8, N), scales, u32(G, N // 8)


_NAME_ID = dict(q=1, k=2, v=3, o=4, gate=5, up=6, down=7, lm_head=8)


@dataclass
class _Linear:
    """one launch: a (possibly fused) weight writing into out[:, col0 : col0 + N]"""
    w: ops.QuantWeight
    col0: int
    ws: torch.Tensor
    fmt: str = ""


class Decoder:
    """One rank of a (tensor-parallel) decoder.  `host` gives exact weights (tests); otherwise weights are
    random blocks generated on the device (bench)."""

    def __init__(self, client: ops.B200Client, cfg: ModelConfig, scheme: str, batch: int = 1, max_ctx: int = 512,
                 host: Optional[HostModel] = None, seed: int = 0xB200, tp_rank: int = 0, tp_world: int = 1, group=None,
                 paged: bool = False, block_size: int = 16, emulate_shard: bool = False, kv_dtype: str = "f32"):
        """paged: KV cache as block pools + block table (reference InferenceConfig.paged_attention / block_size = 16,
        src/config/inference.rs:94-98; forward_with_paged_kv_cache, src/engine/batch_decode.rs:137-147) instead of one
        contiguous [max_ctx] region per sequence.  emulate_shard: build rank tp_rank's shard of a tp_world-way tensor-parallel
        model but run it ALONE on this GPU through the same fused-exchange kernels (world-1 communicator): the per-rank
        latency structure of TP-N measured on one GPU (tools / profiling only; the logits are those of the shard).
        The block table is pre-populated with a shuffled assignment of the pool's
        blocks; a scheduler may overwrite `block_table` / `slot_mapping` between steps (blazr_b200/batch.py builds them).
        kv_dtype: "f32" (default) or "f16" KV cache; f16 halves the cache and stores f16_rn(clamp(x, +-65504)) of every K / V
        element (include/b200q.h, b200q_attn_decode_kv)."""
        assert 1 <= batch <= 256
        if kv_dtype not in KV_DTYPES:
            raise ValueError(f"kv_dtype {kv_dtype!r}: one of {sorted(KV_DTYPES)}")
        self.kv_dtype = kv_dtype
        kv_t = KV_DTYPES[kv_dtype][0]
        # M <= 4: dp4a matvec on int8 activation records (bit-exact contract); M > 4 (batched decode, reference
        # src/engine/batch_decode.rs:115-147): tcgen05 dequant-GEMM on f32 activations (1e-2 tolerance contract)
        self.wide = batch > 4
        assert not (self.wide and tp_world > 1), "batched decode is single-GPU in this round"
        if paged:
            max_ctx = -(-max_ctx // block_size) * block_size   # whole blocks
        self.c, self.cfg, self.scheme, self.M, self.max_ctx = client, cfg, scheme, batch, max_ctx
        self.rank, self.world, self.group = tp_rank, tp_world, group
        dev = client.device
        self.dev = dev
        H, hd = cfg.hidden, cfg.head_dim
        pl = tp.plan(H, cfg.n_heads, cfg.n_kv_heads, hd, cfg.ffn, cfg.vocab, tp_rank, tp_world)  # tensor_parallel.rs:61-101
        self.plan = pl
        self.nh, self.nkv = pl.n_heads, pl.n_kv_heads
        self.qd, self.kvd = self.nh * hd, self.nkv * hd
        f0, f1 = pl.ffn_rows
        self.ff = f1 - f0
        v0, v1 = pl.vocab_rows
        self.v0, self.v1 = v0, v1
        self.weight_bytes = 0
        self.layers = []
        M = batch
        import os as _os
        # fused SwiGLU epilogue (b200q_matmul_q8_swiglu): gate|up rows interleaved per tile at upload, the gate|up matvec writes the
        # down projection's activation records itself -- one launch and one kernel boundary less per layer.  ggml formats only
        # (the INT4 layouts pack 8 output rows per word), gate and up of one format, F % 64 == 0.
        self.swiglu_epi_wanted = ((not self.wide) and _os.environ.get("B200Q_SWIGLU_EPI", "1") != "0" and self.ff % 64 == 0
                                  and _os.environ.get("B200Q_FUSED_SWIGLU", "0") == "0")
        for i in range(cfg.n_layers):
            # formats come from the weights themselves when a host model (tests, GGUF files) is given
            fm = {p_: host.layers[i][p_].fmt for p_ in ("q", "k", "v", "o", "gate", "up", "down")} if host else layer_formats(cfg, scheme, i)
            lay = {}
            # column-parallel q | k | v (rows of this rank's heads), fused where formats agree
            lay["qkv"] = self._fused(i, [("q", fm["q"], cfg.n_heads * hd, pl.q_rows[0], self.qd),
                                         ("k", fm["k"], cfg.n_kv_heads * hd, pl.kv_rows[0], self.kvd),
                                         ("v", fm["v"], cfg.n_kv_heads * hd, pl.kv_rows[0], self.kvd)], H, host)
            # decode matvecs (M <= 4): a Q4_K q|k group followed by a Q6_K v (Q4_K_M files: about half of the layers) is ONE
            # dual-format launch (b200q_weight_set_pair) instead of two; the tcgen05 paths keep the separate launches
            lay["qkv_mv"] = lay["qkv"]
            qk = lay["qkv"]
            if (len(qk) == 2 and not self.wide and _os.environ.get("B200Q_DUAL", "1") != "0" and qk[0].w.N % 128 == 0
                    and (qk[0].fmt, qk[1].fmt) == ("Q4_K", "Q6_K")):
                qk[0].w.set_pair(qk[1].w)
                lay["qkv_mv"] = [qk[0]]
            # row-parallel o: K slice = this rank's heads
            lay["o"] = self._fused(i, [("o", fm["o"], H, 0, H)], cfg.n_heads * hd, host, kslice=pl.o_cols)
            lay["swiglu_epi"] = self.swiglu_epi_wanted and fm["gate"] == fm["up"] and fm["gate"] in synth.GGML
            lay["gu"] = self._fused(i, [("gate", fm["gate"], cfg.ffn, f0, self.ff), ("up", fm["up"], cfg.ffn, f0, self.ff)], H, host,
                                    interleave=lay["swiglu_epi"])
            lay["down"] = self._fused(i, [("down", fm["down"], H, 0, H)], cfg.ffn, host, kslice=(f0, f1))
            an = host.layers[i]["attn_norm"] if host else np.ones(H, np.float32)
            mn = host.layers[i]["mlp_norm"] if host else np.ones(H, np.float32)
            lay["attn_norm"] = torch.from_numpy(an).to(dev)
            lay["mlp_norm"] = torch.from_numpy(mn).to(dev)
            if paged:  # block pools [num_blocks][block_size][nkv][hd]
                nblk = M * (-(-max_ctx // block_size))
                lay["ck"] = torch.zeros((nblk, block_size, self.nkv, hd), dtype=kv_t, device=dev)
                lay["cv"] = torch.zeros((nblk, block_size, self.nkv, hd), dtype=kv_t, device=dev)
            else:
                lay["ck"] = torch.zeros((M, max_ctx, self.nkv, hd), dtype=kv_t, device=dev)
                lay["cv"] = torch.zeros((M, max_ctx, self.nkv, hd), dtype=kv_t, device=dev)
            self.layers.append(lay)
        self.kv_cache_bytes = sum(lay[c].numel() * lay[c].element_size() for lay in self.layers for c in ("ck", "cv"))
        self.final_norm = torch.from_numpy(host.final_norm if host else np.ones(H, np.float32)).to(dev)
        self.rope = torch.from_numpy(rope_table(max_ctx, hd, cfg.rope_theta, cfg.rope_freq_factors)).to(dev)
        # decode attention: the single-CTA kernel holds every score of a (head, sequence) in shared memory; past its limit the
        # split-context kernels run over one workspace shared by all layers (they run in sequence on one stream)
        self.attn_split = max_ctx > int(ops.lib().b200q_attn_decode_max_ctx())
        self.attn_ws = None
        if self.attn_split:
            nbytes = int(ops.lib().b200q_attn_split_workspace_bytes(self.nh, self.nkv, hd, max_ctx, M))
            if nbytes == 0:
                raise ValueError(f"split-context attention does not support head_dim {hd}")
            self.attn_ws = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        self.head = self._fused(-1, [("lm_head", host.lm_head.fmt if host else head_format(scheme), cfg.vocab, v0, v1 - v0)], H, host)
        if host is not None:
            self.embed = torch.from_numpy(host.embed).to(dev)
        else:
            g = torch.Generator(device=dev)
            g.manual_seed(seed + 7)
            self.embed = torch.randn((cfg.vocab, H), device=dev, generator=g).to(torch.float16)
        # activations / scratch (all addresses stable: the step is graph-capturable)
        f32 = dict(dtype=torch.float32, device=dev)
        self.h = torch.zeros((M, H), **f32)
        self.h2 = torch.zeros((M, H), **f32)  # residual stream ping-pong (the fused add+norm is not in-place)
        self.delta = torch.zeros((M, H), **f32)
        self.delta2 = torch.zeros((M, H), **f32)  # down_proj output (the fused o->norm reads delta while down writes)
        self.qkv = torch.zeros((M, self.qd + 2 * self.kvd), **f32)
        self.gu = torch.zeros((M, 2 * self.ff), **f32)
        if tp_world == 1:
            self.logits_local = torch.zeros((M, v1 - v0), **f32)
            self.logits = self.logits_local
        else:
            assert v1 > v0, "vocabulary too small for this TP degree"
            vs = tp.vocab_shard_rows(cfg.vocab, tp_world)   # same on every rank; columns beyond this rank's rows stay -inf
            self.logits_local = torch.full((M, vs), float("-inf"), **f32)
            self.logits = torch.zeros((tp_world, M, vs), **f32)
        self.ids = torch.zeros(M, dtype=torch.int64, device=dev)
        self.pos = torch.zeros(M, dtype=torch.int32, device=dev)
        self.paged, self.block_size = paged, block_size
        if paged:
            self.max_blocks = -(-max_ctx // block_size)
            self.max_ctx = self.max_blocks * block_size
            perm = np.random.Generator(np.random.PCG64(seed + 99)).permutation(M * self.max_blocks).astype(np.int32)
            self.block_table = torch.from_numpy(perm.reshape(M, self.max_blocks)).to(dev)
            self.slot_mapping = None   # int32 [M] device tensor when a scheduler provides the slots; else derived from block_table / pos
        if self.wide:
            self.xq_h, self.xq_attn, self.xq_ff = (torch.zeros((M, k), **f32) for k in (H, self.qd, self.ff))  # f32 activations
        else:
            act = lambda K: torch.zeros(int(ops.lib().b200q_act_bytes(C.c_int64(K), C.c_int64(M))), dtype=torch.uint8, device=dev)
            self.xq_h, self.xq_attn, self.xq_ff = act(H), act(self.qd), act(self.ff)
        # streaming-order hints: every decode matvec prefetches the head of the next projection's weights into L2 while its own
        # tail drains (qkv -> o -> gate|up -> down -> next layer ... -> lm_head -> layer 0 of the next token)
        if not self.wide and _os.environ.get("B200Q_CHAIN", "0") != "0":  # measured neutral on whole steps (round 2): opt-in
            order = [ln.w for lay in self.layers for key in ("qkv", "o", "gu", "down") for ln in lay[key]] + [ln.w for ln in self.head]
            for a, b in zip(order, order[1:] + order[:1]):
                if a is not b:
                    a.set_next(b)
        # add+norm+quant fused into the prologue of the matvec that consumes it (b200q_matmul_norm): measured +3..6 % tok/s on one
        # GPU.  Needs hidden = 512 * 2^j <= 8192; tensor parallel keeps the separate kernel (it is the exchange's consumer).
        ept = H // 512
        # Tensor parallel: the exchange's consumer is the cluster add+norm+quant kernel and plain matvecs follow.  B200Q_TP_FINISH=1
        # (opt-in) makes the element-wise b200q_allreduce_finish the consumer (delta = f32(sum over ranks)) followed by the same fused
        # norm-prologue / SwiGLU-epilogue matvecs as on one GPU.  Measured (round 2, 70B Q4_K_M): equal at TP2 (6.21 vs 6.17 ms/step),
        # SLOWER on the TP8 shard (3.81 vs 3.50 ms): the per-CTA norm prologue (3.6 us) costs more than the cluster kernel saves.
        self.tp_finish = tp_world > 1 and _os.environ.get("B200Q_TP_FINISH", "0") != "0" and _os.environ.get("B200Q_TP_NCCL", "0") == "0"
        self.fused = (_os.environ.get("B200Q_FUSED", "1") != "0" and not self.wide and (tp_world == 1 or self.tp_finish) and H % 512 == 0 and ept <= 16
                      and (ept & (ept - 1)) == 0)
        self.tp_finish = self.tp_finish and self.fused
        self.fused_swiglu = _os.environ.get("B200Q_FUSED_SWIGLU", "0") != "0" and not self.wide  # measured slower: 148x redundant SiLU
        self.graph = None
        self._host_pos = 0
        # tensor parallel: one-shot NVLink all-reduce of the f64 partial sums (csrc/comm.cu); B200Q_TP_NCCL=1 falls back
        # to torch.distributed (NCCL) all-reduce of f32 partials for comparison
        self.comm = None
        if tp_world > 1 and _os.environ.get("B200Q_TP_NCCL", "0") == "0":
            assert (self.tp_finish or not self.fused) and not self.fused_swiglu
            self.vs = tp.vocab_shard_rows(cfg.vocab, tp_world)
            if emulate_shard:
                self.comm = ops.PeerComm(0, 1, M * H, dev, None, gather_elems=M * self.vs)
            else:
                self.comm = ops.PeerComm(tp_rank, tp_world, M * H, dev, group, gather_elems=M * self.vs)

    # ---- weights ------------------------------------------------------------------------------------
    def _fused(self, layer: int, parts, K: int, host: Optional[HostModel], kslice=None, interleave: bool = False) -> List[_Linear]:
        """parts: (name, fmt, N_full, row0, nrows).  Consecutive parts of equal format share one handle.
        interleave: the two parts are gate and up of one format -> rows in the SwiGLU-epilogue order (ops.gate_up_row_order)."""
        out: List[_Linear] = []
        col = 0
        groups = []
        for p in parts:
            if groups and groups[-1][0][1] == p[1]:
                groups[-1].append(p)
            else:
                groups.append([p])
        for grp in groups:
            fmt = grp[0][1]
            nrows = sum(p[4] for p in grp)
            w = self._upload(layer, grp, fmt, K, host, kslice, interleave=interleave)
            self.weight_bytes += w.canonical_bytes
            out.append(_Linear(w, col, w.workspace(self.M), fmt))
            col += nrows
        return out

    def _upload(self, layer: int, grp, fmt: str, K: int, host: Optional[HostModel], kslice, interleave: bool = False) -> ops.QuantWeight:
        k0, k1 = kslice if kslice is not None else (0, K)
        nrows = sum(p[4] for p in grp)
        if fmt in synth.GGML:
            t = synth.GGML[fmt]
            if host is not None:
                rows = []
                for (name, _, _, r0, nr) in grp:
                    hl = host.lm_head if layer < 0 else host.layers[layer][name]
                    rows.append(hl.data[r0:r0 + nr])
                blocks = np.concatenate(rows, axis=0)
                if interleave:
                    assert len(grp) == 2 and grp[0][4] == grp[1][4]
                    blocks = blocks[ops.gate_up_row_order(grp[0][4])]
                blocks = np.ascontiguousarray(blocks)
            else:  # random blocks generated on the device: any row order is as random as any other
                seed = 0x5EED + 7919 * (layer + 2) + 131 * _NAME_ID[grp[0][0]] + self.rank
                if kslice is not None:
                    return self.c.weight_from_ggml(t, random_ggml_device(fmt, nrows, k1 - k0, seed, self.dev), nrows, k1 - k0)
                blocks = random_ggml_device(fmt, nrows, K, seed, self.dev)
            return self.c.weight_from_ggml(t, blocks, nrows, K, cols=(k0, k1) if kslice is not None else None)
        # AWQ / GPTQ
        if host is None:  # bench: random tensors generated on the device, one fused [nrows, k1 - k0] weight
            seed = 0x5EED + 7919 * (layer + 2) + 131 * _NAME_ID[grp[0][0]] + self.rank
            qw, sc, z = random_int4_device(fmt, nrows, k1 - k0, 128, seed, self.dev)
            dq = ops.DecomposedQuantTensor(qw, sc, z, None, ops.DecomposedQuantMethod(fmt.lower(), 128), (nrows, k1 - k0))
            return self.c.weight_from_decomposed(dq)
        # host models: fuse by concatenating along N
        if host is None:
            host_parts = [_host_linear(fmt, p[4], K, 0x5EED + 31 * (layer + 2) + j + 17 * self.rank) for j, p in enumerate(grp)]
            sl = [(hp, 0, hp.N) for hp in host_parts]
        else:
            sl = [((host.lm_head if layer < 0 else host.layers[layer][p[0]]), p[3], p[4]) for p in grp]
        if fmt == "AWQ":
            gs = sl[0][0].data[3]
            qw = np.concatenate([hp.data[0][:, r0 // 8:(r0 + nr) // 8] for hp, r0, nr in sl], axis=1)
            sc = np.concatenate([hp.data[1][:, r0:r0 + nr] for hp, r0, nr in sl], axis=1)
            zr = np.concatenate([hp.data[2][:, r0:r0 + nr] for hp, r0, nr in sl], axis=1)
            dq = ops.DecomposedQuantTensor(np.ascontiguousarray(qw), np.ascontiguousarray(sc), np.ascontiguousarray(zr), None,
                                           ops.DecomposedQuantMethod("awq", gs), (nrows, K))
            return self.c.weight_from_decomposed(dq, cols=(k0, k1) if kslice is not None else None)
        if fmt == "GPTQ":
            gs = sl[0][0].data[4]
            qw = np.concatenate([hp.data[0][:, r0:r0 + nr] for hp, r0, nr in sl], axis=1)
            sc = np.concatenate([hp.data[1][:, r0:r0 + nr] for hp, r0, nr in sl], axis=1)
            qz = np.concatenate([hp.data[2][:, r0 // 8:(r0 + nr) // 8] for hp, r0, nr in sl], axis=1)
            if kslice is not None:  # K shard: slice the source tensors (groups are contiguous: no act-order here)
                qw, sc, qz = qw[k0 // 8:k1 // 8], sc[k0 // gs:k1 // gs], qz[k0 // gs:k1 // gs]
            dq = ops.DecomposedQuantTensor(np.ascontiguousarray(qw), np.ascontiguousarray(sc), np.ascontiguousarray(qz), None,
                                           ops.DecomposedQuantMethod("gptq", gs), (nrows, k1 - k0))
            return self.c.weight_from_decomposed(dq)
        raise ValueError(fmt)

    # ---- one decode step ------------------------------------------------------------------------------
    def _matvec(self, lins: List[_Linear], xq: torch.Tensor, out: torch.Tensor):
        L = ops.lib()
        st = ops._stream_ptr(self.dev)
        dt = ops.F64 if out.dtype == torch.float64 else ops.F32
        if self.wide:
            for ln in lins:
                ops._check(L.b200q_matmul(ln.w.handle, C.c_void_p(xq.data_ptr()), C.c_int32(ops.F32), C.c_int64(self.M), C.c_int64(xq.stride(0)),
                                          C.c_void_p(out.data_ptr() + 4 * ln.col0), C.c_int32(ops.F32), C.c_int64(out.stride(0)),
                                          C.c_void_p(ln.ws.data_ptr()), C.c_size_t(ln.ws.numel()), st))
            return
        for ln in lins:
            ops._check(L.b200q_matmul_q8(ln.w.handle, C.c_void_p(xq.data_ptr()), C.c_int64(self.M),
                                         C.c_void_p(out.data_ptr() + out.element_size() * ln.col0), C.c_int32(dt), C.c_int64(out.stride(0)),
                                         C.c_void_p(ln.ws.data_ptr()), C.c_size_t(ln.ws.numel()), st))

    def _rowpar(self, lins: List[_Linear], xq: torch.Tensor, out: torch.Tensor) -> bool:
        """row-parallel projection (o_proj / down_proj).  Returns True when the result is left IN FLIGHT in the exchange
        buffers: the matvec pushed its exact f64 row sums to every rank (fused exchange, csrc/comm_dev.cuh) and the next
        add+norm kernel is the consumer that sums them in rank order (bit-identical to the 1-GPU output).  Otherwise `out`
        (f32) holds the projection (1 GPU) or its NCCL all-reduce (B200Q_TP_NCCL=1, comparison only)."""
        if self.comm is not None:
            assert len(lins) == 1
            self.comm.matmul_q8_rowpar(lins[0].w, xq, self.M, self.cfg.hidden, lins[0].ws)
            if self.tp_finish:   # element-wise consumer: out = f32(sum over ranks, rank order, f64); the fused-prologue matvec adds + norms it
                self.comm.allreduce_finish(out)
                return False
            return True
        self._matvec(lins, xq, out)
        if self.world > 1:
            torch.distributed.all_reduce(out, group=self.group)
        return False

    def _allreduce(self, t: torch.Tensor):
        if self.world > 1:
            torch.distributed.all_reduce(t, group=self.group)

    def _attention(self, lay, st):
        """RoPE + KV append + single-query attention + output quantise (contiguous or paged KV cache)"""
        L, cfg, M = ops.lib(), self.cfg, self.M
        P = lambda t: C.c_void_p(t.data_ptr())
        xq, ao = (None, P(self.xq_attn)) if self.wide else (P(self.xq_attn), None)
        kvt = C.c_int32(KV_DTYPES[self.kv_dtype][1])
        if self.attn_split:
            ws, wsb = P(self.attn_ws), C.c_size_t(self.attn_ws.numel())
            if self.paged:
                ops._check(L.b200q_attn_decode_paged_split_kv(P(self.qkv), P(self.pos), P(lay["ck"]), P(lay["cv"]), kvt, P(self.block_table),
                                                              P(self.slot_mapping) if self.slot_mapping is not None else None,
                                                              C.c_int32(self.block_size), C.c_int32(self.max_blocks), P(self.rope), C.c_int32(self.nh),
                                                              C.c_int32(self.nkv), C.c_int32(cfg.head_dim), C.c_int64(M), xq, ao, ws, wsb, st))
            else:
                ops._check(L.b200q_attn_decode_split_kv(P(self.qkv), P(self.pos), P(lay["ck"]), P(lay["cv"]), kvt, P(self.rope), C.c_int32(self.nh),
                                                        C.c_int32(self.nkv), C.c_int32(cfg.head_dim), C.c_int32(self.max_ctx), C.c_int64(M), xq, ao,
                                                        ws, wsb, st))
            return
        if self.paged:
            ops._check(L.b200q_attn_decode_paged_kv(P(self.qkv), P(self.pos), P(lay["ck"]), P(lay["cv"]), kvt, P(self.block_table),
                                                    P(self.slot_mapping) if self.slot_mapping is not None else None, C.c_int32(self.block_size),
                                                    C.c_int32(self.max_blocks), P(self.rope), C.c_int32(self.nh), C.c_int32(self.nkv),
                                                    C.c_int32(cfg.head_dim), C.c_int64(M), xq, ao, st))
        else:
            ops._check(L.b200q_attn_decode_kv(P(self.qkv), P(self.pos), P(lay["ck"]), P(lay["cv"]), kvt, P(self.rope), C.c_int32(self.nh),
                                              C.c_int32(self.nkv), C.c_int32(cfg.head_dim), C.c_int32(self.max_ctx), C.c_int64(M), xq, ao, st))

    def kv_rows(self, lay, seq: int, S: int):
        """(K, V) rows [S, nkv, hd] of positions 0..S-1 of sequence `seq`, whatever the cache layout, in the stored dtype"""
        if not self.paged:
            return lay["ck"][seq, :S], lay["cv"][seq, :S]
        j = torch.arange(S, device=self.dev)
        idx = self.block_table[seq, j // self.block_size].long() * self.block_size + j % self.block_size
        nkv, hd = self.nkv, self.cfg.head_dim
        return lay["ck"].view(-1, nkv, hd)[idx], lay["cv"].view(-1, nkv, hd)[idx]

    def _kv_write(self, lay, seq: int, k: torch.Tensor, v: torch.Tensor):
        """prefill: store K (rotated) / V rows [S, nkv, hd] of sequence `seq` (f32 values; an f16 cache stores kv_round of them)"""
        S = k.shape[0]
        if self.kv_dtype == "f16":
            k, v = kv_round(k), kv_round(v)
        if not self.paged:
            lay["ck"][seq, :S].copy_(k)
            lay["cv"][seq, :S].copy_(v)
            return
        j = torch.arange(S, device=self.dev)
        idx = self.block_table[seq, j // self.block_size].long() * self.block_size + j % self.block_size
        nkv, hd = self.nkv, self.cfg.head_dim
        lay["ck"].view(-1, nkv, hd)[idx] = k
        lay["cv"].view(-1, nkv, hd)[idx] = v

    def _advance(self):
        """host-side mirror of the device position counter: every step (eager or replayed) passes through here, so a
        sequence can never run past the KV cache / RoPE table (the kernel guards too: b200q_decode_error)"""
        if self._host_pos >= self.max_ctx:
            raise RuntimeError(f"decode step at position {self._host_pos} exceeds max_ctx={self.max_ctx}: the KV cache is full "
                               "(build the Decoder with a larger max_ctx)")
        self._host_pos += 1

    def replay(self):
        """one captured decode step (CUDA-graph replay), position-checked on the host"""
        self._advance()
        self.graph.replay()

    def check_device_errors(self):
        """raises if a kernel refused an out-of-range position since the last check (synchronises the device)"""
        flags = C.c_int32(0)
        ops._check(ops.lib().b200q_decode_error(C.byref(flags)))
        if flags.value:
            raise RuntimeError(f"decode kernels reported error flags 0x{flags.value:x} (bit 0: position outside [0, max_ctx))")

    def step(self):
        """ids (device) -> next ids (device); positions advance on the device: graph-replayable."""
        if not torch.cuda.is_current_stream_capturing():
            self._advance()
        L, cfg, M = ops.lib(), self.cfg, self.M
        st = ops._stream_ptr(self.dev)
        P = lambda t: C.c_void_p(t.data_ptr())
        ops._check(L.b200q_embed(P(self.embed), P(self.ids), C.c_int64(cfg.hidden), C.c_int64(M), P(self.h), st))
        hin, hout = self.h, self.h2
        delta = None
        in_flight = False  # TP: the projection ahead left its partial sums in the exchange buffers (see _rowpar)

        def norm(w):
            nonlocal hin, hout
            if in_flight:
                self.comm.allreduce_add_rmsnorm_quant(hin, hout, w, cfg.eps, cfg.hidden, M, xq=self.xq_h)
            else:
                ops._check(L.b200q_add_rmsnorm_quant(P(hin), P(delta) if delta is not None else None, P(hout), P(w), C.c_float(cfg.eps),
                                                     C.c_int64(cfg.hidden), C.c_int64(M), None if self.wide else P(self.xq_h),
                                                     P(self.xq_h) if self.wide else None, st))
            hin, hout = hout, hin

        def matvec_norm(lins, w, out):
            """norm fused into the matvec prologue (one launch per fused weight group; the first writes h_out)"""
            nonlocal hin, hout
            for j, ln in enumerate(lins):
                ops._check(L.b200q_matmul_norm(ln.w.handle, P(hin), P(delta) if delta is not None else None, P(hout) if j == 0 else None, P(w),
                                               C.c_float(cfg.eps), C.c_int64(M), C.c_void_p(out.data_ptr() + 4 * ln.col0), C.c_int32(ops.F32),
                                               C.c_int64(out.stride(0)), C.c_void_p(ln.ws.data_ptr()), C.c_size_t(ln.ws.numel()), st))
            hin, hout = hout, hin

        fused = self.fused
        for li, lay in enumerate(self.layers):
            if fused:
                matvec_norm(lay["qkv_mv"], lay["attn_norm"], self.qkv)
            else:
                norm(lay["attn_norm"])
                self._matvec(lay["qkv_mv"], self.xq_h, self.qkv)
            self._attention(lay, st)
            in_flight = self._rowpar(lay["o"], self.xq_attn, self.delta)
            delta = self.delta
            if lay["swiglu_epi"]:
                # gate|up with the fused SwiGLU epilogue: the matvec writes the down projection's records (xq_ff) itself
                ln = lay["gu"][0]
                if fused:
                    ops._check(L.b200q_matmul_norm_swiglu(ln.w.handle, P(hin), P(delta) if delta is not None else None, P(hout), P(lay["mlp_norm"]),
                                                          C.c_float(cfg.eps), C.c_int64(M), P(self.xq_ff), C.c_void_p(ln.ws.data_ptr()),
                                                          C.c_size_t(ln.ws.numel()), st))
                    hin, hout = hout, hin
                else:
                    norm(lay["mlp_norm"])
                    ops._check(L.b200q_matmul_q8_swiglu(ln.w.handle, P(self.xq_h), C.c_int64(M), P(self.xq_ff), C.c_void_p(ln.ws.data_ptr()),
                                                        C.c_size_t(ln.ws.numel()), st))
                in_flight = self._rowpar(lay["down"], self.xq_ff, self.delta2)
                delta = self.delta2
                continue
            if fused:
                matvec_norm(lay["gu"], lay["mlp_norm"], self.gu)
            else:
                norm(lay["mlp_norm"])
                self._matvec(lay["gu"], self.xq_h, self.gu)
            if self.fused_swiglu:
                for ln in lay["down"]:
                    ops._check(L.b200q_matmul_swiglu(ln.w.handle, P(self.gu), C.c_int64(M), C.c_void_p(self.delta2.data_ptr() + 4 * ln.col0),
                                                     C.c_int32(ops.F32), C.c_int64(self.delta2.stride(0)), C.c_void_p(ln.ws.data_ptr()),
                                                     C.c_size_t(ln.ws.numel()), st))
                self._allreduce(self.delta2)
                delta = self.delta2
            else:
                if self.wide:
                    ops._check(L.b200q_swiglu_f32(P(self.gu), C.c_int64(self.ff), C.c_int64(M), P(self.xq_ff), st))
                else:
                    ops._check(L.b200q_swiglu_quant(P(self.gu), C.c_int64(self.ff), C.c_int64(M), P(self.xq_ff), st))
                in_flight = self._rowpar(lay["down"], self.xq_ff, self.delta2)
                delta = self.delta2
        head_fused = fused and self.comm is None   # the vocabulary-parallel lm_head (gather form) takes ready-made records
        if head_fused:
            matvec_norm(self.head, self.final_norm, self.logits_local)
        else:
            norm(self.final_norm)
        if self.comm is not None:
            # vocabulary-parallel lm_head: logits go straight into every rank's gather area, the arg-max is the consumer
            assert len(self.head) == 1
            self.comm.matmul_q8_gather(self.head[0].w, self.xq_h, M, self.vs, self.head[0].ws)
            self.comm.argmax_gathered(self.vs, M, self.ids, self.pos)
            return
        if not head_fused:
            self._matvec(self.head, self.xq_h, self.logits_local)
        if self.world > 1:
            torch.distributed.all_gather_into_tensor(self.logits, self.logits_local, group=self.group)
            full = self.logits.permute(1, 0, 2).reshape(M, -1).contiguous()  # column r * vs + j = vocabulary id (padding = -inf)
            ops._check(L.b200q_argmax(P(full), C.c_int64(full.shape[1]), C.c_int64(M), P(self.ids), P(self.pos), st))
            self._full_logits = full[:, :cfg.vocab]
        else:
            ops._check(L.b200q_argmax(P(self.logits), C.c_int64(self.logits.shape[1]), C.c_int64(M), P(self.ids), P(self.pos), st))

    def full_logits(self) -> torch.Tensor:
        """[M, vocab] f32 logits of the last step on this rank (TP: assembled from the gather area / the all-gather)"""
        if self.comm is not None:
            g = self.comm.gathered()[:, :self.M * self.vs].reshape(self.world, self.M, self.vs)
            return g.permute(1, 0, 2).reshape(self.M, -1)[:, :self.cfg.vocab].contiguous()
        if self.world > 1:
            return self._full_logits
        return self.logits

    def launches_per_step(self) -> int:
        if getattr(self, "_launches", None):
            return self._launches  # counted by the library during the un-captured warm-up step
        glue = 0 if self.fused else 1
        sw = 0 if self.fused_swiglu else 1
        n = 1 + glue + len(self.head) + 1  # embed, (final norm), head, argmax
        for lay in self.layers:
            n += 2 * glue + len(lay["qkv"]) + (3 if self.attn_split else 1) + len(lay["o"]) + len(lay["gu"]) + sw + len(lay["down"])
        return n

    def capture(self):
        """capture one decode step into a CUDA graph (reference src/engine/cuda_graphs.rs:124-130)"""
        n0 = ops.launch_count()
        self.step()  # un-captured warm-up forward (cuda_graphs.rs:104)
        self._launches = ops.launch_count() - n0
        self.pos.sub_(1)      # the warm-up forward is not part of any sequence: undo its position advance
        self._host_pos -= 1
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream(self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):
            with torch.cuda.graph(g, stream=s):
                self.step()
        torch.cuda.synchronize(self.dev)
        self.graph = g
        return g

    # ---- prefill: one M = S pass over the prompt (reference src/engine/executor_generate.rs:357, batch_engine.rs:172-272) ----
    def prefill(self, prompt, seq: int = 0) -> torch.Tensor:
        """prompt: int64 [S] token ids of sequence `seq`.  Runs every projection ONCE at M = S on the tcgen05 dequant-GEMM
        (b200q_matmul, f32 activations -> f16 tiles, f32 accumulate), fills the KV cache rows [0, S) of that sequence, leaves
        pos[seq] = S and ids[seq] = the greedy next token, and returns the f32 logits [vocab] of the last position.  RoPE and
        the causal attention of the prompt run in torch (SDPA, f16) -- they are not the graded path (SURVEY 7.9); norms,
        SwiGLU and all 7L+1 projections are libb200q kernels.  Tolerance contract: 1e-2 relative on the logits against the f32
        CPU path (the GEMM path quantises weights and activations to f16 tiles)."""
        import torch.nn.functional as Fnn
        cfg, L = self.cfg, ops.lib()
        ids_h = np.asarray(prompt, dtype=np.int64).reshape(-1)
        S = int(ids_h.shape[0])
        if S < 1 or S > self.max_ctx:
            raise ValueError(f"prompt length {S} outside [1, max_ctx={self.max_ctx}]")
        assert 0 <= seq < self.M
        H, hd, nh, nkv, ff = cfg.hidden, cfg.head_dim, self.nh, self.nkv, self.ff
        dev = self.dev
        st = ops._stream_ptr(dev)
        P = lambda t: C.c_void_p(t.data_ptr())
        f32 = dict(dtype=torch.float32, device=dev)
        b = getattr(self, "_pf", None)
        if b is None or b["S"] != S:
            ws_bytes = max(ln.w.workspace_bytes(S) for lay in self.layers for key in ("qkv", "o", "gu", "down") for ln in lay[key])
            b = dict(S=S, h=torch.empty((S, H), **f32), h2=torch.empty((S, H), **f32), xn=torch.empty((S, H), **f32),
                     qkv=torch.empty((S, self.qd + 2 * self.kvd), **f32), attn=torch.empty((S, self.qd), **f32), delta=torch.empty((S, H), **f32),
                     delta2=torch.empty((S, H), **f32), gu=torch.empty((S, 2 * ff), **f32), act=torch.empty((S, ff), **f32),
                     ws=torch.zeros(max(256, ws_bytes), dtype=torch.uint8, device=dev))
            b["xq1"] = torch.zeros(int(L.b200q_act_bytes(C.c_int64(H), C.c_int64(1))), dtype=torch.uint8, device=dev)
            b["h1"] = torch.empty((1, H), **f32)
            b["logits1"] = torch.full((1, self.logits_local.shape[1]), float("-inf"), **f32)
            self._pf = b
        ids_d = torch.from_numpy(ids_h).to(dev)
        ops._check(L.b200q_embed(P(self.embed), P(ids_d), C.c_int64(H), C.c_int64(S), P(b["h"]), st))
        hin, hout = b["h"], b["h2"]
        delta = None
        rope = self.rope[:S]                                   # [S, hd/2, 2]
        cos, sin = rope[:, None, :, 0], rope[:, None, :, 1]    # [S, 1, hd/2]

        def gemm(lins, x, out):
            for ln in lins:
                ops._check(L.b200q_matmul(ln.w.handle, P(x), C.c_int32(ops.F32), C.c_int64(S), C.c_int64(x.stride(0)),
                                          C.c_void_p(out.data_ptr() + 4 * ln.col0), C.c_int32(ops.F32), C.c_int64(out.stride(0)), P(b["ws"]),
                                          C.c_size_t(b["ws"].numel()), st))

        def norm(w):
            nonlocal hin, hout
            ops._check(L.b200q_add_rmsnorm_quant(P(hin), P(delta) if delta is not None else None, P(hout), P(w), C.c_float(cfg.eps), C.c_int64(H),
                                                 C.c_int64(S), None, P(b["xn"]), st))
            hin, hout = hout, hin

        def rot(x):  # adjacent-pair RoPE, same table as the decode kernel
            x2 = x.reshape(S, -1, hd // 2, 2)
            x0, x1 = x2[..., 0], x2[..., 1]
            return torch.stack((x0 * cos - x1 * sin, x0 * sin + x1 * cos), dim=-1).reshape(S, -1, hd)

        for lay in self.layers:
            norm(lay["attn_norm"])
            gemm(lay["qkv"], b["xn"], b["qkv"])
            q = rot(b["qkv"][:, :self.qd])
            k = rot(b["qkv"][:, self.qd:self.qd + self.kvd])
            v = b["qkv"][:, self.qd + self.kvd:].reshape(S, nkv, hd)
            self._kv_write(lay, seq, k, v)
            o = Fnn.scaled_dot_product_attention(q.permute(1, 0, 2)[None].half(), k.permute(1, 0, 2)[None].half(), v.permute(1, 0, 2)[None].half(),
                                                 is_causal=True, enable_gqa=(nh != nkv))
            b["attn"].copy_(o[0].permute(1, 0, 2).reshape(S, self.qd))
            gemm(lay["o"], b["attn"], b["delta"])
            if self.world > 1:
                torch.distributed.all_reduce(b["delta"], group=self.group)   # prefill-size message: NCCL over NVLink
            delta = b["delta"]
            norm(lay["mlp_norm"])
            gemm(lay["gu"], b["xn"], b["gu"])
            sw = L.b200q_swiglu_f32_interleaved if lay["swiglu_epi"] else L.b200q_swiglu_f32
            ops._check(sw(P(b["gu"]), C.c_int64(ff), C.c_int64(S), P(b["act"]), st))
            gemm(lay["down"], b["act"], b["delta2"])
            if self.world > 1:
                torch.distributed.all_reduce(b["delta2"], group=self.group)
            delta = b["delta2"]
        # last position only: final norm + quantise -> lm_head on the decode matvec (M = 1) -> greedy token
        last_h, last_d = hin[S - 1:S], delta[S - 1:S]
        ops._check(L.b200q_add_rmsnorm_quant(P(last_h), P(last_d), P(b["h1"]), P(self.final_norm), C.c_float(cfg.eps), C.c_int64(H), C.c_int64(1),
                                             P(b["xq1"]), None, st))
        for ln in self.head:
            ops._check(L.b200q_matmul_q8(ln.w.handle, P(b["xq1"]), C.c_int64(1), C.c_void_p(b["logits1"].data_ptr() + 4 * ln.col0), C.c_int32(ops.F32),
                                         C.c_int64(b["logits1"].stride(0)), P(ln.ws), C.c_size_t(ln.ws.numel()), st))
        logits = b["logits1"][0]
        if self.world > 1:
            parts = [torch.empty_like(b["logits1"]) for _ in range(self.world)]
            torch.distributed.all_gather(parts, b["logits1"], group=self.group)
            logits = torch.cat([p_[0] for p_ in parts])
        logits = logits[:cfg.vocab]
        self.ids[seq] = torch.argmax(logits)
        self.pos[seq] = S
        self._host_pos = max(self._host_pos, S)
        return logits

    def reset(self, first_ids):
        self.ids.copy_(torch.as_tensor(first_ids, dtype=torch.int64, device=self.dev).reshape(self.M))
        self.pos.zero_()
        self._host_pos = 0

    def generate(self, prompt: np.ndarray, n_new: int, use_graph: bool = True) -> np.ndarray:
        """prompt: int64 [M, S].  Greedy: feeds the prompt token by token (decode steps), then n_new tokens."""
        prompt = np.asarray(prompt, dtype=np.int64).reshape(self.M, -1)
        S = prompt.shape[1]
        if S + n_new - 1 > self.max_ctx:
            raise ValueError(f"prompt ({S}) + new tokens ({n_new}) - 1 = {S + n_new - 1} positions exceed max_ctx={self.max_ctx}")
        if use_graph and self.graph is None:
            self.capture()
        self.reset(prompt[:, 0])
        run = self.replay if use_graph else self.step
        out = []
        for s_ in range(S + n_new - 1):
            run()
            if s_ + 1 < S:
                self.ids.copy_(torch.from_numpy(prompt[:, s_ + 1]).to(self.dev))  # teacher-force the prompt
            else:
                out.append(self.ids.clone())
        torch.cuda.synchronize(self.dev)
        self.check_device_errors()
        return torch.stack(out, dim=1).cpu().numpy()
