"""GGUF file parsing + direct upload of the raw quantized blocks (SURVEY.md section 8f rank 1).

Mirrors the reference loader surface (src/loader/gguf.rs):
    Gguf.open(path)                       boostr::format::Gguf::open            (gguf.rs:29)
    config_from_gguf_metadata(gguf)       gguf.rs:101-306  (same keys, same defaults)
    get_gguf_info(path)                   gguf.rs:309-338, detect_quantization_type :362-385
    load_gguf(client, path)               gguf.rs:20-44: VarMap::from_gguf (tensor names mapped GGUF -> HF, raw blocks
                                          uploaded as stored) -> LoadedModel::load

The parser is self-contained (GGUF v2/v3 little-endian, public spec); tensors are numpy views into one mmap, so
the upload path hands the file's bytes straight to b200q_weight_from_ggml (which repacks on the device).  Tensors
that are not matmul operands but stored quantized (token_embd, rarely norms) go through DequantOps
(B200Client.dequantize), as the reference does (gguf.rs:25 `R::Client: DequantOps<R>`).
"""
from __future__ import annotations

import mmap
import os
import struct
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import numpy as np

GGUF_MAGIC = 0x46554747
# ggml type id -> (name, block elems, block bytes)   (public ggml spec; SURVEY.md Appendix A)
GGML_TYPE_INFO = {
    0: ("F32", 1, 4), 1: ("F16", 1, 2), 2: ("Q4_0", 32, 18), 3: ("Q4_1", 32, 20), 6: ("Q5_0", 32, 22), 7: ("Q5_1", 32, 24),
    8: ("Q8_0", 32, 34), 9: ("Q8_1", 32, 36), 10: ("Q2_K", 256, 84), 11: ("Q3_K", 256, 110), 12: ("Q4_K", 256, 144),
    13: ("Q5_K", 256, 176), 14: ("Q6_K", 256, 210), 15: ("Q8_K", 256, 292), 16: ("IQ2_XXS", 256, 66), 17: ("IQ2_XS", 256, 74),
    18: ("IQ3_XXS", 256, 98), 19: ("IQ1_S", 256, 50), 20: ("IQ4_NL", 32, 18), 21: ("IQ3_S", 256, 110), 22: ("IQ2_S", 256, 82),
    23: ("IQ4_XS", 256, 136), 24: ("I8", 1, 1), 25: ("I16", 1, 2), 26: ("I32", 1, 4), 27: ("I64", 1, 8), 28: ("F64", 1, 8),
    29: ("IQ1_M", 256, 56), 30: ("BF16", 1, 2), 34: ("TQ1_0", 256, 54), 35: ("TQ2_0", 256, 66),
}
_SCALAR = {0: "<B", 1: "<b", 2: "<H", 3: "<h", 4: "<I", 5: "<i", 6: "<f", 7: "<?", 10: "<Q", 11: "<q", 12: "<d"}


class GgufError(ValueError):
    pass


@dataclass
class TensorInfo:
    name: str
    shape: Tuple[int, ...]   # ggml order: ne0 (contiguous, = K for a weight) first
    ggml_type: int
    offset: int              # absolute file offset
    nbytes: int

    @property
    def type_name(self) -> str:
        return GGML_TYPE_INFO[self.ggml_type][0]


class Metadata(dict):
    def architecture(self) -> Optional[str]:
        return self.get("general.architecture")

    def get_u32(self, key) -> Optional[int]:
        v = self.get(key)
        return int(v) if isinstance(v, (int, np.integer)) and not isinstance(v, bool) else None

    def get_f32(self, key) -> Optional[float]:
        v = self.get(key)
        return float(v) if isinstance(v, (float, np.floating)) else None

    def get_array(self, key) -> Optional[list]:
        v = self.get(key)
        return v if isinstance(v, list) else None


class Gguf:
    """Parsed GGUF file: metadata + tensor directory over a read-only mmap."""

    def __init__(self, path: str):
        self.path = path
        self._f = open(path, "rb")
        size = os.fstat(self._f.fileno()).st_size
        if size < 24:
            raise GgufError("file too small to be GGUF")
        self._mm = mmap.mmap(self._f.fileno(), 0, access=mmap.ACCESS_READ)
        self.file_size = size
        self._pos = 0
        magic, self.version = self._unpack("<II")
        if magic != GGUF_MAGIC:
            raise GgufError(f"bad magic 0x{magic:08x} (not a GGUF file)")
        if self.version not in (2, 3):
            raise GgufError(f"unsupported GGUF version {self.version}")
        n_tensors, n_kv = self._unpack("<QQ")
        self._meta = Metadata()
        for _ in range(n_kv):
            key = self._string()
            (vt,) = self._unpack("<I")
            self._meta[key] = self._value(vt)
        self.alignment = int(self._meta.get("general.alignment", 32))
        infos = []
        for _ in range(n_tensors):
            name = self._string()
            (nd,) = self._unpack("<I")
            dims = self._unpack("<" + "Q" * nd)
            t, off = self._unpack("<IQ")
            if t not in GGML_TYPE_INFO:
                raise GgufError(f"tensor {name}: unknown ggml type {t}")
            _, be, bb = GGML_TYPE_INFO[t]
            n = int(np.prod(dims)) if nd else 1
            if dims and dims[0] % be:
                raise GgufError(f"tensor {name}: ne0={dims[0]} is not a multiple of the {GGML_TYPE_INFO[t][0]} block ({be})")
            infos.append((name, tuple(int(d) for d in dims), t, off, n // be * bb))
        data_start = (self._pos + self.alignment - 1) // self.alignment * self.alignment
        self._tensors: Dict[str, TensorInfo] = {}
        for name, dims, t, off, nb in infos:
            if data_start + off + nb > size:
                raise GgufError(f"tensor {name}: data [{data_start + off}, +{nb}) runs past the end of the file")
            self._tensors[name] = TensorInfo(name, dims, t, data_start + off, nb)

    # ---- low-level readers ----
    def _unpack(self, fmt):
        n = struct.calcsize(fmt)
        if self._pos + n > self.file_size:
            raise GgufError("truncated GGUF header")
        v = struct.unpack_from(fmt, self._mm, self._pos)
        self._pos += n
        return v

    def _string(self) -> str:
        (n,) = self._unpack("<Q")
        if self._pos + n > self.file_size:
            raise GgufError("truncated GGUF string")
        s = self._mm[self._pos:self._pos + n].decode("utf-8", errors="replace")
        self._pos += n
        return s

    def _value(self, vt):
        if vt in _SCALAR:
            return self._unpack(_SCALAR[vt])[0]
        if vt == 8:
            return self._string()
        if vt == 9:
            et, cnt = self._unpack("<IQ")
            if et in _SCALAR and et != 7:
                fmt = _SCALAR[et]
                n = struct.calcsize(fmt) * cnt
                arr = np.frombuffer(self._mm, dtype=np.dtype(fmt), count=cnt, offset=self._pos).tolist()
                self._pos += n
                return arr
            return [self._value(et) for _ in range(cnt)]
        raise GgufError(f"unknown metadata value type {vt}")

    # ---- public surface ----
    @classmethod
    def open(cls, path: str) -> "Gguf":
        return cls(path)

    def metadata(self) -> Metadata:
        return self._meta

    def tensor_names(self) -> List[str]:
        return list(self._tensors)

    def tensor_info(self, name: str) -> TensorInfo:
        if name not in self._tensors:
            raise GgufError(f"no tensor named {name}")
        return self._tensors[name]

    def tensor_bytes(self, name: str) -> np.ndarray:
        """raw bytes of the tensor as a zero-copy uint8 view of the mmap"""
        ti = self.tensor_info(name)
        return np.frombuffer(self._mm, dtype=np.uint8, count=ti.nbytes, offset=ti.offset)

    def tensor_rows(self, name: str) -> np.ndarray:
        """[rows, row_bytes] uint8 view (rows = product of the outer dims, row = ne0 elements)"""
        ti = self.tensor_info(name)
        _, be, bb = GGML_TYPE_INFO[ti.ggml_type]
        row_bytes = ti.shape[0] // be * bb
        return self.tensor_bytes(name).reshape(-1, row_bytes)

    def close(self):
        self._mm.close()
        self._f.close()


# GGUF -> HF tensor names (reference gguf.rs:32 "names auto-mapped from GGUF to HF convention")
_LAYER_MAP = {
    "attn_q": "self_attn.q_proj", "attn_k": "self_attn.k_proj", "attn_v": "self_attn.v_proj", "attn_output": "self_attn.o_proj",
    "ffn_gate": "mlp.gate_proj", "ffn_up": "mlp.up_proj", "ffn_down": "mlp.down_proj",
    "attn_norm": "input_layernorm", "ffn_norm": "post_attention_layernorm",
    "ffn_gate_inp": "mlp.gate", "ffn_gate_exps": "mlp.experts.gate_proj", "ffn_up_exps": "mlp.experts.up_proj",
    "ffn_down_exps": "mlp.experts.down_proj",
}


def hf_name(gguf_name: str) -> str:
    if gguf_name == "token_embd.weight":
        return "model.embed_tokens.weight"
    if gguf_name == "output_norm.weight":
        return "model.norm.weight"
    if gguf_name == "output.weight":
        return "lm_head.weight"
    parts = gguf_name.split(".")
    if len(parts) == 4 and parts[0] == "blk" and parts[2] in _LAYER_MAP:
        return f"model.layers.{parts[1]}.{_LAYER_MAP[parts[2]]}.{parts[3]}"
    return gguf_name


@dataclass
class GgufInfo:
    """reference gguf.rs:341-358"""
    architecture: str
    vocab_size: Optional[int]
    hidden_size: Optional[int]
    num_layers: Optional[int]
    num_heads: Optional[int]
    num_kv_heads: Optional[int]
    context_length: Optional[int]
    quantization_type: str
    file_size_bytes: Optional[int]
    is_moe: bool


def detect_quantization_type(g: Gguf) -> str:
    """most frequent tensor type (reference gguf.rs:362-385)"""
    counts: Dict[str, int] = {}
    for n in g.tensor_names():
        t = g.tensor_info(n).type_name
        counts[t] = counts.get(t, 0) + 1
    return max(counts.items(), key=lambda kv: kv[1])[0] if counts else "unknown"


def get_gguf_info(path: str) -> GgufInfo:
    g = Gguf.open(path)
    m = g.metadata()
    arch = m.architecture() or "llama"
    vocab = m.get_u32("general.vocab_size") or m.get_u32(f"{arch}.vocab_size")  # llama.cpp writes the arch-scoped key
    if vocab is None and m.get_array("tokenizer.ggml.tokens") is not None:
        vocab = len(m.get_array("tokenizer.ggml.tokens"))
    info = GgufInfo(arch, vocab, m.get_u32(f"{arch}.embedding_length"), m.get_u32(f"{arch}.block_count"),
                    m.get_u32(f"{arch}.attention.head_count"), m.get_u32(f"{arch}.attention.head_count_kv"),
                    m.get_u32(f"{arch}.context_length"), detect_quantization_type(g), g.file_size,
                    (m.get_u32(f"{arch}.expert_count") or 0) > 0)
    g.close()
    return info


def config_from_gguf_metadata(g: Gguf):
    """ModelConfig from the file's metadata: same keys and defaults as reference gguf.rs:101-200
    (heads 32, kv heads = heads, eps 1e-5, rope base 10000, head_dim = key_length or hidden / heads; a missing
    embedding_length or block_count is an error, gguf.rs:120-130)."""
    from .decode import ModelConfig

    m = g.metadata()
    arch = m.architecture() or "llama"
    vocab = m.get_u32("general.vocab_size") or m.get_u32(f"{arch}.vocab_size")
    if vocab is None:
        toks = m.get_array("tokenizer.ggml.tokens")
        if toks is not None:
            vocab = len(toks)
        elif "token_embd.weight" in g.tensor_names():
            vocab = g.tensor_info("token_embd.weight").shape[1]
        else:
            raise GgufError("cannot determine the vocabulary size")
    hidden = m.get_u32(f"{arch}.embedding_length")
    if hidden is None:
        raise GgufError(f"GGUF missing {arch}.embedding_length")  # reference gguf.rs:122 (an error there too, no default)
    layers = m.get_u32(f"{arch}.block_count")
    if layers is None:
        raise GgufError(f"missing {arch}.block_count")
    heads = m.get_u32(f"{arch}.attention.head_count") or 32
    kv = m.get_u32(f"{arch}.attention.head_count_kv") or heads
    hd = m.get_u32(f"{arch}.attention.key_length") or hidden // heads
    ffn = m.get_u32(f"{arch}.feed_forward_length") or 4 * hidden
    eps = m.get_f32(f"{arch}.attention.layer_norm_rms_epsilon") or 1e-5
    theta = m.get_f32(f"{arch}.rope.freq_base") or 10000.0
    return ModelConfig(m.get("general.name", arch), hidden, layers, heads, kv, hd, ffn, vocab, theta, eps)


SUPPORTED_DECODER_ARCHS = frozenset({"llama", "mistral"})


def rope_freq_factors(g: Gguf, head_dim: int) -> Tuple[float, ...]:
    """the per-frequency RoPE divisors llama.cpp's converter writes as rope_freqs.weight for models trained with
    rope_scaling.rope_type "llama3" (Llama 3.1 / 3.2): F32, shape (head_dim / 2,), finite and positive -- anything else raises"""
    ti = g.tensor_info("rope_freqs.weight")
    if ti.ggml_type != 0:
        raise GgufError(f"rope_freqs.weight: expected F32, got {ti.type_name}")
    if ti.shape != (head_dim // 2,):
        raise GgufError(f"rope_freqs.weight: shape {ti.shape} != ({head_dim // 2},) (head_dim / 2)")
    f = g.tensor_bytes("rope_freqs.weight").view(np.float32)
    if not (np.all(np.isfinite(f)) and np.all(f > 0)):
        raise GgufError("rope_freqs.weight: factors must be finite and positive")
    return tuple(float(x) for x in f)


def _to_f32(g: Gguf, name: str) -> np.ndarray:
    ti = g.tensor_info(name)
    raw = g.tensor_bytes(name)
    if ti.ggml_type == 0:
        return raw.view(np.float32).copy()
    if ti.ggml_type == 1:
        return raw.view(np.float16).astype(np.float32)
    if ti.ggml_type == 30:
        return (raw.view(np.uint16).astype(np.uint32) << 16).view(np.float32)
    raise GgufError(f"{name}: expected a float tensor, got {ti.type_name}")


def host_model_from_gguf(g: Gguf, client=None):
    """HostModel (the structure Decoder and the oracle consume) whose projections are zero-copy views of the file.
    Supported: dense Llama-family decoders -- general.architecture "llama" or "mistral" (llama.cpp stores their Q / K
    rows permuted for the adjacent-pair RoPE the attention operator applies) -- with any ggml weight type the library
    has a kernel for.  Anything else raises (no silent fallback): other architectures (qwen2 / phi3 / gemma use the
    NEOX rotate-half RoPE and projection biases), and files holding tensors this decoder would silently ignore
    (*.bias, stacked *_exps expert tensors -- the latter go through moe_mlp_from_gguf).  The one optional tensor is the
    Llama 3.1 / 3.2 rope_freqs.weight (architecture "llama" only; rope_freq_factors below).
    A quantized token_embd is dequantized on the GPU through `client`."""
    from . import synth
    from .decode import HostLinear, HostModel

    arch = g.metadata().architecture() or "llama"
    if arch not in SUPPORTED_DECODER_ARCHS:
        raise GgufError(f"general.architecture '{arch}' is not supported by the decode harness (supported: {sorted(SUPPORTED_DECODER_ARCHS)}): "
                        "its RoPE layout / biases differ from the Llama family")
    cfg = config_from_gguf_metadata(g)
    names = set(g.tensor_names())
    consumed = {"token_embd.weight", "output_norm.weight", "output.weight"}
    if arch == "llama" and "rope_freqs.weight" in names:
        cfg.rope_freq_factors = rope_freq_factors(g, cfg.head_dim)
        consumed.add("rope_freqs.weight")
    for i in range(cfg.n_layers):
        consumed |= {f"blk.{i}.{n}.weight" for n in ("attn_q", "attn_k", "attn_v", "attn_output", "ffn_gate", "ffn_up", "ffn_down", "attn_norm", "ffn_norm")}
    extra = sorted(names - consumed)
    if extra:
        raise GgufError(f"the file holds {len(extra)} tensor(s) the dense Llama-family decoder does not consume (e.g. {extra[:4]}): "
                        "refusing to load and silently drop them")
    by_type = {v: k for k, v in synth.GGML.items()}

    def linear(name: str, N: int, K: int) -> HostLinear:
        ti = g.tensor_info(name)
        if ti.ggml_type not in by_type:
            raise GgufError(f"{name}: ggml type {ti.type_name} has no B200 kernel yet (supported: {sorted(synth.GGML)})")
        if ti.shape != (K, N):
            raise GgufError(f"{name}: shape {ti.shape} != expected (K={K}, N={N})")
        return HostLinear(by_type[ti.ggml_type], N, K, g.tensor_rows(name))

    H, hd = cfg.hidden, cfg.head_dim
    qd, kvd = cfg.n_heads * hd, cfg.n_kv_heads * hd
    emb_t = g.tensor_info("token_embd.weight")
    if emb_t.ggml_type in (0, 1, 30):
        embed = _to_f32(g, "token_embd.weight").reshape(cfg.vocab, H).astype(np.float16)
    else:
        if client is None:
            raise GgufError("token_embd is quantized: pass a B200Client (DequantOps) to expand it")
        import torch
        if emb_t.ggml_type not in by_type:
            raise GgufError(f"token_embd: ggml type {emb_t.type_name} has no B200 dequantizer yet")
        w = client.weight_from_ggml(emb_t.ggml_type, g.tensor_rows("token_embd.weight"), cfg.vocab, H)
        embed = client.dequantize(w, dtype=torch.float16).cpu().numpy()
        w.free()
    hm = HostModel(cfg, detect_quantization_type(g), embed=embed)
    for i in range(cfg.n_layers):
        p = f"blk.{i}."
        hm.layers.append(dict(
            q=linear(p + "attn_q.weight", qd, H), k=linear(p + "attn_k.weight", kvd, H), v=linear(p + "attn_v.weight", kvd, H),
            o=linear(p + "attn_output.weight", H, qd), gate=linear(p + "ffn_gate.weight", cfg.ffn, H),
            up=linear(p + "ffn_up.weight", cfg.ffn, H), down=linear(p + "ffn_down.weight", H, cfg.ffn),
            attn_norm=_to_f32(g, p + "attn_norm.weight"), mlp_norm=_to_f32(g, p + "ffn_norm.weight")))
    hm.final_norm = _to_f32(g, "output_norm.weight")
    head = "output.weight" if "output.weight" in names else "token_embd.weight"  # tied embeddings (Llama-3.2-1B)
    hm.lm_head = linear(head, cfg.vocab, H)
    return hm


def load_gguf(client, path: str, batch: int = 1, max_ctx: int = 512, tp_rank: int = 0, tp_world: int = 1, group=None, kv_dtype: str = "f32"):
    """reference gguf.rs:20-44: open, derive the config from the metadata, upload every tensor, build the model.
    Returns (Decoder, ModelConfig); kv_dtype "f16" halves the KV cache (Decoder).  Each TP rank uploads only its shard of the mmapped blocks (the reference makes
    every rank read the whole file, regular.rs:152)."""
    from .decode import Decoder

    g = Gguf.open(path)
    hm = host_model_from_gguf(g, client)
    dec = Decoder(client, hm.cfg, hm.scheme, batch=batch, max_ctx=max_ctx, host=hm, tp_rank=tp_rank, tp_world=tp_world, group=group,
                  kv_dtype=kv_dtype)
    return dec, hm.cfg


# ------------------------------------------------------------------------------------------------
# MoE expert tensors (reference executor_cache.rs:218-228: experts are stored STACKED [num_experts, ...] and sliced per
# expert).  GGUF stores them as 3-D tensors blk.N.ffn_{gate,up,down}_exps.weight with ne = (K, N, E): E consecutive
# [N, K] matrices of packed blocks.
# ------------------------------------------------------------------------------------------------
def expert_rows(g: Gguf, name: str) -> List[np.ndarray]:
    """per-expert [N, row_bytes] uint8 views of a stacked expert tensor (zero-copy)"""
    ti = g.tensor_info(name)
    if len(ti.shape) != 3:
        raise GgufError(f"{name}: expected a 3-D stacked expert tensor, got shape {ti.shape}")
    K, N, E = ti.shape
    rows = g.tensor_rows(name)            # [E * N, row_bytes]
    if rows.shape[0] != E * N:
        raise GgufError(f"{name}: {rows.shape[0]} rows for {E} experts of {N} rows")
    return [rows[e * N:(e + 1) * N] for e in range(E)]


def host_experts_from_gguf(g: Gguf, layer: int):
    """[(gate_up_blocks [2 ffn, row_bytes], gate_up_type, down_blocks [hidden, row_bytes], down_type)] per expert: gate and up are
    fused row-wise (gate rows first), which is what the decode path launches once (ops.ExpertWeights.gate_up)"""
    p = f"blk.{layer}."
    tg, tu, td = (g.tensor_info(p + n + ".weight") for n in ("ffn_gate_exps", "ffn_up_exps", "ffn_down_exps"))
    if tg.ggml_type != tu.ggml_type or tg.shape != tu.shape:
        raise GgufError(f"layer {layer}: gate and up expert tensors differ in type or shape (cannot fuse)")
    gate, up, down = (expert_rows(g, p + n + ".weight") for n in ("ffn_gate_exps", "ffn_up_exps", "ffn_down_exps"))
    if not (len(gate) == len(up) == len(down)):
        raise GgufError(f"layer {layer}: expert counts differ")
    return [(np.concatenate([gate[e], up[e]], axis=0), tg.ggml_type, down[e], td.ggml_type) for e in range(len(gate))]


def moe_mlp_from_gguf(client, g: Gguf, layer: int):
    """ops.MoeMlp for one MoE layer of a GGUF file (hidden = K of gate, ffn = N of gate)"""
    from . import ops

    p = f"blk.{layer}."
    hidden, ffn, _ = g.tensor_info(p + "ffn_gate_exps.weight").shape
    experts = []
    il = ffn % 64 == 0   # gate|up rows in the SwiGLU-epilogue order: the grouped gate|up launch activates and quantises too
    order = ops.gate_up_row_order(ffn) if il else None
    for gu_blocks, gt, dn_blocks, dt in host_experts_from_gguf(g, layer):
        gu = client.weight_from_ggml(gt, np.ascontiguousarray(gu_blocks[order] if il else gu_blocks), 2 * ffn, hidden)
        dn = client.weight_from_ggml(dt, np.ascontiguousarray(dn_blocks), hidden, ffn)
        experts.append(ops.ExpertWeights(gu, dn, interleaved=il))
    return ops.MoeMlp(client, experts, ffn, hidden)
