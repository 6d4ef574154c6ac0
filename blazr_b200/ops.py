"""Python harness over the C ABI of libb200q.so (include/b200q.h).

PyTorch is used only for device memory, streams and torch.distributed; every compute call goes through
ctypes into the shared library -- the same entry points a Rust host would bind over FFI
(INTEGRATION.md).  The interface mirrors the reference operator boundary
(``boostr::quant::QuantMatmulOps`` / ``DequantOps`` bounds at reference src/loader/api.rs:25 and
``DecomposedQuantTensor::new`` at src/loader/safetensors/awq.rs:218, gptq.rs:252):

    client = B200Client(device)
    w  = client.weight_from_ggml(ggml_type, raw_blocks, N, K)            # VarMap::from_gguf upload
    w  = client.weight_from_decomposed(DecomposedQuantTensor(...))       # AWQ / GPTQ upload
    y  = client.quant_matmul(x, w)                                       # QuantMatmulOps
    wd = client.dequantize(w)                                            # DequantOps

There is no CPU fallback: if the library is missing, fails to load, or no sm_100 GPU is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200Q_LIB") or os.path.join(_HERE, "lib", "libb200q.so")   # B200Q_LIB: e.g. the TRACE build (csrc/Makefile)

F32, F16, BF16, F64 = 0, 1, 2, 3
_TORCH2DT = {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16, torch.float64: F64}
PATH_AUTO, PATH_MATVEC, PATH_GEMM = 0, 1, 2


class B200QError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"b200q error {code}: {msg}")
        self.code = code


class WeightInfo(C.Structure):
    _fields_ = [
        ("N", C.c_int64), ("K", C.c_int64), ("N_pad", C.c_int64), ("K_pad", C.c_int64),
        ("family", C.c_int32), ("source", C.c_int32), ("ggml_type", C.c_int32), ("group_size", C.c_int32),
        ("sub", C.c_int32), ("has_bias", C.c_int32), ("has_perm", C.c_int32), ("device", C.c_int32),
        ("device_bytes", C.c_int64), ("canonical_bytes", C.c_int64), ("chunk_bytes", C.c_int32),
    ]


# every symbol include/b200q.h declares (tests check the library exports each one)
EXPORTS = [
    "b200q_version", "b200q_last_error", "b200q_device_count", "b200q_weight_from_ggml", "b200q_weight_from_ggml_shard",
    "b200q_weight_from_awq", "b200q_weight_from_gptq", "b200q_weight_from_awq_shard", "b200q_weight_from_gptq_shard", "b200q_weight_free", "b200q_weight_info",
    "b200q_weight_set_bias", "b200q_weight_set_next", "b200q_weight_set_pair", "b200q_shard_range", "b200q_shard_range_blocks", "b200q_workspace_bytes", "b200q_matmul",
    "b200q_act_bytes", "b200q_quantize_act", "b200q_matmul_q8", "b200q_matmul_path", "b200q_dequantize", "b200q_act_unpack",
    "b200q_int_partials", "b200q_launch_count", "b200q_add_rmsnorm_quant", "b200q_swiglu_quant", "b200q_attn_decode", "b200q_attn_decode_paged",
    "b200q_attn_decode_max_ctx", "b200q_attn_split_workspace_bytes", "b200q_attn_decode_split", "b200q_attn_decode_paged_split",
    "b200q_attn_decode_kv", "b200q_attn_decode_paged_kv", "b200q_attn_decode_split_kv", "b200q_attn_decode_paged_split_kv",
    "b200q_argmax", "b200q_decode_error", "b200q_embed", "b200q_matmul_norm", "b200q_matmul_swiglu",
    "b200q_swiglu_f32", "b200q_swiglu_f32_interleaved", "b200q_gate_up_row", "b200q_matmul_q8_swiglu", "b200q_matmul_norm_swiglu", "b200q_moe_matmul_q8_swiglu",
    "b200q_comm_create", "b200q_comm_handle", "b200q_comm_connect", "b200q_allreduce_f64", "b200q_comm_free", "b200q_comm_gather_ptr",
    "b200q_matmul_q8_rowpar", "b200q_allreduce_add_rmsnorm_quant", "b200q_allreduce_finish", "b200q_matmul_q8_gather", "b200q_argmax_gathered", "b200q_allreduce",
    "b200q_bank_create", "b200q_bank_free", "b200q_bank_set", "b200q_bank_get", "b200q_bank_workspace_bytes", "b200q_moe_matmul_q8", "b200q_moe_combine",
]

_lib = None


def lib() -> C.CDLL:
    """Load libb200q.so; fail loudly when it is missing (the product path has no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200QError(-5, f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`")
        L = C.CDLL(LIB_PATH)
        L.b200q_last_error.restype = C.c_char_p
        L.b200q_workspace_bytes.restype = C.c_size_t
        L.b200q_act_bytes.restype = C.c_size_t
        L.b200q_launch_count.restype = C.c_int64
        L.b200q_workspace_bytes.argtypes = [C.c_void_p, C.c_int64]
        L.b200q_act_bytes.argtypes = [C.c_int64, C.c_int64]
        L.b200q_bank_workspace_bytes.restype = C.c_size_t
        L.b200q_bank_workspace_bytes.argtypes = [C.c_void_p, C.c_int64]
        L.b200q_bank_get.restype = C.c_void_p
        L.b200q_weight_set_next.argtypes = [C.c_void_p, C.c_void_p]
        L.b200q_gate_up_row.restype = C.c_int64
        L.b200q_gate_up_row.argtypes = [C.c_int64, C.c_int64]
        L.b200q_attn_decode_max_ctx.restype = C.c_int32
        L.b200q_attn_split_workspace_bytes.restype = C.c_size_t
        L.b200q_attn_split_workspace_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64]
        _lib = L
    return _lib


def _check(rc: int):
    if rc != 0:
        raise B200QError(rc, lib().b200q_last_error().decode())


def _stream_ptr(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _src(a):
    """(pointer, on_device, keepalive) for a numpy array or torch tensor"""
    if isinstance(a, torch.Tensor):
        a = a.contiguous()
        return C.c_void_p(a.data_ptr()), int(a.is_cuda), a
    a = np.ascontiguousarray(a)
    return C.c_void_p(a.ctypes.data), 0, a


def shard_range(total: int, rank: int, world: int, granule: int = 1):
    """reference src/engine/tensor_parallel.rs:61-67 (at `granule` granularity)"""
    s, e = C.c_int64(), C.c_int64()
    _check(lib().b200q_shard_range_blocks(C.c_int64(total), C.c_int64(granule), C.c_int64(rank), C.c_int64(world),
                                          C.byref(s), C.byref(e)))
    return int(s.value), int(e.value)


@dataclass
class DecomposedQuantMethod:
    """mirror of boostr::quant::decomposed::DecomposedQuantMethod::{Awq, Gptq}{group_size}"""
    kind: str  # "awq" | "gptq"
    group_size: int


@dataclass
class DecomposedQuantTensor:
    """mirror of DecomposedQuantTensor::new(qweight, scales, qzeros, g_idx, method, logical_shape)
    (reference awq.rs:218-225, gptq.rs:252-259).  AWQ: qzeros are f32 [K/gs, N] (already unpacked);
    GPTQ: qzeros stay packed u32 [G, N/8]."""
    qweight: np.ndarray
    scales: np.ndarray
    qzeros: np.ndarray
    g_idx: Optional[np.ndarray]
    method: DecomposedQuantMethod
    logical_shape: tuple
    bias: Optional[np.ndarray] = None
    zero_plus_one: int = 1


class QuantWeight:
    """Owning wrapper of an opaque b200q_weight handle (immutable once built)."""

    def __init__(self, handle: C.c_void_p, device: torch.device):
        self._h = handle
        self.device = device
        info = WeightInfo()
        _check(lib().b200q_weight_info(self._h, C.byref(info)))
        self.info = info
        self.N, self.K = int(info.N), int(info.K)
        self.K_pad = int(info.K_pad)
        self.canonical_bytes = int(info.canonical_bytes)
        self._ws = {}

    @property
    def handle(self):
        return self._h

    def workspace_bytes(self, M: int) -> int:
        return int(lib().b200q_workspace_bytes(self._h, C.c_int64(M)))

    def workspace(self, M: int) -> torch.Tensor:
        """Zero-filled scratch for calls with this M (cached per M; one in-flight call per workspace)."""
        ws = self._ws.get(M)
        if ws is None:
            ws = torch.zeros(max(256, self.workspace_bytes(M)), dtype=torch.uint8, device=self.device)
            self._ws[M] = ws
        return ws

    def set_next(self, nxt: Optional["QuantWeight"]):
        """streaming-order hint (include/b200q.h b200q_weight_set_next): the decode matvec on this weight prefetches the head
        of `nxt` into L2.  A reference to `nxt` is kept so the hint can never dangle."""
        _check(lib().b200q_weight_set_next(self._h, nxt.handle if nxt is not None else None))
        self._next = nxt

    def set_pair(self, second: Optional["QuantWeight"]):
        """dual-format pairing (include/b200q.h b200q_weight_set_pair): decode matvecs on this weight also compute `second`
        (another format, same K) into the columns that follow this weight's.  A reference is kept so the pairing cannot dangle."""
        _check(lib().b200q_weight_set_pair(self._h, second.handle if second is not None else None))
        self._pair = second

    def free(self):
        if self._h is not None:
            lib().b200q_weight_free(self._h)
            self._h = None
            self._ws = {}
            self._next = None
            self._pair = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class B200Client:
    """The backend client: implements the QuantMatmulOps / DequantOps surface on one B200."""

    def __init__(self, device=0):
        if not torch.cuda.is_available():
            raise B200QError(-5, "no CUDA device: the B200 path has no CPU fallback")
        self.device = torch.device("cuda", device) if not isinstance(device, torch.device) else device
        self.index = self.device.index or 0
        lib()

    # ---- upload -------------------------------------------------------------------------------
    def weight_from_ggml(self, ggml_type: int, blocks, N: int, K: int, rows=None, cols=None) -> QuantWeight:
        p, on_dev, keep = _src(blocks)
        h = C.c_void_p()
        n0, n1 = rows if rows is not None else (0, N)
        k0, k1 = cols if cols is not None else (0, K)
        with torch.cuda.device(self.device):
            _check(lib().b200q_weight_from_ggml_shard(C.c_int32(ggml_type), p, C.c_int32(on_dev), C.c_int64(N), C.c_int64(K),
                                                      C.c_int64(n0), C.c_int64(n1), C.c_int64(k0), C.c_int64(k1),
                                                      C.c_int32(self.index), _stream_ptr(self.device), C.byref(h)))
        del keep
        return QuantWeight(h, self.device)

    def weight_from_decomposed(self, t: DecomposedQuantTensor, rows=None, cols=None) -> QuantWeight:
        N, K = t.logical_shape
        h = C.c_void_p()
        qw, d1, k1_ = _src(t.qweight)
        sc, d2, k2_ = _src(np.asarray(t.scales, dtype=np.float32) if not isinstance(t.scales, torch.Tensor) else t.scales)
        on_dev = d1
        with torch.cuda.device(self.device):
            if t.method.kind == "awq":
                qz, _, k3_ = _src(np.asarray(t.qzeros, dtype=np.float32) if not isinstance(t.qzeros, torch.Tensor) else t.qzeros)
                n0, n1 = rows if rows is not None else (0, N)
                k0, k1 = cols if cols is not None else (0, K)
                _check(lib().b200q_weight_from_awq_shard(qw, sc, qz, C.c_int32(on_dev), C.c_int32(t.method.group_size), C.c_int64(N),
                                                         C.c_int64(K), C.c_int64(n0), C.c_int64(n1), C.c_int64(k0), C.c_int64(k1),
                                                         C.c_int32(self.index), _stream_ptr(self.device), C.byref(h)))
            elif t.method.kind == "gptq":
                qz, _, k3_ = _src(t.qzeros)
                gi, _, k4_ = _src(np.asarray(t.g_idx, dtype=np.int32)) if t.g_idx is not None else (None, 0, None)
                bi, _, k5_ = _src(np.asarray(t.bias, dtype=np.float32)) if t.bias is not None else (None, 0, None)
                n0, n1 = rows if rows is not None else (0, N)
                k0, k1 = cols if cols is not None else (0, K)
                _check(lib().b200q_weight_from_gptq_shard(qw, sc, qz, gi, bi, C.c_int32(on_dev), C.c_int32(t.method.group_size),
                                                          C.c_int32(t.zero_plus_one), C.c_int64(N), C.c_int64(K), C.c_int64(n0), C.c_int64(n1),
                                                          C.c_int64(k0), C.c_int64(k1), C.c_int32(self.index), _stream_ptr(self.device), C.byref(h)))
            else:
                raise B200QError(-2, f"unknown decomposed method {t.method.kind}")
        return QuantWeight(h, self.device)

    # ---- QuantMatmulOps ----------------------------------------------------------------------------
    def quant_matmul(self, x: torch.Tensor, w: QuantWeight, out: Optional[torch.Tensor] = None, out_dtype=None,
                     path: int = PATH_AUTO, workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Y[..., N] = X[..., K] @ dequant(W)[N, K]^T (+bias).  x: f32 / f16 / bf16 on this device."""
        assert x.is_cuda and x.shape[-1] == w.K, (x.shape, w.K)
        lead = x.shape[:-1]
        x2 = x.reshape(-1, w.K)
        if x2.stride(-1) != 1:
            x2 = x2.contiguous()
        M = x2.shape[0]
        ydt = out_dtype or x.dtype
        if out is None:
            out = torch.empty((M, w.N), dtype=ydt, device=x.device)
        y2 = out.reshape(M, w.N)
        ws = workspace if workspace is not None else w.workspace(M)
        _check(lib().b200q_matmul_path(w.handle, C.c_int32(path), C.c_void_p(x2.data_ptr()), C.c_int32(_TORCH2DT[x2.dtype]),
                                       C.c_int64(M), C.c_int64(x2.stride(0)), C.c_void_p(y2.data_ptr()),
                                       C.c_int32(_TORCH2DT[y2.dtype]), C.c_int64(y2.stride(0)), C.c_void_p(ws.data_ptr()),
                                       C.c_size_t(ws.numel()), _stream_ptr(x.device)))
        return out.reshape(*lead, w.N)

    def quantize_act(self, x: torch.Tensor, perm: Optional[torch.Tensor] = None) -> torch.Tensor:
        x2 = x.reshape(-1, x.shape[-1])
        M, K = x2.shape
        xq = torch.empty(int(lib().b200q_act_bytes(C.c_int64(K), C.c_int64(M))), dtype=torch.uint8, device=x.device)
        _check(lib().b200q_quantize_act(C.c_void_p(x2.data_ptr()), C.c_int32(_TORCH2DT[x2.dtype]), C.c_int64(M), C.c_int64(K),
                                        C.c_int64(x2.stride(0)), C.c_void_p(perm.data_ptr()) if perm is not None else None,
                                        C.c_void_p(xq.data_ptr()), _stream_ptr(x.device)))
        return xq

    def matmul_q8(self, xq: torch.Tensor, M: int, w: QuantWeight, out: Optional[torch.Tensor] = None, out_dtype=torch.float32,
                  workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
        if out is None:
            out = torch.empty((M, w.N), dtype=out_dtype, device=xq.device)
        ws = workspace if workspace is not None else w.workspace(M)
        _check(lib().b200q_matmul_q8(w.handle, C.c_void_p(xq.data_ptr()), C.c_int64(M), C.c_void_p(out.data_ptr()),
                                     C.c_int32(_TORCH2DT[out.dtype]), C.c_int64(out.stride(0)), C.c_void_p(ws.data_ptr()),
                                     C.c_size_t(ws.numel()), _stream_ptr(xq.device)))
        return out

    # ---- DequantOps --------------------------------------------------------------------------------
    def dequantize(self, w: QuantWeight, dtype=torch.float32) -> torch.Tensor:
        out = torch.empty((w.N, w.K), dtype=dtype, device=w.device)
        _check(lib().b200q_dequantize(w.handle, C.c_void_p(out.data_ptr()), C.c_int32(_TORCH2DT[dtype]), _stream_ptr(w.device)))
        return out

    # ---- test hooks (bit-exact contracts) --------------------------------------------------------
    def act_unpack(self, xq: torch.Tensor, M: int, K: int):
        K_pad = (K + 255) // 256 * 256
        q = torch.empty((M, K_pad), dtype=torch.int8, device=xq.device)
        d = torch.empty((M, K_pad // 32), dtype=torch.float32, device=xq.device)
        bs = torch.empty((M, K_pad // 16), dtype=torch.int32, device=xq.device)
        _check(lib().b200q_act_unpack(C.c_void_p(xq.data_ptr()), C.c_int64(M), C.c_int64(K), C.c_void_p(q.data_ptr()),
                                      C.c_void_p(d.data_ptr()), C.c_void_p(bs.data_ptr()), _stream_ptr(xq.device)))
        return q, d, bs

    def int_partials(self, w: QuantWeight, xq: torch.Tensor, M: int) -> torch.Tensor:
        P = w.K_pad // int(w.info.sub)
        out = torch.empty((M, w.N, P), dtype=torch.int32, device=xq.device)
        _check(lib().b200q_int_partials(w.handle, C.c_void_p(xq.data_ptr()), C.c_int64(M), C.c_void_p(out.data_ptr()),
                                        _stream_ptr(xq.device)))
        return out


class ExpertBank:
    """E weights of one format and shape behind a device pointer table (one projection of a stacked expert tensor).
    Members stay owned by their QuantWeight wrappers, which the bank keeps alive."""

    def __init__(self, experts):
        self.experts = list(experts)
        arr = (C.c_void_p * len(self.experts))(*[w.handle for w in self.experts])
        h = C.c_void_p()
        _check(lib().b200q_bank_create(arr, C.c_int32(len(self.experts)), C.byref(h)))
        self._h = h
        self.device = self.experts[0].device
        self.N, self.K, self.K_pad = self.experts[0].N, self.experts[0].K, self.experts[0].K_pad
        self._ws = {}

    @property
    def handle(self):
        return self._h

    def __len__(self):
        return len(self.experts)

    def set(self, e: int, w: QuantWeight):
        _check(lib().b200q_bank_set(self._h, C.c_int32(e), w.handle, _stream_ptr(self.device)))
        self.experts[e] = w

    def workspace(self, n_slots: int) -> torch.Tensor:
        ws = self._ws.get(n_slots)
        if ws is None:
            ws = torch.zeros(max(256, int(lib().b200q_bank_workspace_bytes(self._h, C.c_int64(n_slots)))), dtype=torch.uint8, device=self.device)
            self._ws[n_slots] = ws
        return ws

    def matmul_q8(self, sel: torch.Tensor, xq: torch.Tensor, x_rows: int, x_slot_div: int, out: Optional[torch.Tensor] = None,
                  workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
        """y[s, :] = W[sel[s]] . x[s // x_slot_div]   (sel: device int32 [n_slots]; xq: quantised records of x_rows rows)"""
        assert sel.is_cuda and sel.dtype == torch.int32
        n = sel.numel()
        if out is None:
            out = torch.empty((n, self.N), dtype=torch.float32, device=self.device)
        ws = workspace if workspace is not None else self.workspace(n)
        _check(lib().b200q_moe_matmul_q8(self._h, C.c_void_p(sel.data_ptr()), C.c_int64(n), C.c_void_p(xq.data_ptr()), C.c_int64(x_rows),
                                         C.c_int64(x_slot_div), C.c_void_p(out.data_ptr()), C.c_int32(_TORCH2DT[out.dtype]),
                                         C.c_int64(out.stride(0)), C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()),
                                         _stream_ptr(self.device)))
        return out

    def free(self):
        if self._h is not None:
            lib().b200q_bank_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


@dataclass
class ExpertWeights:
    """mirror of boostr::ExpertWeights (reference src/engine/executor_cache.rs:19,344-348): one expert's projections.
    gate_up is the row-fused [2 * ffn, hidden] weight the decode path launches once: gate rows first, or (interleaved) in
    the SwiGLU-epilogue row order (gate_up_row_order) so the grouped gate|up launch also activates and quantises."""
    gate_up: QuantWeight
    down_proj: QuantWeight
    interleaved: bool = False


class MoeMlp:
    """Decode-time mixture-of-experts MLP over two expert banks (gate|up fused, down), the operator behind
    get_expert_weights / set_expert_weights (reference executor_cache.rs:260,283).  `local` lists the expert ids this
    rank hosts (expert parallelism, SURVEY 8e: each rank runs its local selected experts on the replicated hidden state;
    blazr_b200/tp.py:ep_local_slots masks the non-local slots and the caller all-reduces the partial outputs)."""

    def __init__(self, client: "B200Client", experts, ffn: int, hidden: int, local=None):
        self.client = client
        self.E = len(experts)
        self.ffn, self.hidden = ffn, hidden
        self.local = list(range(self.E)) if local is None else list(local)
        self._experts = list(experts)
        self.interleaved = all(e.interleaved for e in experts) and ffn % 64 == 0
        assert self.interleaved or not any(e.interleaved for e in experts), "a bank mixes interleaved and plain gate|up weights"
        self._bufs = {}
        self.gu = ExpertBank([e.gate_up for e in experts])
        self.down = ExpertBank([e.down_proj for e in experts])

    def get_expert_weights(self, e: int) -> ExpertWeights:
        return self._experts[e]

    def set_expert_weights(self, e: int, w: ExpertWeights):
        self.gu.set(e, w.gate_up)
        self.down.set(e, w.down_proj)
        self._experts[e] = w

    def _buffers(self, T: int, top_k: int, device):
        key = (T, top_k)
        b = self._bufs.get(key)
        if b is None:
            n = T * top_k
            u8 = lambda nbytes: torch.zeros(int(nbytes), dtype=torch.uint8, device=device)
            b = dict(xq=u8(lib().b200q_act_bytes(C.c_int64(self.hidden), C.c_int64(T))), aq=u8(lib().b200q_act_bytes(C.c_int64(self.ffn), C.c_int64(n))),
                     gu=None if self.interleaved else torch.empty((n, 2 * self.ffn), dtype=torch.float32, device=device),
                     y=torch.empty((n, self.hidden), dtype=torch.float32, device=device), out=torch.empty((T, self.hidden), dtype=torch.float32, device=device),
                     ws_gu=u8(max(256, lib().b200q_bank_workspace_bytes(self.gu.handle, C.c_int64(n)))),
                     ws_dn=u8(max(256, lib().b200q_bank_workspace_bytes(self.down.handle, C.c_int64(n)))))
            self._bufs[key] = b
        return b

    def forward_decode(self, x: torch.Tensor, sel: torch.Tensor, gate_w: torch.Tensor) -> torch.Tensor:
        """x [T, hidden] f32, sel [T, top_k] int32 (bank-local expert indices, -1 = not hosted here), gate_w [T, top_k] f32
        -> [T, hidden] f32 (a view of an internal buffer: stable address, CUDA-graph capturable, no allocation after the
        first call of a shape).  Launches: quantise, grouped gate|up with the fused SwiGLU epilogue (interleaved banks; else
        grouped gate|up + SwiGLU), grouped down, weighted combine -- all libb200q kernels."""
        T, top_k = sel.shape
        n = T * top_k
        L = lib()
        P = lambda t_: C.c_void_p(t_.data_ptr())
        st = _stream_ptr(x.device)
        b = self._buffers(T, top_k, x.device)
        x = x.contiguous()
        sel_flat, gw = sel.reshape(-1), gate_w.contiguous()
        _check(L.b200q_quantize_act(P(x), C.c_int32(F32), C.c_int64(T), C.c_int64(self.hidden), C.c_int64(self.hidden), None, P(b["xq"]), st))
        if self.interleaved:
            _check(L.b200q_moe_matmul_q8_swiglu(self.gu.handle, P(sel_flat), C.c_int64(n), P(b["xq"]), C.c_int64(T), C.c_int64(top_k), P(b["aq"]),
                                                P(b["ws_gu"]), C.c_size_t(b["ws_gu"].numel()), st))
        else:
            _check(L.b200q_moe_matmul_q8(self.gu.handle, P(sel_flat), C.c_int64(n), P(b["xq"]), C.c_int64(T), C.c_int64(top_k), P(b["gu"]), C.c_int32(F32),
                                         C.c_int64(2 * self.ffn), P(b["ws_gu"]), C.c_size_t(b["ws_gu"].numel()), st))
            _check(L.b200q_swiglu_quant(P(b["gu"]), C.c_int64(self.ffn), C.c_int64(n), P(b["aq"]), st))
        _check(L.b200q_moe_matmul_q8(self.down.handle, P(sel_flat), C.c_int64(n), P(b["aq"]), C.c_int64(n), C.c_int64(1), P(b["y"]), C.c_int32(F32),
                                     C.c_int64(self.hidden), P(b["ws_dn"]), C.c_size_t(b["ws_dn"].numel()), st))
        _check(L.b200q_moe_combine(P(b["y"]), P(gw), C.c_int64(T), C.c_int64(top_k), C.c_int64(self.hidden), P(b["out"]), st))
        return b["out"]


class _DevView:
    """zero-copy torch view of library-owned device memory (CUDA array interface)"""

    def __init__(self, ptr: int, shape, typestr: str):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 2}


class PeerComm:
    """Tensor-parallel exchange context over NVLink peer memory (include/b200q.h b200q_comm_*).  `group` is only used once,
    to all-gather the CUDA IPC handles; the data path never touches NCCL.  The exchange is fused into the kernels on both
    sides of it: matmul_q8_rowpar (producer) -> allreduce_add_rmsnorm_quant / allreduce_finish (consumer), and
    matmul_q8_gather -> argmax_gathered for the vocabulary-parallel lm_head."""

    def __init__(self, rank: int, world: int, max_elems: int, device: torch.device, group=None, gather_elems: int = 0):
        self.rank, self.world, self.device = rank, world, device
        h = C.c_void_p()
        _check(lib().b200q_comm_create(C.c_int32(rank), C.c_int32(world), C.c_int64(max_elems), C.c_int64(gather_elems), C.c_int32(device.index or 0),
                                       C.byref(h)))
        self._h = h
        mine = (C.c_uint8 * 64)()
        _check(lib().b200q_comm_handle(self._h, mine))
        handles = [bytes(mine)]
        if world > 1:
            import torch.distributed as dist
            handles = [None] * world
            dist.all_gather_object(handles, bytes(mine), group=group)
        buf = (C.c_uint8 * (64 * world)).from_buffer_copy(b"".join(handles))
        _check(lib().b200q_comm_connect(self._h, buf))
        if world > 1:
            import torch.distributed as dist
            dist.barrier(group=group)

    @property
    def handle(self):
        return self._h

    def allreduce(self, src: torch.Tensor, dst: torch.Tensor):
        """stand-alone one-shot all-reduce(sum): dst (f32) = sum over ranks of src (f32 or f64), f64 sum in rank order"""
        assert src.dtype in (torch.float64, torch.float32) and dst.dtype == torch.float32 and src.numel() == dst.numel()
        _check(lib().b200q_allreduce(self._h, C.c_void_p(src.data_ptr()), C.c_int32(F64 if src.dtype == torch.float64 else F32),
                                     C.c_void_p(dst.data_ptr()), C.c_int64(src.numel()), _stream_ptr(self.device)))

    def allreduce_f64(self, src: torch.Tensor, dst: torch.Tensor):
        self.allreduce(src, dst)

    def matmul_q8_rowpar(self, w: "QuantWeight", xq: torch.Tensor, M: int, ld: int, workspace: torch.Tensor):
        """row-parallel matvec whose exact f64 row sums [M, ld] go straight into every rank's exchange slot"""
        _check(lib().b200q_matmul_q8_rowpar(w.handle, C.c_void_p(xq.data_ptr()), C.c_int64(M), self._h, C.c_int64(ld), C.c_void_p(workspace.data_ptr()),
                                            C.c_size_t(workspace.numel()), _stream_ptr(self.device)))

    def allreduce_finish(self, dst: torch.Tensor):
        _check(lib().b200q_allreduce_finish(self._h, C.c_void_p(dst.data_ptr()), C.c_int64(dst.numel()), _stream_ptr(self.device)))

    def allreduce_add_rmsnorm_quant(self, h_in, h_out, norm_w, eps: float, H: int, M: int, xq=None, xnorm=None):
        _check(lib().b200q_allreduce_add_rmsnorm_quant(self._h, C.c_void_p(h_in.data_ptr()), C.c_void_p(h_out.data_ptr()), C.c_void_p(norm_w.data_ptr()),
                                                       C.c_float(eps), C.c_int64(H), C.c_int64(M), C.c_void_p(xq.data_ptr()) if xq is not None else None,
                                                       C.c_void_p(xnorm.data_ptr()) if xnorm is not None else None, _stream_ptr(self.device)))

    def matmul_q8_gather(self, w: "QuantWeight", xq: torch.Tensor, M: int, ld: int, workspace: torch.Tensor):
        _check(lib().b200q_matmul_q8_gather(w.handle, C.c_void_p(xq.data_ptr()), C.c_int64(M), self._h, C.c_int64(ld), C.c_void_p(workspace.data_ptr()),
                                            C.c_size_t(workspace.numel()), _stream_ptr(self.device)))

    def argmax_gathered(self, ld: int, M: int, out_ids: torch.Tensor, pos_inc: Optional[torch.Tensor]):
        _check(lib().b200q_argmax_gathered(self._h, C.c_int64(ld), C.c_int64(M), C.c_void_p(out_ids.data_ptr()),
                                           C.c_void_p(pos_inc.data_ptr()) if pos_inc is not None else None, _stream_ptr(self.device)))

    def gathered(self) -> torch.Tensor:
        """f32 [world, elems_per_rank] view of this rank's gather area (region r = what rank r stored)"""
        ptr, n = C.c_void_p(), C.c_int64()
        _check(lib().b200q_comm_gather_ptr(self._h, C.byref(ptr), C.byref(n)))
        return torch.as_tensor(_DevView(ptr.value, (self.world, n.value), "<f4"), device=self.device)

    def free(self):
        if self._h is not None:
            lib().b200q_comm_free(self._h)
            self._h = None


def gate_up_row_order(F: int) -> np.ndarray:
    """row permutation of the SwiGLU-epilogue layout (include/b200q.h b200q_gate_up_row): interleaved[r] = concat(gate, up)[perm[r]]"""
    r = np.arange(2 * F, dtype=np.int64)
    t, rr = r // 128, r % 128
    return np.where((rr % 8) // 4 == 1, F, 0) + 64 * t + 4 * (rr // 8) + rr % 4


def launch_count() -> int:
    return int(lib().b200q_launch_count())
