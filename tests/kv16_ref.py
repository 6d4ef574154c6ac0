"""Test helper: the f16 KV cache element rule restated in numpy, and the CPU oracle model with an f16 KV cache.

The rule (include/b200q.h, b200q_attn_decode_kv): an appended K / V element is f16_rn(clamp(x, -65504, 65504)) of its f32
value (the rotated k, the raw v), and NaN stores -65504 (the kernels clamp with fmaxf first, which drops the NaN).  Every
later read widens the stored f16 exactly, so the oracle's attention arithmetic is unchanged."""
import numpy as np

from oracle.model import OracleModel


def kv_round_np(x) -> np.ndarray:
    """f16 cache element of f32 value(s) x: numpy's f32 -> f16 conversion rounds to nearest even, as __float2half_rn does"""
    x = np.asarray(x, dtype=np.float32)
    return np.where(np.isnan(x), np.float32(-65504.0), np.clip(x, np.float32(-65504.0), np.float32(65504.0))).astype(np.float16)


class Kv16Rows(list):
    """a layer's K or V cache of the oracle: rows are stored as the f16 cache stores them"""

    def __init__(self, rows=()):
        super().__init__(kv_round_np(r) for r in rows)

    def append(self, row):
        super().append(kv_round_np(row))


class OracleModelKV16(OracleModel):
    """OracleModel whose appended k / v rows go through kv_round_np (the rounded rows are scored and weighted by the same
    step that appends them).  To preload a cache, assign Kv16Rows(rows) to k_cache[layer] / v_cache[layer]."""

    def reset(self):
        super().reset()
        self.k_cache = [Kv16Rows() for _ in self.layers]
        self.v_cache = [Kv16Rows() for _ in self.layers]


def oracle_model(host, flavour: str = "B", kv_dtype: str = "f32") -> OracleModel:
    return OracleModelKV16(host, flavour) if kv_dtype == "f16" else OracleModel(host, flavour)
