"""Test-side restatement of the Llama 3.1 / 3.2 RoPE frequency factors (no product code imported):
- llama3_rope_factors: the rope_freqs.weight values llama.cpp's converter writes for rope_scaling.rope_type == "llama3";
- rope_table_ref: the (cos, sin) table with those factors, for oracle models of such files (OracleModel.rope is replaced by it)."""
import math

import numpy as np


def llama3_rope_factors(head_dim, theta, factor=8.0, low_freq_factor=1.0, high_freq_factor=4.0, original_context=8192):
    """1 for short wavelengths, `factor` for long ones, a smooth blend in between; f32 [head_dim / 2]"""
    freqs = 1.0 / (theta ** (np.arange(0, head_dim, 2, dtype=np.float32) / head_dim))
    low_wavelen, high_wavelen = original_context / low_freq_factor, original_context / high_freq_factor
    out = []
    for f in freqs:
        wavelen = 2 * math.pi / f
        if wavelen < high_wavelen:
            out.append(1.0)
        elif wavelen > low_wavelen:
            out.append(factor)
        else:
            smooth = (original_context / wavelen - low_freq_factor) / (high_freq_factor - low_freq_factor)
            out.append(1 / ((1 - smooth) / factor + smooth))
    return np.asarray(out, dtype=np.float32)


def rope_table_ref(max_ctx, head_dim, theta, factors=None):
    """[max_ctx, hd/2, 2] f32 (cos, sin) of pos * theta^(-2i/hd) / factors[i]: f64, one rounding (ggml's theta / freq_factor)"""
    i = np.arange(head_dim // 2, dtype=np.float64)
    freq = np.power(float(theta), -2.0 * i / head_dim)
    if factors is not None:
        freq = freq / np.asarray(factors, dtype=np.float64).reshape(head_dim // 2)
    ang = np.arange(max_ctx, dtype=np.float64)[:, None] * freq[None, :]
    return np.stack([np.cos(ang), np.sin(ang)], axis=-1).astype(np.float32)


def oracle_with_table(om, max_ctx, factors=None):
    """an OracleModel whose RoPE table covers max_ctx positions and carries the model's frequency factors"""
    om.rope = rope_table_ref(max_ctx, om.cfg.head_dim, om.cfg.rope_theta, factors)
    return om
