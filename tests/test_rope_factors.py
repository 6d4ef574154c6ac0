"""CPU: Llama 3.1 / 3.2 RoPE frequency factors -- the table with and without factors, product vs the oracle's table and the
test-side restatement with factors (tests/rope_ref.py), and
the GGUF loader's handling of the rope_freqs.weight tensor llama.cpp writes for these models."""
import dataclasses

import numpy as np
import pytest

from blazr_b200 import decode, gguf_loader
from gguf_util import write_gguf
from oracle import model as oracle_model
from rope_ref import llama3_rope_factors, rope_table_ref

gguf = pytest.importorskip("gguf")


@pytest.mark.parametrize("hd,theta", [(64, 10000.0), (128, 500000.0)])
def test_no_factors_and_unit_factors_are_bit_identical(hd, theta):
    ref = oracle_model.rope_table(1024, hd, theta)
    assert np.array_equal(decode.rope_table(1024, hd, theta).view(np.uint32), ref.view(np.uint32))
    assert np.array_equal(decode.rope_table(1024, hd, theta, factors=None).view(np.uint32), ref.view(np.uint32))
    ones = tuple([1.0] * (hd // 2))
    assert np.array_equal(decode.rope_table(1024, hd, theta, factors=ones).view(np.uint32), ref.view(np.uint32))


@pytest.mark.parametrize("hd,theta,orig", [(64, 10000.0, 64), (128, 500000.0, 8192)])
def test_product_and_reference_tables_agree_with_factors(hd, theta, orig):
    # the test-side restatement without factors is the oracle's table, bit for bit
    assert np.array_equal(rope_table_ref(4096, hd, theta).view(np.uint32), oracle_model.rope_table(4096, hd, theta).view(np.uint32))
    f = llama3_rope_factors(hd, theta, original_context=orig)
    assert f.min() == 1.0 and f.max() == 8.0 and np.any((f > 1.0) & (f < 8.0)), f   # all three regimes present
    a = decode.rope_table(4096, hd, theta, tuple(float(x) for x in f))
    b = rope_table_ref(4096, hd, theta, tuple(float(x) for x in f))
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    # the factors divide the frequencies: the long-wavelength half of the table turns more slowly than without them
    assert not np.array_equal(a, oracle_model.rope_table(4096, hd, theta))
    i = np.arange(hd // 2, dtype=np.float64)
    ang = 1000.0 * np.power(theta, -2.0 * i / hd) / f.astype(np.float64)
    assert np.array_equal(a[1000, :, 0], np.cos(ang).astype(np.float32))


def _host(seed=5):
    return decode.build_host_model(decode.PRESETS["tiny"], "Q8_0", seed=seed)


def test_loader_accepts_rope_freqs_and_sets_config(tmp_path):
    hm = _host()
    f = llama3_rope_factors(hm.cfg.head_dim, hm.cfg.rope_theta, original_context=64)
    path = str(tmp_path / "l31.gguf")
    write_gguf(path, hm, extra_tensors={"rope_freqs.weight": f})
    h2 = gguf_loader.host_model_from_gguf(gguf_loader.Gguf.open(path))
    assert h2.cfg.rope_freq_factors == tuple(float(x) for x in f)
    # a file without the tensor keeps the unscaled table
    p0 = str(tmp_path / "l3.gguf")
    write_gguf(p0, hm)
    assert gguf_loader.host_model_from_gguf(gguf_loader.Gguf.open(p0)).cfg.rope_freq_factors is None
    # the config field is appended with a default: every preset is unscaled
    assert all(c.rope_freq_factors is None for c in decode.PRESETS.values())
    assert dataclasses.fields(decode.ModelConfig)[-1].name == "rope_freq_factors"


@pytest.mark.parametrize("bad,match", [
    (np.ones(16, dtype=np.float32), "shape"),                                     # hd / 4 values instead of hd / 2
    (np.ones((2, 32), dtype=np.float32), "shape"),
    (np.ones(32, dtype=np.float16), "F32"),
    (np.concatenate([np.ones(31), [0.0]]).astype(np.float32), "positive"),
    (np.concatenate([np.ones(31), [-2.0]]).astype(np.float32), "positive"),
    (np.concatenate([np.ones(31), [np.inf]]).astype(np.float32), "positive"),
])
def test_loader_rejects_malformed_rope_freqs(tmp_path, bad, match):
    hm = _host()
    path = str(tmp_path / "bad.gguf")
    write_gguf(path, hm, extra_tensors={"rope_freqs.weight": bad})
    with pytest.raises(gguf_loader.GgufError, match=match):
        gguf_loader.host_model_from_gguf(gguf_loader.Gguf.open(path))


def test_rope_freqs_only_for_llama(tmp_path):
    """mistral files never carry the tensor: there it stays a stray tensor and is refused"""
    hm = _host()
    path = str(tmp_path / "m.gguf")
    write_gguf(path, hm, arch="mistral", extra_tensors={"rope_freqs.weight": np.ones(32, dtype=np.float32)})
    with pytest.raises(gguf_loader.GgufError, match="does not consume"):
        gguf_loader.host_model_from_gguf(gguf_loader.Gguf.open(path))
