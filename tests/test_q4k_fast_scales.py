"""CPU checks of the arithmetic behind the Q4_K matvec fast path (formats.cuh FmtQ4K::load_unit_at).

The fast path forms a' = d * sc * 2^-24 and b' = dmin * m * 2^-24 with one f16 x f16 -> f32 FMA each (sc and m enter as the
f16 subnormals n * 2^-24), and multiplies the activation scale by 2^24 instead.  The output stays bit-identical to the
generic loader when
  1. every d * n * 2^-24 (d any finite f16, n < 64) is an exact f32, so the FMA does not round;
  2. fl(a' * (dx * 2^24)) == fl(a * dx) for every activation scale the quantiser can produce below 2^104;
  3. the header bit trick yields the same m as the canonical unpack.
"""
import numpy as np


def _finite_f16():
    h = np.arange(1 << 16, dtype=np.uint32).astype(np.uint16).view(np.float16)
    return h[np.isfinite(h)].astype(np.float64)


def test_scaled_scale_is_exact_f32():
    d = _finite_f16()
    n = np.arange(64, dtype=np.float64)
    exact = d[:, None] * n[None, :] * 2.0**-24     # exact in f64: <= 17 significant bits
    assert np.array_equal(exact.astype(np.float32).astype(np.float64), exact)


def test_product_with_rescaled_activation_scale_is_unchanged():
    rng = np.random.default_rng(7)
    d = _finite_f16()
    n = np.arange(64, dtype=np.float64)
    a = (d[:, None] * n[None, :]).astype(np.float32).ravel()
    a_s = (d[:, None] * n[None, :] * 2.0**-24).astype(np.float32).ravel()
    assert np.array_equal(a_s.astype(np.float64) * 2.0**24, a.astype(np.float64))
    # activation scales amax / 127: ordinary, tiny (subnormal) and the largest ones the identity covers
    dx = np.concatenate([
        (rng.random(64) * 10.0 ** rng.integers(-12, 4, 64)).astype(np.float32),
        np.array([1e-45, 1e-40, 1.1754942e-38, 2.0**103, np.nextafter(np.float32(2.0**104), np.float32(0))], np.float32),
    ])
    for x in dx:
        x_s = np.float32(x) * np.float32(2.0**24)
        assert np.isfinite(x_s)
        with np.errstate(over="ignore", under="ignore"):
            assert np.array_equal((a_s * x_s).view(np.uint32), (a * np.float32(x)).view(np.uint32)), x


def test_header_bit_trick_gives_m():
    b1 = np.arange(256, dtype=np.uint32)[:, None, None]
    b2 = np.arange(256, dtype=np.uint32)[None, :, None]
    i = np.arange(8, dtype=np.uint32)[None, None, :]
    m_ref = (b1 >> 6) | (((b2 >> (4 * (i & 1))) & 0xF) << 2)
    f = b1 | ((b2 << (8 - 4 * (i & 1))) & 0xF00)
    assert f.max() < (1 << 12)                      # the f16 operand's high bits stay clear
    assert np.array_equal(f >> 6, m_ref)
