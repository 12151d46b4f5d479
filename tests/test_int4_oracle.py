"""Properties of the NumPy INT4 oracle (restating demo/quantize_int4.cu); tests/test_gpu_kv_ops.py pins it against
the reference kernels' stored outputs (tests/golden/int4_ref_kernels.npz)."""
import numpy as np

from oracle import int4_oracle as Q


def test_pack_layout_high_nibble_is_even_element():
    x = np.zeros((1, 128), dtype=np.float16)
    x[0, 0] = 15.0  # -> code 15 in the HIGH nibble of byte 0 (quantize_int4.cu:137)
    x[0, 3] = 15.0  # -> LOW nibble of byte 1
    p, s, z = Q.quantize_int4(x)
    assert p.shape == (1, 64) and p[0, 0] == 0xF0 and p[0, 1] == 0x0F
    assert s.dtype == np.float16 and z.dtype == np.float16 and float(z[0, 0]) == 0.0
    assert abs(float(s[0, 0]) - 1.0) < 1e-3


def test_round_trip_error_bounded_by_half_step():
    rng = np.random.RandomState(0)
    x = (rng.randn(64, 8, 128) * 3).astype(np.float16)
    p, s, z = Q.quantize_int4(x)
    y = Q.dequantize_int4(p, s, z)
    step = s.astype(np.float32)
    err = np.abs(y.astype(np.float32) - x.astype(np.float32))
    assert (err <= 0.5 * step + 0.02 * np.abs(x).max() / 15 + 1e-2).all()
    codes = Q.unpack_codes(p)
    assert codes.min() == 0 and codes.max() == 15
    # min maps to code 0, max to code 15 in every group
    assert (np.take_along_axis(codes, x.argmin(-1)[..., None], -1) == 0).all()
    assert (np.take_along_axis(codes, x.argmax(-1)[..., None], -1) == 15).all()


def test_dequant_rounding_modes():
    p = np.full((1, 64), 0x7B, dtype=np.uint8)  # codes 7, 11
    s = np.array([[0.333251953125]], dtype=np.float16)
    z = np.array([[-1.7001953125]], dtype=np.float16)
    y = Q.dequantize_int4(p, s, z)                 # as built: fused, one rounding
    y2 = Q.dequantize_int4(p, s, z, fused=False)   # literal source reading: two roundings
    for code, got, got2 in ((7, y[0, 0], y2[0, 0]), (11, y[0, 1], y2[0, 1])):
        assert got == np.float16(np.float64(code) * np.float64(s[0, 0]) + np.float64(z[0, 0]))
        prod = np.float16(np.float32(code) * np.float32(s[0, 0]))
        assert got2 == np.float16(np.float32(prod) + np.float32(z[0, 0]))


def test_constant_group_is_stable():
    x = np.full((2, 128), 0.5, dtype=np.float16)
    p, s, z = Q.quantize_int4(x)
    y = Q.dequantize_int4(p, s, z)
    assert np.abs(y.astype(np.float32) - 0.5).max() < 1e-3
