"""The sub-pixel keypoint step, the parts that need no GPU: the oracle (subpixel_oracle.soft_argmax_points) against closed
forms of the reference's arithmetic, and the argument checks of ssp_soft_argmax_points before any CUDA call."""
import ctypes

import numpy as np
import pytest

import subpixel_oracle as SO

H, W = 20, 30
EPS = 1e-6  # norm_patches' and SpatialSoftArgmax2d's eps
# dx is an fp32 sum of p * p rounded terms with a value near 2, where fp32 spacing is 2^-23 (below 2) / 2^-22 (above): for a
# generic patch its rounding error is a few units of 2^-23, more than 1e-7 and well below the 2e-6 the eps moves a point
FP32_NEAR_2 = 4 * 2.0 ** -23


def refine(heat, x, y, p=5):
    return SO.soft_argmax_points(heat, np.array([[float(x)], [float(y)], [0.5]]), p)


def test_lone_centre_tap_keeps_the_eps():
    """One non-zero tap in the centre: q = 1 there, log q = -inf elsewhere, so e is one-hot and s = 1 / (1 + 1e-6): both
    coordinates move by 2 / (1 + 1e-6) - 2 (about -2e-6, the eps of the soft arg-max)."""
    heat = np.zeros((H, W), np.float32)
    heat[10, 15] = 0.7
    out = refine(heat, 15, 10)
    want = 2 / (1 + EPS) - 2
    assert abs(want + 2e-6) < 1e-11
    np.testing.assert_allclose(out[:2, 0], [15 + want, 10 + want], rtol=0, atol=1e-7)
    assert out[2, 0] == 0.5


@pytest.mark.parametrize("seed", range(4))
def test_symmetric_patch(seed):
    """A patch symmetric about its centre: sum(pos e) = 2 S, so both offsets are 2 S / (S + 1e-6) - 2 with S = sum(e)
    (e = exp(l - max l) = patch / max(patch) here)."""
    a = np.random.default_rng(seed).uniform(0.01, 1, (5, 5))
    a = a + a[::-1] + a[:, ::-1] + a[::-1, ::-1]
    a = (a + a.T).astype(np.float32)
    heat = np.zeros((H, W), np.float32)
    heat[8:13, 13:18] = a
    out = refine(heat, 15, 10)
    S = (a.astype(np.float64) / a.max()).sum()
    want = 2 * S / (S + EPS) - 2
    np.testing.assert_allclose(out[:2, 0], [15 + want, 10 + want], rtol=0, atol=FP32_NEAR_2)
    # a uniform patch: e = 1 exactly
    heat[8:13, 13:18] = 0.2
    out = refine(heat, 15, 10)
    np.testing.assert_allclose(out[:2, 0] - [15, 10], 2 * 25 / (25 + EPS) - 2, rtol=0, atol=FP32_NEAR_2)


def test_two_equal_taps():
    """Equal taps at the centre and one column to the right: e = 1 at both, x moves by 5 / (2 + 1e-6) - 2 and y by
    4 / (2 + 1e-6) - 2."""
    heat = np.zeros((H, W), np.float32)
    heat[10, 15] = heat[10, 16] = 0.3
    out = refine(heat, 15, 10)
    np.testing.assert_allclose(out[:2, 0], [15 + 5 / (2 + EPS) - 2, 10 + 4 / (2 + EPS) - 2], rtol=0, atol=1e-7)


@pytest.mark.parametrize("p", [3, 4, 5, 7])
def test_border_points_see_zero_padding(p):
    """Points within p // 2 of the edges (corners included) give what the same points give in a zero-padded larger map."""
    rng = np.random.default_rng(p)
    heat = rng.uniform(0, 1, (H, W)).astype(np.float32)
    pts = np.array([[0, 0, 0.1], [W - 1, 0, 0.2], [0, H - 1, 0.3], [W - 1, H - 1, 0.4], [1, 7, 0.5], [W - 2, 9, 0.6],
                    [12, 1, 0.7], [14, H - 2, 0.8], [15, 10, 0.9]], np.float64).T
    out = SO.soft_argmax_points(heat, [pts], p)
    m = 9
    big = np.zeros((H + 2 * m, W + 2 * m), np.float32)
    big[m:m + H, m:m + W] = heat
    shifted = pts.copy()
    shifted[:2] += m
    ref = SO.soft_argmax_points(big, shifted, p)
    ref[:2] -= m
    np.testing.assert_allclose(out, ref, rtol=0, atol=1e-12)
    assert np.array_equal(out[2], pts[2])


def test_zero_taps_stay_finite():
    """Zero taps (log = -inf) and a negative tap (clamped to 1e-6 before the log) leave a finite result inside the patch."""
    heat = np.zeros((H, W), np.float32)
    heat[9, 14], heat[10, 15], heat[11, 17], heat[12, 13] = 0.2, 0.5, 0.1, -0.05
    out = refine(heat, 15, 10)
    assert np.isfinite(out).all()
    assert (np.abs(out[:2, 0] - [15, 10]) <= 2).all()


def test_oracle_empty_and_list_forms():
    heat = np.ones((1, H, W), np.float32)
    assert SO.soft_argmax_points(heat, [np.zeros((3, 0))]).shape == (3, 0)
    pts = np.array([[3.0], [4.0], [0.5]])
    a, b = SO.soft_argmax_points(heat, pts), SO.soft_argmax_points(heat, [pts])
    assert np.array_equal(a, b) and pts[0, 0] == 3.0  # the input is not modified


def test_argument_errors_without_gpu():
    """Null pointers and a patch outside 1..15 are refused before any CUDA call."""
    from ssp_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(256)
    assert lib.ssp_soft_argmax_points(None, 1, 8, 8, p, 4, p, 4, 5, None) < 0
    assert b"null pointer" in lib.ssp_last_error()
    assert lib.ssp_soft_argmax_points(p, 1, 8, 8, None, 4, p, 4, 5, None) < 0
    assert b"null pointer" in lib.ssp_last_error()
    assert lib.ssp_soft_argmax_points(p, 1, 8, 8, p, 4, None, 4, 5, None) < 0
    assert b"null pointer" in lib.ssp_last_error()
    for bad in (0, -1, 16):
        assert lib.ssp_soft_argmax_points(p, 1, 8, 8, p, 4, p, 4, bad, None) < 0
        assert b"patch" in lib.ssp_last_error()
    assert lib.ssp_soft_argmax_points(p, 1, 8, 8, p, 4, p, -1, 5, None) < 0
    assert b"bad sizes" in lib.ssp_last_error()
    assert lib.ssp_soft_argmax_points(p, 1, 8, 8, p, 4, p, 0, 5, None) == 0  # nothing to refine: no launch
    I, Hh, Ww = 3, 240, 320
    assert lib.ssp_nms_ws_counts_offset(I, Hh, Ww) + 4 * I <= lib.ssp_nms_ws_bytes(I, Hh, Ww, 1)
