"""Sub-pixel keypoints on the device (ssp_soft_argmax_points) against the oracle (subpixel_oracle.soft_argmax_points):
step.adaptation_step(subpixel=True) at the benchmarked shape, utils.heatmap_to_pts_batch / utils.soft_argmax_points at
several patch sizes with border and corner points, and the front-end binding of dropin.install.  Device and oracle sum in
different orders, so coordinates agree to 2e-5 px rather than bit for bit; counts, order and confidences are exact."""
import types

import numpy as np
import pytest
import torch

import ssp_b200 as S
import subpixel_oracle as SO
from ssp_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda"
I0, REP, N, H, W = 4, 8, 100, 240, 320
TOL = 2e-5


def adaptation_inputs(I0=I0, rep=REP, seed=0):
    """bench.py's homography-adaptation workload: I0 distinct source images of N views of 240x320, their logits rescaled
    rep times to I0 * rep source images, binary valid masks.
    Returns (semi [I,N,65,30,40], homographies [I,N,3,3], valid masks [I,N,H,W]) on the device."""
    base, Hs = synth.adaptation_workload(I0, N, H // 8, W // 8, seed)
    Hinv = torch.from_numpy(np.linalg.inv(Hs).astype(np.float32)).to(DEV)
    semi = torch.cat([torch.from_numpy(base * np.float32(1.0 + 0.05 * k)).to(DEV) for k in range(rep)])
    mask = S.compute_valid_mask(torch.tensor([H, W]), Hinv.reshape(-1, 3, 3), device=DEV).reshape(I0, N, H, W)
    return semi, torch.from_numpy(Hs).to(DEV).repeat(rep, 1, 1, 1), mask.repeat(rep, 1, 1, 1)


@pytest.fixture(scope="module")
def bench_inputs():
    return adaptation_inputs()


@pytest.mark.parametrize("top_k", [600, None])
def test_adaptation_step_subpixel_vs_oracle(bench_inputs, top_k):
    """32 source images x 100 views: subpixel=True keeps the count, order and prob of every point of subpixel=False and
    moves x, y to what the oracle computes on the aggregated heatmap from the unrefined points."""
    semi, Hw, mask = bench_inputs
    base = S.step.adaptation_step(semi, Hw, mask, top_k=top_k, binary_mask=True)
    sub = S.step.adaptation_step(semi, Hw, mask, top_k=top_k, binary_mask=True, subpixel=True)
    agg = S.utils.combine_from_logits_batch(semi, Hw, mask).cpu().numpy()
    assert len(sub) == len(base) == I0 * REP
    moved = 0.0
    for i, (a, b) in enumerate(zip(base, sub)):
        assert a.shape == b.shape and a.shape[0] > 0, i
        if top_k:
            assert a.shape[0] <= top_k
        assert np.array_equal(a[:, 2], b[:, 2]), i
        ref = SO.soft_argmax_points(agg[i], a.T, 5).T
        np.testing.assert_allclose(b[:, :2], ref[:, :2], rtol=0, atol=TOL, err_msg="image %d" % i)
        assert np.array_equal(np.trunc(a[:, :2]), a[:, :2])  # NMS output is integral
        moved = max(moved, float(np.abs(b[:, :2] - a[:, :2]).max()))
    assert moved > 0.1


def border_points(Hh, Ww):
    """Corners, points within 1 or 2 pixels of every edge, one interior point (x, y, conf)."""
    xy = [(0, 0), (Ww - 1, 0), (0, Hh - 1), (Ww - 1, Hh - 1), (1, Hh // 2), (Ww - 2, Hh // 3), (Ww // 2, 1), (Ww // 3, Hh - 2),
          (2, 2), (Ww - 3, Hh - 3), (Ww // 2, Hh // 2)]
    return np.array([[x, y, 0.01 * (k + 1)] for k, (x, y) in enumerate(xy)], np.float64).T


@pytest.mark.parametrize("p", [3, 4, 5, 7, 15])
@pytest.mark.parametrize("kind", ["numpy", "cuda"])
def test_soft_argmax_points_vs_oracle(p, kind):
    """NMS points of a 120x160 heatmap plus border and corner points (zero padding), a numpy [H,W] heatmap or a CUDA
    [1,H,W] tensor (squeezed); the list form in and out.  p = 15 fills all 8 register slots of a lane (225 taps), p = 4
    is an even patch (one more tap before the point than after it)."""
    Hh, Ww = 120, 160
    heat = synth.unique_heatmap(Hh, Ww, 40 + p)
    pts = np.concatenate([S.getPtsFromHeatmap(heat, 0.015, 4), border_points(Hh, Ww)], axis=1)
    arg = heat if kind == "numpy" else torch.from_numpy(heat).to(DEV)[None]
    got = S.soft_argmax_points(arg, [pts], p)
    assert isinstance(got, list) and len(got) == 1 and got[0].dtype == np.float64 and got[0].shape == pts.shape
    ref = SO.soft_argmax_points(heat, pts, p)
    np.testing.assert_allclose(got[0][:2], ref[:2], rtol=0, atol=TOL)
    assert np.array_equal(got[0][2], pts[2])
    assert pts[0, -1] == Ww // 2  # the input is not modified


@pytest.mark.parametrize("K", [0, 1])
def test_soft_argmax_points_tiny(K):
    """K = 1 (the reference squeezes its [1,2] offsets to [2]) and K = 0 (-> [zeros((3, 0))], the reference crashes)."""
    heat = synth.unique_heatmap(40, 50, 3)
    pts = border_points(40, 50)[:, :K]
    got = S.soft_argmax_points(heat, pts)
    assert isinstance(got, list) and len(got) == 1 and got[0].shape == (3, K)
    np.testing.assert_allclose(got[0], SO.soft_argmax_points(heat, pts), rtol=0, atol=TOL)


def test_fortran_ordered_points():
    """np.array([[x, y, c], ...]).T is a column-major [3,K] view: refined like its row-major copy, the input untouched."""
    heat = synth.unique_heatmap(60, 80, 8)
    pts = border_points(60, 80)
    assert pts.flags.f_contiguous and not pts.flags.c_contiguous
    keep = pts.copy()
    got = S.soft_argmax_points(heat, pts, 5)[0]
    np.testing.assert_allclose(got, SO.soft_argmax_points(heat, np.ascontiguousarray(pts), 5), rtol=0, atol=TOL)
    assert np.array_equal(pts, keep)


def test_lone_centre_tap_keeps_the_eps():
    """One non-zero tap in the centre: e is one-hot and s = 1 / (1 + 1e-6), so x and y move by 2 / (1 + 1e-6) - 2, about
    -2e-6 px; a kernel without the eps of the soft arg-max (or of the patch normalisation) is off by more than 1e-7."""
    heat = np.zeros((40, 50), np.float32)
    heat[20, 25] = 0.7
    got = S.soft_argmax_points(heat, np.array([[25.0], [20.0], [0.7]]), 5)[0]
    want = 2 / (1 + 1e-6) - 2
    np.testing.assert_allclose(got[:2, 0], [25 + want, 20 + want], rtol=0, atol=1e-7)


def test_heatmap_to_pts_batch_ragged_counts():
    """Three images with 0 points in the middle one: each image refines its own NMS points, counts read on the device."""
    heats = np.stack([synth.unique_heatmap(96, 128, 5), np.zeros((96, 128), np.float32), synth.unique_heatmap(96, 128, 6)])
    x = torch.from_numpy(heats).to(DEV)
    base = S.heatmap_to_pts_batch(x, 0.015, 4)
    for top_k in (None, 7):
        sub = S.heatmap_to_pts_batch(x, 0.015, 4, top_k=top_k, subpixel=True, patch_size=5)
        assert [s.shape[1] for s in sub] == [min(b.shape[1], top_k or 10 ** 9) for b in base]
        assert sub[1].shape[1] == 0 and base[0].shape[1] > 7
        for i in (0, 2):
            ref = SO.soft_argmax_points(heats[i], base[i][:, :sub[i].shape[1]], 5)
            np.testing.assert_allclose(sub[i], ref, rtol=0, atol=TOL)


def test_frontend_binding():
    """dropin.install(frontend_class=...) binds soft_argmax_points(self, pts, patch_size=5): it reads self.heatmap, sets
    self.pts_subpixel and returns a copy of that list; uninstall() restores the reference's method."""
    class Stub:
        def soft_argmax_points(self, pts, patch_size=5):
            return "ref"

    heat = synth.unique_heatmap(120, 160, 11)
    pts = S.getPtsFromHeatmap(heat, 0.015, 4)
    fe = Stub()
    fe.heatmap = torch.from_numpy(heat).to(DEV)[None]  # export.py: fe.heatmap = the aggregated [1,H,W] heatmap
    bound = S.dropin.install(utils_module=types.ModuleType("fake_utils"), frontend_class=Stub)
    try:
        assert any(b.endswith("soft_argmax_points") for b in bound)
        for p in (5, 3):
            out = fe.soft_argmax_points([pts], patch_size=p) if p != 5 else fe.soft_argmax_points([pts])
            assert isinstance(out, list) and len(out) == 1 and out is not fe.pts_subpixel
            assert out[0] is fe.pts_subpixel[0]
            np.testing.assert_allclose(out[0], SO.soft_argmax_points(heat, pts, p), rtol=0, atol=TOL)
        assert not hasattr(fe, "patches")
    finally:
        S.dropin.uninstall()
    assert fe.soft_argmax_points([pts]) == "ref"
