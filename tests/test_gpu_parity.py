"""GPU parity tests: the CUDA path (through the C ABI, via the reference-signature Python mirror) against the
oracle on the same seeded inputs, and against the golden vectors of the live reference.

Tolerances (north_star): coordinates / pixels / losses / gradients 1e-4 relative on the fp32-grade engines
("fp32" CUDA cores, "bf16x3" tcgen05 split); the single-pass "bf16" tcgen05 engine is stated separately
(BF16_LOSS_RTOL / cosine); masks and NMS keypoint sets bit-exact (tie pixels allowed where noted).
"""
import numpy as np
import pytest
import torch

import ssp_b200 as S
from oracle import ssp_oracle as O
from ssp_b200 import synth

pytestmark = pytest.mark.gpu
S.losses.CHECK_LIST_OVERFLOW = True
TOL = 1e-4
BF16_LOSS_RTOL = 3e-3   # single-pass bf16 inputs: loss scalars
BF16_GRAD_COS = 0.995   # single-pass bf16 inputs: gradient direction
DEV = "cuda"


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def close(a, b, rtol=TOL, atol=1e-6):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else b
    np.testing.assert_allclose(a.astype(np.float64), np.asarray(b, np.float64), rtol=rtol, atol=atol)


def homographies(n, seed, identity_first=False):
    rng = np.random.default_rng(seed)
    Hs = np.stack([np.linalg.inv(synth.sample_homography(rng)) for _ in range(n)])
    if identity_first:
        Hs[0] = np.eye(3)
    return Hs.astype(np.float32), np.linalg.inv(Hs).astype(np.float32)


# ------------------------------------------------------------------ a1 / a10
def test_warp_points(golden):
    g = golden("warp_points")
    close(S.warp_points(cu(g["pts"]), cu(g["H"]), device=DEV), g["out_batched"])
    close(S.warp_points(cu(g["pts"]), cu(g["H"][1]), device=DEV), g["out_single"])
    # CPU tensors + device="cpu": computed on the GPU, returned on the CPU like the reference
    out = S.warp_points(torch.from_numpy(g["pts"]), torch.from_numpy(g["H"]))
    assert out.device.type == "cpu"
    close(out, g["out_batched"])
    fp, fm = S.filter_points(cu(g["pix"]), torch.tensor([64, 48]), return_mask=True)
    assert np.array_equal(fm.cpu().numpy(), g["filt_mask"]) and np.array_equal(fp.cpu().numpy(), g["filt_pts"])
    Hs, _ = homographies(4, 5)
    pts = (synth.uniform((76800, 2), 3) * 2 - 1).astype(np.float32)
    close(S.warp_points(cu(pts), cu(Hs), device=DEV), O.warp_points(pts, Hs), atol=1e-5)
    w, keep = S.warp_points_filter(cu(g["pix"]), cu(np.eye(3, dtype=np.float32)), (64, 48), device=DEV)
    assert np.array_equal(keep.cpu().numpy(), g["filt_mask"])


def test_warp_keypoints_f64():
    kp = np.stack([synth.uniform((1000,), 1) * 640, synth.uniform((1000,), 2) * 480], 1).astype(np.float64)
    Hpix = np.array([[0.9, 0.05, 12.0], [-0.04, 1.1, -7.0], [1e-4, -2e-4, 1.0]])
    w, keep = S.warp_keypoints(kp, Hpix, shape=(480, 640))
    ref = O.warp_keypoints_f64(kp, Hpix)
    np.testing.assert_allclose(w, ref, rtol=1e-12, atol=1e-9)
    assert np.array_equal(keep, O.keep_in_bounds_f64(ref, (480, 640)))


def test_warp_keypoints_f64_golden_and_repeatability(golden):
    """The float64 evaluation twin against the fixture of the live detector_evaluation module: warped points, and the
    reference's compute_repeatability with the CUDA warp + in-bounds masks plugged in (same repeatability and
    localisation error as the reference returned)."""
    g = golden("eval_keypoints")
    shape = tuple(int(v) for v in g["shape"])
    w, keep = S.warp_keypoints(g["kp"][:, :2], g["H"], shape=shape)
    np.testing.assert_allclose(w, g["warped"], rtol=1e-13, atol=1e-10)
    assert np.array_equal(keep, O.keep_in_bounds_f64(g["warped"], shape))
    for k, tag in ((300, ""), (1000, "_1000")):
        rep, loc = O.compute_repeatability(g["kp"], g["warped_prob"], g["H"], shape, keep_k_points=k,
                                           warp_and_keep=lambda p, Hm, shp: S.warp_keypoints(p, Hm, shape=shp))
        assert rep == float(g["repeatability" + tag])
        np.testing.assert_allclose(loc, float(g["loc_err" + tag]), rtol=1e-12)


# ------------------------------------------------------------------ a2
def assert_only_rounding_ties(out, ref, Hinv, tol=2e-3, max_frac=1e-3):
    """Nearest-mode warps: every pixel that differs from the reference must sit on a half-pixel rounding tie of its
    source coordinate (float64 coordinates within `tol` of k + 0.5, or of the -0.5 / size-0.5 in-bounds edge), and such
    pixels must be rare.  Anything else is a real error."""
    B, C, H, W = ref.shape
    diff = (out != ref).any(axis=1)  # [B,H,W]
    assert diff.mean() < max_frac, diff.mean()
    if not diff.any():
        return
    ix, iy = O.sample_coords_f64((H, W), Hinv)
    fx = np.abs((ix[diff] - np.floor(ix[diff])) - 0.5)
    fy = np.abs((iy[diff] - np.floor(iy[diff])) - 0.5)
    on_tie = np.minimum(fx, fy) < tol
    assert on_tie.all(), "%d of %d differing pixels are not rounding ties (worst distance %.4f px)" % (
        (~on_tie).sum(), diff.sum(), np.minimum(fx, fy).max())


def test_inv_warp_golden(golden):
    g = golden("inv_warp")
    close(S.inv_warp_image_batch(cu(g["img"]), cu(g["Hinv"]), device=DEV), g["out_bilinear"], atol=2e-6)
    on = S.inv_warp_image_batch(cu(g["img"]), cu(g["Hinv"]), device=DEV, mode="nearest").cpu().numpy()
    assert_only_rounding_ties(on, g["out_nearest"], g["Hinv"])
    close(S.inv_warp_image(cu(g["img"][0, 0]), cu(g["Hinv"][0]), device=DEV), g["out_single"], atol=2e-6)
    close(S.inv_warp_image_batch(cu(g["img"][:1]), torch.eye(3, device=DEV), device=DEV), g["out_identity"], atol=2e-6)


def test_inv_warp_240x320():
    _, Hinv = homographies(4, 11)
    img = synth.uniform((4, 1, 240, 320), 5)
    for mode in ("bilinear", "nearest"):
        out = S.inv_warp_image_batch(cu(img), cu(Hinv), device=DEV, mode=mode).cpu().numpy()
        ref = O.inv_warp_image_batch(img, Hinv, mode)
        if mode == "bilinear":
            close(out, ref, atol=1e-4)  # 1-ulp coordinate jitter at |x| ~ 320 on a U[0,1) image
        else:
            assert_only_rounding_ties(out, ref, Hinv)


def test_inv_warp_multichannel_strong_warps():
    """Multi-channel images under identity, magnifying and strongly minifying homographies, and a width that is not a
    multiple of 4, against the oracle in both modes."""
    _, Hinv = homographies(6, 13)
    Hinv[0] = np.eye(3)
    Hinv[1] = np.array([[0.3, 0, 0], [0, 0.3, 0], [0, 0, 1]], np.float32)            # 3.3x magnification
    Hinv[2] = np.array([[3.0, 0.4, 0.1], [-0.5, 2.5, 0], [0.2, 0.1, 1]], np.float32)  # strong minification
    img = synth.uniform((6, 2, 240, 320), 6)
    odd = synth.uniform((2, 1, 47, 61), 7)
    for im, Hm, atol in ((img, Hinv, 1e-4), (odd, Hinv[3:5], 1e-5)):
        out = S.inv_warp_image_batch(cu(im), cu(Hm), device=DEV).cpu().numpy()
        close(out, O.inv_warp_image_batch(im, Hm, "bilinear"), atol=atol)
        out = S.inv_warp_image_batch(cu(im), cu(Hm), device=DEV, mode="nearest").cpu().numpy()
        assert_only_rounding_ties(out, O.inv_warp_image_batch(im, Hm, "nearest"), Hm)


def test_inv_warp_100x240x320_oracle():
    """BASELINE size of the warp (100 views of 240x320), bilinear, against the oracle."""
    _, Hinv = homographies(100, 14)
    img = synth.uniform((100, 1, 240, 320), 8)
    out = S.inv_warp_image_batch(cu(img), cu(Hinv), device=DEV).cpu().numpy()
    close(out, O.inv_warp_image_batch(img, Hinv, "bilinear"), atol=1e-4)


# ------------------------------------------------------------------ a3
def test_valid_mask(golden):
    g = golden("valid_mask")
    for r in range(1, 9):
        assert np.array_equal(S.ellipse_kernel(r), g["ellipse_%d" % r])
    for r in (0, 1, 3):
        m = S.compute_valid_mask(torch.tensor([48, 64]), cu(g["Hinv5"]), device=DEV, erosion_radius=r).cpu().numpy()
        assert set(np.unique(m)) <= {0.0, 1.0}
        assert (m != g["mask_r%d" % r]).sum() <= 2, r
    m = S.compute_valid_mask(torch.tensor([240, 320]), cu(g["Hinv2"]), device=DEV, erosion_radius=3).cpu().numpy()
    assert (m != g["mask_240_r3"]).sum() <= 4
    m = S.compute_valid_mask(torch.tensor([48, 64]), torch.eye(3), device=DEV, erosion_radius=3).cpu().numpy()
    assert np.array_equal(m[0], g["mask_identity_r3"][0])
    _, Hinv = homographies(8, 12)
    m = S.compute_valid_mask(torch.tensor([240, 320]), cu(Hinv), device=DEV, erosion_radius=3).cpu().numpy()
    assert (m != O.compute_valid_mask((240, 320), Hinv, 3)).mean() < 1e-4


# ------------------------------------------------------------------ a4
def test_labels_and_masks(golden):
    g = golden("detector")
    for key, out in (("lab_bin", "l3_bin"), ("lab_soft", "l3_soft"), ("lab_tiny", "l3_tiny")):
        close(S.labels2Dto3D(cu(g[key]), 8, add_dustbin=True), g[out], atol=1e-7)
    close(S.labels2Dto3D(cu(g["lab_bin"]), 8, add_dustbin=False), g["l3_nodust"], atol=0)
    close(S.getMasks(cu(g["mask2d"]), 8, device=DEV), g["mask3d"], atol=0)
    with pytest.raises(ValueError):
        S.labels2Dto3D(cu(g["lab_bin"]), 4)


def test_detector_loss(golden):
    g = golden("detector")
    for semi_k, l3_k, lab_k, loss_k, grad_k, gout in (("semi", "l3_bin", "lab_bin", "loss", "dsemi", 1.0),
                                                      ("semi2", "l3_soft", "lab_soft", "loss2", "dsemi2", 2.5)):
        semi = cu(g[semi_k]).requires_grad_(True)
        loss = S.detector_loss(semi, cu(g[l3_k]), cu(g["mask3d"]))
        close(loss, g[loss_k])
        (loss * gout).backward()
        close(semi.grad, g[grad_k], atol=1e-7)
        semi_f = cu(g[semi_k]).requires_grad_(True)      # fused path from the 2-D maps
        loss_f = S.detector_loss_2d(semi_f, cu(g[lab_k]), cu(g["mask2d"]))
        close(loss_f, g[loss_k])
        (loss_f * gout).backward()
        close(semi_f.grad, g[grad_k], atol=1e-7)


def test_detector_loss_pair(golden):
    """Both losses of a training pair in one launch == the two single-loss launches == the reference."""
    g = golden("detector")
    a = cu(g["semi"]).requires_grad_(True)
    b = cu(g["semi2"]).requires_grad_(True)
    la, lb, cm = S.detector_loss_pair_2d(a, cu(g["lab_bin"]), cu(g["mask2d"]), b, cu(g["lab_soft"]), cu(g["mask2d"]))
    close(la, g["loss"]); close(lb, g["loss2"]); close(cm, g["mask3d"], atol=0)
    (la + 2.5 * lb).backward()
    close(a.grad, g["dsemi"], atol=1e-7); close(b.grad, g["dsemi2"], atol=1e-7)


def test_detector_loss_240x320():
    B = 4
    semi = synth.pseudo_normal((B, 65, 30, 40), 7) * 2
    labels = synth.keypoint_labels(B, 240, 320, 8)
    _, Hinv = homographies(B, 13)
    mask2d = O.compute_valid_mask((240, 320), Hinv, 3)[:, None]
    ref, dref = O.detector_loss(semi, O.labels2Dto3D(labels), O.getMasks(mask2d), grad=True)
    s = cu(semi).requires_grad_(True)
    loss = S.detector_loss_2d(s, cu(labels), cu(mask2d))
    loss.backward()
    close(loss, ref)
    close(s.grad, dref, atol=1e-4 * np.abs(dref).max())


# ------------------------------------------------------------------ a6 / a7
def test_flatten_combine(golden):
    g = golden("flatten")
    close(S.flattenDetection(cu(g["semi"])), g["heat"], atol=1e-7)
    close(S.flattenDetection(cu(g["semi"][0])), g["heat3d"], atol=1e-7)
    c = golden("combine")
    out = S.combine_heatmap(cu(c["heat"]), cu(c["Hwarp"][None]), cu(c["mask"]), device=DEV).cpu().numpy()
    assert out.shape == (1, 48, 64)
    assert np.array_equal(np.isnan(out), np.isnan(c["out"]))
    close(np.nan_to_num(out), np.nan_to_num(c["out"]), atol=2e-6)


def test_combine_heatmap_n100():
    N = 100
    Hs, Hinv = homographies(N, 14, identity_first=True)
    heat = synth.uniform((N, 1, 240, 320), 9) * 0.2
    mask = O.compute_valid_mask((240, 320), Hinv, 0)[:, None]
    ref = O.combine_heatmap(heat, Hs[None], mask)
    out = S.combine_heatmap(cu(heat), cu(Hs[None]), cu(mask), device=DEV).cpu().numpy()
    assert not np.isnan(out).any()
    close(out, ref, atol=2e-6)
    both = S.combine_heatmap_batch(cu(np.stack([heat[:, 0], heat[::-1, 0]])), cu(np.stack([Hs, Hs[::-1]])),
                                   cu(np.stack([mask[:, 0], mask[::-1, 0]]))).cpu().numpy()
    close(both[0], ref[0] if ref.ndim == 3 else ref, atol=2e-6)
    close(both[1], both[0], atol=2e-6)  # same set of views in another order


def test_combine_from_logits_signed_heat():
    """flatten fused with the 0/1 mask (sign = mask) + one-gather aggregation == flattenDetection + float-mask aggregation, bit for
    bit, on a narrow image (5 views of 24x40) and at N = 100; at N = 100 the whole adaptation step returns the same keypoints
    either way, and a soft mask is refused loudly (NaN)."""
    def case(I, N, Hc, Wc, seed_h, seed_s, identity_first):
        Hs, Hinv = homographies(I * N, seed_h, identity_first=identity_first)
        semi = cu(synth.pseudo_normal((I, N, 65, Hc, Wc), seed_s))
        mask = S.compute_valid_mask(torch.tensor([8 * Hc, 8 * Wc]), cu(Hinv), device=DEV).reshape(I, N, 8 * Hc, 8 * Wc)
        return semi, cu(Hs).reshape(I, N, 3, 3), mask

    for semi, Hw, mask in (case(1, 5, 3, 5, 32, 10, False), case(2, 100, 30, 40, 33, 12, True)):
        I, N, _, Hc, Wc = semi.shape
        heat = S.flattenDetection(semi.reshape(I * N, 65, Hc, Wc)).reshape(I, N, 8 * Hc, 8 * Wc)
        ref = S.combine_heatmap_batch(heat, Hw, mask)
        got = S.utils.combine_from_logits_batch(semi, Hw, mask)
        assert torch.equal(torch.nan_to_num(ref, nan=-1.0), torch.nan_to_num(got, nan=-1.0)), (I, N)
    assert torch.isnan(S.utils.combine_from_logits_batch(semi, Hw, mask * 0.5)).all()
    a = S.step.adaptation_step(semi, Hw, mask)
    b = S.step.adaptation_step(semi, Hw, mask, binary_mask=True)
    assert len(a) == len(b) == I
    for pa, pb in zip(a, b):
        assert pa.shape == pb.shape and pa.shape[0] <= 600 and np.array_equal(pa, pb)


# ------------------------------------------------------------------ a8 / a9
def test_nms_golden(golden):
    g = golden("nms")
    for key, (h, w, seed, thr, r) in {"pts_120": (120, 160, 61, 0.015, 4), "pts_240": (240, 320, 62, 0.015, 4),
                                      "pts_64": (64, 96, 63, 0.03, 2)}.items():
        pts = S.getPtsFromHeatmap(synth.unique_heatmap(h, w, seed), thr, r)
        assert pts.dtype == np.float64 and pts.shape == g[key].shape and np.array_equal(pts, g[key]), key
    assert np.array_equal(S.getPtsFromHeatmap(g["sparse"], 0.015, 4), g["pts_sparse"])
    one = np.zeros((48, 64), np.float32); one[20, 30] = 0.5
    assert np.array_equal(S.getPtsFromHeatmap(one, 0.015, 4), g["pts_one"])
    empty = S.getPtsFromHeatmap(np.zeros((48, 64), np.float32), 0.015, 4)
    assert empty.shape == (3, 0)
    out, inds = S.nms_fast(g["corners"], 48, 64, 4)
    assert np.array_equal(out, g["nms_fast_out"]) and np.array_equal(inds, g["nms_fast_inds"])


def test_nms_480x640_and_batch():
    heat = synth.unique_heatmap(480, 640, 77)
    ref = O.getPtsFromHeatmap(heat, 0.015, 4)
    assert np.array_equal(S.getPtsFromHeatmap(heat, 0.015, 4), ref)
    # adversarial: a monotone ramp needs one round per pixel along the chain
    ramp = (np.arange(64 * 96, dtype=np.float32).reshape(64, 96) + 1) / (64 * 96)
    assert np.array_equal(S.getPtsFromHeatmap(ramp, 0.015, 4), O.getPtsFromHeatmap(ramp, 0.015, 4))
    # ties: stable-sort order of the oracle
    tied = np.round(synth.uniform((96, 128), 5) * 8).astype(np.float32) / 8
    assert np.array_equal(S.getPtsFromHeatmap(tied, 0.3, 3), O.getPtsFromHeatmap(tied, 0.3, 3))
    stack = np.stack([synth.unique_heatmap(120, 160, s) for s in (1, 2, 3)])
    outs = S.heatmap_to_pts_batch(cu(stack), 0.015, 4)
    for i in range(3):
        assert np.array_equal(outs[i], O.getPtsFromHeatmap(stack[i], 0.015, 4))


@pytest.mark.parametrize("r", [0, 7, 9, 16, 48])
def test_nms_radii_off_the_benchmark(r):
    """Radii 0 and 9..48 run the stencil kernel, 7 the sliding kernel: getPtsFromHeatmap, heatmap_to_pts_batch and nms_fast
    equal the oracle exactly on a tie-free map and on the tied map above, up to the largest radius nms_fast accepts."""
    tied = np.round(synth.uniform((96, 128), 5) * 8).astype(np.float32) / 8
    maps = ((synth.unique_heatmap(96, 128, 40 + r), 0.015), (tied, 0.3))
    for heat, thr in maps:
        assert np.array_equal(S.getPtsFromHeatmap(heat, thr, r), O.getPtsFromHeatmap(heat, thr, r))
        ys, xs = np.nonzero(heat >= thr)
        corners = np.stack([xs, ys, heat[ys, xs]]).astype(np.float64)
        out, inds = S.nms_fast(corners, 96, 128, r)
        ref, rinds = O.nms_fast(corners, 96, 128, r)
        assert np.array_equal(out, ref) and np.array_equal(inds, rinds)
    outs = S.heatmap_to_pts_batch(cu(np.stack([m for m, _ in maps])), 0.015, r)
    for (heat, _), got in zip(maps, outs):
        assert np.array_equal(got, O.getPtsFromHeatmap(heat, 0.015, r))


def test_box_nms(golden):
    g = golden("box_nms")
    out = S.box_nms(cu(g["prob"]), 4, iou=0.1, min_prob=0.01, keep_top_k=1000)
    assert np.array_equal(out.cpu().numpy(), g["out"])
    with pytest.raises(NotImplementedError):
        S.box_nms(cu(g["prob"]), 4)
    prob = (synth.unique_heatmap(240, 320, 5, hi=1.0) * (synth.uniform((240, 320), 6) < 0.2)).astype(np.float32)
    assert np.array_equal(S.box_nms(cu(prob), 4, keep_top_k=1).cpu().numpy(), O.box_nms(prob, 4))


# ------------------------------------------------------------------ a5
ENGINES = ("fp32", "bf16x3", "bf16")


def run_desc(D, Dw, Hm, mv, g3, engine, **kw):
    Dt, Dwt = cu(D).requires_grad_(True), cu(Dw).requires_grad_(True)
    loss, mask, pos, neg = S.descriptor_loss(Dt, Dwt, cu(Hm), mask_valid=None if mv is None else cu(mv), device=DEV,
                                             lamda_d=250, descriptor_dist=4, lambda_d=800, engine=engine, **kw)
    (g3[0] * loss + g3[1] * pos + g3[2] * neg).backward()
    return loss, mask, pos, neg, Dt.grad, Dwt.grad


def grad_check(got, ref, dots, exact):
    """Gradients away from hinge kinks: rows/columns touching a pair within 1e-5 of a margin are excused."""
    got = got.cpu().numpy()
    scale = np.abs(ref).max()
    if exact:
        near = (np.abs(dots - 0.2) < 1e-5) | (np.abs(dots - 1.0) < 1e-5)
        assert near.mean() < 1e-3
        err = np.abs(got - ref).reshape(ref.shape[0], ref.shape[1], -1)
        bad = err.max(axis=1) > 1e-4 * scale
        return bad
    cos = (got * ref).sum() / np.sqrt((got * got).sum() * (ref * ref).sum())
    assert cos > BF16_GRAD_COS, cos
    return None


@pytest.mark.parametrize("engine", ENGINES)
def test_descriptor_loss_small_golden(golden, engine):
    g = golden("desc_small")
    dots = O.descriptor_dots(g["D"], g["Dw"])
    for tag, g3 in (("a", (1.0, 0.0, 0.0)), ("b", tuple(float(x) for x in g["g_b"]))):
        loss, mask, pos, neg, dD, dDw = run_desc(g["D"], g["Dw"], g["H"], g["mv"], g3, engine)
        rt = TOL if engine != "bf16" else BF16_LOSS_RTOL
        close(loss, g["loss_" + tag], rtol=rt); close(pos, g["pos_" + tag], rtol=rt); close(neg, g["neg_" + tag], rtol=rt)
        assert tuple(mask.shape) == g["mask_" + tag].shape
        assert np.array_equal(mask.materialize().cpu().numpy().astype(np.uint8), g["mask_" + tag])
        exact = engine != "bf16"
        bad_r = grad_check(dD, g["dD_" + tag], dots, exact)
        bad_c = grad_check(dDw, g["dDw_" + tag], dots, exact)
        if exact:
            near = (np.abs(dots - 0.2) < 1e-5) | (np.abs(dots - 1.0) < 1e-5)
            assert not (bad_r.reshape(near.shape[0], -1) & ~near.any(axis=2)).any()
            assert not (bad_c.reshape(near.shape[0], -1) & ~near.any(axis=1)).any()


@pytest.mark.parametrize("engine", ENGINES)
def test_descriptor_loss_30x40(golden, engine):
    g = golden("desc_30x40")
    D = synth.unit_descriptors(1, 256, 30, 40, 91, smooth=0.3)
    Dw = synth.unit_descriptors(1, 256, 30, 40, 92, smooth=0.3)
    S_dbg = torch.zeros((1, 1200, 1200), device=DEV)
    loss, mask, pos, neg, dD, dDw = run_desc(D, Dw, g["H"], g["mv"], (1.0, 1.0, 1.0), engine, debug_S=S_dbg)
    rt = TOL if engine != "bf16" else BF16_LOSS_RTOL
    close(loss, g["loss"], rtol=rt); close(pos, g["pos"], rtol=rt); close(neg, g["neg"], rtol=rt)
    assert np.array_equal(mask.materialize().reshape(1, 1200, 1200).sum(-1).cpu().numpy(), g["mask_rowsum"])
    dots = O.descriptor_dots(D, Dw)
    err = np.abs(S_dbg.cpu().numpy() - dots).max()
    assert err < {"fp32": 2e-6, "bf16x3": 2e-5, "bf16": 2e-2}[engine], err
    scale = np.abs(g["dD_sample"]).max()
    if engine != "bf16":
        d1 = np.abs(dD[0, :, ::7, ::9].cpu().numpy() - g["dD_sample"]).max(axis=0)
        d2 = np.abs(dDw[0, :, ::7, ::9].cpu().numpy() - g["dDw_sample"]).max(axis=0)
        assert (d1 > 2e-4 * scale).mean() < 0.02 and (d2 > 2e-4 * scale).mean() < 0.02  # kink rows only


@pytest.mark.parametrize("engine", ENGINES)
def test_descriptor_identity_kat(golden, engine):
    g = golden("desc_identity")
    D = synth.unit_descriptors(1, 256, 30, 40, 91, smooth=0.3)
    loss, _, pos, neg, _, _ = run_desc(D, D.copy(), np.eye(3, dtype=np.float32)[None], np.ones((1, 1, 30, 40), np.float32),
                                       (1.0, 0.0, 0.0), engine)
    rt = TOL if engine != "bf16" else BF16_LOSS_RTOL
    assert abs(float(pos)) < 1e-6
    close(neg, g["neg"], rtol=rt); close(loss, g["loss"], rtol=rt)


@pytest.mark.parametrize("dist", [2.0, 4.0, 6.0, 7.5, 8.0])
def test_descriptor_dist_values(dist):
    """descriptor_dist from well below cell/2 up to the supported maximum (= cell): the sparse positive lists come from a tight
    candidate window, the returned pair mask from the full predicate -- both must agree with the oracle (loss, pos, neg and the
    gradients through all three), including homographies that shrink (several rows share a partner column)."""
    B, Hc, Wc = 3, 12, 16
    D = synth.unit_descriptors(B, 256, Hc, Wc, 131, smooth=0.3)
    Dw = synth.unit_descriptors(B, 256, Hc, Wc, 132, smooth=0.3)
    Hs, _ = homographies(B, 41)
    Hs[1] = np.array([[0.7, 0.0, 0.05], [0.0, 0.7, -0.05], [0.0, 0.0, 1.0]], np.float32)  # shrink: shared partner columns
    mv = (synth.uniform((B, 1, Hc, Wc), 133) < 0.9).astype(np.float32)
    g3 = (1.0, 0.5, 0.25)
    r_loss, r_mask, r_pos, r_neg, r_dD, r_dDw = O.descriptor_loss(D, Dw, Hs, mv, descriptor_dist=dist, grad=g3, return_mask=True)
    ref = {"loss": r_loss, "mask": r_mask, "pos": r_pos, "neg": r_neg, "dD": r_dD, "dDw": r_dDw}
    for engine in ("fp32", "bf16x3"):
        Dt, Dwt = cu(D).requires_grad_(True), cu(Dw).requires_grad_(True)
        loss, mask, pos, neg = S.descriptor_loss(Dt, Dwt, cu(Hs), mask_valid=cu(mv), device=DEV, descriptor_dist=dist, engine=engine)
        (g3[0] * loss + g3[1] * pos + g3[2] * neg).backward()
        m = mask.materialize().reshape(B, Hc * Wc, Hc * Wc).cpu().numpy()
        assert np.array_equal(m, np.asarray(ref["mask"]).reshape(m.shape)), (engine, dist)
        assert m.sum() > 0
        close(loss, ref["loss"], rtol=TOL); close(pos, ref["pos"], rtol=TOL); close(neg, ref["neg"], rtol=TOL)
        for got, want in ((Dt.grad, ref["dD"]), (Dwt.grad, ref["dDw"])):
            scale = np.abs(want).max()
            err = np.abs(got.cpu().numpy() - want).reshape(B, 256, -1).max(axis=1)
            assert (err > 2e-4 * scale).mean() < 0.02, (engine, dist, float((err > 2e-4 * scale).mean()))  # hinge-kink rows only


def test_descriptor_engines_agree_b32():
    """Full BASELINE size (B=32, 240x320): the three engines agree; size-independent properties hold."""
    B = 32
    D = synth.unit_descriptors(B, 256, 30, 40, 101, smooth=0.3)
    Dw = synth.unit_descriptors(B, 256, 30, 40, 102, smooth=0.3)
    Hs, _ = homographies(B, 21)
    mv = (synth.uniform((B, 1, 30, 40), 103) < 0.9).astype(np.float32)
    res = {e: run_desc(D, Dw, Hs, mv, (1.0, 0.5, 0.25), e) for e in ENGINES}
    for e in ("bf16x3", "bf16"):
        rt = TOL if e == "bf16x3" else BF16_LOSS_RTOL
        for i in (0, 2, 3):
            close(res[e][i], res["fp32"][i].detach().cpu().numpy(), rtol=rt)
        for i in (4, 5):
            a, b = res[e][i].cpu().numpy(), res["fp32"][i].cpu().numpy()
            cos = (a * b).sum() / np.sqrt((a * a).sum() * (b * b).sum())
            assert cos > (0.99999 if e == "bf16x3" else BF16_GRAD_COS), (e, i, cos)
    # oracle on a 2-pair slice of the same batch would use another normaliser; instead check linearity in
    # lamda_d (pos_sum scales, neg_sum does not) and mask_valid = 0 (loss 0, sums unchanged)
    Dt, Dwt = cu(D), cu(Dw)
    l1, _, p1, n1 = S.descriptor_loss(Dt, Dwt, cu(Hs), mask_valid=cu(mv), device=DEV, lamda_d=250)
    l2, _, p2, n2 = S.descriptor_loss(Dt, Dwt, cu(Hs), mask_valid=cu(mv), device=DEV, lamda_d=500)
    close(p2, 2 * p1.cpu().numpy()); close(n2, n1.cpu().numpy())
    zero = torch.zeros((B, 1, 30, 40), device=DEV)
    l0, _, p0, n0 = S.descriptor_loss(Dt, Dwt, cu(Hs), mask_valid=zero, device=DEV, lamda_d=250)
    norm_ratio = (mv.sum() + 1.0) / 1.0
    assert float(l0) == 0.0
    close(p0, p1.cpu().numpy() * norm_ratio, rtol=2e-4); close(n0, n1.cpu().numpy() * norm_ratio, rtol=2e-4)


def test_descriptor_kitti_shape():
    """config 4: 376x1240 -> 47x155 cells (Nc = 7285, not a multiple of anything convenient), B = 1."""
    D = synth.unit_descriptors(1, 256, 47, 155, 111, smooth=0.3)
    Dw = synth.unit_descriptors(1, 256, 47, 155, 112, smooth=0.3)
    Hs, _ = homographies(1, 22)
    mv = (synth.uniform((1, 1, 47, 155), 113) < 0.9).astype(np.float32)
    ref = O.descriptor_loss(D, Dw, Hs, mv)
    # coordinates reach 1240 px (fp32 ulp 1.2e-4): pairs within 1e-3 px of the distance threshold may flip
    slack = O.descriptor_boundary_slack(D, Dw, Hs, mv, eps=1e-3)
    for e in ("bf16x3", "fp32"):
        loss, _, pos, neg = S.descriptor_loss(cu(D), cu(Dw), cu(Hs), mask_valid=cu(mv), device=DEV, engine=e)
        close(loss, ref[0], atol=slack + 1e-9); close(pos, ref[2], atol=slack + 1e-9); close(neg, ref[3], atol=slack + 1e-9)


@pytest.mark.parametrize("Hc,Wc,B,engine", [(30, 40, 32, "bf16x3"), (47, 155, 1, "bf16x3"), (47, 155, 4, "bf16x3"),
                                             (60, 80, 2, "bf16x3"), (60, 80, 1, "fp32")])
def test_descriptor_loss_and_gradients_vs_oracle_baseline_sizes(Hc, Wc, B, engine):
    """BASELINE configs 2 / 4 / 5 against the ORACLE (not engine against engine): loss scalars and both gradients of
    g = (1, 0.5, 0.25) at B = 32 of 240x320, KITTI 376x1240 (47x155 cells, B = 1 and 4) and 480x640 (60x80 cells).
    Cells whose gradient is discontinuous at this input (a pair within 1e-5 of a hinge margin, or within 1e-3 px of the
    distance threshold: oracle.descriptor_unstable_cells) are excused and must stay rare; every other cell has to
    agree to 1e-4 of the gradient scale."""
    seed = Hc * 7 + B
    D = synth.unit_descriptors(B, 256, Hc, Wc, 300 + seed, smooth=0.3)
    Dw = synth.unit_descriptors(B, 256, Hc, Wc, 400 + seed, smooth=0.3)
    Hs, _ = homographies(B, 30 + seed)
    mv = (synth.uniform((B, 1, Hc, Wc), 500 + seed) < 0.9).astype(np.float32)
    g3 = (1.0, 0.5, 0.25)
    ref = O.descriptor_loss(D, Dw, Hs, mv, grad=g3)
    slack = O.descriptor_boundary_slack(D, Dw, Hs, mv, eps=1e-3)
    loss, _, pos, neg, dD, dDw = run_desc(D, Dw, Hs, mv, g3, engine)
    close(loss, ref[0], atol=slack + 1e-9); close(pos, ref[2], atol=slack + 1e-9); close(neg, ref[3], atol=slack + 1e-9)
    rows, cols = O.descriptor_unstable_cells(D, Dw, Hs)
    assert rows.mean() < 0.03 and cols.mean() < 0.03
    Nc = Hc * Wc
    for got, want, unstable in ((dD, ref[4], rows), (dDw, ref[5], cols)):
        got = got.cpu().numpy().reshape(B, 256, Nc)
        want = want.reshape(B, 256, Nc)
        scale = np.abs(want).max()
        err = np.abs(got - want).max(axis=1)  # [B, Nc]
        bad = (err > 1e-4 * scale) & ~unstable
        assert not bad.any(), "%d stable cells off by up to %.3g of the gradient scale" % (bad.sum(), (err * ~unstable).max() / scale)
        # the excused cells are wrong by at most one flipped pair each: still the right order of magnitude
        assert err.max() < 600.0 * scale


def test_descriptor_other_channel_count():
    """Dch != 256 routes to the CUDA-core engine (the tcgen05 kernels are specialised for 256 channels)."""
    D = synth.unit_descriptors(2, 64, 10, 12, 121, smooth=0.3)
    Dw = synth.unit_descriptors(2, 64, 10, 12, 122, smooth=0.3)
    Hs, _ = homographies(2, 23)
    ref = O.descriptor_loss(D, Dw, Hs, None, grad=(1, 0, 0))
    loss, _, pos, neg, dD, dDw = run_desc(D, Dw, Hs, None, (1.0, 0.0, 0.0), "bf16x3")
    close(loss, ref[0]); close(pos, ref[2]); close(neg, ref[3])
    close(dD, ref[4], atol=2e-4 * np.abs(ref[4]).max())


# ------------------------------------------------------------------ boundary behaviour
# ------------------------------------------------------------------ 8f rank 1: semantic head
def _sem_check(lr, lab, ignore=133, gout=1.0, full=False):
    """CUDA sem_loss (fused x8 upsample, or full resolution when full=True) against the oracle, loss and gradient."""
    if full:
        pred = O.upsample_bilinear(lr, lab.shape[1:]).astype(np.float32)
    else:
        pred = lr
    ref, dref = O.sem_loss(pred, lab, ignore_index=ignore, grad=True, gout=gout)
    x = cu(pred).requires_grad_(True)
    loss = S.utils.sem_loss(x, cu(lab), DEV, ignore_index=ignore)
    (loss * gout).backward()
    if np.isnan(ref):
        assert torch.isnan(loss).item() and float(x.grad.abs().max()) == 0.0
        return
    close(loss, ref)
    close(x.grad, dref, atol=1e-4 * max(np.abs(dref).max(), 1e-30))


def test_sem_loss_golden(golden):
    g = golden("semantic")
    for lr_k, lab_k, loss_k, d_k, gout in (("lr", "label", "loss", "dlr", 1.0), ("lr2", "label2", "loss2", "dlr2", 0.7)):
        x = cu(g[lr_k]).requires_grad_(True)
        loss = S.utils.sem_loss(x, cu(g[lab_k]), DEV)          # fused upsample: pred is 1/8 of the label size
        close(loss, g[loss_k])
        (loss * gout).backward()
        close(x.grad, g[d_k], atol=1e-4 * np.abs(g[d_k]).max())
        _sem_check(g[lr_k], g[lab_k], gout=gout, full=True)     # full-resolution kernels on the upsampled logits
    with torch.no_grad():                                       # no-grad forward (validation): GRAD=false kernel
        close(S.utils.sem_loss(cu(g["lr"]), cu(g["label"]), DEV), g["loss"])


def test_sem_loss_shapes_and_edges():
    rng = np.random.default_rng(5)
    for (B, C, hc, wc) in ((2, 133, 30, 40), (1, 133, 47, 155), (1, 7, 3, 13), (2, 64, 5, 11), (1, 256, 2, 2), (1, 2, 1, 1)):
        lr = (synth.pseudo_normal((B, C, hc, wc), 11 + C) * 3).astype(np.float32)
        lab = rng.integers(0, C + 1, (B, hc * 8, wc * 8)).astype(np.int64)   # C = ignore_index here
        lab[:, : hc * 2, : wc * 3] = C
        _sem_check(lr, lab, ignore=C, gout=1.3)
        if B * C * hc * wc < 200000:
            _sem_check(lr, lab, ignore=C, gout=1.3, full=True)
    # nothing counted: loss NaN, gradient 0 (torch's mean over nothing)
    lr = synth.pseudo_normal((1, 133, 4, 5), 3).astype(np.float32)
    _sem_check(lr, np.full((1, 32, 40), 133, np.int64))
    _sem_check(lr, np.full((1, 32, 40), 133, np.int64), full=True)
    # logit spread far beyond the fp32 exponent range between neighbouring cells: the shift bound underflows and the
    # per-pixel exact path takes over
    big = synth.pseudo_normal((1, 133, 4, 5), 4).astype(np.float32)
    big[0, :, ::2, ::2] *= 120.0
    lab = rng.integers(0, 133, (1, 32, 40)).astype(np.int64)
    _sem_check(big, lab)
    # int32 labels and a CPU label tensor are accepted (converted), CPU logits are not
    x = cu(lr).requires_grad_(True)
    l = S.utils.sem_loss(x, torch.from_numpy(lab.astype(np.int32)), DEV)
    close(l, O.sem_loss(lr, lab))
    with pytest.raises(RuntimeError):
        S.utils.sem_loss(torch.from_numpy(lr), torch.from_numpy(lab))
    with pytest.raises(RuntimeError):
        S.utils.sem_loss(cu(lr), cu(lab[:, :30]))               # neither the label size nor 1/8 of it


def test_loss_step_semantic():
    """SSp configuration: detector x2 + descriptor + semantic x2 (BASELINE configs[1]) through loss_step and the graph."""
    B = 2
    rng = np.random.default_rng(9)
    ex = {"semi": cu(synth.pseudo_normal((B, 65, 30, 40), 1)), "semi_warp": cu(synth.pseudo_normal((B, 65, 30, 40), 2)),
          "desc": cu(synth.unit_descriptors(B, 256, 30, 40, 3, smooth=0.3)),
          "desc_warp": cu(synth.unit_descriptors(B, 256, 30, 40, 4, smooth=0.3)),
          "labels_2D": cu(synth.keypoint_labels(B, 240, 320, 5)), "warped_labels": cu(synth.keypoint_labels(B, 240, 320, 6)),
          "mask_2D": cu(np.ones((B, 1, 240, 320), np.float32))}
    Hs, Hinv = homographies(B, 31)
    ex["mask_warp_2D"] = cu(O.compute_valid_mask((240, 320), Hinv, 3)[:, None])
    ex["mat_H"] = cu(Hs)
    base = S.step.loss_step(ex["semi"], ex["semi_warp"], ex["desc"], ex["desc_warp"], ex["labels_2D"], ex["warped_labels"],
                            ex["mask_2D"], ex["mask_warp_2D"], ex["mat_H"])
    sp, spw = synth.pseudo_normal((B, 133, 30, 40), 7) * 2, synth.pseudo_normal((B, 133, 30, 40), 8) * 2
    sem, semw = rng.integers(0, 134, (B, 240, 320)), rng.integers(0, 134, (B, 240, 320))
    ex.update(sem_pred=cu(sp), sem_warp_pred=cu(spw), sem=cu(sem), warped_sem=cu(semw))
    r1, d1 = O.sem_loss(sp, sem, grad=True)
    r2, d2 = O.sem_loss(spw, semw, grad=True)
    leaves = {k: ex[k].clone().requires_grad_(True) for k in ("semi", "semi_warp", "desc", "desc_warp", "sem_pred", "sem_warp_pred")}
    out = S.step.loss_step(leaves["semi"], leaves["semi_warp"], leaves["desc"], leaves["desc_warp"], ex["labels_2D"],
                           ex["warped_labels"], ex["mask_2D"], ex["mask_warp_2D"], ex["mat_H"], sem_pred=leaves["sem_pred"],
                           sem=ex["sem"], sem_warp_pred=leaves["sem_warp_pred"], warped_sem=ex["warped_sem"])
    out["loss"].backward()
    close(out["loss_sem"], r1); close(out["loss_sem_warp"], r2)
    close(out["loss"], float(base["loss"]) + float(r1) + float(r2))
    close(leaves["sem_pred"].grad, d1, atol=1e-4 * np.abs(d1).max())
    close(leaves["sem_warp_pred"].grad, d2, atol=1e-4 * np.abs(d2).max())
    S.losses.CHECK_LIST_OVERFLOW = False   # the check is a host sync, not capturable
    try:
        graphed = S.step.GraphedLossStep(ex)
        res = graphed(ex)
        torch.cuda.synchronize()
    finally:
        S.losses.CHECK_LIST_OVERFLOW = True
    close(res["loss"], out["loss"], rtol=1e-5)
    assert len(res["grads"]) == 6
    close(res["grads"][4], d1, atol=1e-4 * np.abs(d1).max())


# ------------------------------------------------------------------ 8f rank 3: sparse descriptors + matching
def test_sample_desc_and_nn_match(golden):
    g = golden("matching")
    coarse = synth.unit_descriptors(1, 256, 15, 20, 111, smooth=0.5)
    coarse2 = (coarse + 0.35 * synth.unit_descriptors(1, 256, 15, 20, 112, smooth=0.5)).astype(np.float32)
    d1 = S.utils.sample_desc_from_points(cu(coarse), g["pts"])
    d2 = S.utils.sample_desc_from_points(cu(coarse2), g["pts2"])
    assert d1.dtype == np.float32 and d1.shape == (256, 90)
    close(d1, g["desc1"], atol=1e-6); close(d2, g["desc2"], atol=1e-6)
    for thr, key in ((0.36, "matches_36"), (0.7, "matches_70")):
        m = S.utils.nn_match_two_way(g["desc1"], g["desc2"], thr)          # numpy in, like the reference
        assert m.dtype == np.float64 and np.array_equal(m[:2], g[key][:2])
        close(m[2], g[key][2], atol=2e-4)   # sqrt(2 - 2 dot) amplifies fp32 rounding of the dot near dist = 0
        m2 = S.utils.nn_match_two_way(cu(d1), cu(d2), thr)                   # device tensors, own descriptors
        assert np.array_equal(m2[:2], g[key][:2])
    assert S.utils.nn_match_two_way(g["desc1"], g["desc2"][:, :0], 0.7).shape == (3, 0)
    assert S.utils.sample_desc_from_points(cu(coarse), np.zeros((3, 0))).shape == (256, 0)
    # HPatches-size case (BASELINE configs[4]): 1000 x 1000 keypoints at 480x640 against the oracle
    big = synth.unit_descriptors(1, 256, 60, 80, 121, smooth=0.4)
    big2 = (big + 0.5 * synth.unit_descriptors(1, 256, 60, 80, 122, smooth=0.4)).astype(np.float32)
    p1 = np.stack([np.round(synth.uniform((1000,), 123) * 639), np.round(synth.uniform((1000,), 124) * 479), synth.uniform((1000,), 125)])
    p2 = p1[:, ::-1][:, :937].copy()
    e1, e2 = S.utils.sample_desc_from_points(cu(big), p1), S.utils.sample_desc_from_points(cu(big2), p2)
    close(e1, O.sample_desc_from_points(big, p1), atol=1e-6)
    ref = O.nn_match_two_way(e1, e2, 0.7)
    got = S.utils.nn_match_two_way(e1, e2, 0.7)
    same = set(map(tuple, ref[:2].T.astype(int))) ^ set(map(tuple, got[:2].T.astype(int)))
    assert len(same) <= 2 and ref.shape[1] > 300       # near-tie distances may flip between BLAS and the kernel


def test_abi_errors():
    from ssp_b200 import _lib
    lib = _lib.load()
    assert lib.ssp_warp_points_mask(None, 4, None, 1, 0.0, 0.0, None, None, None) < 0
    assert b"null" in lib.ssp_last_error()
    x = torch.zeros((1, 1, 12, 16), device=DEV)
    with pytest.raises(RuntimeError):
        S.labels2Dto3D(torch.zeros((1, 1, 12, 12), device=DEV), 8)   # H, W must be multiples of 8
    with pytest.raises(ValueError):
        S.inv_warp_image_batch(x, torch.eye(3, device=DEV), device=DEV, mode="bicubic")
    with pytest.raises(RuntimeError):
        S.descriptor_loss(torch.zeros((1, 256, 4, 4)), torch.zeros((1, 256, 4, 4)), torch.eye(3)[None])  # CPU tensors


def test_loss_step_and_adaptation_step():
    B = 2
    semi = cu(synth.pseudo_normal((B, 65, 30, 40), 1)).requires_grad_(True)
    semi_w = cu(synth.pseudo_normal((B, 65, 30, 40), 2)).requires_grad_(True)
    D = cu(synth.unit_descriptors(B, 256, 30, 40, 3, smooth=0.3)).requires_grad_(True)
    Dw = cu(synth.unit_descriptors(B, 256, 30, 40, 4, smooth=0.3)).requires_grad_(True)
    Hs, Hinv = homographies(B, 31)
    lab, labw = synth.keypoint_labels(B, 240, 320, 5), synth.keypoint_labels(B, 240, 320, 6)
    m = np.ones((B, 1, 240, 320), np.float32)
    mw = O.compute_valid_mask((240, 320), Hinv, 3)[:, None]
    out = S.step.loss_step(semi, semi_w, D, Dw, cu(lab), cu(labw), cu(m), cu(mw), cu(Hs))
    out["loss"].backward()
    ref_det = O.detector_loss(semi.detach().cpu().numpy(), O.labels2Dto3D(lab), O.getMasks(m))
    ref_detw = O.detector_loss(semi_w.detach().cpu().numpy(), O.labels2Dto3D(labw), O.getMasks(mw))
    ref_desc = O.descriptor_loss(D.detach().cpu().numpy(), Dw.detach().cpu().numpy(), Hs, O.getMasks(mw)[:, None])
    close(out["loss_det"], ref_det); close(out["loss_det_warp"], ref_detw); close(out["loss_desc"], ref_desc[0])
    close(out["loss"], float(ref_det) + float(ref_detw) + float(ref_desc[0]))
    assert all(t.grad is not None and torch.isfinite(t.grad).all() for t in (semi, semi_w, D, Dw))
    # the one-node fused step (default) and the three-node autograd composition give the same values and gradients
    twins = [t.detach().clone().requires_grad_(True) for t in (semi, semi_w, D, Dw)]
    out2 = S.step.loss_step(twins[0], twins[1], twins[2], twins[3], cu(lab), cu(labw), cu(m), cu(mw), cu(Hs), fused=False)
    out2["loss"].backward()
    close(out2["loss"], out["loss"], rtol=1e-6)
    for a, b in zip(twins, (semi, semi_w, D, Dw)):
        close(a.grad, b.grad, rtol=1e-5, atol=1e-6 * float(b.grad.abs().max()))
    assert out2["positive_dist"].requires_grad and not out["positive_dist"].requires_grad
    # homography adaptation, N = 10 views of one image
    N = 10
    Hs, Hinv = homographies(N, 32, identity_first=True)
    semis = synth.pseudo_normal((N, 65, 30, 40), 7) * 3
    masks = O.compute_valid_mask((240, 320), Hinv, 0)
    pts = S.step.adaptation_step(cu(semis), cu(Hs), cu(masks), conf_thresh=0.015, nms_dist=4, top_k=600)[0]
    agg = O.combine_heatmap(O.flattenDetection(semis), Hs[None], masks[:, None])
    ref = O.getPtsFromHeatmap(agg[0] if agg.ndim == 3 else agg, 0.015, 4).transpose()[:600]
    assert pts.shape == ref.shape
    # aggregated heat values differ in the last ulp between CPU and GPU summation: compare the sets
    assert np.array_equal(pts[:, :2], ref[:, :2]) or len(set(map(tuple, pts[:, :2])) ^ set(map(tuple, ref[:, :2]))) <= 4


# ------------------------------------------------------------------ 8f rank 4: label warping / GPU collate
def test_warp_labels_golden(golden):
    """datasets/data_tools.warpLabels of the live reference (fixture), single image and batched, incl. the bilinear label map
    and the last-wins rule for points that land on one pixel."""
    g = golden("warp_labels")
    for i in range(2):
        o = S.warpLabels(g["pts"], 48, 64, torch.from_numpy(g["H"][i]), bilinear=True)
        assert np.array_equal(o["labels"].numpy(), g["labels_%d" % i])
        close(o["warped_pnts"], g["warped_pnts_%d" % i], atol=2e-5)
        close(o["res"], g["res_%d" % i], atol=2e-5)
        close(o["labels_bi"], g["labels_bi_%d" % i], atol=2e-5)
    both = S.warp_labels_batch([g["pts"], g["pts"][:50]], 48, 64, torch.from_numpy(g["H"]), bilinear=True)
    assert np.array_equal(both["labels"][0].cpu().numpy(), g["labels_0"])
    ref1 = O.warp_labels(g["pts"][:50], 48, 64, g["H"][1], bilinear=True)
    assert np.array_equal(both["labels"][1].cpu().numpy(), ref1["labels"])
    close(both["labels_bi"][1], ref1["labels_bi"], atol=2e-5)
    close(both["res"][1], ref1["res"], atol=2e-5)
    close(both["warped_pnts"][1], ref1["warped_pnts"], atol=2e-5)


def test_warp_labels_240x320_collisions_and_collate():
    """BASELINE-size images with 600 keypoints each (top_k of the export) and deliberate duplicates: same maps as the oracle;
    the collate helper returns the reference's batch keys with the right shapes."""
    B, H, W = 4, 240, 320
    Hs, Hinv = homographies(B, 41)
    pts = []
    for b in range(B):
        p = np.stack([np.floor(synth.uniform((600,), 50 + b) * W), np.floor(synth.uniform((600,), 60 + b) * H)], 1)
        p[300:320] = p[:20]  # duplicates: the later copy wins (same value here, but exercises the winner path)
        p[320:330] = p[100:110] + np.array([0.4, 0.3])  # truncated to the same integer pixel as the originals
        pts.append(p)
    out = S.warp_labels_batch(pts, H, W, torch.from_numpy(Hs), bilinear=True)
    for b in range(B):
        ref = O.warp_labels(pts[b], H, W, Hs[b], bilinear=True)
        wp = ref["warped_pnts"].astype(np.float64)
        close(out["warped_pnts"][b], ref["warped_pnts"], atol=2e-4)
        # a warped coordinate within 1e-3 of k + 0.5 (rounding tie) or of an integer (truncation tie of the bilinear base) may
        # legitimately land one pixel over between two fp32 evaluations of the pixel homography: such points are excused
        frac = wp - np.floor(wp)
        ties = int(((np.abs(frac - 0.5) < 1e-3) | (frac < 1e-3) | (frac > 1 - 1e-3)).any(axis=1).sum())
        lab = out["labels"][b].cpu().numpy()
        assert (lab != ref["labels"]).sum() <= 2 * ties
        same = (lab == ref["labels"])[0]
        assert (np.abs(out["res"][b].cpu().numpy() - ref["res"]).max(axis=2)[same] < 2e-4).all()
        bad_bi = np.abs(out["labels_bi"][b].cpu().numpy() - ref["labels_bi"]) > 2e-4
        assert bad_bi.sum() <= 8 * ties
    img = cu(synth.uniform((B, 1, H, W), 70))
    col = S.step.collate_warped_pair(img, pts, torch.from_numpy(Hs), erosion_radius=3, bilinear=True)
    assert col["warped_img"].shape == (B, 1, H, W) and col["warped_res"].shape == (B, 2, H, W)
    assert col["warped_valid_mask"].shape == (B, 1, H, W) and col["warped_labels_bi"].shape == (B, 1, H, W)
    close(col["warped_img"], O.inv_warp_image_batch(img.cpu().numpy(), np.linalg.inv(Hs).astype(np.float32), "bilinear"), atol=1e-4)
    assert torch.equal(col["warped_labels"], out["labels"])


# ------------------------------------------------------------------ 8f rank 2: sparse descriptor loss
def test_sparse_descriptor_loss_golden(golden):
    """Kernels on the index lists of the live reference: its losses and (sampled) gradients; then the drop-in
    batch_descriptor_loss_sparse under the reference's RNG seeds returns the reference's own numbers."""
    g = golden("sparse_loss")
    D = synth.unit_descriptors(3, 256, 30, 40, 151, smooth=0.3)
    Dw = synth.unit_descriptors(3, 256, 30, 40, 152, smooth=0.3)
    Dt, Dwt = cu(D).requires_grad_(True), cu(Dw).requires_grad_(True)
    loss, pos, neg = S.sparse.sparse_loss_from_lists(Dt, Dwt, g["matches_a"], g["matches_b"], g["non_a"], g["non_b"], 250)
    close(loss, g["loss"]); close(pos, g["pos"]); close(neg, g["neg"])
    gv = g["g"]
    (float(gv[0]) * loss + float(gv[1]) * pos + float(gv[2]) * neg).backward()
    scale = np.abs(g["dD_sample"]).max()
    close(Dt.grad[:, :, ::3, ::4], g["dD_sample"], atol=1e-4 * scale); close(Dwt.grad[:, :, ::3, ::4], g["dDw_sample"], atol=1e-4 * scale)
    np.testing.assert_allclose(float(Dt.grad.abs().sum()), float(g["dD_abs_sum"]), rtol=1e-4)
    torch.manual_seed(int(g["seed_torch"]))
    np.random.seed(int(g["seed_numpy"]))
    l2, none, p2, n2 = S.batch_descriptor_loss_sparse(cu(D), cu(Dw), torch.from_numpy(g["H"]), device=DEV, lamda_d=250)
    assert none is None
    close(l2, g["loss"]); close(p2, g["pos"]); close(n2, g["neg"])
    l1 = S.descriptor_loss_sparse(cu(D[0]), cu(Dw[0]), torch.from_numpy(g["H"][0]), device=DEV)
    assert len(l1) == 3 and float(l1[0]) > 0


def test_sparse_descriptor_loss_b32_oracle():
    """BASELINE batch (32 pairs, 30x40 cells, 1000 matches x 10 non-matches each) against the oracle, with gradients."""
    B = 32
    D = synth.unit_descriptors(B, 256, 30, 40, 161, smooth=0.3)
    Dw = synth.unit_descriptors(B, 256, 30, 40, 162, smooth=0.3)
    Hs, _ = homographies(B, 51)
    torch.manual_seed(5)
    np.random.seed(6)
    lists = [S.sparse.sample_correspondences(torch.from_numpy(Hs[i]), 30, 40) for i in range(B)]
    ma, mb, na, nb = (torch.stack([l[j] for l in lists]).numpy() for j in range(4))
    ref = O.sparse_descriptor_loss(D, Dw, ma, mb, na, nb, 250, grad=(1.0, 0.5, 0.25))
    Dt, Dwt = cu(D).requires_grad_(True), cu(Dw).requires_grad_(True)
    loss, pos, neg = S.sparse.sparse_loss_from_lists(Dt, Dwt, ma, mb, na, nb, 250)
    close(loss, ref[0]); close(pos, ref[1]); close(neg, ref[2])
    (loss + 0.5 * pos + 0.25 * neg).backward()
    for got, want in ((Dt.grad, ref[3]), (Dwt.grad, ref[4])):
        close(got, want, atol=1e-4 * np.abs(want).max())
