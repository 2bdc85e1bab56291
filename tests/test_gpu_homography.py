"""The device homography sampler (homography.HomographySampler, ssp_sample_homography) against the reference's sampler
(homography_oracle.sample_homography_np): the law of every component, all components at the training and export parameters,
the structure of a draw, reproducibility from a saved state, and the two step-level users -- step.adaptation_views and
step.collate_warped_pair(sampler=...) -- against the oracle on the homographies they drew.

Distribution tests run at fixed seeds, so their outcome is deterministic; their thresholds are set so that a correct sampler
fails them with probability below 1e-6 (Bonferroni-corrected where one test makes several comparisons).
"""
import numpy as np
import pytest
import torch
from scipy import stats

import homography_oracle as HO
import ssp_b200 as S
from oracle import ssp_oracle as O
from ssp_b200 import synth
from test_gpu_parity import assert_only_rounding_ties

pytestmark = pytest.mark.gpu
P_FAIL = 1e-6
DEV = "cuda"
ONLY = dict(perspective=False, scaling=False, rotation=False, translation=False, allow_artifacts=True)


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def host(t):
    return t.detach().cpu().numpy()


def draw(sampler, B, **params):
    hom, inv = sampler.sample(B, **params)
    torch.cuda.synchronize()
    return host(hom), host(inv)


def ks_ok(x, cdf, n_tests=1):
    p = stats.kstest(x, cdf).pvalue
    assert p > P_FAIL / n_tests, p


# ------------------------------------------------------------------ one component at a time
def test_perspective_only():
    """pd, hl, hr ~ truncnorm(-2, 2, 0, amplitude / 2), read off the corners of the sampled quadrilateral."""
    s = S.HomographySampler(11, DEV)
    hom, _ = draw(s, 20000, **dict(ONLY, perspective=True, perspective_amplitude_x=0.2, perspective_amplitude_y=0.3,
                                  patch_ratio=0.85))
    c = HO.corners(hom)
    m, e = 0.075, 0.925
    hl, hr, pd = c[:, 0, 0] - m, c[:, 2, 0] - e, c[:, 0, 1] - m
    np.testing.assert_allclose(c[:, 1, 0] - m, hl, atol=1e-5)
    np.testing.assert_allclose(c[:, 3, 0] - e, hr, atol=1e-5)
    np.testing.assert_allclose(c[:, 1, 1] - e, -pd, atol=1e-5)
    for x, sd in ((pd, 0.15), (hl, 0.1), (hr, 0.1)):
        ks_ok(x, stats.truncnorm(-2, 2, loc=0, scale=sd).cdf, 3)
    assert stats.spearmanr(hl, hr)[0] ** 2 * len(hl) < stats.chi2.isf(P_FAIL, 1)


def test_scaling_only():
    """Scale 1 with probability 1 / n_scales (the reference's prepended 1), otherwise truncnorm(-2, 2, 1, amplitude / 2)."""
    s = S.HomographySampler(12, DEV)
    B, n_scales = 20000, 5
    hom, _ = draw(s, B, **dict(ONLY, scaling=True, scaling_amplitude=0.2, n_scales=n_scales, patch_ratio=0.85))
    c = HO.corners(hom)
    scale = (c[:, 2, 0] - c[:, 0, 0]) / 0.85
    atom = np.abs(scale - 1) < 2e-6
    k = int(atom.sum())
    assert stats.binom.cdf(k, B, 1 / n_scales) > P_FAIL / 4 and stats.binom.sf(k - 1, B, 1 / n_scales) > P_FAIL / 4, k
    ks_ok(scale[~atom], stats.truncnorm(-2, 2, loc=1, scale=0.1).cdf, 2)
    np.testing.assert_allclose(c.mean(axis=1), 0.5, atol=1e-5)  # about the centre


def test_translation_only():
    """Uniform on [-min(pts2), min(1 - pts2)] per axis: [-margin, margin] for the centred patch."""
    s = S.HomographySampler(13, DEV)
    hom, _ = draw(s, 20000, **dict(ONLY, translation=True, patch_ratio=0.6))
    c = HO.corners(hom)
    t = c[:, 0] - 0.2
    np.testing.assert_allclose(c[:, 2] - 0.8, t, atol=1e-5)
    for ax in range(2):
        ks_ok(t[:, ax], stats.uniform(loc=-0.2, scale=0.4).cdf, 2)
    assert stats.spearmanr(t[:, 0], t[:, 1])[0] ** 2 * len(t) < stats.chi2.isf(P_FAIL, 1)


def rotation_angles(hom, patch_ratio):
    """The reference rotates row vectors by [[cos a, -sin a], [sin a, cos a]] on the right: a clockwise turn by a."""
    c = HO.corners(hom) - 0.5
    h = patch_ratio / 2
    return np.angle(np.exp(-1j * (np.arctan2(c[:, 0, 1], c[:, 0, 0]) - np.arctan2(-h, -h))))


@pytest.mark.parametrize("n_angles", [25, 24])
def test_rotation_only(n_angles):
    """Every angle is one of linspace(-max_angle, max_angle, n_angles), uniformly (chi-square); the reference's appended 0 is
    never chosen, so with an even n_angles no angle is 0."""
    s = S.HomographySampler(14, DEV)
    B = 25000
    hom, _ = draw(s, B, **dict(ONLY, rotation=True, n_angles=n_angles, max_angle=1.57, patch_ratio=0.85))
    a = rotation_angles(hom, 0.85)
    grid = np.linspace(-1.57, 1.57, n_angles)
    idx = np.abs(a[:, None] - grid[None]).argmin(1)
    assert np.abs(a - grid[idx]).max() < 1e-5
    counts = np.bincount(idx, minlength=n_angles)
    assert stats.chisquare(counts).pvalue > P_FAIL, counts
    if n_angles % 2 == 0:
        assert np.abs(a).min() > 0.05


# ------------------------------------------------------------------ all components against the vectorised oracle
@pytest.mark.parametrize("which", ["train", "export"])
def test_all_components_vs_oracle(which):
    """Two-sample KS of the eight corner coordinates against the oracle, Bonferroni-corrected over the eight."""
    params = HO.WARP_PARAMS if which == "train" else HO.EXPORT_PARAMS
    s = S.HomographySampler(15, DEV)
    B = 40000
    hom, _ = draw(s, B, **params)
    np.random.seed(16)
    ref = HO.corners(np.linalg.inv(HO.sample_homography_np(n=B, **params)))
    got = HO.corners(hom)
    for j in range(4):
        for ax in range(2):
            p = stats.ks_2samp(got[:, j, ax], ref[:, j, ax]).pvalue
            assert p > P_FAIL / 8, (j, ax, p)


# ------------------------------------------------------------------ structure
def test_inverse_identities_and_finite():
    s = S.HomographySampler(17, DEV)
    for params in (HO.WARP_PARAMS, HO.EXPORT_PARAMS):
        hom, inv = draw(s, 100000, **params)
        assert np.isfinite(hom).all() and np.isfinite(inv).all()
        prod = np.einsum("nij,njk->nik", inv.astype(np.float64), hom.astype(np.float64))
        assert np.abs(prod - np.eye(3)).max() < 1e-5
    hom, inv = draw(s, 1000, group=100, **HO.WARP_PARAMS)
    eye = np.eye(3, dtype=np.float32)
    for i in range(1000):
        assert np.array_equal(hom[i], eye) == (i % 100 == 0), i
        assert np.array_equal(inv[i], eye) == (i % 100 == 0), i


def test_state_reproduces_and_advances():
    s = S.HomographySampler(123, DEV)
    st = s.get_state()
    assert host(st).tolist() == [123, 0]
    a = draw(s, 300, **HO.WARP_PARAMS)  # three blocks: the last one advances the counter once
    assert host(s.get_state()).tolist() == [123, 1]
    b = draw(s, 300, **HO.WARP_PARAMS)
    assert not np.array_equal(a[0], b[0])
    s.set_state(st)
    for x, y in zip(a + b, draw(s, 300, **HO.WARP_PARAMS) + draw(s, 300, **HO.WARP_PARAMS)):
        assert np.array_equal(x, y)
    assert not np.array_equal(draw(S.HomographySampler(124, DEV), 300, **HO.WARP_PARAMS)[0], a[0])


def test_uncorrelated_with_correspondence_sampler():
    """A DeviceSampler and a HomographySampler with the same seed and launch counter: the non-match cell k of image 0 and
    the first draw of homography k come from different Philox counters (rank correlation of 10 000 pairs)."""
    n = 10000
    d = S.sparse.DeviceSampler(5, DEV)
    _, ib, _ = d.sample(torch.eye(3, device=DEV)[None], 30, 40, 1000, 10)
    h = S.HomographySampler(5, DEV)
    hom, _ = draw(h, n, **dict(ONLY, perspective=True, perspective_amplitude_x=0.2, perspective_amplitude_y=0.2,
                               patch_ratio=0.85))
    pd = HO.corners(hom)[:, 0, 1] - 0.075
    r = stats.spearmanr(host(ib)[0, 1000:1000 + n], pd)[0]
    assert r * r * n < stats.chi2.isf(P_FAIL, 1), r


# ------------------------------------------------------------------ step level, against the oracle on the drawn homographies
def test_adaptation_views_vs_oracle():
    """I = 2 source images, N = 100 views at 240x320 with the export parameters: views against O.inv_warp_image_batch, masks
    against O.compute_valid_mask; then adaptation_step on synthetic logits consumes the result directly (the name swap of
    export.py:284-287) and returns what it returns on the same tensors through the two-array aggregation."""
    I, N, H, W = 2, 100, 240, 320
    img = cu(synth.uniform((I, 1, H, W), 21))
    out = S.step.adaptation_views(img, S.HomographySampler(22, DEV), num=N, **HO.EXPORT_PARAMS)
    torch.cuda.synchronize()
    assert out["image"].shape == (I, N, H, W) and out["valid_mask"].shape == (I, N, H, W)
    hom, inv = host(out["homographies"]), host(out["inv_homographies"])
    assert hom.shape == (I, N, 3, 3) and inv.shape == (I, N, 3, 3)
    for i in range(I):
        assert np.array_equal(hom[i, 0], np.eye(3)) and not np.array_equal(hom[i, 1], np.eye(3))
        views = O.inv_warp_image_batch(np.repeat(host(img)[i:i + 1], N, 0), inv[i], "bilinear")
        np.testing.assert_allclose(host(out["image"][i]), views[:, 0], rtol=0, atol=1e-4)
        mask = O.compute_valid_mask((H, W), inv[i], 0)
        assert_only_rounding_ties(host(out["valid_mask"][i])[:, None], mask[:, None], inv[i])
    semi = cu(synth.pseudo_normal((I, N, 65, H // 8, W // 8), 23) * 3)
    pts = S.step.adaptation_step(semi, out["homographies"], out["valid_mask"], binary_mask=True)
    same = S.step.adaptation_step(semi.clone(), cu(hom), out["valid_mask"].clone(), binary_mask=False)
    for a, b in zip(pts, same):
        assert np.array_equal(a, b)
    agg = O.combine_heatmap(O.flattenDetection(host(semi[0])), hom[0][None], host(out["valid_mask"][0])[:, None])
    ref = O.getPtsFromHeatmap(agg[0] if agg.ndim == 3 else agg, 0.015, 4).transpose()[:600]
    assert len(set(map(tuple, pts[0][:, :2])) ^ set(map(tuple, ref[:, :2]))) <= 4


def test_adaptation_views_graph_replay():
    """adaptation_views captured in a CUDA graph: replay k equals eager call k from the same state bit for bit, and every
    replay draws fresh homographies."""
    I, N, H, W = 2, 100, 240, 320
    img = cu(synth.uniform((I, 1, H, W), 24))
    s = S.HomographySampler(25, DEV)
    S.step.adaptation_views(img, s, num=N, **HO.EXPORT_PARAMS)  # warm-up: grids and module loads
    torch.cuda.synchronize()
    st = s.get_state()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        static = S.step.adaptation_views(img, s, num=N, **HO.EXPORT_PARAMS)
    s.set_state(st)  # capture does not run the kernels, but keep the start explicit
    replays = []
    for _ in range(3):
        g.replay()
        replays.append({k: v.clone() for k, v in static.items()})
    torch.cuda.synchronize()
    s.set_state(st)
    eager = [S.step.adaptation_views(img, s, num=N, **HO.EXPORT_PARAMS) for _ in range(3)]
    torch.cuda.synchronize()
    assert not torch.equal(replays[0]["homographies"], replays[1]["homographies"])
    for k, (r, e) in enumerate(zip(replays, eager)):
        for key in ("image", "valid_mask", "homographies", "inv_homographies"):
            assert torch.equal(r[key], e[key]), (k, key)


def test_collate_warped_pair_with_sampler_vs_oracle():
    """B = 32 training pairs at 240x320: the kernel's inv_homographies against the float64 host inverse of the drawn
    homographies, the warped image, labels and valid mask against the oracle on the drawn homographies."""
    B, H, W = 32, 240, 320
    img = cu(synth.uniform((B, 1, H, W), 31))
    pts = [np.stack([np.floor(synth.uniform((300,), 32 + b) * W), np.floor(synth.uniform((300,), 80 + b) * H)], 1)
           for b in range(B)]
    col = S.step.collate_warped_pair(img, pts, erosion_radius=3, bilinear=True, sampler=S.HomographySampler(33, DEV),
                                     **HO.WARP_PARAMS)
    torch.cuda.synchronize()
    hom, inv = host(col["homographies"]), host(col["inv_homographies"])
    want = np.linalg.inv(hom.astype(np.float64))
    rel = np.abs(inv - want).max(axis=(1, 2)) / np.abs(want).max(axis=(1, 2))
    assert rel.max() < 1e-6, rel.max()
    np.testing.assert_allclose(host(col["warped_img"]), O.inv_warp_image_batch(host(img), inv, "bilinear"), rtol=0,
                               atol=1e-4)
    for b in range(B):
        ref = O.warp_labels(pts[b], H, W, hom[b], bilinear=True)
        wp = ref["warped_pnts"].astype(np.float64)
        frac = wp - np.floor(wp)
        ties = int(((np.abs(frac - 0.5) < 1e-3) | (frac < 1e-3) | (frac > 1 - 1e-3)).any(axis=1).sum())
        lab = host(col["warped_labels"][b])
        assert (lab != ref["labels"]).sum() <= 2 * ties, b
        same = (lab == ref["labels"])[0]
        assert (np.abs(host(col["warped_res"][b]).transpose(1, 2, 0) - ref["res"]).max(axis=2)[same] < 2e-4).all(), b
        assert (np.abs(host(col["warped_labels_bi"][b]) - ref["labels_bi"]) > 2e-4).sum() <= 8 * ties, b
    mask = host(col["warped_valid_mask"])[:, 0]
    assert (mask != O.compute_valid_mask((H, W), inv, 3)).mean() < 1e-4
