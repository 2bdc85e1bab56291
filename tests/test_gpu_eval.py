"""The pair evaluation on the GPU (csrc/eval.cu, utils.evaluate_pairs, match_step(homographies=...)) against the numpy
oracle (tests/eval_oracle.py, RANSAC replayed from the device's draws), the live reference's repeatability fixture and
OpenCV.  Inputs are seeded synthetic HPatches-like pairs at 480 x 640: a pixel homography from HomographySampler, an
inlier fraction w of the keypoints warped by it plus 0.5 px noise, uniform points for the rest; descriptors are perturbed
copies for the correspondences and random unit vectors otherwise."""

import numpy as np
import pytest
import torch

import eval_oracle as E
import ssp_b200 as S
from ssp_b200 import _lib, synth, utils
from ssp_b200.homography import HomographySampler

pytestmark = pytest.mark.gpu
SHAPE = (480, 640)
M = utils.RANSAC_HYPOTHESES
# px: |mean_dist(ours) - mean_dist(cv2.findHomography(RANSAC))| on well-conditioned pairs (eval_oracle.depth_ratio >= 0.5,
# >= 20 correspondences), calibrated on the CPU by tests/test_eval_host.py::test_oracle_ransac_close_to_opencv
CV_TOL = 1.5
WELL_CONDITIONED_DEPTH_RATIO = 0.5


def pixel_homographies(P, seed):
    hom, _ = HomographySampler(seed, "cuda").sample(P, perspective_amplitude_x=0.2, perspective_amplitude_y=0.2,
                                                    patch_ratio=0.85, allow_artifacts=True)
    return [utils.homography_scaling_torch(hom[p].cpu(), *SHAPE).double().numpy() for p in range(P)]


def unit(x):
    return x / np.linalg.norm(x, axis=0, keepdims=True)


def synthetic_pair(H, w, K, seed, noise=0.5):
    """pts [3,K1], warped_pts [3,K2], desc [256,K1], warped_desc [256,K2]: round(w K) correspondences (integer positions,
    as NMS gives) inside both images."""
    rng = np.random.default_rng(seed)
    src = np.stack([rng.integers(0, SHAPE[1], 8 * K), rng.integers(0, SHAPE[0], 8 * K)], 1).astype(np.float64)
    p = np.c_[src, np.ones(len(src))] @ H.T
    dst = p[:, :2] / p[:, 2:] + rng.normal(0, noise, (len(src), 2))
    ok = (dst[:, 0] >= 0) & (dst[:, 0] < SHAPE[1]) & (dst[:, 1] >= 0) & (dst[:, 1] < SHAPE[0]) & (p[:, 2] > 0)
    n_in = min(int(round(w * K)), int(ok.sum()))
    src, dst = src[ok][:n_in], dst[ok][:n_in]
    out1 = np.stack([rng.integers(0, SHAPE[1], K - n_in), rng.integers(0, SHAPE[0], K - n_in)], 1).astype(np.float64)
    out2 = np.stack([rng.integers(0, SHAPE[1], K - n_in), rng.integers(0, SHAPE[0], K - n_in)], 1).astype(np.float64)
    d = unit(rng.normal(size=(256, K)))
    d2 = np.concatenate([unit(d[:, :n_in] + 0.3 * unit(rng.normal(size=(256, n_in)))), unit(rng.normal(size=(256, K - n_in)))], 1)
    a = np.concatenate([src, out1])
    b = np.concatenate([np.round(dst), out2])
    conf = lambda n: rng.uniform(0.015, 1.0, n)
    perm = rng.permutation(K)
    return (np.c_[a, conf(K)].T, np.c_[b, conf(K)][perm].T, d.astype(np.float32), d2[:, perm].astype(np.float32))


def device_matches(pairs):
    """The cross-check matches of evaluate_pairs (the matcher is deterministic): P arrays [3,L]."""
    K = max(max(p[2].shape[1], p[3].shape[1]) for p in pairs)
    pad = lambda d: np.pad(d, ((0, 0), (0, K - d.shape[1])))
    d1 = torch.from_numpy(np.stack([pad(p[2]) for p in pairs])).cuda()
    d2 = torch.from_numpy(np.stack([pad(p[3]) for p in pairs])).cuda()
    return utils.nn_match_two_way_batch(d1, d2, float("inf"), counts1=[p[2].shape[1] for p in pairs],
                                        counts2=[p[3].shape[1] for p in pairs])


def run_ransac(pairs, matches, n_sets=1, subset_dist=1.2, seed=0):
    """ssp_ransac_homography with its test outputs: dict of numpy arrays."""
    P = len(pairs)
    K = max(max(p[0].shape[1], p[1].shape[1]) for p in pairs)
    R = max(256, (max(m.shape[1] for m in matches) + 255) // 256 * 256)
    pts = np.zeros((2, P, 3, K))
    mm = np.zeros((P, 3, R))
    for p, (a, b, _, _) in enumerate(pairs):
        pts[0, p, :, :a.shape[1]], pts[1, p, :, :b.shape[1]] = a, b
        mm[p, :, :matches[p].shape[1]] = matches[p]
    cu = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    d_pts, d_m = cu(pts), cu(mm)
    nm = cu(np.array([m.shape[1] for m in matches], np.int32))
    n = n_sets * P
    H, ninl, mask, best = (torch.empty((n, 9), dtype=torch.float64, device="cuda"), torch.empty(n, dtype=torch.int32, device="cuda"),
                           torch.empty((n, R), dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.int32, device="cuda"))
    samples = torch.empty((n, M, 4), dtype=torch.int32, device="cuda")
    hyp = torch.empty((n, M), dtype=torch.int32, device="cuda")
    nbytes = _lib.load().ssp_ransac_homography_ws_bytes(n, M)
    ws = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    p_ = _lib.ptr
    _lib.call("ssp_ransac_homography", p_(d_pts[0]), K, p_(d_pts[1]), K, p_(d_m), p_(nm), R, P, n_sets, subset_dist, M, 3.0,
              seed, p_(H), p_(ninl), p_(mask), p_(best), p_(samples), p_(hyp), p_(ws), nbytes, _lib.stream_of(H))
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in dict(H=H, ninl=ninl, mask=mask, best=best, samples=samples, hyp=hyp).items()}


def subset(m, set_, dist=1.2):
    return m if set_ == 0 else m[:, m[2] < dist]


def check_against_oracle(pairs, matches, out, n_sets=1):
    P = len(pairs)
    for q in range(n_sets * P):
        p, set_ = q % P, q // P
        m = subset(matches[p], set_)
        src, dst = E.match_coords(pairs[p][0], pairs[p][1], m)
        L = src.shape[0]
        samp = out["samples"][q]
        r = E.ransac(src, dst, samp)
        if L < 4:
            assert (samp == -1).all() and (out["hyp"][q] == -1).all() and out["best"][q] == -1
            assert np.isnan(out["H"][q]).all() and out["ninl"][q] == 0
            continue
        assert ((samp >= 0) & (samp < L)).all()
        assert all(len(set(s)) == 4 for s in samp.tolist())
        # hypothesis by hypothesis: same rejections; counts equal up to matches within 1e-9 relative of the threshold
        dev, ref = out["hyp"][q].astype(np.int64), r["count"]
        assert np.array_equal(dev == -1, ref == -1)
        near = (np.abs(r["d2"] - 9.0) <= 1e-9 * 9.0).sum(axis=1)
        assert (np.abs(dev - ref) <= near).all(), q
        assert out["best"][q] == r["best"], q
        if r["H"] is None:
            assert np.isnan(out["H"][q]).all()
            continue
        Hr = r["H"].reshape(9)
        assert np.abs(out["H"][q] - Hr).max() <= 1e-9 * np.abs(Hr).max(), (q, out["H"][q], Hr)
        assert out["ninl"][q] == out["mask"][q].sum() == r["mask"].sum()
        assert np.array_equal(out["mask"][q, :L].astype(bool), r["mask"])


def make_pairs(P, seed, w_lo=0.3, w_hi=0.9, K=600):
    Hs = pixel_homographies(P, seed)
    rng = np.random.default_rng(seed)
    ws = rng.uniform(w_lo, w_hi, P)
    return Hs, [synthetic_pair(Hs[p], ws[p], K, 1000 * seed + p) for p in range(P)]


def test_ransac_hypothesis_by_hypothesis():
    Hs, pairs = make_pairs(6, 1)
    matches = device_matches(pairs)
    out = run_ransac(pairs, matches, n_sets=2)
    check_against_oracle(pairs, matches, out, n_sets=2)
    again = run_ransac(pairs, matches, n_sets=2)
    for k in out:
        assert np.array_equal(out[k], again[k], equal_nan=k == "H"), k
    other = run_ransac(pairs, matches, n_sets=2, seed=7)
    assert not np.array_equal(other["samples"], out["samples"])


def test_ransac_finds_h():
    """w >= 0.3: a correct sampler misses an all-inlier sample of 2000 with p < 1e-7; correctness at 3 px on all 32."""
    Hs, pairs = make_pairs(32, 2, 0.3, 0.9)
    matches = device_matches(pairs)
    out = run_ransac(pairs, matches)
    for p in range(32):
        assert E.mean_corner_dist(Hs[p], out["H"][p].reshape(3, 3), SHAPE) <= 3.0, p


def test_ransac_small_and_degenerate():
    """0, 4 and 5 matches; a point repeated (every sample degenerate); all points on one line."""
    Hs, base = make_pairs(1, 3, 0.9, 0.9, K=50)
    a, b, _, _ = base[0]
    m = device_matches(base)[0]
    cases = [m[:, :0], m[:, :4], m[:, :5]]
    dup = m[:, :12].copy()
    dup[0], dup[1] = dup[0, 0], dup[1, 0]
    cases.append(dup)
    line_a = a.copy()
    line_a[1] = 100.0  # every image-1 point on y = 100
    pairs = [base[0]] * 4 + [(line_a, b, None, None)]
    cases.append(m[:, :20])
    out = run_ransac(pairs, cases)
    check_against_oracle(pairs, cases, out)
    assert out["best"][0] == -1 and out["best"][3] == -1 and out["best"][4] == -1
    assert (out["hyp"][3] == -1).all() and (out["hyp"][4] == -1).all()


def test_ransac_against_opencv():
    """64 pairs, w in [0.3, 0.9]; compared on the well-conditioned ones (moderate perspective: under strong perspective the
    corner distance extrapolates far from the points and the DLT refit and OpenCV's LM step differ by several px)."""
    cv2 = pytest.importorskip("cv2")
    Hs, pairs = make_pairs(64, 4, 0.3, 0.9)
    matches = device_matches(pairs)
    out = run_ransac(pairs, matches)
    used = 0
    for p in range(64):
        if E.depth_ratio(Hs[p], SHAPE) < WELL_CONDITIONED_DEPTH_RATIO:
            continue
        used += 1
        src, dst = E.match_coords(pairs[p][0], pairs[p][1], matches[p])
        Hc, _ = cv2.findHomography(src, dst, cv2.RANSAC)
        ours = E.mean_corner_dist(Hs[p], out["H"][p].reshape(3, 3), SHAPE)
        theirs = E.mean_corner_dist(Hs[p], Hc, SHAPE)
        for t in (3.0, 5.0):
            if abs(ours - t) > CV_TOL and abs(theirs - t) > CV_TOL:
                assert (ours <= t) == (theirs <= t), (p, ours, theirs)
        if ours < 5 and theirs < 5:
            assert abs(ours - theirs) <= CV_TOL, (p, ours, theirs)
    assert used >= 24, used


def test_repeatability_golden(golden):
    g = golden("eval_keypoints")
    shape = tuple(int(v) for v in g["shape"])
    P = 1
    kp, wp = g["kp"].T, g["warped_prob"].T
    rng = np.random.default_rng(0)
    d1, d2 = unit(rng.normal(size=(256, kp.shape[1]))), unit(rng.normal(size=(256, wp.shape[1])))
    for k, tag in ((300, ""), (1000, "_1000")):
        r = utils.evaluate_pairs([kp], [wp], [d1], [d2], g["H"][None], shape, keep_k_points=k)
        assert r["repeatability"][0] == float(g["repeatability" + tag])
        np.testing.assert_allclose(r["localization_err"][0], float(g["loc_err" + tag]), rtol=1e-12)


def test_evaluate_pairs_against_oracle_chain():
    """8 pairs, ragged counts, an empty image and a pair with fewer than 4 matches; npz layout for half of them."""
    Hs, pairs = make_pairs(8, 5, 0.3, 0.9)
    K = [600, 350, 900, 3, 600, 0, 800, 120]
    pairs = [tuple(x[:, :K[p]] for x in pr) for p, pr in enumerate(pairs)]
    for mode in ("ransac", "gt"):
        args = ([pr[0] if p % 2 else pr[0].T for p, pr in enumerate(pairs)], [pr[1] for pr in pairs],
                [pr[2] if p % 2 else pr[2].T for p, pr in enumerate(pairs)], [pr[3] for pr in pairs], np.stack(Hs), SHAPE)
        r = utils.evaluate_pairs(*args, map_inliers=mode, seed=3)
        again = utils.evaluate_pairs(*args, map_inliers=mode, seed=3)
        for k in r:
            if k == "inliers":
                assert all(np.array_equal(a, b) for a, b in zip(r[k], again[k]))
            else:
                assert np.array_equal(r[k], again[k], equal_nan=True), k
        matches = device_matches(pairs)
        dev = run_ransac(pairs, matches, n_sets=2, seed=3)
        check_against_oracle(pairs, matches, dev, n_sets=2)
        for p in range(8):
            o = E.evaluate_pair(pairs[p][0], pairs[p][1], Hs[p], SHAPE, matches[p], dev["samples"][p], dev["samples"][8 + p],
                                map_inliers=mode)
            assert r["repeatability"][p] == o["repeatability"], p
            np.testing.assert_allclose(r["localization_err"][p], o["localization_err"], rtol=1e-12)
            np.testing.assert_allclose(r["mean_dist"][p], o["mean_dist"], rtol=1e-7, atol=1e-7)
            assert np.array_equal(r["correctness"][p], o["correctness"]) or abs(o["mean_dist"] - 3) < 1e-6
            assert r["matching_score"][p] == o["matching_score"], p
            np.testing.assert_allclose(r["ap"][p], o["ap"], rtol=1e-12, atol=1e-15)
            assert np.array_equal(r["inliers"][p], o["inliers"])
            np.testing.assert_allclose(r["homography"][p], o["homography"], rtol=1e-9,
                                       atol=1e-9 * np.nanmax(np.abs(o["homography"])) if p not in (3, 5) else 0)
        assert np.isnan(r["mean_dist"][5]) and r["ap"][5] == 0 and r["repeatability"][5] == 0
        assert np.isnan(r["homography"][3]).all() and not r["correctness"][3].any()


def export_inputs(P, seed):
    semi = synth.adaptation_workload(1, 2 * P, 60, 80, seed)[0][0]
    desc = synth.unit_descriptors(P, 256, 60, 80, 31 + seed, smooth=0.4).astype(np.float64)
    dw = desc + 0.5 * synth.unit_descriptors(P, 256, 60, 80, 32 + seed, smooth=0.4)
    dw /= np.sqrt((dw * dw).sum(axis=1, keepdims=True))
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return cu(semi[:P]), cu(desc.astype(np.float32)), cu(semi[P:]), cu(dw.astype(np.float32))


@pytest.mark.parametrize("nn_thresh,top_k", [(0.7, 1000), (3.0, 300)])
def test_match_step_with_homographies(nn_thresh, top_k):
    semi, desc, semi_w, desc_w = export_inputs(3, 0)
    Hs = np.stack(pixel_homographies(3, 9))
    plain = S.step.match_step(semi, desc, semi_w, desc_w, top_k=top_k, nn_thresh=nn_thresh)
    ev = S.step.match_step(semi, desc, semi_w, desc_w, top_k=top_k, nn_thresh=nn_thresh, homographies=Hs, seed=5)
    ref = utils.evaluate_pairs([r["pts"] for r in ev], [r["warped_pts"] for r in ev], [r["desc"] for r in ev],
                               [r["warped_desc"] for r in ev], Hs, SHAPE, seed=5)
    for p in range(3):
        for k in plain[p]:
            assert np.array_equal(plain[p][k], ev[p][k]), k
        for k, v in ref.items():
            assert np.array_equal(np.asarray(ev[p]["metrics"][k]), np.asarray(v[p]), equal_nan=True), k
