"""The pair evaluation without a GPU: argument checks of its three entry points and of utils.evaluate_pairs (all raised
before any CUDA call), and the numpy oracle's AP and DLT refit against sklearn and OpenCV."""
import ctypes

import numpy as np
import pytest

import eval_oracle as E
from ssp_b200 import _lib, synth, utils

p = ctypes.c_void_p(16)


def test_ransac_argument_errors():
    lib = _lib.load()
    nbytes = lib.ssp_ransac_homography_ws_bytes(2, 2000)
    assert nbytes == 2 * 2000 * (9 * 8 + 4)
    ok = [p, 1000, p, 1000, p, p, 1024, 1, 2, 1.2, 2000, 3.0, 0, p, p, p, p, None, None, p, nbytes, None]

    def err(i, v, text):
        args = list(ok)
        args[i] = v
        assert lib.ssp_ransac_homography(*args) < 0
        assert text in lib.ssp_last_error()

    err(0, None, b"null pointer")
    err(5, None, b"null pointer")
    err(6, 8193, b"the limit is 8192")
    err(10, 0, b"hypotheses")
    err(10, -5, b"hypotheses")
    err(8, 3, b"n_sets")
    err(11, 0.0, b"threshold")
    err(20, nbytes - 1, b"workspace too small")


def test_eval_entry_point_argument_errors():
    lib = _lib.load()
    assert lib.ssp_eval_repeatability(p, 1000, p, p, 1000, None, 1000, 4, p, 480, 640, 1000, 3.0, p, None) < 0
    assert b"null pointer" in lib.ssp_last_error()
    assert lib.ssp_eval_repeatability(p, 1000, p, p, 1000, p, 1000, 4, p, 480, 640, 0, 3.0, p, None) < 0
    assert b"keep_k" in lib.ssp_last_error()
    assert lib.ssp_eval_repeatability(p, 9000, p, p, 9000, p, 9000, 4, p, 480, 640, 9000, 3.0, p, None) < 0
    assert b"shared memory" in lib.ssp_last_error()
    assert lib.ssp_eval_repeatability(p, 1000, p, p, 900, p, 1000, 4, p, 480, 640, 1000, 3.0, p, None) < 0
    assert b"exceeds a point capacity" in lib.ssp_last_error()
    thr = (ctypes.c_double * 3)(1, 3, 5)
    args = [p, 1000, p, p, 1000, p, 1000, 4, p, 480, 640, p, p, 1024, 1.2, p, p, p, 0, thr, 3, p, None]
    for i, v, text in ((6, 1001, b"exceeds a point capacity"), (12, None, b"null pointer"), (13, 8448, b"the limit is 8192"), (20, 9, b"correctness thresholds"),
                       (18, 2, b"map_gt"), (19, None, b"null pointer")):
        a = list(args)
        a[i] = v
        assert lib.ssp_eval_match_metrics(*a) < 0, i
        assert text in lib.ssp_last_error()


def pair(K1=5, K2=6):
    rng = np.random.default_rng(K1 * 7 + K2)
    return (np.c_[rng.uniform(0, 60, (K1, 2)), rng.uniform(0, 1, (K1, 1))].T,
            np.c_[rng.uniform(0, 60, (K2, 2)), rng.uniform(0, 1, (K2, 1))].T,
            rng.normal(size=(256, K1)), rng.normal(size=(256, K2)))


def test_evaluate_pairs_argument_errors():
    a, b, da, db = pair()
    H = np.eye(3)[None]
    with pytest.raises(ValueError, match="map_inliers"):
        utils.evaluate_pairs([a], [b], [da], [db], H, (64, 64), map_inliers="cv")
    with pytest.raises(ValueError, match="1 to 8 thresholds"):
        utils.evaluate_pairs([a], [b], [da], [db], H, (64, 64), correctness_thresh=tuple(range(1, 10)))
    with pytest.raises(ValueError, match="keep_k_points"):
        utils.evaluate_pairs([a], [b], [da], [db], H, (64, 64), keep_k_points=0)
    with pytest.raises(ValueError, match="neither"):
        utils.evaluate_pairs([a], [b], [da[:, :4]], [db], H, (64, 64))
    with pytest.raises(ValueError, match="P > 0"):
        utils.evaluate_pairs([a], [b, b], [da], [db], H, (64, 64))
    with pytest.raises(ValueError, match="homographies for"):
        utils.evaluate_pairs([a], [b], [da], [db], np.eye(3)[None].repeat(2, 0), (64, 64))
    big = np.zeros((3, 8193))
    with pytest.raises(ValueError, match="at most 8192"):
        utils.evaluate_pairs([big], [b], [np.zeros((256, 8193))], [db], H, (64, 64))


def test_oracle_ap_equals_sklearn():
    metrics = pytest.importorskip("sklearn.metrics")
    rng = np.random.default_rng(3)
    for t in range(200):
        n = int(rng.integers(1, 60))
        scores = rng.integers(0, 6, n).astype(np.float64) * 0.25  # many ties
        labels = rng.random(n) < rng.uniform(0.05, 0.95)
        if not labels.any():
            assert E.average_precision(labels, scores) == 0.0
            continue
        assert abs(E.average_precision(labels, scores) - metrics.average_precision_score(labels, scores)) < 1e-12, t


def in_image_correspondences(rng, n, noise, shape=(480, 640)):
    """n source points uniform in the image whose true warps land inside image 2 (and in front of the camera), the
    warps plus Gaussian noise, and the pixel homography."""
    Hn = np.linalg.inv(synth.sample_homography(rng))
    H = utils.homography_scaling(Hn, shape[0], shape[1])
    src = np.stack([rng.uniform(0, shape[1], 4 * n), rng.uniform(0, shape[0], 4 * n)], 1)
    w = np.c_[src, np.ones(len(src))] @ H.T
    dst = w[:, :2] / w[:, 2:]
    k = (dst[:, 0] >= 0) & (dst[:, 0] < shape[1]) & (dst[:, 1] >= 0) & (dst[:, 1] < shape[0]) & (w[:, 2] > 0)
    src, dst = src[k][:n], dst[k][:n]
    return src, dst + rng.normal(0, noise, dst.shape), H


def test_oracle_refit_exact():
    rng = np.random.default_rng(11)
    done = 0
    while done < 50:
        src, dst, H = in_image_correspondences(rng, 40, 0.0)
        if len(src) < 8:
            continue
        Ho = E.normalised_dlt(src, dst)
        np.testing.assert_allclose(Ho, H / H[2, 2], rtol=1e-9, atol=1e-9 * np.abs(H / H[2, 2]).max())
        done += 1


# the regime where the corner distance compares estimators: moderate perspective and enough correspondences
WELL_CONDITIONED_DEPTH_RATIO = 0.5
WELL_CONDITIONED_POINTS = 20


def test_oracle_refit_close_to_opencv():
    """0.5 px noise, 8 to 400 in-image correspondences of synth.sample_homography pairs at 480 x 640 (seeds 0-9, 3000
    draws): the normalised DLT against cv2.findHomography(src, dst, 0) (the same DLT followed by 10 Levenberg-Marquardt
    iterations), by the mean corner distance between the two estimates, on the cases where both lie within 5 px of the truth.
    In the well-conditioned regime (eval_oracle.depth_ratio >= 0.5, >= 20 correspondences) this loop measures, with opencv
    4.13, at most 0.773 px apart over 1976 cases (median 0.044 px); the same recipe on seeds 20-39 gave at most 0.815 px
    over 3874 cases.  Bound 1.0 px.  Outside the regime the difference is not usefully bounded (up to 4.06 px in this loop,
    5.76 px on seeds 20-39: under strong perspective the corners extrapolate far from the points), so comparisons against
    OpenCV are restricted to it."""
    cv2 = pytest.importorskip("cv2")
    worst, used = 0.0, 0
    for seed in range(10):
        rng = np.random.default_rng(seed)
        for _ in range(300):
            src, dst, H = in_image_correspondences(rng, int(rng.integers(8, 400)), 0.5)
            if len(src) < WELL_CONDITIONED_POINTS or E.depth_ratio(H, (480, 640)) < WELL_CONDITIONED_DEPTH_RATIO:
                continue
            Ho = E.normalised_dlt(src, dst)
            Hc, _ = cv2.findHomography(src, dst, 0)
            if E.mean_corner_dist(H, Ho, (480, 640)) < 5 and E.mean_corner_dist(H, Hc, (480, 640)) < 5:
                worst = max(worst, E.mean_corner_dist(Hc, Ho, (480, 640)))
                used += 1
    assert used > 1500 and worst < 1.0, (used, worst)


def ransac_pair(rng, w, K=600, shape=(480, 640)):
    """A pair like tests/test_gpu_eval.py's: integer keypoints, true correspondences warped with 0.5 px noise and rounded,
    a fraction 1 - w of unrelated matches.  Returns (H, src [L,2], dst [L,2], number of true correspondences)."""
    Hn = np.linalg.inv(synth.sample_homography(rng, perspective_amplitude_x=0.2, perspective_amplitude_y=0.2,
                                               patch_ratio=0.85))
    H = utils.homography_scaling(Hn, shape[0], shape[1])
    src = np.stack([rng.integers(0, shape[1], 8 * K), rng.integers(0, shape[0], 8 * K)], 1).astype(np.float64)
    p = np.c_[src, np.ones(len(src))] @ H.T
    dst = p[:, :2] / p[:, 2:] + rng.normal(0, 0.5, (len(src), 2))
    ok = (dst[:, 0] >= 0) & (dst[:, 0] < shape[1]) & (dst[:, 1] >= 0) & (dst[:, 1] < shape[0]) & (p[:, 2] > 0)
    n_in = min(int(round(w * K * 0.7)), int(ok.sum()))
    n_out = int(round(n_in * (1 - w) / w))
    rand = lambda n: np.stack([rng.integers(0, shape[1], n), rng.integers(0, shape[0], n)], 1).astype(np.float64)
    return H, np.r_[src[ok][:n_in], rand(n_out)], np.r_[np.round(dst[ok][:n_in]), rand(n_out)], n_in


def test_oracle_ransac_close_to_opencv():
    """The RANSAC of tests/test_gpu_eval.py's OpenCV comparison, calibrated here: the oracle's RANSAC (the device's rules,
    2000 quadruples drawn with numpy) against cv2.findHomography(src, dst, cv2.RANSAC), 600 seeded pairs with inlier
    fraction w in [0.3, 0.9], by |mean_dist(ours) - mean_dist(cv2)| on the well-conditioned pairs where both are below 5 px.
    Measured with opencv 4.13: this loop gives at most 0.524 px over 391 pairs (median 0.028 px); an independent 600-pair
    run with other draws gave at most 1.11 px over 413 pairs.  Bound 1.5 px, the CV_TOL of tests/test_gpu_eval.py.  The two
    estimators differ by their draws, the LM step and, through both, the inlier sets."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(0)
    worst, used = 0.0, 0
    for _ in range(600):
        H, src, dst, n_in = ransac_pair(rng, rng.uniform(0.3, 0.9))
        if n_in < WELL_CONDITIONED_POINTS or E.depth_ratio(H, (480, 640)) < WELL_CONDITIONED_DEPTH_RATIO:
            continue
        samples = np.stack([rng.choice(len(src), 4, replace=False) for _ in range(2000)])
        r = E.ransac(E.staged(src), E.staged(dst), samples)
        Hc, _ = cv2.findHomography(src, dst, cv2.RANSAC)
        ours, theirs = E.mean_corner_dist(H, r["H"], (480, 640)), E.mean_corner_dist(H, Hc, (480, 640))
        if ours < 5 and theirs < 5:
            worst = max(worst, abs(ours - theirs))
            used += 1
    assert used > 300 and worst < 1.5, (used, worst)


def test_oracle_ransac_rules():
    """The sample checks on hand-made quadruples: a collinear triple and a flipped orientation are rejected; a proper
    sample solves exactly."""
    src = np.array([[0, 0], [10, 0], [0, 10], [10, 10], [20, 0], [5, 5]], np.float64)
    H = np.array([[1.1, 0.05, 3], [-0.02, 0.95, -2], [1e-4, 2e-5, 1]])
    w = np.c_[src, np.ones(6)] @ H.T
    dst = E.staged(w[:, :2] / w[:, 2:])
    samples = np.array([[0, 1, 2, 3], [0, 1, 4, 2], [0, 3, 5, 1], [0, 1, 3, 2]])
    r = E.ransac(src, dst, samples)
    assert r["count"][1] == -1 and r["count"][2] == -1  # (0,1,4) and (0,3,5) collinear
    assert r["count"][0] == 6 and r["count"][3] == 6 and r["best"] == 0
    flip = dst.copy()
    flip[3] = dst[2]
    flip[2] = dst[3]  # swapping two targets breaks the orientation test
    assert E.ransac(src, flip, samples[:1])["count"][0] == -1
