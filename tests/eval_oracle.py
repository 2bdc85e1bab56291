"""numpy float64 restatement of the pair evaluation (utils.evaluate_pairs, csrc/eval.cu) -- test infrastructure.

Repeatability is oracle.ssp_oracle.compute_repeatability (pinned by the live reference's fixture).  The rest restates
evaluation.py of the reference lineage (not pinned by a fixture): RANSAC on the cross-check matches, corner distance and
correctness, matching score, NN mAP.  The RANSAC here takes the drawn quadruples as an input, so it replays the device's
draws; every hypothesis is recomputed from them with the same rules (OpenCV's collinearity and orientation checks, the
partial-pivoting 4-point solve, the inlier test), and the refit is OpenCV's normalised DLT (eigenvector of the smallest
eigenvalue of L^T L), without its Levenberg-Marquardt step."""
import numpy as np

FLT_EPSILON = float(np.finfo(np.float32).eps)
DBL_EPSILON = float(np.finfo(np.float64).eps)


def staged(points):
    """Coordinates as the device stages them for RANSAC: rounded to fp32, computed on in float64."""
    return np.asarray(points, dtype=np.float64).astype(np.float32).astype(np.float64)


def _collinear(x, y):
    """haveCollinearPoints over every triple of the 4 points, x / y [N,4] fp32 values: [N] bool."""
    out = np.zeros(x.shape[0], dtype=bool)
    for i in (2, 3):
        for j in range(1, i):
            for k in range(j):
                dx1 = (x[:, j].astype(np.float32) - x[:, i].astype(np.float32)).astype(np.float64)
                dy1 = (y[:, j].astype(np.float32) - y[:, i].astype(np.float32)).astype(np.float64)
                dx2 = (x[:, k].astype(np.float32) - x[:, i].astype(np.float32)).astype(np.float64)
                dy2 = (y[:, k].astype(np.float32) - y[:, i].astype(np.float32)).astype(np.float64)
                out |= np.abs(dx2 * dy1 - dy2 * dx1) <= FLT_EPSILON * (((np.abs(dx1) + np.abs(dy1)) + np.abs(dx2)) +
                                                                       np.abs(dy2))
    return out


def _det3(xa, ya, xb, yb, xc, yc):
    return (xa * (yb - yc) - ya * (xb - xc)) + (xb * yc - xc * yb)


def _orientation_ok(x1, y1, x2, y2):
    neg = np.zeros(x1.shape[0], dtype=np.int64)
    for a, b, c in ((0, 1, 2), (1, 2, 3), (0, 2, 3), (0, 1, 3)):
        dA = _det3(x1[:, a], y1[:, a], x1[:, b], y1[:, b], x1[:, c], y1[:, c])
        dB = _det3(x2[:, a], y2[:, a], x2[:, b], y2[:, b], x2[:, c], y2[:, c])
        neg += dA * dB < 0
    return (neg == 0) | (neg == 4)


def perspective_transform(x, y, u, v):
    """The 4-point solve of csrc/perspective.cuh for N problems at once ([N,4] each): partial-pivoting elimination of the
    8x9 system, h33 = 1.  Returns [N,9] (non-finite where a pivot is zero)."""
    N = x.shape[0]
    a = np.zeros((N, 8, 9))
    z, o = np.zeros((N, 4)), np.ones((N, 4))
    a[:, 0::2] = np.stack([x, y, o, z, z, z, -u * x, -u * y, u], axis=2)
    a[:, 1::2] = np.stack([z, z, z, x, y, o, -v * x, -v * y, v], axis=2)
    rows = np.arange(N)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for k in range(8):
            p = k + np.argmax(np.abs(a[:, k:, k]), axis=1)  # first maximum, as the strict > of the device loop
            tmp = a[rows, k].copy()
            a[rows, k] = a[rows, p]
            a[rows, p] = tmp
            piv = 1.0 / a[:, k, k]
            f = a[:, k + 1:, k] * piv[:, None]
            a[:, k + 1:, k + 1:] -= f[:, :, None] * a[:, k:k + 1, k + 1:]
        H = np.zeros((N, 9))
        for k in range(7, -1, -1):
            s = a[:, k, 8].copy()
            for c in range(k + 1, 8):
                s -= a[:, k, c] * H[:, c]
            H[:, k] = s / a[:, k, k]
    H[:, 8] = 1.0
    return H


def reprojection_d2(Hs, src, dst):
    """[N,L] squared reprojection distances of the matches under N hypotheses, and the [N,L] mask |w| > FLT_EPSILON."""
    x, y = src[:, 0][None], src[:, 1][None]
    h = [Hs[:, c][:, None] for c in range(9)]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        w = h[6] * x + h[7] * y + h[8]
        ok = np.abs(w) > FLT_EPSILON
        dx = (h[0] * x + h[1] * y + h[2]) / w - dst[:, 0][None]
        dy = (h[3] * x + h[4] * y + h[5]) / w - dst[:, 1][None]
        return dx * dx + dy * dy, ok


def ransac(src, dst, samples, thresh=3.0):
    """RANSAC on matches src -> dst ([L,2] float64, already `staged`) with the given quadruples samples [M,4].
    Returns dict(count [M] (-1: rejected sample), hyps [M,9], d2 [M,L], valid_w [M,L], best, H [3,3] or None, mask [L])."""
    L, M = src.shape[0], samples.shape[0]
    count = np.full(M, -1, dtype=np.int64)
    hyps = np.full((M, 9), np.nan)
    d2 = np.full((M, L), np.inf)
    vw = np.zeros((M, L), dtype=bool)
    if L >= 4:
        s = samples.astype(np.int64)
        x1, y1, x2, y2 = src[s, 0], src[s, 1], dst[s, 0], dst[s, 1]
        ok = ~_collinear(x1, y1) & ~_collinear(x2, y2) & _orientation_ok(x1, y1, x2, y2)
        H = perspective_transform(x1, y1, x2, y2)
        ok &= np.isfinite(H).all(axis=1)
        hyps[ok] = H[ok]
        d2[ok], vw[ok] = reprojection_d2(H[ok], src, dst)
        inl = vw & (d2 <= thresh * thresh)
        count[ok] = inl[ok].sum(axis=1)
    best = int(np.argmax(count)) if M else -1
    res = {"count": count, "hyps": hyps, "d2": d2, "valid_w": vw, "best": best, "H": None, "mask": np.zeros(L, bool)}
    if L < 4 or count[best] < 4:
        res["best"] = -1
        return res
    mask = vw[best] & (d2[best] <= thresh * thresh)
    Hr = normalised_dlt(src[mask], dst[mask])
    if Hr is None:
        res["best"] = -1
        return res
    res["H"], res["mask"] = Hr, mask
    return res


def normalised_dlt(src, dst):
    """OpenCV's homography DLT (HomographyEstimatorCallback::runKernel): per-axis centroid and mean absolute deviation
    normalisation, the eigenvector of the smallest eigenvalue of L^T L, denormalised, h33 = 1.  None when degenerate."""
    src, dst = np.asarray(src, np.float64), np.asarray(dst, np.float64)
    n = src.shape[0]
    cM, cm = src.mean(axis=0), dst.mean(axis=0)
    sM, sm = np.abs(src - cM).sum(axis=0), np.abs(dst - cm).sum(axis=0)
    if (sM < DBL_EPSILON).any() or (sm < DBL_EPSILON).any():
        return None
    sM, sm = n / sM, n / sm
    X, Y = (src[:, 0] - cM[0]) * sM[0], (src[:, 1] - cM[1]) * sM[1]
    x, y = (dst[:, 0] - cm[0]) * sm[0], (dst[:, 1] - cm[1]) * sm[1]
    z, o = np.zeros(n), np.ones(n)
    Lx = np.stack([X, Y, o, z, z, z, -x * X, -x * Y, -x], axis=1)
    Ly = np.stack([z, z, z, X, Y, o, -y * X, -y * Y, -y], axis=1)
    LtL = Lx.T @ Lx + Ly.T @ Ly
    _, V = np.linalg.eigh(LtL)
    H0 = V[:, 0].reshape(3, 3)
    inv2 = np.array([[1 / sm[0], 0, cm[0]], [0, 1 / sm[1], cm[1]], [0, 0, 1]])
    n1 = np.array([[sM[0], 0, -cM[0] * sM[0]], [0, sM[1], -cM[1] * sM[1]], [0, 0, 1]])
    H = inv2 @ H0 @ n1
    H = H / H[2, 2]
    return H if np.isfinite(H).all() else None


def mean_corner_dist(H, Hest, shape):
    """evaluation.py's corner distance: mean over the 4 image corners of ||pi(H c) - pi(Hest c)||; NaN without estimate."""
    if Hest is None:
        return float("nan")
    Hh, W = shape
    c = np.array([[0, 0, 1], [0, Hh - 1, 1], [W - 1, 0, 1], [W - 1, Hh - 1, 1]], dtype=np.float64)
    a, b = c @ np.asarray(H).T, c @ np.asarray(Hest).T
    return float(np.mean(np.linalg.norm(a[:, :2] / a[:, 2:] - b[:, :2] / b[:, 2:], axis=1)))


def depth_ratio(H, shape):
    """min / max of |w| of H at the four image corners: 1 for an affine map, small when the perspective is strong.  With
    ratio >= 0.5 (the depth varies at most 2x over the image) the corner distance is well conditioned: the DLT refit and
    OpenCV's DLT + Levenberg-Marquardt agree to within 1 px there (tests/test_eval_host.py), while below it the corners
    extrapolate far from the points and the two differ by up to ~6 px on the same correspondences."""
    Hh, W = shape
    c = np.array([[0, 0, 1], [0, Hh - 1, 1], [W - 1, 0, 1], [W - 1, Hh - 1, 1]], dtype=np.float64) @ np.asarray(H).T
    return float(np.abs(c[:, 2]).min() / np.abs(c[:, 2]).max())


def backwarp_count(pts2, H, shape):
    """K2': points of image 2 whose warpLabels back-warp (integer truncation, fp32 warp in warp_points_mask_kernel's
    order, filter_points' inclusive bounds) by fp32(H^-1) lies inside the image."""
    if pts2.shape[1] == 0:
        return 0
    h = np.linalg.inv(np.asarray(H, np.float64)).astype(np.float32).reshape(9)
    x = np.trunc(pts2[0]).astype(np.float32)
    y = np.trunc(pts2[1]).astype(np.float32)
    f32 = np.float32

    def row(a, b, c):  # fmaf(b, y, a * x) + c, the fma emulated in float64 (exact product, one rounding)
        return (f32(b) * y.astype(np.float64) + (f32(a) * x).astype(np.float64)).astype(f32) + f32(c)

    Z = row(h[6], h[7], h[8])
    ox, oy = row(h[0], h[1], h[2]) / Z, row(h[3], h[4], h[5]) / Z
    Hh, W = shape
    return int(((ox >= 0) & (ox <= f32(W) - 1) & (oy >= 0) & (oy <= f32(Hh) - 1)).sum())


def average_precision(labels, scores):
    """sklearn's average_precision_score: (1 / #pos) sum over positives i of TP(s >= s_i) / N(s >= s_i); 0 without
    positives."""
    labels, scores = np.asarray(labels, bool), np.asarray(scores, np.float64)
    if not labels.any():
        return 0.0
    ge = scores[None, :] >= scores[labels][:, None]
    return float(np.mean((ge & labels[None, :]).sum(axis=1) / ge.sum(axis=1)))


def gt_labels(pts1, pts2, matches, H, dist=3.0):
    """evaluation.py getInliers: ||pi(H p1) - p2|| < dist for each match."""
    i, j = matches[0].astype(int), matches[1].astype(int)
    p = np.stack([pts1[0, i], pts1[1, i], np.ones(len(i))], axis=1) @ np.asarray(H).T
    w = p[:, :2] / p[:, 2:]
    return np.linalg.norm(w - np.stack([pts2[0, j], pts2[1, j]], axis=1), axis=1) < dist


def match_coords(pts1, pts2, matches):
    i, j = matches[0].astype(int), matches[1].astype(int)
    return staged(np.stack([pts1[0, i], pts1[1, i]], 1)), staged(np.stack([pts2[0, j], pts2[1, j]], 1))


def evaluate_pair(pts1, pts2, H, shape, matches, samples, map_samples=None, keep_k_points=1000, distance_thresh=3,
                  correctness_thresh=(1, 3, 5), map_nn_thresh=1.2, map_inliers="ransac", thresh=3.0):
    """Every metric of one pair from its cross-check matches [3,L] (index 1, index 2, distance) and the device's RANSAC draws
    (samples [M,4] for all matches, map_samples for the mAP matches)."""
    from oracle import ssp_oracle as O
    rep, loc = O.compute_repeatability(pts1.T, pts2.T, H, shape, keep_k_points=keep_k_points,
                                       distance_thresh=distance_thresh)
    src, dst = match_coords(pts1, pts2, matches)
    r = ransac(src, dst, samples, thresh)
    md = mean_corner_dist(H, r["H"], shape)
    K = pts1.shape[1] + backwarp_count(pts2, H, shape)
    score = 2.0 * int(r["mask"].sum()) / K if K else 0.0
    sub = matches[:, matches[2] < map_nn_thresh]
    if map_inliers == "gt":
        lab, r2 = gt_labels(pts1, pts2, sub, H), None
    else:
        r2 = ransac(*match_coords(pts1, pts2, sub), map_samples, thresh)
        lab = r2["mask"]
    ap = average_precision(lab, -sub[2]) if sub.shape[1] else 0.0
    return {"repeatability": rep, "localization_err": loc, "mean_dist": md,
            "correctness": np.array([md <= t for t in correctness_thresh]), "matching_score": score, "ap": ap,
            "homography": r["H"] if r["H"] is not None else np.full((3, 3), np.nan), "inliers": r["mask"],
            "ransac": r, "map_ransac": r2}
