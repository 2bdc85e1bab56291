"""Restatement of the reference's sample_homography_np (utils/homographies.py:12-141) at the arguments of its call sites:
shape [2, 2], shift -1, allow_artifacts=True, translation_overflow 0 (the oracle of homography.HomographySampler).

Two details differ from what the reference's own comments suggest, and the live reference's draws in tests/golden pin them:
pts1 is the unit square (not the patch), and the candidate lists are indexed with arange(n), so the prepended scale 1 is
eligible and the last drawn scale is not, and the appended angle 0 is never chosen.

n = 1 makes the reference's exact calls on numpy's global RNG (scipy truncnorm .rvs(1), np.random.randint(n, size=1),
np.random.uniform(low, high, 1)) and reproduces its homographies; n > 1 draws each quantity as an array of n: the same
distribution at vectorised speed, not the same stream.
"""
import numpy as np
from scipy.stats import truncnorm

WARP_PARAMS = dict(translation=True, rotation=True, scaling=True, perspective=True, scaling_amplitude=0.2,
                   perspective_amplitude_x=0.2, perspective_amplitude_y=0.2, patch_ratio=0.85, max_angle=1.57,
                   allow_artifacts=True)  # the training pair (configs' warped_pair.params)
EXPORT_PARAMS = dict(WARP_PARAMS)
del EXPORT_PARAMS["max_angle"]  # the export config leaves max_angle at its default pi / 2


def solve_persp(p1, p2):
    """cv2.getPerspectiveTransform in float64 on [n,4,2] corner arrays -> [n,3,3]."""
    p1, p2 = p1.astype(np.float64), p2.astype(np.float64)
    n = p1.shape[0]
    A = np.zeros((n, 8, 8))
    b = np.zeros((n, 8))
    for i in range(4):
        x, y, u, v = p1[:, i, 0], p1[:, i, 1], p2[:, i, 0], p2[:, i, 1]
        A[:, 2 * i] = np.stack([x, y, np.ones(n), 0 * x, 0 * x, 0 * x, -u * x, -u * y], 1)
        A[:, 2 * i + 1] = np.stack([0 * x, 0 * x, 0 * x, x, y, np.ones(n), -v * x, -v * y], 1)
        b[:, 2 * i], b[:, 2 * i + 1] = u, v
    h = np.linalg.solve(A, b[:, :, None])[:, :, 0]
    return np.concatenate([h, np.ones((n, 1))], 1).reshape(n, 3, 3)


def sample_homography_np(shape=(2, 2), shift=-1, perspective=True, scaling=True, rotation=True, translation=True,
                         n_scales=5, n_angles=25, scaling_amplitude=0.1, perspective_amplitude_x=0.1,
                         perspective_amplitude_y=0.1, patch_ratio=0.5, max_angle=np.pi / 2, allow_artifacts=False,
                         translation_overflow=0., n=1):
    """[3,3] for n = 1 (the reference's return value), else [n,3,3]: the sampled transform of pts1 onto pts2, before the
    callers' inversion."""
    assert allow_artifacts and translation_overflow == 0 and list(shape) == [2, 2] and shift == -1
    pts1 = np.array([[0., 0.], [0., 1.], [1., 1.], [1., 0.]])
    margin = (1 - patch_ratio) / 2
    pts2 = np.repeat((margin + np.array([[0, 0], [0, patch_ratio], [patch_ratio, patch_ratio], [patch_ratio, 0]]))[None],
                     n, 0)
    if perspective:
        ty = truncnorm(-2, 2, loc=0, scale=perspective_amplitude_y / 2)
        tx = truncnorm(-2, 2, loc=0, scale=perspective_amplitude_x / 2)
        pd, hl, hr = ty.rvs(n), tx.rvs(n), tx.rvs(n)
        pts2 += np.stack([np.stack([hl, pd], 1), np.stack([hl, -pd], 1), np.stack([hr, pd], 1), np.stack([hr, -pd], 1)], 1)
    if scaling:
        ts = truncnorm(-2, 2, loc=1, scale=scaling_amplitude / 2)
        scales = np.concatenate([np.ones((n, 1)), ts.rvs(n * n_scales).reshape(n, n_scales)], 1)
        center = np.mean(pts2, axis=1, keepdims=True)
        s = scales[np.arange(n), np.random.randint(n_scales, size=n)]
        pts2 = (pts2 - center) * s[:, None, None] + center
    if translation:
        t_min, t_max = np.min(pts2, axis=1), np.min(1 - pts2, axis=1)
        pts2 += np.stack([np.random.uniform(-t_min[:, 0], t_max[:, 0], n), np.random.uniform(-t_min[:, 1], t_max[:, 1], n)],
                         1)[:, None, :]
    if rotation:
        angles = np.concatenate([np.linspace(-max_angle, max_angle, num=n_angles), [0.]])
        a = angles[np.random.randint(n_angles, size=n)]
        center = np.mean(pts2, axis=1, keepdims=True)
        rot = np.stack([np.cos(a), -np.sin(a), np.sin(a), np.cos(a)], 1).reshape(n, 2, 2)
        pts2 = np.matmul(pts2 - center, rot) + center
    H = solve_persp(np.float32(pts1 * 2 - 1)[None].repeat(n, 0), np.float32(pts2 * 2 - 1))
    return H[0] if n == 1 else H


def dataset_homographies(n, seed, params=WARP_PARAMS, identity_first=False):
    """What tests/golden/make_golden.py stores: n draws under np.random.seed(seed), inverted like datasets/Coco.py:345
    (identity first like Coco.py:271); returns fp32 (homographies, inv_homographies)."""
    np.random.seed(seed)
    Hs = np.linalg.inv(np.stack([sample_homography_np(**params) for _ in range(n)]))
    if identity_first:
        Hs[0] = np.eye(3)
    return Hs.astype(np.float32), np.linalg.inv(Hs).astype(np.float32)


def corners(homographies):
    """The sampled corners pts2 (unit-square coordinates, [n,4,2]) recovered from the callers' homographies: their inverse
    maps the corners of [-1, 1]^2 onto 2 pts2 - 1."""
    Hd = np.linalg.inv(np.asarray(homographies, np.float64))
    c = np.array([[-1., -1., 1.], [-1., 1., 1.], [1., 1., 1.], [1., -1., 1.]])
    w = np.einsum("nij,kj->nki", Hd, c)
    return (w[..., :2] / w[..., 2:] + 1) / 2
