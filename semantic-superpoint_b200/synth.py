"""Synthetic input generators shared by tests and bench.py (SURVEY 8d).  numpy only, no product logic.

splitmix64-based generators are pure integer arithmetic, hence bit-identical on every machine: golden
fixtures for large cases store only outputs and regenerate their inputs from a seed.
"""
import numpy as np


def _splitmix64(idx):
    z = (idx + np.uint64(0x9E3779B97F4A7C15)).astype(np.uint64)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def uniform(shape, seed):
    """U[0,1) float32 array, bit-reproducible (24 random mantissa bits per element)."""
    n = int(np.prod(shape))
    with np.errstate(over="ignore"):
        idx = np.arange(n, dtype=np.uint64) + np.uint64(seed) * np.uint64(0x100000001B3)
        bits = _splitmix64(idx) >> np.uint64(40)
    return (bits.astype(np.float32) / np.float32(1 << 24)).reshape(shape)


def pseudo_normal(shape, seed):
    """Zero-mean, roughly unit-variance values from the sum of four uniforms (exact arithmetic, reproducible)."""
    u = sum(uniform(shape, seed * 4 + k).astype(np.float64) for k in range(4))
    return ((u - 2.0) * np.sqrt(3.0)).astype(np.float32)


def unit_descriptors(B, Dch, Hc, Wc, seed, smooth=0.0):
    """[B,Dch,Hc,Wc] float32, L2-normalised over channels (like the descriptor head, SuperPointNet_gauss2.py:64-65).
    smooth in [0,1) mixes in a shared component so that many pairs exceed the 0.2 negative margin."""
    x = pseudo_normal((B, Dch, Hc, Wc), seed).astype(np.float64)
    if smooth > 0:
        shared = pseudo_normal((B, Dch, 1, 1), seed + 7919).astype(np.float64)
        x = (1 - smooth) * x + smooth * shared
    x /= np.sqrt((x * x).sum(axis=1, keepdims=True))
    return x.astype(np.float32)


def keypoint_labels(B, H, W, seed, p=0.005):
    """Bernoulli(p) binary keypoint maps [B,1,H,W]."""
    return (uniform((B, 1, H, W), seed) < p).astype(np.float32)


def unique_heatmap(H, W, seed, hi=0.05):
    """Tie-free heatmap in [0, hi): a random permutation of H*W distinct fp32 levels."""
    key = uniform((H * W,), seed).astype(np.float64) + np.arange(H * W) * 1e-12
    order = np.argsort(key, kind="stable")
    vals = (np.arange(H * W, dtype=np.float64) + 0.5) / (H * W) * hi
    out = np.empty(H * W, np.float32)
    out[order] = vals.astype(np.float32)
    assert len(np.unique(out)) == H * W
    return out.reshape(H, W)


def sample_homography(rng, shift=-1, perspective=True, scaling=True, rotation=True, translation=True, n_scales=5,
                      n_angles=25, scaling_amplitude=0.2, perspective_amplitude_x=0.2, perspective_amplitude_y=0.2,
                      patch_ratio=0.85, max_angle=1.57, allow_artifacts=True):
    """Random homography in [-1,1]^2 coordinates in the manner of utils/homographies.py:12-141
    (sample_homography_np): perspective / scale / translation / rotation of a centred patch, then the
    4-point transform.  Input generation only; uses `rng` (numpy Generator) instead of scipy.truncnorm."""
    def tnorm(scale, size=None):
        v = rng.normal(0.0, scale, size=size)
        return np.clip(v, -2 * scale, 2 * scale)

    margin = (1 - patch_ratio) / 2
    pts1 = margin + np.array([[0, 0], [0, patch_ratio], [patch_ratio, patch_ratio], [patch_ratio, 0]], dtype=np.float64)
    pts2 = pts1.copy()
    if perspective:
        if not allow_artifacts:
            perspective_amplitude_x = min(perspective_amplitude_x, margin)
            perspective_amplitude_y = min(perspective_amplitude_y, margin)
        pd = tnorm(perspective_amplitude_y / 2)
        hl = tnorm(perspective_amplitude_x / 2)
        hr = tnorm(perspective_amplitude_x / 2)
        pts2 += np.array([[hl, pd], [hl, -pd], [hr, pd], [hr, -pd]])
    if scaling:
        scales = np.concatenate([1 + tnorm(scaling_amplitude / 2, n_scales), [1.0]])
        center = pts2.mean(axis=0, keepdims=True)
        scaled = (pts2 - center)[None] * scales[:, None, None] + center
        valid = np.arange(n_scales + 1) if allow_artifacts else np.where(
            ((scaled >= 0) & (scaled < 1)).all(axis=(1, 2)))[0]
        pts2 = scaled[valid[rng.integers(0, len(valid))]]
    if translation:
        t_min, t_max = pts2.min(axis=0), (1 - pts2).min(axis=0)  # translation_overflow = 0 (homographies.py:100-105)
        lo, hi = -t_min, t_max  # like numpy's legacy uniform, lo > hi is allowed (artifacts enabled)
        pts2 += (lo + (hi - lo) * rng.random(2))[None]
    if rotation:
        angles = np.concatenate([np.linspace(-max_angle, max_angle, n_angles), [0.0]])
        center = pts2.mean(axis=0, keepdims=True)
        rot = np.stack([np.cos(angles), -np.sin(angles), np.sin(angles), np.cos(angles)], axis=1).reshape(-1, 2, 2)
        rotated = np.matmul((pts2 - center)[None], rot) + center
        valid = np.arange(n_angles + 1) if allow_artifacts else np.where(
            ((rotated >= 0) & (rotated < 1)).all(axis=(1, 2)))[0]
        pts2 = rotated[valid[rng.integers(0, len(valid))]]
    # [0,1]^2 patch coordinates -> [-1,1]^2 (the reference's shape=[2,2], shift=-1)
    pts1 = pts1 * 2.0 + shift
    pts2 = pts2 * 2.0 + shift
    A, bvec = [], []
    for (x, y), (u, v) in zip(pts1, pts2):
        A.append([x, y, 1, 0, 0, 0, -u * x, -u * y]); bvec.append(u)
        A.append([0, 0, 0, x, y, 1, -v * x, -v * y]); bvec.append(v)
    h = np.linalg.solve(np.array(A), np.array(bvec))
    Hm = np.append(h, 1.0).reshape(3, 3)
    return Hm  # pts1 -> pts2, as cv2.getPerspectiveTransform(pts1, pts2) (homographies.py:140); callers invert it


def adaptation_workload(I0, N, Hc, Wc, seed=0):
    """Host inputs of bench.py's homography-adaptation workload: logits semi [I0,N,65,Hc,Wc] (3 x pseudo-normal) and
    homographies [I0,N,3,3] of N views per source image, the identity first (float32)."""
    rng = np.random.default_rng(500 + seed)
    Hs = np.stack([[np.linalg.inv(sample_homography(rng, max_angle=3.14 / 2)) for _ in range(N)] for _ in range(I0)])
    Hs[:, 0] = np.eye(3)
    return pseudo_normal((I0, N, 65, Hc, Wc), 7000 + seed) * 3, Hs.astype(np.float32)
