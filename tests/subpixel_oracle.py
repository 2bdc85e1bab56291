"""Restatement of the reference's sub-pixel keypoint step, SuperPointFrontend_torch.soft_argmax_points
(models/model_wrap.py:212-248), in numpy fp32 (the oracle of utils.soft_argmax_points and of
step.adaptation_step(subpixel=True)).  The shipped COCO export config runs it between NMS and top-k
(configs/magicpoint_coco_export.yaml:44-45, export.py:309-314).

Operation order of the reference, per point (x, y, conf) of the [3,K] float64 NMS output, p = patch_size:
  1. extract_patch_from_points (utils/losses.py): np.pad(heat, p // 2, 'constant')[yi:yi+p, xi:xi+p] with
     (xi, yi) = (x, y).astype(int), one Python slice per point;
  2. norm_patches: d = sum(patch) + 1e-6, q = patch / d;
  3. do_log: q[q < 0] = 1e-6, l = log(q) (a zero tap gives -inf);
  4. torchgeometry 0.1.2 SpatialSoftArgmax2d(normalized_coordinates=False): e = exp(l - max l), s = 1 / (sum e + 1e-6),
     dx = sum((pos_x * e) * s), dy = sum((pos_y * e) * s), pos_x / pos_y the column / row of linspace(0, p - 1, p);
  5. float64: x = (x + dx) - p // 2, y likewise; conf unchanged.
"""
import numpy as np


def soft_argmax_points(heatmap, pts, patch_size=5):
    """heatmap [H,W] (anything np.squeeze makes [H,W]), pts [3,K] float64 or a one-element list of it -> refined [3,K]
    float64 (a new array)."""
    if isinstance(pts, (list, tuple)):
        pts = pts[0]
    out = np.array(pts, dtype=np.float64)
    K = out.shape[1]
    if K == 0:
        return out
    p = int(patch_size)
    half = p // 2
    heat = np.pad(np.squeeze(np.asarray(heatmap, dtype=np.float32)), half, "constant")
    ij = out[:2].T.astype(int)
    patches = np.stack([heat[y:y + p, x:x + p] for x, y in ij]).reshape(K, p * p)
    f = np.float32
    d = patches.sum(axis=1, keepdims=True, dtype=f) + f(1e-6)
    q = patches / d
    q[q < 0] = f(1e-6)
    with np.errstate(divide="ignore"):
        l = np.log(q)
    with np.errstate(invalid="ignore"):
        e = np.exp(l - l.max(axis=1, keepdims=True))
    s = f(1.0) / (e.sum(axis=1, keepdims=True, dtype=f) + f(1e-6))
    pos = np.linspace(0, p - 1, p, dtype=f)
    pos_x, pos_y = np.tile(pos, p), np.repeat(pos, p)
    dx = ((pos_x * e) * s).sum(axis=1, dtype=f)
    dy = ((pos_y * e) * s).sum(axis=1, dtype=f)
    out[0] = (out[0] + dx.astype(np.float64)) - half
    out[1] = (out[1] + dy.astype(np.float64)) - half
    return out
