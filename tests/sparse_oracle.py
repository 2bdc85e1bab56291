"""CPU oracle of the deterministic half of the sparse loss's correspondence sampling -- TEST INFRASTRUCTURE, NOT PRODUCT.

The device sampler (sparse.DeviceSampler, ssp_sparse_sample) draws its matches from the candidate pairs of every image; this
module restates how the reference finds them, in numpy fp32 on top of oracle.ssp_oracle.warp_points.  It is pinned by
tests/test_sparse_sampler_host.py against the index lists the live reference sampled (tests/golden/sparse_loss.npz) and
against the host sampler (sparse.sample_correspondences); tests/test_gpu_sparse_step.py checks the device sampler with it.
"""
import numpy as np

from oracle.ssp_oracle import f32, warp_points


def sparse_candidates(H, Hc, Wc):
    """The deterministic half of sample_correspondences (sparse_loss.py:170-200 with correspondence_finder.py:191-240) in
    fp32: every cell (u, v) of a Hc x Wc grid warped by scale_homography_torch(H, shift -1) = T^-1 H T, rounded half to even,
    kept when 0 <= p <= (Wc-1, Hc-1).  H [3,3] in normalised coordinates.  Returns a dict:
      a, b   int64 [M]: the candidate pairs (cell index u + v*Wc in each image), in row-major order of a
      b_all  int64 [Hc*Wc]: the rounded warp of every cell (-1 where it is not kept)
      tie    [Hc*Wc]: distance of the unrounded warp to the nearest rounding tie (x.5) over both coordinates, inf if not finite
      bound  [Hc*Wc]: distance of the unrounded warp to the nearest edge of the kept region [-0.5, Wc-0.5] x [-0.5, Hc-0.5]
    A 1-ulp difference in the warp can only move a cell whose tie distance is tiny (the bounds of the kept region are ties
    themselves), so a sampler computed in another operation order agrees on every cell with tie > a small tolerance."""
    trans = np.array([[2.0 / Wc, 0.0, -1], [0.0, 2.0 / Hc, -1], [0.0, 0.0, 1.0]], dtype=f32)
    Hcell = (np.linalg.inv(trans).astype(f32) @ np.asarray(H, f32).reshape(3, 3) @ trans).astype(f32)
    vv, uu = np.meshgrid(np.arange(Hc), np.arange(Wc), indexing="ij")
    uv = np.stack([uu.ravel(), vv.ravel()], axis=1).astype(f32)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        p = warp_points(uv, Hcell)
        r = np.round(p)  # half to even, like torch.round
        keep = np.all(np.isfinite(p), axis=1) & np.all((r >= 0) & (r <= np.array([Wc - 1, Hc - 1], f32)), axis=1)
        frac = np.abs(p - np.floor(p) - 0.5).astype(np.float64)
        tie = np.where(np.all(np.isfinite(p), axis=1), frac.min(axis=1), np.inf)
        lo, hi = p + 0.5, np.array([Wc - 0.5, Hc - 0.5], f32) - p
        bound = np.where(np.all(np.isfinite(p), axis=1), np.abs(np.concatenate([lo, hi], axis=1)).min(axis=1), np.inf)
    b_all = np.full(Hc * Wc, -1, np.int64)
    b_all[keep] = (r[keep, 0] + r[keep, 1] * Wc).astype(np.int64)
    a = np.nonzero(keep)[0].astype(np.int64)
    return {"a": a, "b": b_all[a], "b_all": b_all, "tie": tie, "bound": bound.astype(np.float64)}
