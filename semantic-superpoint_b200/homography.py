"""Homography sampling on the device (SURVEY 8f rank 4).

reference: utils/homographies.py:12-141 `sample_homography_np`, called in the DataLoader workers once per training pair
(datasets/Coco.py:342-347) and `num` times per source image for homography adaptation (Coco.py:261-277), always with
shape [2, 2], shift -1 and allow_artifacts=True, then inverted by the caller.  HomographySampler draws from the same
distribution with the kernel ssp_sample_homography (csrc/homography.cu) and returns both the callers' `homographies` and
their inverses: no host RNG, no host inverse, no host synchronisation.  Its draws are not the reference's RNG stream.
"""
import math

import torch

from ._lib import call, ptr, stream_of
from .rng import DeviceRng

PERSPECTIVE, SCALING, ROTATION, TRANSLATION = 1, 2, 4, 8


class HomographySampler(DeviceRng):
    """Batches of homographies drawn on the device: Philox4x32-10 keyed by (seed, homography index, launch counter), with
    the state handling of rng.DeviceRng (eager calls and graph replays draw fresh homographies; get_state() / set_state()
    reproduce them bit for bit).  A DeviceSampler built from the same seed draws unrelated numbers."""

    def sample(self, B, group=0, shape=(2, 2), shift=-1, perspective=True, scaling=True, rotation=True, translation=True,
               n_scales=5, n_angles=25, scaling_amplitude=0.1, perspective_amplitude_x=0.1, perspective_amplitude_y=0.1,
               patch_ratio=0.5, max_angle=math.pi / 2, allow_artifacts=False, translation_overflow=0.0, **config):
        """B homographies with sample_homography_np's keyword arguments and defaults (other keys are ignored, like the
        reference's **config).  Returns (homographies, inv_homographies), fp32 [B,3,3] on the device: homographies is the
        inverse of the sampled transform, as the dataset stores it (Coco.py:345).  group > 0: every index that is a
        multiple of group is the identity, the first view of each source image in homography adaptation (Coco.py:271)."""
        if not allow_artifacts:
            raise NotImplementedError("HomographySampler: only allow_artifacts=True (what every shipped config uses)")
        if translation_overflow != 0:
            raise NotImplementedError("HomographySampler: only translation_overflow=0 (what every shipped config uses)")
        if [int(s) for s in shape] != [2, 2] or shift != -1:
            raise NotImplementedError("HomographySampler: only shape [2, 2] and shift -1 (normalised coordinates)")
        flags = ((PERSPECTIVE if perspective else 0) | (SCALING if scaling else 0) | (ROTATION if rotation else 0) |
                 (TRANSLATION if translation else 0))
        B = int(B)
        hom = torch.empty((B, 3, 3), dtype=torch.float32, device=self.device)
        inv = torch.empty_like(hom)
        call("ssp_sample_homography", B, flags, int(n_scales), int(n_angles), float(scaling_amplitude),
             float(perspective_amplitude_x), float(perspective_amplitude_y), float(patch_ratio), float(max_angle), int(group),
             ptr(self.state), ptr(hom), ptr(inv), stream_of(hom))
        return hom, inv
