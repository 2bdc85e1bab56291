"""Runs the homography-adaptation step (32 source images x 100 views) and the warp kernels a few times at BASELINE sizes:
target of `ncu` launch lists / --set full captures (scripts/gpu_run.sh launches_adapt)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import ssp_b200 as S
from ssp_b200 import synth

dev = torch.device("cuda")
I, N, Hc, Wc = int(os.environ.get("ADAPT_I", "32")), 100, 30, 40
rng = np.random.default_rng(0)
Hs = np.stack([[np.linalg.inv(synth.sample_homography(rng, max_angle=1.57)) for _ in range(N)] for _ in range(4)]).astype(np.float32)
Hs[:, 0] = np.eye(3)
Hw = torch.from_numpy(Hs).to(dev).repeat(I // 4, 1, 1, 1)
Hinv = torch.from_numpy(np.linalg.inv(Hs).astype(np.float32)).to(dev).repeat(I // 4, 1, 1, 1)
g = torch.Generator(device=dev)
g.manual_seed(0)
semi = torch.randn((I, N, 65, Hc, Wc), device=dev, generator=g) * 3
shape_t = torch.tensor([240, 320])
img = torch.rand((100, 1, 240, 320), device=dev, generator=g)
pts = torch.rand((76800, 2), device=dev, generator=g) * 2 - 1
for rep in range(2):
    mask = S.compute_valid_mask(shape_t, Hinv.reshape(-1, 3, 3), device=dev).reshape(I, N, 240, 320)
    mask3 = S.compute_valid_mask(shape_t, Hinv[0], device=dev, erosion_radius=3)
    out = S.step.adaptation_step(semi, Hw, mask, binary_mask=True)
    w = S.inv_warp_image_batch(img, Hinv[0], device=dev)
    wn = S.inv_warp_image_batch(img, Hinv[0], device=dev, mode="nearest")
    wp = S.warp_points(pts, Hinv[0], device=dev)
torch.cuda.synchronize()
print("done", len(out), out[0].shape)
