"""Times the device homography sampler and its two step-level users, and the reference's scalar sampler on the host, and
writes JSON to an output directory:

  sampler          HomographySampler.sample (ssp_sample_homography) at B = 32 (one training batch) and B = 3200 (32 source
                   images x 100 views), training parameters
  adaptation_views step.adaptation_views at I = 32, N = 100, 240x320, export parameters: eager and CUDA-graph replay
  collate          step.collate_warped_pair at B = 32, 240x320, 300 keypoints per image: with a HomographySampler and with
                   homographies sampled on the host (its host inverse)
  host_sampler     the reference's sample_homography_np call sequence (tests/homography_oracle.py at n = 1) on this host's
                   CPU, per homography, with the torch / BLAS thread count

Device numbers are CUDA events over --steps calls after --warmup calls; the GPU name and power limit are read in the same run.

    python scripts/bench_homography.py OUT_DIR [--steps 200] [--warmup 20]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import homography_oracle as HO  # noqa: E402
import ssp_b200 as S  # noqa: E402
from bench_sparse_step import gpu_info  # noqa: E402
from ssp_b200 import synth  # noqa: E402


def time_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    res = {"gpu": gpu_info(), "steps": a.steps, "warmup": a.warmup}
    s = S.HomographySampler(0, "cuda")

    res["sampler_ms"] = {str(B): time_ms(lambda: s.sample(B, **HO.WARP_PARAMS), a.steps, a.warmup) for B in (32, 3200)}

    I, N, H, W = 32, 100, 240, 320
    img = torch.from_numpy(synth.uniform((I, 1, H, W), 1)).cuda()
    views = lambda: S.step.adaptation_views(img, s, num=N, **HO.EXPORT_PARAMS)  # noqa: E731
    eager = time_ms(views, a.steps, a.warmup)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        views()
    graph = time_ms(g.replay, a.steps, a.warmup)
    res["adaptation_views_ms"] = {"I": I, "N": N, "eager": eager, "graph": graph, "images_per_s_graph": I / graph * 1e3}

    B = 32
    img = torch.from_numpy(synth.uniform((B, 1, H, W), 2)).cuda()
    pts = [np.stack([np.floor(synth.uniform((300,), 10 + b) * W), np.floor(synth.uniform((300,), 60 + b) * H)], 1)
           for b in range(B)]
    dev = lambda: S.step.collate_warped_pair(img, pts, sampler=s, **HO.WARP_PARAMS)  # noqa: E731

    def host():
        Hs = np.linalg.inv(np.stack([HO.sample_homography_np(**HO.WARP_PARAMS) for _ in range(B)]))
        return S.step.collate_warped_pair(img, pts, torch.from_numpy(Hs.astype(np.float32)))

    steps = max(a.steps // 10, 5)
    res["collate_ms"] = {"B": B, "sampler": time_ms(dev, steps, a.warmup), "host_sampled": time_ms(host, steps, 2)}

    np.random.seed(0)
    n = 200
    t0 = time.perf_counter()
    for _ in range(n):
        HO.sample_homography_np(**HO.WARP_PARAMS)
    res["host_sampler_ms_per_homography"] = (time.perf_counter() - t0) / n * 1e3
    res["host_threads"] = {"torch": torch.get_num_threads(), "cpu_count": os.cpu_count()}

    with open(os.path.join(a.out, "bench_homography.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    print("gpu: %s, power limit %s" % (res["gpu"]["name"], res["gpu"]["power_limit"]))


if __name__ == "__main__":
    main()
