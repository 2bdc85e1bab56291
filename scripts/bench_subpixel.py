"""Times the sub-pixel keypoint step (ssp_soft_argmax_points) and writes JSON to an output directory:

  adaptation_step  step.adaptation_step at I = 32 source images x N = 100 views of 240x320 (bench.py's workload, binary
                   masks, top-k 600) with subpixel False and True, alternated call by call in the same run: a host clock
                   around each call (the call ends in the keypoint read-back, a device synchronise) and CUDA events
                   around the same call
  kernel           ssp_soft_argmax_points alone on 32 images x 600 points of that workload's aggregated heatmaps, patch 5,
                   CUDA events: over eager launches through the ctypes binding, and over a CUDA graph of back-to-back
                   launches (kernel time without the host)
  host_arm         the reference's per-image refinement of 600 points on this host's CPU (tests/subpixel_oracle.py: one
                   Python slice per patch like extract_patch_from_points, numpy fp32 arithmetic), with the thread counts

The GPU name and power limit are read in the same run.

    python scripts/bench_subpixel.py OUT_DIR [--pairs 100] [--warmup 5]
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

import ssp_b200 as S  # noqa: E402
import subpixel_oracle as SO  # noqa: E402
from bench_sparse_step import gpu_info  # noqa: E402
from ssp_b200 import _lib  # noqa: E402
from ssp_b200 import synth  # noqa: E402

TOP_K, PATCH = 600, 5
I0, REP, N, H_IMG, W_IMG = 4, 8, 100, 240, 320


def adaptation_inputs():
    """bench.py's homography-adaptation workload on the device: I0 distinct source images x N views, logits rescaled REP
    times to 32 source images, binary valid masks from compute_valid_mask."""
    base, Hs = synth.adaptation_workload(I0, N, H_IMG // 8, W_IMG // 8)
    Hinv = torch.from_numpy(np.linalg.inv(Hs).astype(np.float32)).cuda()
    semi = torch.cat([torch.from_numpy(base * np.float32(1.0 + 0.05 * k)).cuda() for k in range(REP)])
    mask = S.compute_valid_mask(torch.tensor([H_IMG, W_IMG]), Hinv.reshape(-1, 3, 3), device="cuda")
    return semi, torch.from_numpy(Hs).cuda().repeat(REP, 1, 1, 1), mask.reshape(I0, N, H_IMG, W_IMG).repeat(REP, 1, 1, 1)


def stats(v):
    v = np.asarray(v)
    return {"median": float(np.median(v)), "mean": float(v.mean()), "min": float(v.min()), "max": float(v.max()),
            "n": int(v.size)}


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--pairs", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    res = {"gpu": gpu_info(), "pairs": a.pairs, "warmup": a.warmup}
    semi, Hw, mask = adaptation_inputs()
    I = semi.shape[0]

    def step(sub):
        return S.step.adaptation_step(semi, Hw, mask, top_k=TOP_K, binary_mask=True, subpixel=sub, patch_size=PATCH)

    for _ in range(a.warmup):
        step(False), step(True)
    host = {False: [], True: []}
    dev = {False: [], True: []}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(a.pairs):
        for sub in (False, True):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record()
            pts = step(sub)
            e1.record()
            host[sub].append((time.perf_counter() - t0) * 1e3)
            torch.cuda.synchronize()
            dev[sub].append(e0.elapsed_time(e1))
    res["adaptation_step_ms"] = {"I": I, "N": semi.shape[1], "top_k": TOP_K, "patch_size": PATCH,
                                 "host_clock": {"subpixel_false": stats(host[False]), "subpixel_true": stats(host[True])},
                                 "cuda_events": {"subpixel_false": stats(dev[False]), "subpixel_true": stats(dev[True])},
                                 "added_ms_median_host_clock": float(np.median(host[True]) - np.median(host[False])),
                                 "added_ms_median_events": float(np.median(dev[True]) - np.median(dev[False])),
                                 "keypoints_per_image": [int(p.shape[0]) for p in pts]}

    # the kernel alone: the unrefined top-600 points of every image in the NMS layout [I, 3, 600], counts on the device
    agg = S.utils.combine_from_logits_batch(semi, Hw, mask)
    base = S.heatmap_to_pts_batch(agg, 0.015, 4, top_k=TOP_K)
    buf = np.zeros((I, 3, TOP_K))
    for i, p in enumerate(base):
        buf[i, :, :p.shape[1]] = p
    pts_d = torch.from_numpy(buf).cuda()
    counts = torch.tensor([p.shape[1] for p in base], dtype=torch.int32).cuda()
    H, W = agg.shape[1:]

    def launch():  # refines in place: every launch starts from the previous one's points (same work per launch)
        _lib.call("ssp_soft_argmax_points", _lib.ptr(agg), I, H, W, _lib.ptr(pts_d), TOP_K, _lib.ptr(counts), TOP_K, PATCH,
                  _lib.stream_of(agg))

    n_eager, per_graph, replays = 2000, 100, 50
    events_ms(launch, 50)
    eager = events_ms(launch, n_eager)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(per_graph):
            launch()
    g.replay()
    graph = events_ms(g.replay, replays) / per_graph
    res["kernel_us"] = {"images": I, "points": int(counts.sum()), "patch_size": PATCH, "eager_launch": eager * 1e3,
                        "graph_back_to_back": graph * 1e3, "eager_launches": n_eager, "graph_launches": per_graph * replays}

    # host arm: the oracle's per-image refinement of 600 points (what the reference's method does per source image)
    agg_h = agg.cpu().numpy()
    t = []
    for i, p in enumerate(base):
        t0 = time.perf_counter()
        SO.soft_argmax_points(agg_h[i], p, PATCH)
        t.append((time.perf_counter() - t0) * 1e3)
    res["host_arm_ms_per_image"] = stats(t)
    res["host_threads"] = {"torch": torch.get_num_threads(), "cpu_count": os.cpu_count()}

    with open(os.path.join(a.out, "bench_subpixel.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    print("gpu: %s, power limit %s" % (res["gpu"]["name"], res["gpu"]["power_limit"]))


if __name__ == "__main__":
    main()
