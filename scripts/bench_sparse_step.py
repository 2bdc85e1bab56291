"""Times the sparse-loss training step (the loss of the shipped configs) three ways and writes JSON to an output directory:

  host     detector pair + sparse.batch_descriptor_loss_sparse with host sampling (sampler=None), forward + backward, eager:
           what the drop-in runs today
  device   loss_step(descriptor_loss="sparse") with a DeviceSampler, eager
  graph    the same step captured by GraphedLossStep and replayed

at B = 32 of 240x320 (bench.host_inputs, K = 1000, n = 10) and at KITTI B = 4 of 376x1240.  For each run: pairs/s from CUDA
events over --steps steps after --warmup steps, and, in a separate pass, the time of every C-ABI entry point from CUDA events
around each call (_lib.profile_begin).  The GPU name and power limit are read in the same run.

    python scripts/bench_sparse_step.py OUT_DIR [--steps 200] [--warmup 20]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import ssp_b200 as S  # noqa: E402
from ssp_b200 import _lib, synth  # noqa: E402

K, N_PER = 1000, 10


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [c.strip() for c in out.split(",")]
    except Exception as e:  # noqa: BLE001
        name, power, clock = torch.cuda.get_device_name(0), "unknown (%s)" % e, "unknown"
    return {"name": name, "power_limit": power, "sm_clock_max": clock, "torch_name": torch.cuda.get_device_name(0)}


def kitti_inputs(B, seed):
    Hc, Wc = 47, 155
    H, W = 8 * Hc, 8 * Wc
    rng = np.random.default_rng(seed)
    Hs = np.stack([np.linalg.inv(synth.sample_homography(rng)) for _ in range(B)]).astype(np.float32)
    return {"semi": synth.pseudo_normal((B, 65, Hc, Wc), seed * 10 + 1),
            "semi_warp": synth.pseudo_normal((B, 65, Hc, Wc), seed * 10 + 2),
            "desc": synth.unit_descriptors(B, 256, Hc, Wc, seed * 10 + 3, smooth=0.3),
            "desc_warp": synth.unit_descriptors(B, 256, Hc, Wc, seed * 10 + 4, smooth=0.3),
            "labels_2D": synth.keypoint_labels(B, H, W, seed * 10 + 5),
            "warped_labels": synth.keypoint_labels(B, H, W, seed * 10 + 6),
            "mat_H": Hs, "inv_H": np.linalg.inv(Hs).astype(np.float32)}


def device_inputs(h):
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in h.items()}
    B, _, H, W = d["labels_2D"].shape
    d["mask_2D"] = torch.ones((B, 1, H, W), device="cuda")
    d["mask_warp_2D"] = S.compute_valid_mask(torch.tensor([H, W]), d["inv_H"], device="cuda", erosion_radius=3).unsqueeze(1)
    return d


LEAVES = ("semi", "semi_warp", "desc", "desc_warp")


def host_step(d, _state):
    lv = [d[k].detach().requires_grad_(True) for k in LEAVES]
    l0, l1, _ = S.utils.detector_loss_pair_2d(lv[0], d["labels_2D"], d["mask_2D"], lv[1], d["warped_labels"],
                                              d["mask_warp_2D"])
    ld, _, _, _ = S.batch_descriptor_loss_sparse(lv[2], lv[3], d["mat_H"], device="cuda", lamda_d=250,
                                                 num_matching_attempts=K, num_masked_non_matches_per_match=N_PER)
    (l0 + l1 + ld).backward()


def device_step(d, state):
    lv = [d[k].detach().requires_grad_(True) for k in LEAVES]
    out = S.step.loss_step(*lv, d["labels_2D"], d["warped_labels"], d["mask_2D"], d["mask_warp_2D"], d["mat_H"],
                           descriptor_loss="sparse", sampler=state["sampler"], num_matching_attempts=K,
                           num_masked_non_matches_per_match=N_PER)
    out["loss"].backward()


def graph_step(d, state):
    if "graph" not in state:
        state["graph"] = S.step.GraphedLossStep(d, descriptor_loss="sparse", sampler=state["sampler"],
                                                num_matching_attempts=K, num_masked_non_matches_per_match=N_PER)
    state["graph"].replay()


def time_path(fn, d, steps, warmup):
    state = {"sampler": S.sparse.DeviceSampler(0, "cuda")}
    for _ in range(warmup):
        fn(d, state)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn(d, state)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    B = d["semi"].shape[0]
    # separate pass: CUDA events around every C-ABI entry point (eager paths; a replay makes no such calls)
    per_call = {}
    if fn is not graph_step:
        prof_steps = 20
        _lib.profile_begin()
        for _ in range(prof_steps):
            fn(d, state)
        per_call = {k: {"calls_per_step": n / prof_steps, "ms_per_step": t / prof_steps}
                    for k, (n, t) in sorted(_lib.profile_end().items())}
    return {"ms_per_step": ms, "pairs_per_s": B / ms * 1e3, "steps": steps, "warmup": warmup, "per_entry_point": per_call}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse_step.py measures on a CUDA device; none is available")
    if args.steps < 100:
        raise SystemExit("--steps must be at least 100")
    os.makedirs(args.out_dir, exist_ok=True)
    res = {"gpu": gpu_info(), "K": K, "n": N_PER, "runs": {}}
    for name, h in (("240x320_b32", bench.host_inputs(bench.B_PER_GPU, 0)), ("kitti_376x1240_b4", kitti_inputs(4, 0))):
        d = device_inputs(h)
        for path, fn in (("host", host_step), ("device", device_step), ("graph", graph_step)):
            r = time_path(fn, d, args.steps, args.warmup)
            res["runs"]["%s/%s" % (name, path)] = r
            print("%-22s %-6s %9.1f pairs/s  %8.3f ms/step" % (name, path, r["pairs_per_s"], r["ms_per_step"]), flush=True)
            for k, v in sorted(r["per_entry_point"].items(), key=lambda kv: -kv[1]["ms_per_step"]):
                print("    %-32s %5.1f calls %8.4f ms" % (k, v["calls_per_step"], v["ms_per_step"]), flush=True)
    res["gpu_after"] = gpu_info()
    path = os.path.join(args.out_dir, "bench_sparse_step.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: round(v["pairs_per_s"], 1) for k, v in res["runs"].items()}))
    print("gpu: %s, power limit %s" % (res["gpu"]["name"], res["gpu"]["power_limit"]))


if __name__ == "__main__":
    main()
