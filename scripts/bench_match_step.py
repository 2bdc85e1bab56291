"""Times the batched descriptor export (step.match_step) and its tensor-core matcher, and writes JSON to an output directory:

  match_step   32 pairs of 480x640 (logits of synth.adaptation_workload, desc_warp = normalised(desc + 0.5 other)), top-k
               1000 and all points: host clock around the call (it ends in the read-back, a device synchronise); CUDA
               events around every entry point of one call (the device part before the read-back); the read-back of a
               buffer of the same size on its own, into page-locked memory (what match_step does) and into pageable memory
  matcher      ssp_nn_match_batch alone on that workload's descriptors, CUDA events over >= 100 launches after warm-up,
               against ssp_nn_match (fp32 CUDA cores) looped over the same pairs: algorithmic TFLOP/s (2 K1 K2 256) and the
               share of the data sheet's 2,250 TFLOP/s BF16 with the three MMA passes counted
  per_pair     the drop-in path the stock export runs per pair (getPtsFromHeatmap x2, sample_desc_from_points x2,
               nn_match_two_way), host clock over the 32 pairs
  oracle       the reference chain in numpy (oracle/) for one pair on this host's CPU, with its thread count

The GPU name and power limit are read in the same run.

    python scripts/bench_match_step.py OUT_DIR [--pairs 32] [--launches 100]
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
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import ssp_b200 as S  # noqa: E402
from bench_sparse_step import gpu_info  # noqa: E402
from oracle import ssp_oracle as O  # noqa: E402
from ssp_b200 import _lib  # noqa: E402
from ssp_b200 import synth  # noqa: E402
from ssp_b200 import utils as U  # noqa: E402

HC, WC, CONF, NMS, THR = 60, 80, 0.015, 4, 0.7
BF16_PEAK = 2250.0  # TFLOP/s, dense BF16, HGX B200 data sheet per GPU


def workload(P):
    semi = synth.adaptation_workload(1, 2 * P, HC, WC)[0][0]
    desc = synth.unit_descriptors(P, 256, HC, WC, 41, smooth=0.4).astype(np.float64)
    dw = desc + 0.5 * synth.unit_descriptors(P, 256, HC, WC, 42, smooth=0.4)
    dw /= np.sqrt((dw * dw).sum(axis=1, keepdims=True))
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return cu(semi[:P]), cu(desc.astype(np.float32)), cu(semi[P:]), cu(dw.astype(np.float32))


def stats(v):
    v = np.asarray(v, dtype=np.float64)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()), "n": int(v.size)}


def host_ms(fn, n):
    out = []
    for _ in range(n):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t) * 1e3)
    return stats(out)


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def device_inputs(semi, desc, semi_w, desc_w, top_k):
    """match_step's stages 1-3 by hand: the sampled descriptors [2P,256,kmax] and the per-image counts (device, capped)."""
    P = semi.shape[0]
    heat = S.flattenDetection(torch.cat([semi, semi_w])).view(2 * P, 8 * HC, 8 * WC)
    pts, counts, cdev = U._nms_batch(heat, CONF, NMS)
    cnt = [min(c, top_k) for c in counts] if top_k else counts
    kmax = max(cnt)
    d_all = torch.empty((2 * P, 256, kmax), dtype=torch.float32, device="cuda")
    for h, d in enumerate((desc, desc_w)):
        _lib.call("ssp_sample_desc_batch", _lib.ptr(d), _lib.ptr(pts[h * P:]), pts.shape[2], _lib.ptr(cdev[h * P:]), kmax, P,
                  256, HC, WC, 8, _lib.ptr(d_all[h * P:]), _lib.stream_of(d))
    return d_all, cnt, cdev, kmax


def bench_matcher(d_all, cnt, cdev, kmax, P, launches):
    planes = U._pack_planes(d_all)
    R = planes.shape[2]
    matches = torch.empty((P, 3, R), dtype=torch.float64, device="cuda")
    nmatch = torch.empty((P,), dtype=torch.int32, device="cuda")
    run = lambda: U._nn_match_planes(planes[:, :P], planes[:, P:], cdev[:P], cdev[P:], kmax, THR, matches, nmatch)
    flops = float(sum(2.0 * cnt[p] * cnt[P + p] * 256 for p in range(P)))
    for _ in range(5):
        run()
    tc_ms = events_ms(run, launches)
    # fp32 CUDA-core matcher on the same pairs, one call per pair (what nn_match_two_way launches)
    d1 = [d_all[p, :, :cnt[p]].contiguous() for p in range(P)]
    d2 = [d_all[P + p, :, :cnt[P + p]].contiguous() for p in range(P)]
    best = torch.empty((2 * R,), dtype=torch.int64, device="cuda")

    def simt():
        for p in range(P):
            if cnt[p] and cnt[P + p]:
                _lib.call("ssp_nn_match", _lib.ptr(d1[p]), _lib.ptr(d2[p]), 256, cnt[p], cnt[P + p], _lib.ptr(best[:cnt[p]]),
                          _lib.ptr(best[R:R + cnt[P + p]]), _lib.stream_of(best))
    simt()
    simt_ms = events_ms(simt, max(3, launches // 20))
    tf = lambda ms: flops / (ms * 1e-3) / 1e12
    return {"pairs": P, "points_mean": float(np.mean(cnt)), "gflop": flops / 1e9, "launches": launches,
            "tc_ms": tc_ms, "tc_tflops": tf(tc_ms), "tc_share_of_bf16_peak_3pass": 3 * tf(tc_ms) / BF16_PEAK,
            "simt_fp32_ms": simt_ms, "simt_fp32_tflops": tf(simt_ms), "speedup": simt_ms / tc_ms}


def per_pair(semi, desc, semi_w, desc_w, top_k):
    for p in range(semi.shape[0]):
        pts = [S.getPtsFromHeatmap(S.flattenDetection(s[p]).squeeze(0), CONF, NMS)[:, :top_k] for s in (semi, semi_w)]
        ds = [S.utils.sample_desc_from_points(d[p:p + 1], q) for d, q in zip((desc, desc_w), pts)]
        S.utils.nn_match_two_way(ds[0], ds[1], THR)


def oracle_pair(semi, desc, semi_w, desc_w, top_k):
    t = time.perf_counter()
    pts = [O.getPtsFromHeatmap(O.flattenDetection(s[0].cpu().numpy())[0], CONF, NMS)[:, :top_k] for s in (semi, semi_w)]
    ds = [O.sample_desc_from_points(d[:1].cpu().numpy(), q) for d, q in zip((desc, desc_w), pts)]
    O.nn_match_two_way(ds[0], ds[1], THR)
    return (time.perf_counter() - t) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--pairs", type=int, default=32)
    ap.add_argument("--launches", type=int, default=100)
    a = ap.parse_args()
    P = a.pairs
    inputs = workload(P)
    res = {"gpu": gpu_info(), "workload": "%d pairs of 480x640, conf %.3f, NMS %d, nn_thresh %.1f" % (P, CONF, NMS, THR),
           "host_threads": {"torch": torch.get_num_threads(), "cpu_count": os.cpu_count(),
                            "OMP_NUM_THREADS": os.environ.get("OMP_NUM_THREADS")}}
    for top_k in (1000, None):
        key = "top_k_%s" % (top_k or "all")
        call = lambda: S.step.match_step(*inputs, conf_thresh=CONF, nms_dist=NMS, top_k=top_k, nn_thresh=THR)
        out = call()
        call()
        r = {"match_step_host_ms": host_ms(call, 7)}
        _lib.profile_begin()
        call()
        prof = _lib.profile_end()
        r["match_step_entry_points_ms"] = {k: v[1] for k, v in prof.items()}
        r["match_step_device_ms_excl_nms"] = sum(v[1] for k, v in prof.items() if k != "ssp_nms_fast")
        nbytes = sum(o[k].nbytes for o in out for k in o)
        buf = torch.empty((nbytes,), dtype=torch.uint8, device="cuda")
        pinned = torch.empty((nbytes,), dtype=torch.uint8, pin_memory=True)
        r["readback_bytes"] = nbytes
        r["readback_pinned_ms"] = host_ms(lambda: pinned.copy_(buf), 5)
        r["readback_pageable_ms"] = host_ms(lambda: buf.cpu(), 5)
        r["matches_mean"] = float(np.mean([o["matches"].shape[1] for o in out]))
        d_all, cnt, cdev, kmax = device_inputs(*inputs, top_k)
        r["matcher"] = bench_matcher(d_all, cnt, cdev, kmax, P, a.launches)
        del d_all
        per_pair(*inputs, top_k)
        r["per_pair_dropin_host_ms"] = host_ms(lambda: per_pair(*inputs, top_k), 2)
        r["oracle_one_pair_cpu_ms"] = oracle_pair(*inputs, top_k)
        res[key] = r
        print(key, json.dumps(r), flush=True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "r3_bench_match.json"), "w") as f:
        json.dump(res, f, indent=1)
    print("gpu: %s, power limit %s" % (res["gpu"]["name"], res["gpu"]["power_limit"]))


if __name__ == "__main__":
    main()
