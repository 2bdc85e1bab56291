"""Times the pair evaluation (utils.evaluate_pairs, step.match_step(homographies=...)) and writes JSON to an output directory:

  workload     32 pairs of 480x640 (logits of synth.adaptation_workload, desc_warp = normalised(desc + 0.5 other), pixel
               homographies from HomographySampler), at top-k 1000 and at all points
  host_ms      median host clock around the synchronising call: plain match_step, match_step(homographies=...) and
               evaluate_pairs on match_step's returned arrays
  entry_ms     CUDA events around every entry point of one evaluate_pairs call (median over the timed calls)
  ransac       the RANSAC entry point's achieved float64 rate: 20 operations per (hypothesis, match) inlier test (3 fma
               chains of 2, 1 reciprocal, 2 fma, 1 multiply-add) over its CUDA-event time (score + refit kernels)
  reference    the per-pair host path of evaluation.py on this host's CPU -- cv2.BFMatcher(crossCheck) + findHomography(RANSAC)
               twice, sklearn average_precision_score, numpy repeatability (oracle) -- if cv2 and sklearn import

The GPU name and power limit are read in the same run.

    python scripts/bench_eval.py OUT_DIR [--pairs 32] [--reps 20]
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
from bench_match_step import workload, stats  # noqa: E402
from bench_sparse_step import gpu_info  # noqa: E402
from oracle import ssp_oracle as O  # noqa: E402
from ssp_b200 import _lib  # noqa: E402
from ssp_b200 import utils as U  # noqa: E402
from ssp_b200.homography import HomographySampler  # noqa: E402

SHAPE = (480, 640)
OPS_PER_TEST = 20


def host_ms(fn, n):
    out = []
    for _ in range(n):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t) * 1e3)
    return stats(out)


def reference_arm(res, Hs):
    try:
        import cv2
        from sklearn.metrics import average_precision_score
    except ImportError as e:
        return {"status": "not run (%s)" % e}
    t = time.perf_counter()
    for p, r in enumerate(res):
        kp, wk = r["pts"].T, r["warped_pts"].T
        O.compute_repeatability(kp, wk, Hs[p], SHAPE, keep_k_points=1000, distance_thresh=3)
        bf = cv2.BFMatcher(cv2.NORM_L2, crossCheck=True)
        ms = bf.match(np.ascontiguousarray(r["desc"].T), np.ascontiguousarray(r["warped_desc"].T))
        if len(ms) >= 4:
            a = kp[[m.queryIdx for m in ms], :2]
            b = wk[[m.trainIdx for m in ms], :2]
            cv2.findHomography(a, b, cv2.RANSAC)
            d = np.array([m.distance for m in ms])
            sub = d < 1.2
            if sub.sum() >= 4:
                _, inl = cv2.findHomography(a[sub], b[sub], cv2.RANSAC)
                if inl is not None and inl.sum():
                    average_precision_score(inl.ravel(), d[sub].max() - d[sub])
    ms_total = (time.perf_counter() - t) * 1e3
    return {"status": "run", "ms_total": ms_total, "ms_per_pair": ms_total / len(res), "cpu_threads": os.cpu_count(),
            "cv2": cv2.__version__}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--pairs", type=int, default=32)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    P = a.pairs
    semi, desc, semi_w, desc_w = workload(P)
    hom, _ = HomographySampler(11, "cuda").sample(P, perspective_amplitude_x=0.2, perspective_amplitude_y=0.2,
                                                  patch_ratio=0.85, allow_artifacts=True)
    Hs = np.stack([U.homography_scaling_torch(hom[p].cpu(), *SHAPE).double().numpy() for p in range(P)])
    out = {"gpu": gpu_info(), "pairs": P, "shape": SHAPE, "hypotheses": U.RANSAC_HYPOTHESES, "runs": {}}
    for top_k in (1000, None):
        run = lambda **kw: S.step.match_step(semi, desc, semi_w, desc_w, top_k=top_k, **kw)
        res = run(homographies=Hs)
        args = ([r["pts"] for r in res], [r["warped_pts"] for r in res], [r["desc"] for r in res],
                [r["warped_desc"] for r in res], Hs, SHAPE)
        ev = lambda: U.evaluate_pairs(*args)
        for f in (run, lambda: run(homographies=Hs), ev):
            f()
        r = {"points_mean": float(np.mean([x["pts"].shape[1] for x in res] + [x["warped_pts"].shape[1] for x in res])),
             "host_ms": {"match_step": host_ms(run, a.reps), "match_step_eval": host_ms(lambda: run(homographies=Hs), a.reps),
                         "evaluate_pairs": host_ms(ev, a.reps)}}
        prof = []
        for _ in range(a.reps):
            _lib.profile_begin()
            ev()
            prof.append(_lib.profile_end())
        r["entry_ms"] = {k: float(np.median([pp[k][1] for pp in prof])) for k in prof[0]}
        m = ev()
        L = sum(int(x.shape[0]) for x in m["inliers"])  # the cross-check matches; the mAP problems' matches below
        K = max(max(x["desc"].shape[1], x["warped_desc"].shape[1]) for x in res)
        pad = lambda d: np.pad(d, ((0, 0), (0, K - d.shape[1])))
        mm = U.nn_match_two_way_batch(torch.from_numpy(np.stack([pad(x["desc"]) for x in res])).cuda(),
                                      torch.from_numpy(np.stack([pad(x["warped_desc"]) for x in res])).cuda(), 1.2,
                                      counts1=[x["desc"].shape[1] for x in res], counts2=[x["warped_desc"].shape[1] for x in res])
        L_sub = sum(x.shape[1] for x in mm)
        ops = float(OPS_PER_TEST) * U.RANSAC_HYPOTHESES * (L + L_sub)
        t_r = r["entry_ms"]["ssp_ransac_homography"]
        r["ransac"] = {"matches_all": L, "matches_map": L_sub, "gflop": ops / 1e9, "ms": t_r,
                       "tflops_fp64": ops / (t_r * 1e-3) / 1e12}
        r["mean"] = {k: float(np.nanmean(np.asarray(m[k], dtype=np.float64))) for k in
                     ("repeatability", "localization_err", "mean_dist", "matching_score", "ap")}
        r["mean"]["correctness"] = np.asarray(m["correctness"]).mean(axis=0).tolist()
        r["reference"] = reference_arm(res, Hs)
        out["runs"]["top_k_%s" % (top_k or "all")] = r
        print(json.dumps({k: r[k] for k in ("points_mean", "host_ms", "entry_ms", "ransac")}), flush=True)
    with open(os.path.join(a.out, "bench_eval.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["gpu"]))


if __name__ == "__main__":
    main()
