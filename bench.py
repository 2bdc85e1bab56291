"""bench.py -- loss-step pairs/s @240x320 B32 (BASELINE.json metric) on N GPUs of one node.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...       # the CPU path (oracle port) on the box's host cores
    python bench.py --dump-outputs DIR ...     # also write the outputs of the last timed step as DIR/<name>.npy

A "step" is one pass of the hot path over one batch: detector loss on both images + dense descriptor loss,
forward and backward, on 32 synthetic 240x320 pairs per GPU (head outputs `semi`/`desc` are the inputs; the
conv backbone is not on this path).  Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H_IMG, W_IMG, HC, WC, DCH, B_PER_GPU = 240, 320, 30, 40, 256, 32
NC = HC * WC
METRIC = "loss-step pairs/s @240x320 B32"
N_ADAPT = 100


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "src": "fallback"}


def host_inputs(B, seed):
    """One batch of synthetic loss-step inputs as numpy arrays (SURVEY 8d)."""
    from ssp_b200 import synth
    rng = np.random.default_rng(seed)
    Hs = np.stack([np.linalg.inv(synth.sample_homography(rng)) for _ in range(B)]).astype(np.float32)
    return {
        "semi": synth.pseudo_normal((B, 65, HC, WC), seed * 10 + 1),
        "semi_warp": synth.pseudo_normal((B, 65, HC, WC), seed * 10 + 2),
        "desc": synth.unit_descriptors(B, DCH, HC, WC, seed * 10 + 3, smooth=0.3),
        "desc_warp": synth.unit_descriptors(B, DCH, HC, WC, seed * 10 + 4, smooth=0.3),
        "labels_2D": synth.keypoint_labels(B, H_IMG, W_IMG, seed * 10 + 5),
        "warped_labels": synth.keypoint_labels(B, H_IMG, W_IMG, seed * 10 + 6),
        "mat_H": Hs,
        "inv_H": np.linalg.inv(Hs).astype(np.float32),
    }


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------
def host_threads():
    """Give the CPU path every host core (torchrun exports OMP_NUM_THREADS=1, which would throttle the BLAS behind the
    oracle port) and return the thread count actually in effect."""
    n = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=n)
        got = [p.get("num_threads") for p in threadpool_info() if p.get("user_api") in ("blas", "openmp")]
        return max(got) if got else n
    except Exception:  # noqa: BLE001
        return int(os.environ.get("OMP_NUM_THREADS", n))


def cpu_loss_step(inp):
    from oracle import ssp_oracle as O
    B = inp["semi"].shape[0]
    m2 = np.ones((B, 1, H_IMG, W_IMG), np.float32)
    mw2 = O.compute_valid_mask((H_IMG, W_IMG), inp["inv_H"], 3)[:, None]
    m3, mw3 = O.getMasks(m2), O.getMasks(mw2)
    l1, _ = O.detector_loss(inp["semi"], O.labels2Dto3D(inp["labels_2D"]), m3, grad=True)
    l2, _ = O.detector_loss(inp["semi_warp"], O.labels2Dto3D(inp["warped_labels"]), mw3, grad=True)
    r = O.descriptor_loss(inp["desc"], inp["desc_warp"], inp["mat_H"], mw3[:, None], grad=(1.0, 0.0, 0.0))
    return float(l1) + float(l2) + float(r[0])


def cpu_baseline(sample_pairs, reps):
    inp = host_inputs(sample_pairs, 99)
    threads = host_threads()
    cpu_loss_step(inp)  # warm-up (BLAS threads, page faults)
    t0 = time.perf_counter()
    for _ in range(reps):
        cpu_loss_step(inp)
    dt = (time.perf_counter() - t0) / reps
    return {"value": sample_pairs / dt, "unit": "pairs/s", "cores": threads, "host_cores": os.cpu_count(), "kind": "port",
            "sample": "%d pairs of 240x320 per step (fwd+bwd, numpy/BLAS oracle port of the reference path; the reference "
                      "itself materialises a 1.47 GB/pair product and ran ~1 pair/s on 8 cores), %d reps" % (sample_pairs, reps)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pairs = 2  # BASELINE configs[0]: the reference's own CPU-runnable case
    threads = host_threads()
    inp = host_inputs(pairs, 99)
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_loss_step(inp)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_loss_step(inp)
    dt = time.perf_counter() - t0
    val = pairs * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "loss step (detector x2 + dense descriptor, fwd+bwd), bounded sample of %d pairs 240x320 per step" % pairs},
        "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": threads, "host_cores": os.cpu_count(), "kind": "port",
                         "sample": "%d pairs per step, %d steps, %d BLAS threads" % (pairs, args.steps, threads)},
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 5.0:  # nvidia-smi can take a second to produce its first line
                time.sleep(0.05)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 8 for i in range(4) if r[4 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


DUMP_MAX_BYTES = 64 * 10**6
DUMP_SAMPLE = 1 << 22  # elements kept of a larger output (the two descriptor gradients, 9.8 M elements each at B32)


def dump_outputs(path, out):
    """Write what one loss step returns -- the loss scalars and the gradients of the four head outputs -- to path/<name>.npy in
    float32.  An output of more than DUMP_SAMPLE elements is reduced to the same seeded sample of its flattened elements in
    every run, so that the files of two builds can be compared element for element."""
    grads = dict(zip(("grad_semi", "grad_semi_warp", "grad_desc", "grad_desc_warp"), out["grads"]))
    arrays = {k: v for k, v in out.items() if k != "grads"}
    arrays.update(grads)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    for k, a in arrays.items():
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            arrays[k] = a.reshape(-1)[idx]
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, total
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    # keep stdout clean for the ONE JSON line: libraries (NCCL banner, warnings) write to stderr meanwhile
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import ssp_b200 as S
    from ssp_b200 import _lib, dist as sdist

    rank, world, local = sdist.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    placement = sdist.bind_to_gpu_numa_node(local)  # before the pinned staging buffers are allocated (first touch)
    group = True if world > 1 else None
    S.set_descriptor_engine(args.engine)
    B = B_PER_GPU
    NSETS = 3  # 3 x 138 MB of inputs rotate, > 126 MB L2: every step reads its inputs from HBM

    host_sets = [host_inputs(B, 1000 * rank + s) for s in range(NSETS)]
    keys = ["semi", "semi_warp", "desc", "desc_warp", "labels_2D", "warped_labels", "mat_H", "inv_H"]
    pinned = [{k: torch.from_numpy(hs[k]).pin_memory() for k in keys} for hs in host_sets]
    dsets = []
    for p in pinned:
        d = {k: p[k].to(dev) for k in keys}
        d["mask_2D"] = torch.ones((B, 1, H_IMG, W_IMG), device=dev)
        d["mask_warp_2D"] = S.compute_valid_mask(torch.tensor([H_IMG, W_IMG]), d["inv_H"], device=dev, erosion_radius=3).unsqueeze(1)
        dsets.append(d)
    for p, d in zip(pinned, dsets):
        p["mask_2D"] = d["mask_2D"].cpu().pin_memory()
        p["mask_warp_2D"] = d["mask_warp_2D"].cpu().pin_memory()
    in_keys = ["semi", "semi_warp", "desc", "desc_warp", "labels_2D", "warped_labels", "mask_2D", "mask_warp_2D", "mat_H"]
    h2d_bytes = sum(pinned[0][k].numel() * pinned[0][k].element_size() for k in in_keys)

    def step(d):
        """One eager step; returns what GraphedLossStep.replay() returns: the loss scalars and "grads" of the four leaves."""
        leaves = [d[k].detach().requires_grad_(True) for k in ("semi", "semi_warp", "desc", "desc_warp")]
        out = S.step.loss_step(leaves[0], leaves[1], leaves[2], leaves[3], d["labels_2D"], d["warped_labels"], d["mask_2D"],
                               d["mask_warp_2D"], d["mat_H"], dist_group=group)
        out["loss"].backward()
        out["grads"] = [l.grad for l in leaves]
        return out

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # kernels per step, counted on one eager step
    step(dsets[0])
    k0 = _lib.kernel_count
    step(dsets[0])
    kernels_per_step = _lib.kernel_count - k0
    use_graph = not args.no_graph  # with world > 1 the exchange kernel is captured inside the graph like any other kernel
    if use_graph:
        # fwd+bwd of the whole step captured once per input set and replayed: the step is ~25 short kernels
        graphs = [S.step.GraphedLossStep(d, dist_group=group) for d in dsets]
        run = lambda i: graphs[i % NSETS].replay()
    else:
        run = lambda i: step(dsets[i % NSETS])
    for i in range(max(args.warmup, 3)):
        run(i)
    barrier()

    # ---- timed region: K steps, device-resident inputs, CUDA events on the launching stream
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps):
        out = run(i)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    kernels = kernels_per_step * args.steps
    ms = sdist.max_over_ranks(ms, dev)
    value = B * world * args.steps / (ms * 1e-3)
    loss_val = float(out["loss"])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)  # before any later phase reuses the buffers

    # ---- everything below is secondary to the timed region above: if a later phase fails (or, with several ranks, a peer
    #      is lost and rank 0 would wait forever) the line is still printed, with e2e / roofline marked as failed
    import threading
    import traceback
    emitted = threading.Event()

    def emit(line):
        if emitted.is_set():
            return
        emitted.set()
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.write(1, (json.dumps(line) + "\n").encode())

    def bail(reason):
        if rank == 0:
            emit({"metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
                  "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                  "vs_baseline": None, "dtype": args.engine, "data": "synthetic",
                  "config": {"workload": "SSp loss step: detector loss x2 + dense descriptor loss, fwd+bwd, 32 pairs of 240x320 per GPU",
                             "per_gpu_pairs": B, "global_pairs": B * world, "engine": args.engine, "cuda_graph": use_graph},
                  "e2e": {"value": None, "unit": "pairs/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4, "error": reason},
                  "gpu_launches": kernels, "clocks": None, "roofline": None, "loss": loss_val, "incomplete": reason})
        sys.stderr.flush()
        os._exit(3)  # a phase failed (CUDA error, lost peer): the partial line above is diagnostic, the run is NOT ok

    if world > 1 and rank == 0:
        wd = threading.Timer(200.0, bail, args=("watchdog: a phase after the timed region did not finish (peer rank lost?)",))
        wd.daemon = True
        wd.start()
    try:
        # ---- e2e: same step through the public API from pinned HOST buffers, H2D inside the timed region
        #      (double-buffered on a copy stream), loss scalar read back every step
        copy_stream = torch.cuda.Stream(device=dev)
        if use_graph:
            slots = [S.step.GraphedLossStep(dsets[0], dist_group=group) for _ in range(2)]
            bufs = [g.static for g in slots]
        else:
            bufs = [{k: torch.empty_like(dsets[0][k]) for k in in_keys} for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]

        def upload(i):
            slot = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[slot])
                for k in in_keys:
                    bufs[slot][k].copy_(pinned[i % NSETS][k], non_blocking=True)
                ready[slot].record(copy_stream)

        def run_slot(slot):
            return slots[slot].replay()["loss"] if use_graph else step(bufs[slot])["loss"]

        def e2e_loop(n):
            for f in freed:
                f.record()
            upload(0)
            last = 0.0
            for i in range(n):
                slot = i % 2
                if i + 1 < n:
                    upload(i + 1)
                torch.cuda.current_stream().wait_event(ready[slot])
                l = run_slot(slot)
                freed[slot].record()
                last = float(l)  # device -> host read of the step's result
            return last

        e2e_loop(3)
        barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        e2e_loop(args.steps)
        e1.record()
        barrier()
        e2e_ms = sdist.max_over_ranks(max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0)), dev)
        e2e_val = B * world * args.steps / (e2e_ms * 1e-3)

        # ---- roofline of the dominant kernel: per-entry-point CUDA-event durations over K more steps
        # Every entry point is bracketed by CUDA events on its launching stream.  Launched eagerly, the GPU would finish each
        # kernel long before the host issues the next one, and the interval between the two events would then contain the
        # host's launch latency (tensor-map encoding, ctypes): a spin kernel in front of every step lets the host run ahead,
        # so the step's kernels execute back to back and the event pairs enclose kernel time only.
        _lib.profile_begin()
        for i in range(args.steps):
            torch.cuda._sleep(int(3.0e6))  # ~1.5 ms of device spin: longer than the host needs to enqueue one step
            step(dsets[i % NSETS])
        torch.cuda.synchronize()
        prof = _lib.profile_end()  # {entry point: (calls, total ms)}
        clocks = sampler.stop()  # sampled every 20 ms from before the timed region to the end of the profiled steps (same workload)
        # the exchange kernel's duration in these eager, event-bracketed steps is time spent WAITING for the slowest peer (the
        # ranks drift apart without the graph), not work: reported separately, never the "dominant kernel"
        xchg = prof.pop("ssp_loss_exchange", None)
        total_prof = sum(v[1] for v in prof.values())
        shares = {k: {"calls_per_step": v[0] / args.steps, "us_per_call": 1e3 * v[1] / v[0], "share": v[1] / total_prof}
                  for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}
        top = next(iter(shares))
        if xchg is not None:
            shares["ssp_loss_exchange"] = {"calls_per_step": xchg[0] / args.steps, "us_per_call": 1e3 * xchg[1] / xchg[0], "share": None,
                                           "note": "peer wait in the eager profiling pass; inside the replayed graph the step costs ms_per_step"}
        pk = peaks()
        flops_pair = 2.0 * NC * NC * DCH
        bound_tbl = {
            "ssp_desc_dense_fwd_tc": ("tensor", flops_pair * B),
            "ssp_desc_bits_gemm_tc_pair": ("tensor", 2 * flops_pair * B),  # both indicator GEMMs (dD, dDw) in one launch
            "ssp_desc_bits_gemm_tc_planes": ("tensor", flops_pair * B), "ssp_desc_pos_fwd_planes": ("hbm", 2.0 * B * NC * DCH * 4),
            "ssp_desc_dense_fwd_simt": ("tensor", flops_pair * B), "ssp_desc_bits_gemm_simt": ("tensor", flops_pair * B),
            "ssp_desc_pack": ("hbm", B * NC * DCH * 4 * 2.0), "ssp_desc_pos_fwd": ("hbm", 2.0 * B * NC * DCH * 4),
            "ssp_desc_pos_coef": ("hbm", 8.0 * B * NC * 16 * 4),
            "ssp_detector_loss_fwd_pair": ("hbm", 2 * B * (65 * NC * 4 + 2 * H_IMG * W_IMG * 4.0)),
            "ssp_detector_loss_bwd_pair": ("hbm", 2 * B * (2 * 65 * NC * 4 + 2 * H_IMG * W_IMG * 4.0)),
            "ssp_desc_pack2": ("hbm", 2 * B * NC * DCH * 4 * 2.0), "ssp_desc_pack2_geometry": ("hbm", 2 * B * NC * DCH * 4 * 2.0),
            "ssp_step_bwd_prologue": ("hbm", 2 * B * (2 * 65 * NC * 4 + 2 * H_IMG * W_IMG * 4.0) + 8.0 * B * NC * 16 * 4),
        }
        bound_tbl["ssp_desc_pos_apply"] = ("hbm", 2.0 * 3.0 * B * NC * DCH * 4)
        # the roofline is reported for the dominant KERNEL of the dense contraction / its data movement
        kind, work = bound_tbl.get(top, ("hbm", 0.0))
        dur_s = shares[top]["us_per_call"] * 1e-6
        if kind == "tensor":
            achieved, peak, unit = work / dur_s / 1e12, pk["bf16_tflops"], "TFLOP/s"
        else:
            achieved, peak, unit = work / dur_s / 1e9, pk["hbm_gbs"], "GB/s"
        # DRAM traffic of that kernel from the committed ncu --set full capture of this same command (per launch)
        traffic = None
        kern_of = {"ssp_desc_bits_gemm_tc_pair": "desc_bits_gemm_tc_kernel", "ssp_desc_bits_gemm_tc_planes": "desc_bits_gemm_tc_kernel",
                   "ssp_desc_dense_fwd_tc": "desc_dense_fwd_tc_kernel",
                   "ssp_desc_pack2": "desc_pack_kernel", "ssp_detector_loss_fwd_pair": "detector_loss_fwd_kernel",
                   "ssp_desc_pack2_geometry": "desc_pack_geometry_kernel", "ssp_step_bwd_prologue": "step_bwd_prologue_kernel",
                   "ssp_desc_pos_fwd_planes": "desc_pos_fwd_planes_kernel"}
        tpath = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
        if top in kern_of and os.path.exists(tpath) and args.engine == "bf16x3":
            traffic = json.load(open(tpath)).get(kern_of[top], {}).get("dram_bytes_per_launch")
        roofline = {"kernel": top, "bound": kind, "achieved": achieved, "peak": peak, "unit": unit, "frac": achieved / peak,
                    "traffic": traffic, "traffic_source": "profiles/r2_ncu_traffic.json (ncu --set full of this command, DRAM read + write bytes per launch)" if traffic else None, "peak_source": pk["src"] + (" burst bf16" if kind == "tensor" else " copy"),
                    "us_per_launch": shares[top]["us_per_call"],
                    "note": "algorithmic 2*Nc^2*256 flop per pair x 32 pairs per launch; bf16x3 issues 3 (fwd) / 2 (bwd) MMAs per "
                            "algorithmic MAC, so its ceiling is 1/3 (1/2) of the bf16 peak"}

        # ---- second headline of BASELINE.json: homography adaptation images/s (N=100), measured in the same run
        extra = {}
        if not args.no_adapt:
            extra = bench_adaptation(torch, S, dev, rank, world, sdist, barrier, args)
        if world == 1 and not args.no_variants:
            try:
                extra["variants"] = bench_variants(torch, S, dsets, args)
            except Exception as e:  # noqa: BLE001
                extra["variants"] = {"error": repr(e)}
        if not args.no_semantic and world == 1:  # auxiliary timing, single GPU only
            try:
                extra.update(bench_semantic(torch, S, dev, dsets, group, world, sdist, barrier, args.steps))
            except Exception as e:  # auxiliary measurement: never lose the headline line to it
                extra["with_semantic_head"] = {"error": repr(e)}

        if rank == 0:
            cpu = cpu_baseline(8, 2) if world == 1 and not args.no_cpu else None
            line = {
                "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"bf16x3": "bf16x3 (hi/lo split bf16 on tcgen05, fp32 accumulate, fp32-grade)", "bf16": "bf16", "fp32": "f32"}[args.engine],
                "data": "synthetic",
                "config": {"workload": "SSp loss step: detector loss x2 + dense descriptor loss, fwd+bwd, 32 pairs of 240x320 per GPU "
                                       "(Nc=1200 cells, 256-d), inputs = head outputs resident in HBM",
                           "per_gpu_pairs": B, "global_pairs": B * world, "engine": args.engine, "cuda_graph": use_graph,
                           "l2": "3 input sets x 138 MB rotate (> 126 MB L2)", "exchange": ("one peer-memory kernel per step (P2P stores over NVLink + flags, %s backend)" % sdist.get_exchange(True).backend) if world > 1 else "none",
                           "host_placement": placement},
                "e2e": {"value": e2e_val, "unit": "pairs/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                        "ms_per_step": e2e_ms / args.steps, "note": "pinned host inputs (head outputs + labels + masks), double-buffered H2D on a copy stream, loss read back per step; PCIe-bound"},
                "gpu_launches": kernels, "clocks": clocks, "roofline": roofline, "kernel_shares": shares, "loss": loss_val,
            }
            if cpu is not None:
                line["cpu_baseline"] = cpu
            line.update(extra)
            emit(line)
        if world > 1:
            ex = sdist.get_exchange(True)
            ex.check()  # raises if any exchange of the run timed out waiting for a peer
            torch.cuda.synchronize()
            # captured graphs go first: with the all-reduce fallback they hold NCCL kernels, and tearing the communicator down
            # under live graphs blocks forever (seen at N=2: line printed, processes never exit)
            import gc
            graphs = slots = None  # noqa: F841
            gc.collect()
            torch.cuda.synchronize()
            sdist.close_exchanges()
            torch.distributed.barrier()
            if ex.backend != "p2p":
                # everything is measured, checked and printed; NCCL's own teardown after graph capture is not worth a hang
                t = threading.Timer(20.0, lambda: os._exit(0))
                t.daemon = True
                t.start()
            torch.distributed.destroy_process_group()
    except Exception as e:  # noqa: BLE001 -- a sticky CUDA error cannot be recovered, only reported
        traceback.print_exc()
        bail("phase after the timed region failed: %r" % (e,))


def bench_variants(torch, S, dsets, args):
    """The same step on the other code paths, graph replay, CUDA events (ms per step): the single-pass bf16 engine (tensor
    operands rounded to bf16: loss within 3e-3, not the product path), the exact fp32 CUDA-core engine, fused=False
    (detector and descriptor losses as separately differentiable autograd nodes) and the reference's multi_task_loss terms
    (gradient through positive_dist / negative_dist instead of loss_desc, Train_model_heatmap_all.py:355-359)."""
    out = {}
    steps = max(5, min(args.steps, 20))
    MT = ("loss_det", "loss_det_warp", "positive_dist", "negative_dist")  # the reference's multi_task_loss terms, unit weights
    for name, engine, fused, keys in (("bf16_single_pass", "bf16", True, None), ("fp32_cuda_cores", "fp32", True, None),
                                      ("bf16x3_unfused", "bf16x3", False, None), ("bf16x3_multitask_terms", "bf16x3", False, MT)):
        S.set_descriptor_engine(engine)
        try:
            graphs = [S.step.GraphedLossStep(d, fused=fused, loss_keys=keys) for d in dsets]
            for i in range(3):
                graphs[i % len(graphs)].replay()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                graphs[i % len(graphs)].replay()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"ms_per_step": ms, "pairs_per_s": B_PER_GPU / (ms * 1e-3)}
            del graphs
        finally:
            S.set_descriptor_engine(args.engine)
    return out


def bench_semantic(torch, S, dev, dsets, group, world, sdist, barrier, steps):
    """Same loss step with the semantic head of the SSp configuration added (SURVEY 8f rank 1): two cross entropies over
    133 classes whose x8 bilinear upsample is fused into the loss (inputs: the 1/8-resolution head outputs + int64 label
    maps).  Reported next to the headline, which stays the five north-star pieces."""
    gen = torch.Generator(device=dev)
    gen.manual_seed(7)
    B = dsets[0]["semi"].shape[0]
    sets = []
    for d in dsets:
        e = dict(d)
        e["sem_pred"] = torch.randn((B, 133, HC, WC), device=dev, generator=gen) * 2
        e["sem_warp_pred"] = torch.randn((B, 133, HC, WC), device=dev, generator=gen) * 2
        e["sem"] = torch.randint(0, 134, (B, H_IMG, W_IMG), device=dev, generator=gen)
        e["warped_sem"] = torch.randint(0, 134, (B, H_IMG, W_IMG), device=dev, generator=gen)
        sets.append(e)
    graphs = [S.step.GraphedLossStep(e, dist_group=group) for e in sets]
    for i in range(3):
        graphs[i % len(graphs)].replay()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        out = graphs[i % len(graphs)].replay()
    e1.record()
    barrier()
    ms = sdist.max_over_ranks(e0.elapsed_time(e1), dev)
    return {"with_semantic_head": {"pairs_per_s": B * world * steps / (ms * 1e-3), "ms_per_step": ms / steps,
                                   "loss": float(out["loss"]), "loss_sem": float(out["loss_sem"]),
                                   "workload": "detector x2 + descriptor + semantic CE x2 (133 classes, fused x8 upsample), fwd+bwd"}}


def cpu_adaptation(n_images):
    """The reference's export hot loop on the host (oracle port): flattenDetection -> combine_heatmap -> getPtsFromHeatmap
    -> top-600 for N = 100 views per source image.  Returns images/s."""
    from oracle import ssp_oracle as O
    from ssp_b200 import synth
    rng = np.random.default_rng(77)
    Hs = np.stack([np.linalg.inv(synth.sample_homography(rng, max_angle=3.14 / 2)) for _ in range(N_ADAPT)])
    Hs[0] = np.eye(3)
    Hinv = np.linalg.inv(Hs).astype(np.float32)
    semi = synth.pseudo_normal((N_ADAPT, 65, HC, WC), 7100) * 3
    mask = O.compute_valid_mask((H_IMG, W_IMG), Hinv, 0)[:, None]
    t0 = time.perf_counter()
    for _ in range(n_images):
        heat = O.flattenDetection(semi)
        agg = O.combine_heatmap(heat, Hs.astype(np.float32)[None], mask)
        pts = O.getPtsFromHeatmap(agg[0], 0.015, 4)
        pts = pts.transpose()[:600]
    return n_images / (time.perf_counter() - t0)


def bench_adaptation(torch, S, dev, rank, world, sdist, barrier, args, images_per_step=32, steps=6):
    """Second headline of BASELINE.json: homography-adaptation images/s (N = 100 views per source image),
    export_detector_homoAdapt hot loop: flattenDetection -> combine_heatmap -> getPtsFromHeatmap -> top-k.  Source images
    are sharded over ranks (no collective).  Reports value (logits resident in HBM), e2e (pinned host logits + homographies
    uploaded inside the timed region, keypoints read back), the roofline of its dominant kernel and the CPU port."""
    from ssp_b200 import _lib, synth
    I0, N = 4, N_ADAPT  # 4 distinct synthetic source images, replicated (rescaled logits) to images_per_step
    rep = max(1, images_per_step // I0)
    rng = np.random.default_rng(500 + rank)
    Hs = np.stack([[np.linalg.inv(synth.sample_homography(rng, max_angle=3.14 / 2)) for _ in range(N)] for _ in range(I0)])
    Hs[:, 0] = np.eye(3)
    Hs = Hs.astype(np.float32)
    Hinv = torch.from_numpy(np.linalg.inv(Hs).astype(np.float32)).to(dev)
    shape_t = torch.tensor([H_IMG, W_IMG])
    sets, host_sets = [], []
    for s in range(2):  # 2 sets, each far larger than L2
        semi_h = np.concatenate([synth.pseudo_normal((I0, N, 65, HC, WC), 7000 + 10 * rank + s) * 3 * (1.0 + 0.05 * k) for k in range(rep)])
        host_sets.append(torch.from_numpy(semi_h).pin_memory())
        mask = S.compute_valid_mask(shape_t, Hinv.reshape(-1, 3, 3), device=dev).reshape(I0, N, H_IMG, W_IMG)
        sets.append((host_sets[-1].to(dev), mask.repeat(rep, 1, 1, 1)))
    Hw = torch.from_numpy(Hs).to(dev).repeat(rep, 1, 1, 1)
    Hw_host = Hw.cpu().pin_memory()
    Hinv_host = Hinv.repeat(rep, 1, 1, 1).cpu().pin_memory()
    I = I0 * rep
    for s in range(2):
        pts = S.step.adaptation_step(sets[s][0], Hw, sets[s][1], binary_mask=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        pts = S.step.adaptation_step(sets[i % 2][0], Hw, sets[i % 2][1], binary_mask=True)
    e1.record()
    barrier()
    ms = sdist.max_over_ranks(e0.elapsed_time(e1), dev)
    value = I * world * steps / (ms * 1e-3)

    # ---- e2e: pinned host logits + homographies -> device inside the timed region; the valid masks are rebuilt on the device
    #      from the uploaded inverse homographies (the reference builds them in the dataset workers), keypoints come back
    semi_d = torch.empty_like(sets[0][0])
    def e2e_step(i):
        semi_d.copy_(host_sets[i % 2], non_blocking=True)
        hw = Hw_host.to(dev, non_blocking=True)
        hinv = Hinv_host.to(dev, non_blocking=True)
        mask = S.compute_valid_mask(shape_t, hinv.reshape(-1, 3, 3), device=dev).reshape(I, N, H_IMG, W_IMG)
        return S.step.adaptation_step(semi_d, hw, mask, binary_mask=True)
    e2e_step(0)
    barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        pts = e2e_step(i)
    torch.cuda.synchronize()
    barrier()
    e2e_ms = sdist.max_over_ranks(1e3 * (time.perf_counter() - t0), dev)
    h2d = semi_d.numel() * 4 + Hw_host.numel() * 4 * 2
    d2h = int(sum(p.size for p in pts) * 8)

    # ---- roofline of the dominant kernel (per-entry-point CUDA events over the same steps)
    _lib.profile_begin()
    for i in range(steps):
        S.step.adaptation_step(sets[i % 2][0], Hw, sets[i % 2][1], binary_mask=True)
    prof = _lib.profile_end()
    tot = sum(v[1] for v in prof.values())
    shares = {k: {"calls_per_step": v[0] / steps, "us_per_call": 1e3 * v[1] / v[0], "share": v[1] / tot}
              for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}
    px = H_IMG * W_IMG * 4.0
    algo = {"ssp_combine_heatmap": I * (2 * N + 1) * px, "ssp_combine_heatmap_tiled": I * (2 * N + 1) * px,
            "ssp_combine_heatmap_bits": I * (2 * N + 1) * px, "ssp_combine_heatmap_signed": I * (N + 1) * px,
            "ssp_flatten_detection_masked": I * N * (65 * NC * 4.0 + 2 * px),
            "ssp_flatten_detection": I * N * (65 * NC * 4.0 + px), "ssp_nms_fast": I * (px + 12.0 * 600),
            "ssp_mask_pack_bits": I * N * (px + px / 32)}
    top = next(iter(shares))
    pk = peaks()
    dur = shares[top]["us_per_call"] * 1e-6
    ach = algo.get(top, 0.0) / dur / 1e9
    roof = {"kernel": top, "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
            "traffic": None, "peak_source": pk["src"] + " copy", "us_per_launch": shares[top]["us_per_call"],
            "note": "algorithmic bytes per source image (SURVEY 8d): flatten 61.9 MB + combine (2N+1)*H*W*4 = 61.75 MB + NMS 0.3 MB "
                    "= 124 MB; whole pipeline = %.3f of the HBM peak" % (124.0e6 * value / world / 1e9 / pk["hbm_gbs"])}
    out = {"metric": "homography-adapt imgs/s (N=100)", "value": value, "unit": "images/s", "n_gpus": world,
           "images_per_step_per_gpu": I, "steps": steps, "ms_per_step": ms / steps, "scaling": "weak", "dtype": "f32",
           "keypoints_first_image": int(pts[0].shape[0]),
           "config": {"workload": "export_detector_homoAdapt hot loop: flatten + aggregate + NMS + top-600 for 100 warped views of 240x320 per source image, "
                                  "%d source images per step per GPU, detector logits resident in HBM" % I,
                      "l2": "2 logit sets x %.0f MB rotate (> 126 MB L2)" % (semi_d.numel() * 4 / 1e6)},
           "e2e": {"value": I * world * steps / (e2e_ms * 1e-3), "unit": "images/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": d2h,
                   "ms_per_step": e2e_ms / steps,
                   "note": "pinned host logits of the 100 views + homographies uploaded every step, valid masks rebuilt on the device, keypoints read back; PCIe-bound"},
           "roofline": roof, "kernel_shares": shares}
    if rank == 0 and world == 1 and not args.no_cpu:
        v = cpu_adaptation(2)
        out["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": host_threads(), "host_cores": os.cpu_count(), "kind": "port",
                               "sample": "2 source images x 100 views (numpy oracle port of flattenDetection + combine_heatmap + getPtsFromHeatmap)"}
    return {"homography_adaptation": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--engine", default="bf16x3", choices=["bf16x3", "bf16", "fp32"])
    ap.add_argument("--no-adapt", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--graph-multi", action="store_true", help="(default now) kept for compatibility")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip the timings of the other engines / fused=False")
    ap.add_argument("--no-semantic", action="store_true", help="skip the auxiliary step timing with the semantic head")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss scalars and input gradients of the last timed step "
                    "(rank 0) to DIR/<name>.npy; the inputs are seeded, so runs with the same arguments are comparable")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
