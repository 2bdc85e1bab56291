"""The fused loss step -- the path bench.py times: step.GraphedLossStep over losses.LossStepFn, bf16x3 engine, B = 32 of
240x320 -- against oracle.loss_step, eager and replayed from a CUDA graph; the launch paths only this step runs (the mask
folded into the indicator words, lambda_loss applied inside the coefficient kernel, the fused backward prologue, the
standalone coefficient launch when only the descriptors need a gradient); graph replay with new inputs and the
determinism it relies on; the descriptor kernels at the edges of their tiles; and the two NaN signals the step documents
(sparse-list overflow, a soft mask on the fused step).

Tolerances are those of tests/test_gpu_parity.py (DESIGN.md section 2): 1e-4 on the fp32-grade engines, with the
pair-mask boundary slack on the descriptor scalars and the cells next to a hinge kink or the distance threshold excused
in the descriptor gradients; the single-pass bf16 engine at BF16_LOSS_RTOL / BF16_GRAD_COS.
"""
import contextlib

import numpy as np
import pytest
import torch

import bench
import ssp_b200 as S
from oracle import ssp_oracle as O
from ssp_b200 import synth

pytestmark = pytest.mark.gpu
TOL = 1e-4
BF16_LOSS_RTOL = 3e-3
BF16_GRAD_COS = 0.995
DEV = "cuda"
LEAVES = ("semi", "semi_warp", "desc", "desc_warp")
SCALARS = ("loss", "loss_det", "loss_det_warp", "loss_desc", "positive_dist", "negative_dist")
MULTI_TASK = ("loss_det", "loss_det_warp", "positive_dist", "negative_dist")  # the reference's multi_task_loss terms


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def host(t):
    return t.detach().cpu().numpy()


@contextlib.contextmanager
def overflow_check(on):
    """losses.CHECK_LIST_OVERFLOW is a module global (test_gpu_parity turns it on at import); a host sync cannot be
    captured into a graph."""
    old = S.losses.CHECK_LIST_OVERFLOW
    S.losses.CHECK_LIST_OVERFLOW = on
    try:
        yield
    finally:
        S.losses.CHECK_LIST_OVERFLOW = old


# ------------------------------------------------------------------ inputs and oracle, cached per input set
_sets, _oracle = {}, {}


def bench_set(s):
    """bench.host_inputs(32, s) on the device, with the masks run_ours builds: mask_2D all ones, mask_warp_2D the valid mask
    of the inverse homography eroded by 3."""
    key = ("bench", s)
    if key not in _sets:
        h = bench.host_inputs(bench.B_PER_GPU, s)
        d = {k: cu(h[k]) for k in LEAVES + ("labels_2D", "warped_labels", "mat_H", "inv_H")}
        d["mask_2D"] = torch.ones((bench.B_PER_GPU, 1, bench.H_IMG, bench.W_IMG), device=DEV)
        d["mask_warp_2D"] = S.compute_valid_mask(torch.tensor([bench.H_IMG, bench.W_IMG]), d["inv_H"], device=DEV,
                                                 erosion_radius=3).unsqueeze(1)
        _sets[key] = d
    return _sets[key]


def mild_homographies(B, seed):
    """Near-identity homographies (normalised coordinates): every grid, down to 2x3 cells, keeps positive pairs."""
    rng = np.random.default_rng(seed)
    Hs = np.tile(np.eye(3), (B, 1, 1))
    Hs[:, :2, :2] += rng.uniform(-0.08, 0.08, (B, 2, 2))
    Hs[:, :2, 2] = rng.uniform(-0.15, 0.15, (B, 2))
    Hs[:, 2, :2] = rng.uniform(-0.03, 0.03, (B, 2))
    return Hs.astype(np.float32)


def random_homographies(B, seed):
    rng = np.random.default_rng(seed)
    return np.stack([np.linalg.inv(synth.sample_homography(rng)) for _ in range(B)]).astype(np.float32)


def shrink(f):
    """Scale by f about the image centre (normalised coordinates): 1/f^2 rows share the neighbourhood of one column."""
    return np.diag([f, f, 1.0]).astype(np.float32)


def synth_set(name, B, Hc, Wc, seed, Hs=None, mask_warp=None, mix=0.12):
    """Loss-step inputs at any grid.  desc_warp = normalise(independent + mix * desc): bench's independent descriptors put
    almost no pair above the 0.2 negative margin; mix = 0.12 puts about one pair in a hundred there, so the negative hinge
    and its coefficients carry weight while pairs within 1e-5 of the margin stay rare.  mask_warp: a [B,1,8Hc,8Wc] array,
    or None for the valid mask of the inverse homographies eroded by 3 (as run_ours builds it)."""
    key = ("synth", name)
    if key not in _sets:
        H, W = 8 * Hc, 8 * Wc
        Hs = random_homographies(B, seed) if Hs is None else np.asarray(Hs, np.float32)
        D = synth.unit_descriptors(B, 256, Hc, Wc, seed * 10 + 3, smooth=0.5)
        Dw = synth.unit_descriptors(B, 256, Hc, Wc, seed * 10 + 4, smooth=0.5) + np.float32(mix) * D
        Dw /= np.sqrt((Dw.astype(np.float64) ** 2).sum(axis=1, keepdims=True)).astype(np.float32)
        d = {"semi": cu(synth.pseudo_normal((B, 65, Hc, Wc), seed * 10 + 1)),
             "semi_warp": cu(synth.pseudo_normal((B, 65, Hc, Wc), seed * 10 + 2)), "desc": cu(D), "desc_warp": cu(Dw),
             "labels_2D": cu(synth.keypoint_labels(B, H, W, seed * 10 + 5, p=0.02)),
             "warped_labels": cu(synth.keypoint_labels(B, H, W, seed * 10 + 6, p=0.02)),
             "mat_H": cu(Hs), "mask_2D": torch.ones((B, 1, H, W), device=DEV)}
        if mask_warp is None:
            mask_warp = host(S.compute_valid_mask(torch.tensor([H, W]), cu(np.linalg.inv(Hs).astype(np.float32)), device=DEV,
                                                  erosion_radius=3).unsqueeze(1))
        d["mask_warp_2D"] = cu(np.asarray(mask_warp, np.float32))
        _sets[key] = d
    return _sets[key]


def mix_for(Nc):
    """A row meets Nc columns, and the pairs within 1e-5 of the 0.2 margin (excused in the gradient check) grow with Nc times
    the share of pairs near the margin: more mixing on tiny grids (which then still have negatives), less on KITTI."""
    return 0.4 if Nc < 128 else (0.12 if Nc < 4096 else 0.05)


def holey_mask(B, Hc, Wc, seed):
    """Binary pixel mask with scattered zero pixels: getMasks zeroes about one cell in six."""
    return (synth.uniform((B, 1, 8 * Hc, 8 * Wc), seed) > 0.003).astype(np.float32)


def oracle_step(key, d, lamda_d=250.0, descriptor_dist=4.0, lambda_loss=1.0, weighting="uniform"):
    """oracle.loss_step on input set `d` (named `key`) with the pair-mask slack and the unstable cells of its descriptors,
    computed once per set and parameters: engines and eager / graph runs share it."""
    kw = dict(lamda_d=lamda_d, descriptor_dist=descriptor_dist, lambda_loss=lambda_loss, weighting=weighting)
    ck = (key, tuple(sorted(kw.items())))
    if ck not in _oracle:
        a = {k: host(v) for k, v in d.items()}
        ref = O.loss_step(*(a[k] for k in ("semi", "semi_warp", "desc", "desc_warp", "labels_2D", "warped_labels", "mask_2D",
                                           "mask_warp_2D", "mat_H")), **kw)
        mv = O.getMasks(a["mask_warp_2D"])[:, None]
        ref["slack"] = O.descriptor_boundary_slack(a["desc"], a["desc_warp"], a["mat_H"], mv, lamda_d=lamda_d,
                                                   descriptor_dist=descriptor_dist, eps=1e-3, per_term=True)
        ref["unstable"] = O.descriptor_unstable_cells(a["desc"], a["desc_warp"], a["mat_H"], descriptor_dist=descriptor_dist)
        _oracle[ck] = ref
    return _oracle[ck]


# ------------------------------------------------------------------ running the step
def run_eager(d, engine="bf16x3", fused=True, loss_keys=None, grad_on=LEAVES, **kw):
    """One eager step; returns what GraphedLossStep.replay() returns (loss scalars + "grads" of the four head outputs)."""
    leaves = {k: d[k].detach().requires_grad_(k in grad_on) for k in LEAVES}
    out = S.step.loss_step(leaves["semi"], leaves["semi_warp"], leaves["desc"], leaves["desc_warp"], d["labels_2D"],
                           d["warped_labels"], d["mask_2D"], d["mask_warp_2D"], d["mat_H"], engine=engine, fused=fused, **kw)
    total = out["loss"] if not loss_keys else sum(out[k] for k in loss_keys)
    total.backward()
    res = {k: v.detach() for k, v in out.items()}
    res["grads"] = [leaves[k].grad for k in LEAVES]
    return res


def graphed(d, **kw):
    with overflow_check(False):
        g = S.step.GraphedLossStep(d, **kw)
    torch.cuda.synchronize()
    return g


def snap(out):
    """A copy of a replay's outputs (the next replay of the same graph overwrites them)."""
    res = {k: v.clone() for k, v in out.items() if k != "grads"}
    res["grads"] = [None if g is None else g.clone() for g in out["grads"]]
    return res


def assert_identical(a, b, what):
    for k in SCALARS:
        assert torch.equal(a[k], b[k]), (what, k, float(a[k]), float(b[k]))
    for i, (x, y) in enumerate(zip(a["grads"], b["grads"])):
        assert torch.equal(x, y), (what, LEAVES[i], float((x - y).abs().max()))


# ------------------------------------------------------------------ comparing with the oracle
def close(a, b, rtol=TOL, atol=1e-6, what=""):
    a = host(a) if isinstance(a, torch.Tensor) else np.asarray(a)
    np.testing.assert_allclose(a.astype(np.float64), np.asarray(b, np.float64), rtol=rtol, atol=atol, err_msg=str(what))


def check_scalars(out, ref, lambda_loss=1.0, weighting="uniform", rtol=TOL, what=""):
    """Detector scalars at TOL; descriptor scalars (and the totals containing them) at rtol plus the pair-mask slack of
    each term."""
    s_loss, s_pos, s_neg = ref["slack"]
    slack = {"loss": lambda_loss * s_loss if weighting == "uniform" else s_pos + s_neg, "loss_det": 0.0,
             "loss_det_warp": 0.0, "loss_desc": s_loss, "positive_dist": s_pos, "negative_dist": s_neg}
    for k in SCALARS:
        close(out[k], ref[k], rtol=rtol if k not in ("loss_det", "loss_det_warp") else TOL, atol=slack[k] + 1e-9,
              what=(what, k))


def check_desc_grad(got, want, unstable, what=""):
    """Per cell (max over the 256 channels) within 1e-4 of the gradient scale; cells whose gradient is discontinuous at this
    input (oracle.descriptor_unstable_cells) are excused, must stay rare and still be of the right magnitude."""
    B = want.shape[0]
    got = host(got).reshape(B, want.shape[1], -1)
    want = want.reshape(B, want.shape[1], -1)
    scale = np.abs(want).max()
    assert scale > 0, what
    err = np.abs(got - want).max(axis=1)
    bad = (err > 1e-4 * scale) & ~unstable
    assert not bad.any(), "%s: %d stable cells off by up to %.3g of the gradient scale" % (
        what, bad.sum(), (err * ~unstable).max() / scale)
    assert unstable.mean() < 0.03 or unstable.sum() <= 2, (what, unstable.sum())
    assert err.max() < 600.0 * scale, what


def cosine(a, b):
    a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
    return float((a * b).sum() / np.sqrt((a * a).sum() * (b * b).sum()))


def check_step(out, ref, engine="bf16x3", lambda_loss=1.0, weighting="uniform", grad_on=LEAVES, what=""):
    exact = engine != "bf16"
    check_scalars(out, ref, lambda_loss, weighting, rtol=TOL if exact else BF16_LOSS_RTOL, what=what)
    rows, cols = ref["unstable"]
    for i, k in enumerate(LEAVES):
        got, want = out["grads"][i], ref["grads"][i]
        if k not in grad_on:
            assert got is None, (what, k)
        elif k.startswith("semi"):  # the detector loss does not depend on the descriptor engine
            close(got, want, atol=1e-4 * np.abs(want).max(), what=(what, k))
        elif exact:
            check_desc_grad(got, want, rows if k == "desc" else cols, what=(what, k))
        else:
            c = cosine(host(got), want)
            assert c > BF16_GRAD_COS, (what, k, c)


def max_list_lengths(Hs, Hc, Wc, dist):
    """Longest positive-pair row list and column list of the oracle's pair mask."""
    m, _ = O.descriptor_pair_mask(Hs, Hc, Wc, 8, dist)
    return int(m.sum(axis=2).max()), int(m.sum(axis=1).max())


# ------------------------------------------------------------------ the benchmarked step
@pytest.mark.parametrize("mode", ["eager", "graph"])
def test_bench_step_vs_oracle(mode):
    """bench.py's step on its own inputs (B = 32, 30x40 cells, bf16x3, fused), eager and replayed, against the oracle."""
    d = bench_set(0)
    ref = oracle_step("bench0", d)
    if mode == "eager":
        with overflow_check(True):
            out = run_eager(d)
    else:
        out = graphed(d).replay()
    torch.cuda.synchronize()
    check_step(out, ref, what=mode)


# (name, B, Hc, Wc, homographies, engine, fused, weighting, lamda_d, descriptor_dist, lambda_loss)
CASES = {
    # long row lists (4 partners: the full-list branch of the coefficient kernel) on the fold path, lambda_loss != 1
    # through gscale
    "rows_lambda0.25_dist7.5": (4, 30, 40, "random", "bf16x3", True, "uniform", 800.0, 7.5, 0.25),
    "rows_lambda3_dist8": (4, 30, 40, "random", "bf16x3", True, "uniform", 800.0, 8.0, 3.0),
    # 0.3x shrink: column lists longer than 4 (pos_coef_cols<DESC_MAXP>)
    "cols_shrink0.3": (3, 30, 40, "shrink0.3", "bf16x3", True, "uniform", 250.0, 4.0, 1.5),
    "kitti_47x155": (3, 47, 155, "random", "bf16x3", True, "uniform", 250.0, 4.0, 2.0),
    "bf16_fused": (4, 30, 40, "random", "bf16", True, "uniform", 250.0, 4.0, 0.5),
    "fp32_fused": (4, 30, 40, "random", "fp32", True, "uniform", 250.0, 4.0, 3.0),
    "multitask_unfused": (4, 30, 40, "random", "bf16x3", False, "multi_task", 250.0, 4.0, 1.0),
}


def case_inputs(name):
    B, Hc, Wc, hs = CASES[name][:4]
    seed = 10 + sorted(CASES).index(name)
    Hs = random_homographies(B, seed)
    if hs == "shrink0.3":
        Hs[0] = shrink(0.3)
        Hs[1] = shrink(0.3) @ mild_homographies(1, seed)[0]
    return name, synth_set(name, B, Hc, Wc, seed, Hs=Hs, mix=mix_for(Hc * Wc))


@pytest.mark.parametrize("mode", ["eager", "graph"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_step_variants_vs_oracle(name, mode):
    B, Hc, Wc, hs, engine, fused, weighting, lamda_d, dist, lam = CASES[name]
    key, d = case_inputs(name)
    rmax, cmax = max_list_lengths(host(d["mat_H"]), Hc, Wc, dist)
    assert rmax <= 16 and cmax <= 16
    if name.startswith("rows"):
        assert rmax >= 4, rmax  # a filled 4th slot sends a row to pos_coef_rows<DESC_MAXP>
    if name.startswith("cols"):
        assert cmax > 4, cmax
    ref = oracle_step(key, d, lamda_d, dist, lam, weighting)
    kw = dict(engine=engine, fused=fused, lamda_d=lamda_d, descriptor_dist=dist, lambda_loss=lam)
    keys = MULTI_TASK if weighting == "multi_task" else None
    if mode == "eager":
        with overflow_check(True):
            out = run_eager(d, loss_keys=keys, **kw)
    else:
        out = graphed(d, loss_keys=keys, **kw).replay()
    torch.cuda.synchronize()
    if weighting == "multi_task":
        # out["loss"] is the uniform total whatever is differentiated; the oracle's is the multi-task one
        close(out["loss"], float(ref["loss_det"]) + float(ref["loss_det_warp"]) + lam * float(ref["loss_desc"]),
              atol=lam * ref["slack"][0] + 1e-9, what="uniform total")
        out = dict(out, loss=out["loss_det"] + out["loss_det_warp"] + out["positive_dist"] + out["negative_dist"])
    check_step(out, ref, engine, lam, weighting, what=(name, mode))


@pytest.mark.parametrize("grad_on", [("desc", "desc_warp"), ("semi", "semi_warp")], ids=["descriptors", "logits"])
def test_step_partial_gradients(grad_on):
    """Only the descriptors need a gradient: the fold backward launches the coefficient kernel on its own (alpha, srow and
    the bitsC transpose included) instead of the fused prologue.  Only the logits: the detector-only backward."""
    key, d = case_inputs("rows_lambda3_dist8")
    lamda_d, dist, lam = CASES["rows_lambda3_dist8"][7:]
    ref = oracle_step(key, d, lamda_d, dist, lam)
    with overflow_check(True):
        out = run_eager(d, grad_on=grad_on, lamda_d=lamda_d, descriptor_dist=dist, lambda_loss=lam)
    torch.cuda.synchronize()
    check_step(out, ref, lambda_loss=lam, grad_on=grad_on, what=grad_on)


def test_step_all_zero_warp_mask():
    """mask_warp_2D = 0 everywhere: loss_desc is 0 and both descriptor gradients are exactly zero (every column is folded
    out of the indicator words and every positive coefficient carries mv = 0); pos / neg and the detector terms are
    unchanged in kind and still match the oracle."""
    B, Hc, Wc = 3, 30, 40
    d = synth_set("zero_mask", B, Hc, Wc, 31, mask_warp=np.zeros((B, 1, 8 * Hc, 8 * Wc), np.float32))
    ref = oracle_step("zero_mask", d, lambda_loss=2.0)
    assert float(ref["loss_desc"]) == 0.0 and float(ref["positive_dist"]) > 0 and float(ref["negative_dist"]) > 0
    for engine in ("bf16x3", "fp32"):
        with overflow_check(True):
            out = run_eager(d, engine=engine, lambda_loss=2.0)
        torch.cuda.synchronize()
        assert float(out["loss_desc"]) == 0.0, engine
        for i in (2, 3):
            assert bool((out["grads"][i] == 0).all()), (engine, LEAVES[i])
        check_scalars(out, ref, 2.0, what=engine)
        for i in (0, 1):
            close(out["grads"][i], ref["grads"][i], atol=1e-4 * max(np.abs(ref["grads"][i]).max(), 1e-30), what=(engine, i))


# ------------------------------------------------------------------ graph replay with new inputs, determinism
def test_graph_reload_replays_new_inputs():
    """bench's e2e pattern: a graph captured on set A, then load(B) -> replay == the oracle for B, then load(A) -> replay is
    bit-identical to the first replay of A (nothing of B is left behind in the graph's buffers)."""
    A, Bset = bench_set(0), bench_set(1)
    g = graphed(A)
    first = snap(g.replay())
    g.load(Bset)
    second = snap(g.replay())
    g.load(A)
    third = g.replay()
    torch.cuda.synchronize()
    check_step(second, oracle_step("bench1", Bset), what="set B")
    assert_identical(first, third, "A after B")
    assert not torch.equal(first["grads"][2], second["grads"][2])


def test_graph_slots_with_copy_stream():
    """Two graphs alive at once, as in bench's e2e phase: the next input set is uploaded from pinned host memory into one
    slot's static buffers on a copy stream while the other slot replays.  Every slot result equals the eager step on the
    set it was given."""
    sets = [bench_set(0), bench_set(1)]
    with overflow_check(True):
        eager = [snap(run_eager(d)) for d in sets]
    keys = S.step.GraphedLossStep.IN_KEYS
    pinned = [{k: d[k].cpu().pin_memory() for k in keys} for d in sets]
    slots = [graphed(sets[0]) for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    order = [1, 0, 0, 1, 1, 0]  # input set of step i; slot i % 2 sees both sets, in both orders

    def upload(i):
        slot = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[slot])
            for k in keys:
                slots[slot].static[k].copy_(pinned[order[i]][k], non_blocking=True)
            ready[slot].record(copy_stream)

    for f in freed:
        f.record()
    upload(0)
    results = []
    for i in range(len(order)):
        slot = i % 2
        if i + 1 < len(order):
            upload(i + 1)
        torch.cuda.current_stream().wait_event(ready[slot])
        results.append(snap(slots[slot].replay()))
        freed[slot].record()
    torch.cuda.synchronize()
    for i, r in enumerate(results):
        assert_identical(r, eager[order[i]], "step %d (slot %d, set %d)" % (i, i % 2, order[i]))


@pytest.mark.parametrize("engine", ["bf16x3", "bf16", "fp32"])
def test_step_deterministic(engine):
    """Fixed summation order (DESIGN section 3): the same eager step twice, and the same graph replayed twice, give
    bit-identical scalars and gradients, and the replay equals the eager step."""
    d = bench_set(0)
    with overflow_check(True):
        a = snap(run_eager(d, engine=engine))
        b = run_eager(d, engine=engine)
    assert_identical(a, b, "eager")
    g = graphed(d, engine=engine)
    r1 = snap(g.replay())
    r2 = g.replay()
    torch.cuda.synchronize()
    assert_identical(r1, r2, "replay")
    assert_identical(a, r1, "eager vs replay")


def test_backward_twice_over_retained_graph():
    """Two backward(retain_graph=True) calls over one graph give the same gradients: the backward leaves the saved pair
    lists as the forward wrote them.  Bit-identical on descriptor_loss (each engine) and the fused dense step, whose
    summation order is fixed; within 1e-5 of the largest element on the fused sparse step, whose scatter backward adds
    with fp32 atomics."""
    d = bench_set(0)
    mv = S.getMasks(d["mask_warp_2D"], 8, device=DEV).unsqueeze(1)

    def step(**kw):
        return lambda *leaves: S.step.loss_step(*leaves, d["labels_2D"], d["warped_labels"], d["mask_2D"], d["mask_warp_2D"],
                                                d["mat_H"], **kw)["loss"]

    def desc(engine):
        def run(semi, semi_w, D, Dw):
            loss, _, pos, neg = S.descriptor_loss(D, Dw, d["mat_H"], mask_valid=mv, device=DEV, engine=engine)
            return loss + 0.5 * pos + 0.25 * neg
        return run

    cases = [("descriptor_loss " + e, desc(e), 0.0) for e in ("bf16x3", "bf16", "fp32")]
    cases += [("fused dense step", step(), 0.0),
              ("fused sparse step", step(descriptor_loss="sparse", sampler=S.sparse.DeviceSampler(11, DEV)), 1e-5)]
    for what, run, rtol in cases:
        leaves = [d[k].detach().requires_grad_(True) for k in LEAVES]
        total = run(*leaves)
        grads = []
        for _ in range(2):
            for t in leaves:
                t.grad = None
            total.backward(retain_graph=True)
            grads.append([t.grad for t in leaves])
        torch.cuda.synchronize()
        for name, a, b in zip(LEAVES, *grads):
            assert (a is None) == (b is None), (what, name)
            if a is not None:
                assert float((a - b).abs().max()) <= rtol * float(a.abs().max()), (what, name)


# ------------------------------------------------------------------ tile edges of the descriptor kernels
# Hc x Wc: exact multiples of 256 cells (no padding rows), 264 (a 16-wide last column tile: 8 cells per CTA in the TMA
# box), 255, 1023, and fewer than 128 cells (the second CTA of a pair holds only padding)
EDGE_SHAPES = [(16, 16), (16, 32), (11, 24), (15, 17), (31, 33), (5, 7), (2, 3)]
EDGE_CASES = [(hc, wc, b) for hc, wc in EDGE_SHAPES for b in (1, 3)] + [(5, 7, 75)]  # B = 75: 75 items on 74 clusters


def edge_inputs(Hc, Wc, B, masked):
    seed = 1000 + 37 * Hc + Wc + B
    Hs = mild_homographies(B, seed)
    Hs[1::2] = random_homographies(B, seed)[1::2]
    mask = holey_mask(B, Hc, Wc, seed) if masked else np.ones((B, 1, 8 * Hc, 8 * Wc), np.float32)
    name = "edge_%dx%d_b%d_%s" % (Hc, Wc, B, "holes" if masked else "ones")
    return name, synth_set(name, B, Hc, Wc, seed, Hs=Hs, mask_warp=mask, mix=mix_for(Hc * Wc))


_edge_desc = {}


def oracle_desc(name, d, g3):
    if name not in _edge_desc:
        D, Dw, Hs = host(d["desc"]), host(d["desc_warp"]), host(d["mat_H"])
        mv = O.getMasks(host(d["mask_warp_2D"]))[:, None]
        ref = O.descriptor_loss(D, Dw, Hs, mv, grad=g3)
        slack = O.descriptor_boundary_slack(D, Dw, Hs, mv, eps=1e-3, per_term=True)
        _edge_desc[name] = (ref, slack, O.descriptor_unstable_cells(D, Dw, Hs), mv)
    return _edge_desc[name]


@pytest.mark.parametrize("engine", ["bf16x3", "fp32", "bf16"])
@pytest.mark.parametrize("Hc,Wc,B", EDGE_CASES)
def test_descriptor_tile_edges(Hc, Wc, B, engine):
    """descriptor_loss (unfused, g = (1, 0.5, 0.25)) and the fused step, with a mask with holes and an all-ones mask."""
    exact = engine != "bf16"
    rt = TOL if exact else BF16_LOSS_RTOL
    g3 = (1.0, 0.5, 0.25)
    for masked in (True, False):
        name, d = edge_inputs(Hc, Wc, B, masked)
        (loss_r, _, pos_r, neg_r, dD_r, dDw_r), slack, (rows, cols), mv = oracle_desc(name, d, g3)
        assert float(pos_r) > 0 and float(neg_r) > 0, name
        what = (name, engine)
        Dt, Dwt = d["desc"].detach().requires_grad_(True), d["desc_warp"].detach().requires_grad_(True)
        with overflow_check(True):
            loss, _, pos, neg = S.descriptor_loss(Dt, Dwt, d["mat_H"], mask_valid=cu(mv), device=DEV, engine=engine)
            (g3[0] * loss + g3[1] * pos + g3[2] * neg).backward()
        torch.cuda.synchronize()
        for got, want, sl, k in zip((loss, pos, neg), (loss_r, pos_r, neg_r), slack, ("loss", "pos", "neg")):
            close(got, want, rtol=rt, atol=sl + 1e-9, what=(what, k))
        for got, want, unstable, k in ((Dt.grad, dD_r, rows, "dD"), (Dwt.grad, dDw_r, cols, "dDw")):
            if exact:
                check_desc_grad(got, want, unstable, what=(what, k))
            else:
                assert cosine(host(got), want) > BF16_GRAD_COS, (what, k)
        ref = oracle_step(name, d, lambda_loss=1.5)
        with overflow_check(True):
            out = run_eager(d, engine=engine, lambda_loss=1.5)
        torch.cuda.synchronize()
        check_step(out, ref, engine, 1.5, what=(what, "fused"))


# ------------------------------------------------------------------ documented NaN signals
def test_list_overflow_is_nan_and_raises_when_checked():
    """A 0.1x shrink at descriptor_dist = 4 puts far more than 16 rows next to one column: the sparse lists overflow (the
    list writes are bounds-checked), the loss is NaN on both the unfused and the fused path, and CHECK_LIST_OVERFLOW
    turns the count into an exception."""
    B, Hc, Wc = 2, 30, 40
    Hs = np.stack([shrink(0.1), shrink(0.1) @ mild_homographies(1, 5)[0]])
    assert max_list_lengths(Hs, Hc, Wc, 4.0)[1] > 16
    d = synth_set("overflow", B, Hc, Wc, 41, Hs=Hs, mask_warp=np.ones((B, 1, 8 * Hc, 8 * Wc), np.float32))
    leaves = [d[k].detach().requires_grad_(True) for k in LEAVES]

    def unfused(engine):
        return S.descriptor_loss(leaves[2], leaves[3], d["mat_H"], device=DEV, engine=engine)

    def fused(engine):  # forward only: the signal is the loss
        return S.step.loss_step(*leaves, d["labels_2D"], d["warped_labels"], d["mask_2D"], d["mask_warp_2D"], d["mat_H"],
                                engine=engine)

    for engine in ("bf16x3", "fp32"):
        with overflow_check(False):
            loss, _, pos, _ = unfused(engine)
            out = fused(engine)
        torch.cuda.synchronize()
        assert torch.isnan(loss).item() and torch.isnan(pos).item(), engine
        assert torch.isnan(out["loss"]).item() and torch.isnan(out["loss_desc"]).item(), engine
        with overflow_check(True):
            with pytest.raises(RuntimeError, match="overflowed"):
                unfused(engine)
            with pytest.raises(RuntimeError, match="overflowed"):
                fused(engine)


def test_soft_mask_fused_nan_unfused_matches_oracle():
    """A non-binary mask_warp_2D cannot be folded into the indicator words: the fused step poisons its loss with NaN; the
    same input on fused=False (alpha * Dw packed per column) matches the oracle."""
    B, Hc, Wc = 3, 30, 40
    Hs = random_homographies(B, 51)
    mask = host(S.compute_valid_mask(torch.tensor([8 * Hc, 8 * Wc]), cu(np.linalg.inv(Hs).astype(np.float32)), device=DEV,
                                     erosion_radius=3).unsqueeze(1))
    soft = synth.uniform((B, 1, Hc, Wc), 52) < 0.3
    corner = mask[:, :, ::8, ::8]  # a view: the first pixel of every cell
    corner[soft] *= 0.5            # about 30 % of the cells: getMasks gives those that are valid 0.5
    assert 0.0 < ((O.getMasks(mask) != 0) & (O.getMasks(mask) != 1)).mean() < 0.5
    d = synth_set("soft_mask", B, Hc, Wc, 51, Hs=Hs, mask_warp=mask)
    with overflow_check(True):
        fused = run_eager(d)
        unfused = run_eager(d, fused=False)
    torch.cuda.synchronize()
    assert torch.isnan(fused["loss"]).item() and torch.isnan(fused["loss_desc"]).item()
    check_step(unfused, oracle_step("soft_mask", d), what="fused=False")
