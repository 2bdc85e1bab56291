"""The sparse loss step on device-sampled correspondences: sparse.DeviceSampler (ssp_sparse_sample) against the candidate
oracle (sparse_oracle.sparse_candidates), the structure and distribution of its draws, its reproducibility from a saved
state, and loss_step(descriptor_loss="sparse") eager and replayed from a CUDA graph against the oracle on the lists it drew.

Candidate sets may differ from the oracle only at cells whose warp lies within TIE_EPS of a rounding tie (the device and
numpy compute T^-1 H T and the warp in different operation orders).  Distribution tests run at fixed seeds, so their outcome
is deterministic; their thresholds are set so that a correct sampler fails them with probability below 1e-6.
"""
import numpy as np
import pytest
import torch
from scipy import stats

import bench
import ssp_b200 as S
from oracle import ssp_oracle as O
from sparse_oracle import sparse_candidates
from ssp_b200 import synth
from test_gpu_loss_step import bench_set, cu, host, mild_homographies, random_homographies, shrink, synth_set

pytestmark = pytest.mark.gpu
TOL = 1e-4
TIE_EPS = 1e-3
P_FAIL = 1e-6
DEV = "cuda"
LEAVES = ("semi", "semi_warp", "desc", "desc_warp")
SCALARS = ("loss", "loss_det", "loss_det_warp", "loss_desc", "positive_dist", "negative_dist")


def draw(sampler, Hs, Hc, Wc, K=1000, n=10):
    ia, ib, M = sampler.sample(cu(np.asarray(Hs, np.float32)), Hc, Wc, K, n)
    torch.cuda.synchronize()
    return host(ia).astype(np.int64), host(ib).astype(np.int64), host(M).astype(np.int64)


def zoom_homographies(B, seed):
    """The inverse of test_gpu_loss_step's 0.3x shrink (a 3.3x zoom about the centre; mat_H maps cells of the image to
    cells of the warped image): only the middle 0.3 of each axis lands inside, M is about 0.09 of the cells (M < K at
    30x40), and the draws with replacement fill the rest."""
    Hs = np.stack([np.linalg.inv(shrink(0.3)) for _ in range(B)])
    Hs[1:] = Hs[1:] @ mild_homographies(B - 1, seed)
    return Hs.astype(np.float32)


def check_candidates(H, Hc, Wc, M, pairs, every):
    """pairs (a, b) drawn for one image: all candidates of the oracle; every=True: the set is the oracle's whole set.  Only
    cells within TIE_EPS of a rounding tie may differ."""
    c = sparse_candidates(H, Hc, Wc)
    ours = set(zip(c["a"].tolist(), c["b"].tolist()))
    loose = np.nonzero(c["tie"] < TIE_EPS)[0]
    assert abs(int(M) - c["a"].size) <= loose.size, (M, c["a"].size, loose.size)
    drawn = set(pairs)
    diff = {a for a, _ in (drawn - ours if not every else drawn ^ ours)}
    assert diff <= set(loose.tolist()), sorted(diff - set(loose.tolist()))[:10]
    return c


# ------------------------------------------------------------------ candidates
def candidate_cases():
    h = bench.host_inputs(bench.B_PER_GPU, 0)["mat_H"]
    return {"bench_30x40_b32": (h, 30, 40), "kitti_47x155_b3": (random_homographies(3, 61), 47, 155),
            "60x80_b4": (random_homographies(4, 62), 60, 80)}


@pytest.mark.parametrize("name", ["bench_30x40_b32", "kitti_47x155_b3", "60x80_b4"])
def test_candidates_vs_oracle(name):
    """M[b] and the drawn pairs agree with sparse_candidates; with K above the cell count every candidate is drawn, so the
    drawn set is the whole candidate set."""
    Hs, Hc, Wc = candidate_cases()[name]
    s = S.sparse.DeviceSampler(1, DEV)
    ia, ib, M = draw(s, Hs, Hc, Wc)
    ia_all, ib_all, M_all = draw(s, Hs, Hc, Wc, K=Hc * Wc + 1, n=0)
    assert np.array_equal(M, M_all)
    for b in range(len(Hs)):
        check_candidates(Hs[b], Hc, Wc, M[b], list(zip(ia[b, :1000].tolist(), ib[b, :1000].tolist())), every=False)
        check_candidates(Hs[b], Hc, Wc, M_all[b], list(zip(ia_all[b].tolist(), ib_all[b].tolist())), every=True)


# ------------------------------------------------------------------ structure of a draw
def test_structure_m_at_least_k():
    """M >= K: the K matches are distinct candidates; non_a repeats matches_a n times; non_b lies in [0, Nc)."""
    Hc, Wc, K, n = 30, 40, 600, 10
    Hs = mild_homographies(4, 71)
    ia, ib, M = draw(S.sparse.DeviceSampler(2, DEV), Hs, Hc, Wc, K, n)
    assert ia.shape == (4, K + K * n) and np.all(M >= K), M
    for b in range(4):
        assert len(np.unique(ia[b, :K])) == K
        c = check_candidates(Hs[b], Hc, Wc, M[b], list(zip(ia[b, :K].tolist(), ib[b, :K].tolist())), every=False)
        assert np.array_equal(ia[b, K:], np.repeat(ia[b, :K], n))
        assert ib[b, K:].min() >= 0 and ib[b, K:].max() < Hc * Wc
        assert c["a"].size >= K


def test_structure_m_below_k():
    """M < K (zoom_homographies): the first M matches are every candidate once, the total is K, every repeat is a candidate."""
    Hc, Wc, K, n = 30, 40, 1000, 3
    Hs = zoom_homographies(3, 72)
    ia, ib, M = draw(S.sparse.DeviceSampler(3, DEV), Hs, Hc, Wc, K, n)
    assert np.all(M < K) and np.all(M > 0), M
    for b in range(3):
        m = int(M[b])
        first = list(zip(ia[b, :m].tolist(), ib[b, :m].tolist()))
        assert len(set(first)) == m
        check_candidates(Hs[b], Hc, Wc, m, first, every=True)
        assert set(zip(ia[b, m:K].tolist(), ib[b, m:K].tolist())) <= set(first)
        assert np.array_equal(ia[b, K:], np.repeat(ia[b, :K], n))
        assert ib[b, K:].min() >= 0 and ib[b, K:].max() < Hc * Wc


# ------------------------------------------------------------------ distribution
def test_inclusion_frequency():
    """M >= K: over 400 draws every candidate is among the K matches with frequency K/M (binomial per candidate; the
    threshold is Bonferroni-corrected over the candidates)."""
    Hc, Wc, K, draws = 30, 40, 300, 400
    Hs = mild_homographies(2, 73)
    s = S.sparse.DeviceSampler(4, DEV)
    counts = np.zeros((2, Hc * Wc))
    for _ in range(draws):
        ia, _, M = draw(s, Hs, Hc, Wc, K, 0)
        for b in range(2):
            np.add.at(counts[b], ia[b], 1)
    for b in range(2):
        m = int(M[b])
        p = K / m
        cand = counts[b] > 0
        assert cand.sum() == m
        z = np.abs(counts[b][cand] - draws * p) / np.sqrt(draws * p * (1 - p))
        assert z.max() < stats.norm.isf(P_FAIL / (2 * m)), (b, z.max())
        # the first rank is a uniform candidate too
    first = np.zeros(Hc * Wc)
    for _ in range(draws):
        ia, _, M = draw(s, Hs[:1], Hc, Wc, K, 0)
        first[ia[0, 0]] += 1
    assert first.sum() == draws and first.max() <= stats.binom.isf(P_FAIL / Hc / Wc, draws, 1.0 / int(M[0]))


def test_non_match_cells_uniform():
    """Chi-square of non_b over the cells: 40 draws x 4 images x 10 000 non-matches at 30x40."""
    Hc, Wc = 30, 40
    Hs = random_homographies(4, 74)
    s = S.sparse.DeviceSampler(5, DEV)
    counts = np.zeros(Hc * Wc)
    for _ in range(40):
        _, ib, _ = draw(s, Hs, Hc, Wc)
        counts += np.bincount(ib[:, 1000:].ravel(), minlength=Hc * Wc)
    e = counts.sum() / counts.size
    chi = ((counts - e) ** 2 / e).sum()
    assert stats.chi2.sf(chi, counts.size - 1) > P_FAIL, chi


def test_with_replacement_fill_uniform():
    """M < K: the K - M fill draws are uniform over the M candidates (chi-square over 60 draws of 3 images)."""
    Hc, Wc, K = 30, 40, 1000
    Hs = zoom_homographies(3, 75)
    s = S.sparse.DeviceSampler(6, DEV)
    chis = [np.zeros(Hc * Wc) for _ in range(3)]
    for _ in range(60):
        ia, _, M = draw(s, Hs, Hc, Wc, K, 0)
        for b in range(3):
            np.add.at(chis[b], ia[b, int(M[b]):], 1)
    for b in range(3):
        m = int(M[b])
        c = chis[b][chis[b] > 0]
        assert c.size == m
        e = c.sum() / m
        chi = ((c - e) ** 2 / e).sum()
        assert stats.chi2.sf(chi, m - 1) > P_FAIL / 3, (b, chi, m)


# ------------------------------------------------------------------ reproducibility
def test_state_reproduces_and_advances():
    Hs = bench.host_inputs(4, 3)["mat_H"]
    s = S.sparse.DeviceSampler(123, DEV)
    st = s.get_state()
    assert host(st).tolist() == [123, 0]
    a = draw(s, Hs, 30, 40)
    assert host(s.get_state()).tolist() == [123, 1]  # one launch advances the counter by one
    b = draw(s, Hs, 30, 40)
    assert not np.array_equal(a[0], b[0]) and not np.array_equal(a[1], b[1])
    s.set_state(st)
    assert torch.equal(s.get_state(), st)
    a2 = draw(s, Hs, 30, 40)
    b2 = draw(s, Hs, 30, 40)
    for x, y in zip(a + b, a2 + b2):
        assert np.array_equal(x, y)
    other = draw(S.sparse.DeviceSampler(124, DEV), Hs, 30, 40)
    assert not np.array_equal(other[1], a[1])
    assert s.empty_images() == 0


def test_graph_replays_equal_eager_calls():
    """Replay k of a captured sparse step equals eager step k from the same starting state: lists and loss scalars bit for
    bit, gradients within fp32 reordering (the scatter backward uses atomics).  Replays draw fresh lists."""
    d = bench_set(0)
    s = S.sparse.DeviceSampler(7, DEV)
    st = s.get_state()
    g = S.step.GraphedLossStep(d, descriptor_loss="sparse", sampler=s)
    assert torch.equal(s.get_state(), st)  # the warm-up steps restore the state
    replays = [snap(g.replay()) for _ in range(3)]
    torch.cuda.synchronize()
    s.set_state(st)
    eager = [snap(run_eager(d, sampler=s)) for _ in range(3)]
    torch.cuda.synchronize()
    assert not torch.equal(replays[0]["lists"][0], replays[1]["lists"][0])
    for k, (r, e) in enumerate(zip(replays, eager)):
        for x, y in zip(r["lists"], e["lists"]):
            assert torch.equal(x, y), k
        for key in SCALARS:
            assert torch.equal(r[key], e[key]), (k, key)
        for i, (x, y) in enumerate(zip(r["grads"], e["grads"])):
            scale = float(y.abs().max())
            assert float((x - y).abs().max()) <= 1e-5 * scale, (k, LEAVES[i])


# ------------------------------------------------------------------ the step against the oracle
def run_eager(d, grad_on=LEAVES, loss_keys=None, sem=False, **kw):
    leaves = {k: d[k].detach().requires_grad_(k in grad_on) for k in LEAVES}
    extra = {}
    if sem:
        extra = {"sem_pred": d["sem_pred"].detach().requires_grad_(True), "sem": d["sem"],
                 "sem_warp_pred": d["sem_warp_pred"].detach().requires_grad_(True), "warped_sem": d["warped_sem"]}
    out = S.step.loss_step(leaves["semi"], leaves["semi_warp"], leaves["desc"], leaves["desc_warp"], d["labels_2D"],
                           d["warped_labels"], d["mask_2D"], d["mask_warp_2D"], d["mat_H"], descriptor_loss="sparse",
                           **extra, **kw)
    total = out["loss"] if not loss_keys else sum(out[k] for k in loss_keys)
    total.backward()
    res = {k: v.detach() for k, v in out.items()}
    res["grads"] = [leaves[k].grad for k in LEAVES]
    if sem:
        res["grads"] += [extra["sem_pred"].grad, extra["sem_warp_pred"].grad]
    res["lists"] = kw["sampler"].last
    return res


def snap(out):
    res = {k: v.clone() for k, v in out.items() if k not in ("grads", "lists")}
    res["grads"] = [None if g is None else g.clone() for g in out["grads"]]
    res["lists"] = tuple(t.clone() for t in out["lists"])
    return res


def oracle_sparse_step(d, lists, K, lamda_d=250.0, lambda_loss=1.0, weighting="uniform", sem=False):
    """O.detector_loss x2 + O.sparse_descriptor_loss on the drawn lists (+ O.sem_loss x2): scalars and gradients."""
    a = {k: host(v) for k, v in d.items()}
    ia, ib = host(lists[0]).astype(np.int64), host(lists[1]).astype(np.int64)
    l0, g0 = O.detector_loss(a["semi"], O.labels2Dto3D(a["labels_2D"]), O.getMasks(a["mask_2D"]), grad=True)
    l1, g1 = O.detector_loss(a["semi_warp"], O.labels2Dto3D(a["warped_labels"]), O.getMasks(a["mask_warp_2D"]), grad=True)
    gw = (lambda_loss, 0.0, 0.0) if weighting == "uniform" else (0.0, 1.0, 1.0)
    ld, pos, neg, dD, dDw = O.sparse_descriptor_loss(a["desc"], a["desc_warp"], ia[:, :K], ib[:, :K], ia[:, K:], ib[:, K:],
                                                     lamda_d, grad=gw)
    total = float(l0) + float(l1) + (lambda_loss * float(ld) if weighting == "uniform" else float(pos) + float(neg))
    ref = {"loss": total, "loss_det": l0, "loss_det_warp": l1, "loss_desc": ld, "positive_dist": pos, "negative_dist": neg,
           "grads": [g0, g1, dD, dDw], "flip": hard_count_slack(a["desc"], a["desc_warp"], ia[:, K:], ib[:, K:])}
    if sem:
        r1, d1 = O.sem_loss(a["sem_pred"], a["sem"], grad=True)
        r2, d2 = O.sem_loss(a["sem_warp_pred"], a["warped_sem"], grad=True)
        ref["loss"] += float(r1) + float(r2)
        ref.update(loss_sem=r1, loss_sem_warp=r2)
        ref["grads"] += [d1, d2]
    return ref


def hard_count_slack(D, Dw, na, nb, eps=1e-5):
    """A non-match dot within eps of the 0.2 margin may fall on either side of it in fp32: it moves the hard-negative count
    of its image by one, which scales that image's non-match mean and coefficients by up to 1/(hard + 1).  Returns the
    largest such relative change over the batch (0 when no dot is that close)."""
    B, Dch = D.shape[:2]
    A, Bm = D.reshape(B, Dch, -1).astype(np.float64), Dw.reshape(B, Dch, -1).astype(np.float64)
    worst = 0.0
    for b in range(B):
        dn = (A[b][:, na[b]] * Bm[b][:, nb[b]]).sum(0)
        near = int((np.abs(dn - 0.2) < eps).sum())
        worst = max(worst, near / (int((dn > 0.2).sum()) + 1.0))
    return worst


def check_vs_oracle(out, ref, what):
    """Scalars at TOL, gradients at TOL of their largest element; the descriptor terms also get the hard-count slack."""
    flip = ref["flip"]
    assert flip < 0.01, (what, flip)
    for k in SCALARS + tuple(k for k in ("loss_sem", "loss_sem_warp") if k in ref):
        rtol = TOL + (flip if k in ("loss", "loss_desc", "negative_dist") else 0.0)
        np.testing.assert_allclose(float(out[k]), float(ref[k]), rtol=rtol, atol=1e-7, err_msg=str((what, k)))
    for i, (got, want) in enumerate(zip(out["grads"], ref["grads"])):
        scale = np.abs(want).max()
        assert scale > 0, (what, i)
        atol = (TOL + (flip if i in (2, 3) else 0.0)) * scale
        np.testing.assert_allclose(host(got), want, rtol=0, atol=atol, err_msg=str((what, i)))


def sem_inputs(d, seed):
    B, _, Hc, Wc = d["semi"].shape
    rng = np.random.default_rng(seed)
    d = dict(d)
    d["sem_pred"] = cu(synth.pseudo_normal((B, 133, Hc, Wc), seed + 1) * 2)
    d["sem_warp_pred"] = cu(synth.pseudo_normal((B, 133, Hc, Wc), seed + 2) * 2)
    d["sem"] = cu(rng.integers(0, 134, (B, 8 * Hc, 8 * Wc)))
    d["warped_sem"] = cu(rng.integers(0, 134, (B, 8 * Hc, 8 * Wc)))
    return d


# (inputs, lamda_d, lambda_loss, fused, weighting, semantic, K, n)
STEP_CASES = {
    "bench_b32": ("bench", 250.0, 1.0, True, "uniform", False, 1000, 10),
    "kitti_47x155_b3": ("kitti", 250.0, 1.0, True, "uniform", False, 1000, 10),
    "zoom_m_below_k": ("zoom", 250.0, 1.5, True, "uniform", False, 1000, 10),
    "lambda_loss2.5_lamda_d100": ("synth", 100.0, 2.5, True, "uniform", False, 1000, 10),
    "multitask_unfused": ("synth", 250.0, 1.0, False, "multi_task", False, 500, 4),
    "semantic": ("synth", 250.0, 0.5, True, "uniform", True, 1000, 10),
}


def step_inputs(kind):
    if kind == "bench":
        return bench_set(0)
    if kind == "kitti":
        return synth_set("sparse_kitti", 3, 47, 155, 81, mix=0.3)
    if kind == "zoom":
        return synth_set("sparse_zoom", 3, 30, 40, 82, Hs=zoom_homographies(3, 82), mix=0.3)
    return synth_set("sparse_synth", 4, 30, 40, 83, mix=0.3)


@pytest.mark.parametrize("mode", ["eager", "graph"])
@pytest.mark.parametrize("name", sorted(STEP_CASES))
def test_sparse_step_vs_oracle(name, mode):
    """Read back the drawn lists and compare the six scalars and the four gradients with O.detector_loss x2 plus
    O.sparse_descriptor_loss on those lists (+ the semantic cross entropies) at 1e-4."""
    kind, lamda_d, lam, fused, weighting, sem, K, n = STEP_CASES[name]
    d = step_inputs(kind)
    if sem:
        d = sem_inputs(d, 84)
    s = S.sparse.DeviceSampler(8, DEV)
    keys = ("loss_det", "loss_det_warp", "positive_dist", "negative_dist") if weighting == "multi_task" else None
    kw = dict(sampler=s, lamda_d=lamda_d, lambda_loss=lam, fused=fused, num_matching_attempts=K,
              num_masked_non_matches_per_match=n)
    if mode == "eager":
        out = run_eager(d, loss_keys=keys, sem=sem, **kw)
    else:
        example = {k: d[k] for k in S.step.GraphedLossStep.IN_KEYS + (S.step.GraphedLossStep.SEM_KEYS if sem else ())}
        g = S.step.GraphedLossStep(example, loss_keys=keys, descriptor_loss="sparse", **kw)
        g.replay()
        out = g.replay()  # the second replay: its own fresh lists
    torch.cuda.synchronize()
    ia, _, M = out["lists"]
    assert ia.shape == (d["semi"].shape[0], K + K * n)
    if kind == "zoom":
        assert bool((M < K).all()), M
    ref = oracle_sparse_step(d, out["lists"], K, lamda_d, lam, weighting, sem)
    if weighting == "multi_task":
        np.testing.assert_allclose(float(out["loss"]), float(ref["loss_det"]) + float(ref["loss_det_warp"]) +
                                   lam * float(ref["loss_desc"]), rtol=TOL)
        out = dict(out, loss=out["loss_det"] + out["loss_det_warp"] + out["positive_dist"] + out["negative_dist"])
    check_vs_oracle(out, ref, (name, mode))


def test_batch_descriptor_loss_sparse_device_sampler():
    """The drop-in's entry point with sampler= takes the device path; the host path is unchanged without it."""
    d = step_inputs("synth")
    s = S.sparse.DeviceSampler(9, DEV)
    D, Dw = d["desc"].detach().requires_grad_(True), d["desc_warp"].detach().requires_grad_(True)
    loss, none, pos, neg = S.batch_descriptor_loss_sparse(D, Dw, d["mat_H"], device=DEV, lamda_d=250, sampler=s)
    (loss + 0.5 * pos + 0.25 * neg).backward()
    torch.cuda.synchronize()
    ia, ib, _ = (host(t).astype(np.int64) for t in s.last)
    K = 1000
    r = O.sparse_descriptor_loss(host(d["desc"]), host(d["desc_warp"]), ia[:, :K], ib[:, :K], ia[:, K:], ib[:, K:], 250,
                                 grad=(1.0, 0.5, 0.25))
    assert none is None
    for got, want in zip((loss, pos, neg), r[:3]):
        np.testing.assert_allclose(float(got.detach()), float(want), rtol=TOL)
    for got, want in ((D.grad, r[3]), (Dw.grad, r[4])):
        np.testing.assert_allclose(host(got), want, rtol=0, atol=TOL * np.abs(want).max())


# ------------------------------------------------------------------ NaN signal
def test_empty_image_is_nan_and_raises_when_checked():
    """A homography that maps no cell inside: M = 0, the loss of the fused and the unfused step is NaN, the flag counts the
    image, and CHECK_EMPTY_IMAGES turns it into an exception."""
    d = dict(step_inputs("synth"))
    Hs = host(d["mat_H"]).copy()
    Hs[1] = np.array([[1, 0, 5.0], [0, 1, 5.0], [0, 0, 1]], np.float32)  # 2.5 image widths to the right and down
    d["mat_H"] = cu(Hs)
    s = S.sparse.DeviceSampler(10, DEV)
    for fused in (True, False):
        out = run_eager(d, sampler=s, fused=fused)
        torch.cuda.synchronize()
        assert int(out["lists"][2][1]) == 0 and int(out["lists"][2][0]) > 0
        for k in ("loss", "loss_desc", "positive_dist", "negative_dist"):
            assert torch.isnan(out[k]).item(), (fused, k)
        assert not torch.isnan(out["loss_det"]).item()
    assert s.empty_images() == 2
    old = S.sparse.CHECK_EMPTY_IMAGES
    S.sparse.CHECK_EMPTY_IMAGES = True
    try:
        with pytest.raises(RuntimeError, match="maps no cell"):
            s.sample(d["mat_H"], 30, 40)
    finally:
        S.sparse.CHECK_EMPTY_IMAGES = old
