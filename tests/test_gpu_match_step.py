"""The batched descriptor export on the GPU: step.match_step (NMS -> descriptors -> two-way matches of P image pairs in one
call) and utils.nn_match_two_way_batch (the tensor-core matcher), against the live reference's fixtures, the oracle and the
single-image functions.

The matcher multiplies bf16 hi / lo splits (three MMA passes), so its dot products carry ~1e-6 of error where the reference's
float32 BLAS carries its own: a row or column whose two best candidates (or whose best candidate and the threshold) lie
closer than that may legitimately resolve either way.  `check_matches` excuses exactly those, from exact float64 dots."""
import numpy as np
import pytest
import torch

import ssp_b200 as S
from oracle import ssp_oracle as O
from ssp_b200 import synth

pytestmark = pytest.mark.gpu
DEV = "cuda"
DELTA = 2e-5  # excusal margin in dot-product units


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def unit_cols(D, K, seed):
    x = synth.pseudo_normal((D, K), seed).astype(np.float64)
    return (x / np.sqrt((x * x).sum(0, keepdims=True))).astype(np.float32)


def related(d1, K2, seed, noise=0.5):
    """K2 descriptors: a shuffled subset of d1's columns plus noise, renormalised (many mutual matches, some not)."""
    perm = np.argsort(synth.uniform((max(d1.shape[1], K2),), seed))[:K2] % d1.shape[1]
    x = d1[:, perm].astype(np.float64) + noise * unit_cols(d1.shape[0], K2, seed + 1)
    return (x / np.sqrt((x * x).sum(0, keepdims=True))).astype(np.float32)


def _excused(G, thr):
    if G.shape[1] > 1:
        top = -np.partition(-G, 1, axis=1)[:, :2]
        gap = top[:, 0] - top[:, 1]
    else:
        top, gap = G[:, :1], np.full(G.shape[0], np.inf)
    return (gap < DELTA) | (np.abs(top[:, 0] - (1.0 - thr * thr / 2.0)) < DELTA)


def check_matches(got, d1, d2, thr):
    """got vs O.nn_match_two_way(d1, d2, thr): the same index pairs except at excused rows / columns and their partners
    (at most 0.5 % of the rows excused), squared distances within 4e-5, increasing index-1 order."""
    ref = O.nn_match_two_way(d1, d2, thr)
    assert got.dtype == np.float64 and got.shape[0] == 3
    n1, n2 = d1.shape[1], d2.shape[1]
    if n1 == 0 or n2 == 0:
        assert got.shape == (3, 0)
        return
    G = d1.astype(np.float64).T @ d2.astype(np.float64)
    er, ec = _excused(G, thr), _excused(G.T, thr)
    assert er.sum() <= 0.005 * n1 + 1, (er.sum(), n1)
    rows = set(np.flatnonzero(er).tolist()) | set(G[:, ec].argmax(0).tolist())
    cols = set(np.flatnonzero(ec).tolist()) | set(G[er].argmax(1).tolist())
    a = {(int(i), int(j)): s for i, j, s in got.T}
    b = {(int(i), int(j)): s for i, j, s in ref.T}
    for i, j in a.keys() ^ b.keys():
        assert i in rows or j in cols, (i, j, (i, j) in a)
    for k in a.keys() & b.keys():
        assert abs(a[k] ** 2 - b[k] ** 2) <= 4e-5, (k, a[k], b[k])
    assert np.all(np.diff(got[0]) > 0)
    assert len(a.keys() & b.keys()) >= 0.99 * len(b) - 2


# ------------------------------------------------------------------ nn_match_two_way_batch
def test_batch_matcher_golden(golden):
    """Index pairs of the live reference's fixture, at P = 1 and as three copies with columns past the counts."""
    g = golden("matching")
    d1, d2 = g["desc1"], g["desc2"]
    pad1 = np.concatenate([d1, unit_cols(256, 37, 901)], axis=1)
    pad2 = np.concatenate([d2, unit_cols(256, 300, 902)], axis=1)
    for thr, key in ((0.36, "matches_36"), (0.7, "matches_70")):
        (m,) = S.utils.nn_match_two_way_batch(cu(d1[None]), cu(d2[None]), thr)
        assert np.array_equal(m[:2], g[key][:2])
        np.testing.assert_allclose(m[2], g[key][2], atol=2e-4)
        ms = S.utils.nn_match_two_way_batch(cu(np.stack([pad1] * 3)), cu(np.stack([pad2] * 3)), thr,
                                            counts1=[90] * 3, counts2=torch.tensor([73] * 3, device=DEV))
        for mm in ms:
            assert np.array_equal(mm[:2], g[key][:2])
            assert np.array_equal(mm, ms[0])


def test_batch_matcher_against_oracle():
    """8 pairs of 1000 x 937 points (the HPatches export's top-k size)."""
    P, K1, K2 = 8, 1000, 937
    d1 = np.stack([unit_cols(256, K1, 1000 + p) for p in range(P)])
    d2 = np.stack([related(d1[p], K2, 2000 + 7 * p) for p in range(P)])
    out = S.utils.nn_match_two_way_batch(cu(d1), cu(d2), 0.7)
    assert len(out) == P
    for p in range(P):
        assert out[p].shape[1] > 100
        check_matches(out[p], d1[p], d2[p], 0.7)


def test_batch_matcher_ragged_counts():
    """Ragged pairs around the 128-point tiles, up to 6000 points; columns past a pair's count hold unrelated descriptors."""
    K = 6000
    c1 = [0, 1, 127, 128, 129, 255, 256, 257, 6000]
    c2 = [5, 1, 300, 129, 128, 1000, 256, 257, 6000]
    P = len(c1)
    d1 = np.stack([unit_cols(256, K, 3000 + p) for p in range(P)])
    d2 = np.stack([np.concatenate([related(d1[p][:, :max(c1[p], 1)], c2[p], 4000 + p), unit_cols(256, K - c2[p], 5000 + p)],
                                  axis=1) for p in range(P)])
    out = S.utils.nn_match_two_way_batch(cu(d1), cu(d2), 0.7, counts1=c1, counts2=c2)
    for p in range(P):
        check_matches(out[p], d1[p][:, :c1[p]], d2[p][:, :c2[p]], 0.7)
    assert out[0].shape == (3, 0) and out[1].shape[1] <= 1 and out[-1].shape[1] > 1000


def test_batch_matcher_exact_cases():
    """Duplicate descriptors: the lowest index wins both ways.  A permutation: every point matches its partner."""
    base = unit_cols(256, 200, 77)
    a = np.r_[np.arange(200), [0, 5, 5, 199]]
    b = np.r_[np.argsort(synth.uniform((200,), 78)), [7, 7, 0, 150]]
    d1, d2 = base[:, a], base[:, b]
    (m,) = S.utils.nn_match_two_way_batch(cu(d1[None]), cu(d2[None]), 0.7)
    first_col = {}
    for j, v in enumerate(b):
        first_col.setdefault(int(v), j)
    want = [(i, first_col[int(v)]) for i, v in enumerate(a) if i == int(np.flatnonzero(a == v)[0])]
    assert [tuple(x) for x in m[:2].T.astype(int)] == want
    assert np.all(m[2] < 5e-3)
    perm = np.argsort(synth.uniform((1500,), 79))
    d1 = unit_cols(256, 1500, 80)
    (m,) = S.utils.nn_match_two_way_batch(cu(d1[None]), cu(d1[:, perm][None]), 0.7)
    inv = np.argsort(perm)
    assert np.array_equal(m[0], np.arange(1500)) and np.array_equal(m[1], inv)


# ------------------------------------------------------------------ match_step
def export_inputs(P, Hc, Wc, seed):
    semi = synth.adaptation_workload(1, 2 * P, Hc, Wc, seed)[0][0]
    desc = synth.unit_descriptors(P, 256, Hc, Wc, 31 + seed, smooth=0.4).astype(np.float64)
    other = synth.unit_descriptors(P, 256, Hc, Wc, 32 + seed, smooth=0.4)
    dw = desc + 0.5 * other
    dw /= np.sqrt((dw * dw).sum(axis=1, keepdims=True))
    return cu(semi[:P]), cu(desc.astype(np.float32)), cu(semi[P:]), cu(dw.astype(np.float32))


@pytest.mark.parametrize("top_k", [None, 1000])
def test_match_step_equals_per_image_calls(top_k):
    """480 x 640, 4 pairs: points and descriptors of the single-image functions bit for bit, matches against the oracle."""
    semi, desc, semi_w, desc_w = export_inputs(4, 60, 80, 0)
    out = S.step.match_step(semi, desc, semi_w, desc_w, conf_thresh=0.015, nms_dist=4, top_k=top_k, nn_thresh=0.7)
    assert len(out) == 4
    for p, r in enumerate(out):
        for key, s, d in (("", semi, desc), ("warped_", semi_w, desc_w)):
            pts = S.getPtsFromHeatmap(S.flattenDetection(s[p]).squeeze(0), 0.015, 4)[:, :top_k]
            assert pts.shape[1] > (900 if top_k else 4000)
            assert np.array_equal(r[key + "pts"], pts)
            ref = S.utils.sample_desc_from_points(d[p:p + 1], pts)
            assert r[key + "desc"].dtype == np.float32 and np.array_equal(r[key + "desc"], ref)
        check_matches(r["matches"], r["desc"], r["warped_desc"], 0.7)
    again = S.step.match_step(semi, desc, semi_w, desc_w, top_k=top_k)
    for r, r2 in zip(out, again):
        for k in r:
            assert np.array_equal(r[k], r2[k]), k


def test_match_step_against_oracle_chain():
    """240 x 320, 3 pairs, every stage in the oracle: flattenDetection, getPtsFromHeatmap, sample_desc_from_points,
    nn_match_two_way (points matched by position, descriptors to 1e-6)."""
    semi, desc, semi_w, desc_w = export_inputs(3, 30, 40, 5)
    out = S.step.match_step(semi, desc, semi_w, desc_w)
    for p, r in enumerate(out):
        order, ref_desc = [], []
        for key, s, d in (("", semi, desc), ("warped_", semi_w, desc_w)):
            ref = O.getPtsFromHeatmap(O.flattenDetection(s[p].cpu().numpy())[0], 0.015, 4)
            got = r[key + "pts"]
            pos = {(x, y): i for i, (x, y) in enumerate(ref[:2].T)}
            assert got.shape == ref.shape and set(pos) == {(x, y) for x, y in got[:2].T}
            idx = np.array([pos[(x, y)] for x, y in got[:2].T])
            np.testing.assert_allclose(got[2], ref[2, idx], atol=1e-6)
            rd = O.sample_desc_from_points(d[p:p + 1].cpu().numpy(), ref)
            np.testing.assert_allclose(r[key + "desc"], rd[:, idx], atol=1e-6)
            order.append(idx)
            ref_desc.append(rd)
        m = r["matches"].copy()
        m[0], m[1] = order[0][m[0].astype(int)], order[1][m[1].astype(int)]
        m = m[:, np.argsort(m[0])]
        check_matches(m, ref_desc[0], ref_desc[1], 0.7)


def test_match_step_empty_and_uneven():
    """P = 1 with an image without points (K1 != K2 = 0), and a batch where no image has a point."""
    semi, desc, semi_w, desc_w = export_inputs(1, 30, 40, 9)
    blank = torch.zeros_like(semi_w)
    blank[:, 64] = 50.0  # all mass on the dustbin: an empty heatmap
    (r,) = S.step.match_step(semi, desc, blank, desc_w)
    assert r["pts"].shape[1] > 100 and r["desc"].shape == (256, r["pts"].shape[1])
    assert r["warped_pts"].shape == (3, 0) and r["warped_desc"].shape == (256, 0) and r["matches"].shape == (3, 0)
    (r,) = S.step.match_step(blank, desc, blank, desc_w)
    assert r["pts"].shape == (3, 0) and r["desc"].shape == (256, 0) and r["matches"].shape == (3, 0)
    rs = S.step.match_step(torch.cat([semi, semi]), torch.cat([desc, desc]), torch.cat([semi_w, semi]),
                           torch.cat([desc_w, desc]), top_k=300)
    assert rs[0]["pts"].shape[1] == 300 and rs[1]["matches"].shape[1] == 300  # an image against itself matches fully
