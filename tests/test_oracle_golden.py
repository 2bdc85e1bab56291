"""oracle/ssp_oracle.py against outputs of the live reference (tests/golden/*.npz, made by make_golden.py).
This is the pin of the oracle: the reference itself has no fixtures for the path (SURVEY 4 / 8c)."""
import numpy as np

from oracle import ssp_oracle as O
from ssp_b200 import synth

TOL = 1e-4  # relative, the north_star tolerance for coordinates / pixels / losses / gradients


def close(a, b, rtol=TOL, atol=1e-6):
    np.testing.assert_allclose(np.asarray(a, np.float64), np.asarray(b, np.float64), rtol=rtol, atol=atol)


def test_warp_points(golden):
    g = golden("warp_points")
    close(O.warp_points(g["pts"], g["H"]), g["out_batched"])
    close(O.warp_points(g["pts"], g["H"][1]), g["out_single"])
    fp, fm = O.filter_points(g["pix"], [64, 48], return_mask=True)
    assert np.array_equal(fm, g["filt_mask"]) and np.array_equal(fp, g["filt_pts"])


def test_inv_warp(golden):
    g = golden("inv_warp")
    close(O.inv_warp_image_batch(g["img"], g["Hinv"], "bilinear"), g["out_bilinear"], atol=2e-6)
    on = O.inv_warp_image_batch(g["img"], g["Hinv"], "nearest")
    assert (on != g["out_nearest"]).mean() < 1e-3  # nearest ties at exact half pixels may flip
    close(O.inv_warp_image_batch(g["img"][0, 0], g["Hinv"][0])[0, 0], g["out_single"], atol=2e-6)
    close(O.inv_warp_image_batch(g["img"][:1], np.eye(3, dtype=np.float32)), g["out_identity"], atol=2e-6)


def test_valid_mask_and_ellipse(golden):
    g = golden("valid_mask")
    for r in range(1, 9):
        assert np.array_equal(O.ellipse_kernel(r), g["ellipse_%d" % r]), r
    for r in (0, 1, 3):
        m = O.compute_valid_mask((48, 64), g["Hinv5"], r)
        assert (m != g["mask_r%d" % r]).sum() <= 2, r
    m = O.compute_valid_mask((240, 320), g["Hinv2"], 3)
    assert (m != g["mask_240_r3"]).sum() <= 4
    assert np.array_equal(O.compute_valid_mask((48, 64), np.eye(3), 3), g["mask_identity_r3"])


def test_labels_and_detector_loss(golden):
    g = golden("detector")
    close(O.labels2Dto3D(g["lab_bin"]), g["l3_bin"])
    close(O.labels2Dto3D(g["lab_soft"]), g["l3_soft"])
    close(O.labels2Dto3D(g["lab_tiny"]), g["l3_tiny"])
    close(O.labels2Dto3D(g["lab_bin"], add_dustbin=False), g["l3_nodust"])
    close(O.getMasks(g["mask2d"]), g["mask3d"])
    loss, d = O.detector_loss(g["semi"], g["l3_bin"], g["mask3d"], grad=True)
    close(loss, g["loss"])
    close(d, g["dsemi"], atol=1e-7)
    loss2, d2 = O.detector_loss(g["semi2"], g["l3_soft"], g["mask3d"], grad=True)
    close(loss2, g["loss2"])
    close(d2 * g["g2"], g["dsemi2"], atol=1e-7)


def test_flatten_and_combine(golden):
    g = golden("flatten")
    close(O.flattenDetection(g["semi"]), g["heat"])
    close(O.flattenDetection(g["semi"][0]), g["heat3d"])
    c = golden("combine")
    out = O.combine_heatmap(c["heat"], c["Hwarp"][None], c["mask"])
    assert np.array_equal(np.isnan(out), np.isnan(c["out"]))
    close(np.nan_to_num(out), np.nan_to_num(c["out"]), atol=2e-6)


def test_nms(golden):
    g = golden("nms")
    for key, (h, w, seed, thr, r) in {"pts_120": (120, 160, 61, 0.015, 4), "pts_240": (240, 320, 62, 0.015, 4),
                                      "pts_64": (64, 96, 63, 0.03, 2)}.items():
        pts = O.getPtsFromHeatmap(synth.unique_heatmap(h, w, seed), thr, r)
        assert pts.dtype == np.float64 and np.array_equal(pts, g[key]), key
    assert np.array_equal(O.getPtsFromHeatmap(g["sparse"], 0.015, 4), g["pts_sparse"])
    one = np.zeros((48, 64), np.float32); one[20, 30] = 0.5
    assert np.array_equal(O.getPtsFromHeatmap(one, 0.015, 4), g["pts_one"])
    assert O.getPtsFromHeatmap(np.zeros((48, 64), np.float32), 0.015, 4).shape == (3, 0)
    out, inds = O.nms_fast(g["corners"], 48, 64, 4)
    assert np.array_equal(out, g["nms_fast_out"]) and np.array_equal(inds, g["nms_fast_inds"])


def test_box_nms(golden):
    g = golden("box_nms")
    assert np.array_equal(O.box_nms(g["prob"], 4, 0.1, 0.01), g["out"])


def test_descriptor_loss_small(golden):
    g = golden("desc_small")
    for tag, gr in (("a", (1.0, 0.0, 0.0)), ("b", tuple(g["g_b"]))):
        loss, mask, pos, neg, dD, dDw = O.descriptor_loss(g["D"], g["Dw"], g["H"], g["mv"], grad=gr, return_mask=True)
        close(loss, g["loss_" + tag]); close(pos, g["pos_" + tag]); close(neg, g["neg_" + tag])
        assert np.array_equal(mask.astype(np.uint8), g["mask_" + tag])
        scale = np.abs(g["dD_" + tag]).max()
        close(dD, g["dD_" + tag], atol=1e-4 * scale)
        close(dDw, g["dDw_" + tag], atol=1e-4 * scale)


def test_descriptor_loss_30x40(golden):
    g = golden("desc_30x40")
    D = synth.unit_descriptors(1, 256, 30, 40, 91, smooth=0.3)
    Dw = synth.unit_descriptors(1, 256, 30, 40, 92, smooth=0.3)
    loss, mask, pos, neg, dD, dDw = O.descriptor_loss(D, Dw, g["H"], g["mv"], grad=(1, 1, 1), return_mask=True)
    close(loss, g["loss"]); close(pos, g["pos"]); close(neg, g["neg"])
    assert np.array_equal(mask.reshape(1, 1200, 1200).sum(-1), g["mask_rowsum"])
    scale = np.abs(g["dD_sample"]).max()
    close(dD[0, :, ::7, ::9], g["dD_sample"], atol=2e-4 * scale)
    close(dDw[0, :, ::7, ::9], g["dDw_sample"], atol=2e-4 * scale)


def test_descriptor_identity_kat(golden):
    """identical descriptors + identity homography: the positive term vanishes (reference's informal KAT)."""
    g = golden("desc_identity")
    D = synth.unit_descriptors(1, 256, 30, 40, 91, smooth=0.3)
    loss, _, pos, neg = O.descriptor_loss(D, D.copy(), np.eye(3)[None], np.ones((1, 1, 30, 40), np.float32))
    close(pos, g["pos"], atol=1e-7); close(neg, g["neg"]); close(loss, g["loss"])
    assert abs(float(pos)) < 1e-6


def test_loss_step_composition_and_gradients():
    """oracle.loss_step at a tiny shape: its scalars are those of detector_loss / descriptor_loss on getMasks of the two
    masks, the total follows the chosen weighting, and each of the four gradients is the derivative of that total
    (central differences along a fixed direction, in float64 around the fp32 inputs)."""
    B, Hc, Wc = 2, 3, 4
    inp = {"semi": synth.pseudo_normal((B, 65, Hc, Wc), 1), "semi_warp": synth.pseudo_normal((B, 65, Hc, Wc), 2),
           "desc": synth.unit_descriptors(B, 256, Hc, Wc, 3, smooth=0.3),
           "desc_warp": synth.unit_descriptors(B, 256, Hc, Wc, 4, smooth=0.3),
           "labels_2D": synth.keypoint_labels(B, 8 * Hc, 8 * Wc, 5, p=0.05),
           "warped_labels": synth.keypoint_labels(B, 8 * Hc, 8 * Wc, 6, p=0.05),
           "mask_2D": np.ones((B, 1, 8 * Hc, 8 * Wc), np.float32),
           "mask_warp_2D": np.ones((B, 1, 8 * Hc, 8 * Wc), np.float32),
           "mat_H": np.stack([np.eye(3), [[0.9, 0.05, 0.1], [0.0, 1.1, -0.05], [0.0, 0.0, 1.0]]]).astype(np.float32)}
    inp["mask_warp_2D"][0, 0, 3, 12] = 0    # one pixel: getMasks zeroes cell (0, 1)
    inp["mask_warp_2D"][1, 0, 16:, :8] = 0  # cell (2, 0)
    mw3 = O.getMasks(inp["mask_warp_2D"])
    assert mw3.sum() == B * Hc * Wc - 2
    ld = O.detector_loss(inp["semi"], O.labels2Dto3D(inp["labels_2D"]), O.getMasks(inp["mask_2D"]))
    ldw = O.detector_loss(inp["semi_warp"], O.labels2Dto3D(inp["warped_labels"]), mw3)
    desc = O.descriptor_loss(inp["desc"], inp["desc_warp"], inp["mat_H"], mw3[:, None], lamda_d=250, descriptor_dist=6)
    assert float(desc[2]) > 0  # positive pairs exist
    keys = ("semi", "semi_warp", "desc", "desc_warp")
    for weighting, lam in (("uniform", 2.5), ("multi_task", 1.0)):
        kw = dict(descriptor_dist=6, lambda_loss=lam, weighting=weighting)
        r = O.loss_step(**inp, **kw)
        assert float(r["loss_det"]) == float(ld) and float(r["loss_det_warp"]) == float(ldw)
        assert (float(r["loss_desc"]), float(r["positive_dist"]), float(r["negative_dist"])) == tuple(float(x) for x in (desc[0], desc[2], desc[3]))
        terms = (lam * float(desc[0]),) if weighting == "uniform" else (float(desc[2]), float(desc[3]))
        close(r["loss"], float(ld) + float(ldw) + sum(terms))
        for i, k in enumerate(keys):
            v = synth.pseudo_normal(inp[k].shape, 40 + i).astype(np.float64)
            eps = (3e-2 if k.startswith("semi") else 1e-3) / np.abs(v).max()  # the detector loss is smooth, the hinges are not

            def total(t):
                moved = dict(inp)
                moved[k] = (inp[k].astype(np.float64) + t * v).astype(np.float32)
                return float(O.loss_step(**moved, **kw)["loss"])

            fd = (total(eps) - total(-eps)) / (2 * eps)
            an = float((r["grads"][i].astype(np.float64) * v).sum())
            assert r["grads"][i].shape == inp[k].shape
            noise = 3 * float(np.spacing(np.float32(abs(r["loss"])))) / (2 * eps)  # the fp32 rounding of three scalars
            np.testing.assert_allclose(an, fd, rtol=1e-3, atol=noise, err_msg="%s %s" % (weighting, k))


def test_semantic_head(golden):
    """SURVEY 8f rank 1: x8 bilinear upsample (reference model forward) + CrossEntropyLoss(ignore_index=133)."""
    g = golden("semantic")
    close(O.upsample_bilinear(g["lr"], g["label"].shape[1:])[:, ::7], g["full_sample"], atol=1e-6)
    for lr_k, lab_k, loss_k, d_k, ds_k, gout in (("lr", "label", "loss", "dlr", "dfull_sample", 1.0),
                                                 ("lr2", "label2", "loss2", "dlr2", "dfull2_sample", float(g["g2"]))):
        loss, d = O.sem_loss(g[lr_k], g[lab_k], grad=True, gout=gout)
        close(loss, g[loss_k], rtol=1e-5)
        close(d, g[d_k], atol=1e-4 * np.abs(g[d_k]).max())
        full = O.upsample_bilinear(g[lr_k], g[lab_k].shape[1:])
        loss_f, d_f = O.sem_loss(full, g[lab_k], grad=True, gout=gout)   # full-resolution entry of the same oracle
        close(loss_f, g[loss_k], rtol=1e-5)
        sy, sx = (5, 7) if lr_k == "lr" else (3, 5)
        close(d_f[:, ::9, ::sy, ::sx], g[ds_k], atol=1e-4 * np.abs(g[ds_k]).max())


def _matching_inputs():
    coarse = synth.unit_descriptors(1, 256, 15, 20, 111, smooth=0.5)
    coarse2 = (coarse + 0.35 * synth.unit_descriptors(1, 256, 15, 20, 112, smooth=0.5)).astype(np.float32)
    return coarse, coarse2


def test_sparse_descriptors_and_matching(golden):
    """SURVEY 8f rank 3: sample_desc_from_points + nn_match_two_way (models/model_wrap.py:295-313, 451-494)."""
    g = golden("matching")
    coarse, coarse2 = _matching_inputs()
    close(O.sample_desc_from_points(coarse, g["pts"]), g["desc1"], atol=1e-6)
    close(O.sample_desc_from_points(coarse2, g["pts2"]), g["desc2"], atol=1e-6)
    for thr, key in ((0.36, "matches_36"), (0.7, "matches_70")):
        m = O.nn_match_two_way(g["desc1"], g["desc2"], thr)
        assert np.array_equal(m[:2], g[key][:2])
        close(m[2], g[key][2], atol=1e-6)
    assert g["matches_36"].shape[1] < g["matches_70"].shape[1]
    assert O.nn_match_two_way(g["desc1"], g["desc2"][:, :0], 0.7).shape == (3, 0)
    assert O.sample_desc_from_points(coarse, np.zeros((3, 0))).shape == (256, 0)


def test_warp_labels_oracle(golden):
    """SURVEY 8f rank 4 (oracle pinned ahead of the kernels): datasets/data_tools.warpLabels incl. the bilinear label map."""
    g = golden("warp_labels")
    for i in range(2):
        o = O.warp_labels(g["pts"], 48, 64, g["H"][i], bilinear=True)
        assert np.array_equal(o["labels"], g["labels_%d" % i])
        close(o["warped_pnts"], g["warped_pnts_%d" % i], atol=2e-5)
        close(o["res"], g["res_%d" % i], atol=2e-5)
        close(o["labels_bi"], g["labels_bi_%d" % i], atol=2e-5)
        assert o["labels"].sum() <= o["warped_pnts"].shape[0]  # collisions keep one label per pixel


def test_eval_keypoints_and_repeatability(golden):
    """8a-a10 evaluation side: detector_evaluation.warp_keypoints and the repeatability masks, as run by the reference's own
    compute_repeatability on synthetic detections (fixture generated from the live module)."""
    g = golden("eval_keypoints")
    shape = tuple(int(v) for v in g["shape"])
    np.testing.assert_array_equal(O.warp_keypoints_f64(g["kp"][:, :2], g["H"]), g["warped"])
    rep, loc = O.compute_repeatability(g["kp"], g["warped_prob"], g["H"], shape, keep_k_points=300)
    assert rep == float(g["repeatability"]) and loc == float(g["loc_err"])
    rep, loc = O.compute_repeatability(g["kp"], g["warped_prob"], g["H"], shape, keep_k_points=1000)
    assert rep == float(g["repeatability_1000"]) and loc == float(g["loc_err_1000"])


def test_sparse_descriptor_loss_oracle_and_sampler(golden):
    """8f rank 2: the oracle's evaluation of the sparse loss on the index lists the live reference sampled (captured inside its own
    call), incl. gradients; and the product's host-side sampler reproduces those lists call for call under the same RNG
    state (torch + numpy seeds), including the padding branch (image 1 matches only 232 distinct cells)."""
    import torch
    from ssp_b200 import sparse, synth
    g = golden("sparse_loss")
    D = synth.unit_descriptors(3, 256, 30, 40, 151, smooth=0.3)
    Dw = synth.unit_descriptors(3, 256, 30, 40, 152, smooth=0.3)
    r = O.sparse_descriptor_loss(D, Dw, g["matches_a"], g["matches_b"], g["non_a"], g["non_b"], 250, grad=tuple(g["g"]))
    close(r[0], g["loss"], rtol=1e-6); close(r[1], g["pos"], rtol=1e-6); close(r[2], g["neg"], rtol=1e-6)
    close(r[3][:, :, ::3, ::4], g["dD_sample"], atol=1e-6); close(r[4][:, :, ::3, ::4], g["dDw_sample"], atol=1e-6)
    np.testing.assert_allclose(np.abs(r[3]).sum(), float(g["dD_abs_sum"]), rtol=1e-5)
    torch.manual_seed(int(g["seed_torch"]))
    np.random.seed(int(g["seed_numpy"]))
    for i in range(3):
        l = sparse.sample_correspondences(torch.from_numpy(g["H"][i]), 30, 40, 1000, 10)
        for got, key in zip(l, ("matches_a", "matches_b", "non_a", "non_b")):
            assert np.array_equal(got.numpy(), g[key][i]), (i, key)
    assert len(np.unique(g["matches_a"][1])) < 1000  # the padded image
