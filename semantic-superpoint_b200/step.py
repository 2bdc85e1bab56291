"""The hot loops of the reference, expressed over the kernels (no backbone: heads' outputs come in).

loss_step          = Train_model_heatmap_all.train_val_sample lines 295-365 (detector loss x2 + descriptor loss,
                     optionally the two semantic cross entropies of the SSp configuration)
adaptation_step    = export.export_detector_homoAdapt_gpu lines 304-323 (flatten -> aggregate -> NMS [-> sub-pixel] -> top-k)
match_step         = export.export_descriptor lines 66-189 for a batch of image pairs (flatten -> NMS -> descriptors -> matches),
                     optionally followed by evaluation.py's metrics of the pairs (utils.evaluate_pairs)
The first two are free of host synchronisation except the final keypoint read-back of adaptation_step; match_step
synchronises twice (NMS counts, read-back).
"""
import numpy as np
import torch

from . import _lib
from . import utils as U
from ._lib import call, ptr


def loss_step(semi, semi_warp, desc, desc_warp, labels_2D, warped_labels, mask_2D, mask_warp_2D, mat_H,
              lamda_d=250, descriptor_dist=4, lambda_loss=1.0, engine=None, dist_group=None, side_stream=None,
              sem_pred=None, sem=None, sem_warp_pred=None, warped_sem=None, fused=True, descriptor_loss="dense",
              sampler=None, num_matching_attempts=1000, num_masked_non_matches_per_match=10):
    """Returns dict(loss, loss_det, loss_det_warp, loss_desc, positive_dist, negative_dist[, loss_sem, loss_sem_warp]).

    loss = loss_det + loss_det_warp [+ loss_sem + loss_sem_warp] + lambda_loss * loss_desc
    (uniform weighting, Train_model_heatmap_all.py:361-365).  The semantic terms (config data.semantic, :304,:320-324)
    are added when sem_pred / sem (and the warped twins) are given; sem_pred may be the full-resolution logits or the
    1/8-resolution head output (fused upsample, see utils.sem_loss).
    side_stream: unused (kept for compatibility).
    fused=True: the step is one autograd node and only `loss` carries gradient; the component scalars are
    values for logging.  Pass fused=False to differentiate through loss_det / positive_dist / negative_dist separately
    (the reference's multi_task_loss weighting, Train_model_heatmap_all.py:355-359).
    descriptor_loss="sparse": the descriptor term is the sparse loss of the shipped configs (sparse_loss.py:65-284,
    Train_model_heatmap_all.py:333-347) on lists that `sampler` (a sparse.DeviceSampler) draws on the device with
    num_matching_attempts matches and num_masked_non_matches_per_match non-matches per match; descriptor_dist and engine
    do not apply.  Single GPU only.
    """
    if descriptor_loss == "sparse":
        return _sparse_loss_step(semi, semi_warp, desc, desc_warp, labels_2D, warped_labels, mask_2D, mask_warp_2D, mat_H,
                                 lamda_d, lambda_loss, dist_group, sem_pred, sem, sem_warp_pred, warped_sem, fused, sampler,
                                 num_matching_attempts, num_masked_non_matches_per_match)
    if descriptor_loss != "dense":
        raise ValueError("descriptor_loss must be 'dense' or 'sparse', got %r" % (descriptor_loss,))
    if fused:
        # fast path: the whole step is one autograd node (no scalar-glue kernels), see losses.LossStepFn; with dist_group
        # set, one peer-memory exchange kernel makes the normalisers global (dist.LossExchange)
        from .losses import LossStepFn, get_descriptor_engine
        Hm = mat_H if mat_H.dim() == 3 else mat_H.unsqueeze(0)
        loss, loss_det, loss_det_warp, loss_desc, pos, neg = LossStepFn.apply(
            semi, labels_2D, mask_2D, semi_warp, warped_labels, mask_warp_2D, desc, desc_warp,
            Hm.to(device=semi.device, dtype=torch.float32).contiguous(), float(lamda_d), float(descriptor_dist),
            float(lambda_loss), engine or get_descriptor_engine(), dist_group)
        return _result(loss, loss_det, loss_det_warp, loss_desc, pos, neg,
                       _sem_losses(sem_pred, sem, sem_warp_pred, warped_sem, dist_group))
    # separately differentiable components (the reference's multi_task_loss weighting); with dist_group each loss runs
    # its own exchange kernel
    # both detector losses in one launch each way; getMasks(mask_warp_2D) comes out of the same kernel
    loss_det, loss_det_warp, mask_cells = U.detector_loss_pair_2d(semi, labels_2D, mask_2D, semi_warp, warped_labels,
                                                                  mask_warp_2D, dist_group=dist_group)
    mask_desc = mask_cells.unsqueeze(1)
    kw = {"dist_group": dist_group}
    if engine is not None:
        kw["engine"] = engine
    loss_desc, _mask, pos, neg = U.descriptor_loss(desc, desc_warp, mat_H, mask_valid=mask_desc, device=semi.device,
                                                   lamda_d=lamda_d, descriptor_dist=descriptor_dist, **kw)
    sem_terms = _sem_losses(sem_pred, sem, sem_warp_pred, warped_sem, dist_group)
    loss = loss_det + loss_det_warp + lambda_loss * loss_desc
    return _result(loss, loss_det, loss_det_warp, loss_desc, pos, neg, sem_terms)


def _sem_losses(sem_pred, sem, sem_warp_pred, warped_sem, dist_group=None):
    """(loss_sem, loss_sem_warp), or None without semantic terms."""
    if sem_pred is None:
        return None
    return U.sem_loss(sem_pred, sem, dist_group=dist_group), U.sem_loss(sem_warp_pred, warped_sem, dist_group=dist_group)


def _result(loss, loss_det, loss_det_warp, loss_desc, pos, neg, sem_terms):
    """loss_step's result dict; the semantic terms, if any, are added to the total."""
    out = {}
    if sem_terms is not None:
        out["loss_sem"], out["loss_sem_warp"] = sem_terms
        loss = loss + sem_terms[0] + sem_terms[1]
    out.update({"loss": loss, "loss_det": loss_det, "loss_det_warp": loss_det_warp, "loss_desc": loss_desc,
                "positive_dist": pos, "negative_dist": neg})
    return out


def _sparse_loss_step(semi, semi_warp, desc, desc_warp, labels_2D, warped_labels, mask_2D, mask_warp_2D, mat_H, lamda_d,
                      lambda_loss, dist_group, sem_pred, sem, sem_warp_pred, warped_sem, fused, sampler, K, n):
    """loss_step(descriptor_loss="sparse"): sampler launch, detector pair, sparse loss; no host sync, no host RNG."""
    from .sparse import DeviceSampler, SparseDescriptorLossFn
    if dist_group is not None:
        raise NotImplementedError("loss_step: the sparse descriptor loss runs on one GPU (dist_group is not supported)")
    if not isinstance(sampler, DeviceSampler):
        raise ValueError("loss_step(descriptor_loss='sparse') needs sampler=sparse.DeviceSampler(seed, device)")
    K = int(K)
    ia, ib, M = sampler.sample(mat_H, desc.shape[2], desc.shape[3], K, n)
    if fused:
        from .losses import SparseLossStepFn
        loss, loss_det, loss_det_warp, loss_desc, pos, neg = SparseLossStepFn.apply(
            semi, labels_2D, mask_2D, semi_warp, warped_labels, mask_warp_2D, desc, desc_warp, ia, ib, M, K, float(lamda_d),
            float(lambda_loss))
    else:
        loss_det, loss_det_warp, _ = U.detector_loss_pair_2d(semi, labels_2D, mask_2D, semi_warp, warped_labels, mask_warp_2D)
        loss_desc, pos, neg = SparseDescriptorLossFn.apply(desc, desc_warp, ia, ib, K, ia.shape[1] - K, float(lamda_d), M)
        loss = loss_det + loss_det_warp + lambda_loss * loss_desc
    return _result(loss, loss_det, loss_det_warp, loss_desc, pos, neg, _sem_losses(sem_pred, sem, sem_warp_pred, warped_sem))


@torch.no_grad()
def adaptation_step(semi, inv_homographies, mask_2D, conf_thresh=0.015, nms_dist=4, top_k=600, binary_mask=False,
                    subpixel=False, patch_size=5):
    """semi [I,N,65,Hc,Wc] (or [N,65,Hc,Wc]), inv_homographies [I,N,3,3], mask_2D [I,N,H,W] -> list of [K,3] arrays
    (x, y, prob), K <= top_k, per source image.
    mask_2D is the stack of valid masks of the warped views; binary_mask=True promises a 0/1 mask (compute_valid_mask's output,
    what the export path always passes): the mask is folded into the flattened heatmap as its sign and the aggregation gathers
    one array instead of two (bit-identical results; a non-binary mask then yields NaN heatmaps).
    subpixel=True (the export config's model.subpixel.enable, export.py:309-314) refines x and y of the kept points by
    utils.soft_argmax_points on the aggregated heatmap with patch_size, on the device before the read-back; count, order
    and prob are those of subpixel=False."""
    if semi.dim() == 4:
        semi, inv_homographies = semi.unsqueeze(0), inv_homographies.reshape(1, -1, 3, 3)
        mask_2D = mask_2D.reshape(1, semi.shape[1], mask_2D.shape[-2], mask_2D.shape[-1])
    I, N, C, Hc, Wc = semi.shape
    if binary_mask:
        agg = U.combine_from_logits_batch(semi, inv_homographies, mask_2D)
    else:
        heat = U.flattenDetection(semi.reshape(I * N, C, Hc, Wc)).reshape(I, N, Hc * 8, Wc * 8)
        agg = U.combine_heatmap_batch(heat, inv_homographies, mask_2D)
    pts = U.heatmap_to_pts_batch(agg, conf_thresh, nms_dist, top_k=top_k, subpixel=subpixel, patch_size=patch_size)
    return [p.transpose() for p in pts]


@torch.no_grad()
def match_step(semi, desc, semi_warp, desc_warp, conf_thresh=0.015, nms_dist=4, top_k=None, nn_thresh=0.7,
               homographies=None, shape_eval=None, **eval_kw):
    """The descriptor export of P image pairs (export.py:66-189, export_descriptor) as one call: keypoints, descriptors and
    two-way matches of every pair.  semi, semi_warp [P,65,Hc,Wc] logits; desc, desc_warp [P,256,Hc,Wc] coarse descriptors
    (the head's normalised output); CUDA tensors.  Returns P dicts with
      pts, warped_pts      [3,K] float64 (x, y, conf), confidence-descending, K <= top_k (None: every NMS point)
      desc, warped_desc    [256,K] float32
      matches              [3,L] float64 (index in pts, index in warped_pts, distance), increasing index-1 order
    equal, pair by pair, to getPtsFromHeatmap(flattenDetection(semi[p]), conf_thresh, nms_dist)[:, :top_k],
    sample_desc_from_points(desc[p:p+1], pts), the same for the warped image, and nn_match_two_way(desc, warped_desc,
    nn_thresh), the matching on the tensor cores (nn_match_two_way_batch).  Two host synchronisations: the NMS reads its
    counts (which also size every later buffer) and the single read-back of all results.
    homographies [P,3,3] (pixel coordinates, image 1 -> image 2) runs utils.evaluate_pairs on the device buffers before the
    read-back (same host synchronisations, no descriptor round trip) and adds "metrics" to every result: that pair's entries
    of evaluate_pairs' dict.  shape_eval (H, W) defaults to the image shape; eval_kw are evaluate_pairs' keywords.  The
    evaluation's cross-check matches reuse the export's matcher launch when nn_thresh > 2 (every distance is <= 2), else
    one more ssp_nn_match_batch runs without a threshold; the export's own results do not change."""
    U._check_nn_thresh(nn_thresh)
    P, C, Hc, Wc = semi.shape
    if C != 65 or tuple(semi_warp.shape) != (P, C, Hc, Wc):
        raise ValueError("match_step: semi and semi_warp must be [P,65,Hc,Wc], got %s and %s"
                         % (tuple(semi.shape), tuple(semi_warp.shape)))
    if desc.shape[1] != 256 or tuple(desc.shape) != (P, 256, Hc, Wc) or tuple(desc_warp.shape) != (P, 256, Hc, Wc):
        raise ValueError("match_step: desc and desc_warp must be [P,256,Hc,Wc] (the tensor-core matcher takes 256-dimensional "
                         "descriptors), got %s and %s" % (tuple(desc.shape), tuple(desc_warp.shape)))
    _lib.require_cuda(semi, desc, semi_warp, desc_warp)
    dev = semi.device
    st = _lib.stream_of(semi)
    H, W = Hc * 8, Wc * 8
    if homographies is not None:
        params = U._eval_params(**eval_kw)
        shape_eval = (H, W) if shape_eval is None else tuple(int(v) for v in shape_eval)
        Hs_host = U._homography_pairs(homographies, P)
        Hs = torch.from_numpy(Hs_host).pin_memory().to(dev, non_blocking=True)
    # 1. both flattened heatmaps into the halves of one [2P,1,H,W] buffer
    heat = torch.empty((2 * P, 1, H, W), dtype=torch.float32, device=dev)
    for h, s in enumerate((semi, semi_warp)):
        call("ssp_flatten_detection", ptr(_lib.f32c(s.detach(), dev)), P, Hc, Wc, ptr(heat[h * P:(h + 1) * P]), st)
    # 2. one NMS over the 2P heatmaps (host sync 1: the counts)
    pts, counts, counts_dev = U._nms_batch(heat.view(2 * P, H, W), conf_thresh, nms_dist)
    cnt = [min(c, top_k) for c in counts] if top_k is not None else counts
    kmax = max(cnt)
    if kmax == 0:
        empty = {"pts": np.zeros((3, 0)), "desc": np.zeros((256, 0)), "warped_pts": np.zeros((3, 0)),
                 "warped_desc": np.zeros((256, 0)), "matches": np.zeros((3, 0))}
        out = [{k: v.copy() for k, v in empty.items()} for _ in range(P)]
        if homographies is not None:
            keys = ("keep_k_points", "distance_thresh", "correctness_thresh", "map_nn_thresh", "map_inliers", "seed")
            m = U.evaluate_pairs([r["pts"] for r in out], [r["warped_pts"] for r in out], [r["desc"] for r in out],
                                 [r["warped_desc"] for r in out], Hs_host[:, 0].reshape(P, 3, 3), shape_eval,
                                 **dict(zip(keys, params)))
            _attach_metrics(out, m)
        return out
    R = (kmax + 255) // 256 * 256
    # every result lands in one device buffer, read back with one copy
    sizes = {"pts": 2 * P * 3 * kmax * 8, "desc": 2 * P * 256 * kmax * 4, "matches": P * 3 * R * 8, "nmatch": P * 4}
    if homographies is not None:
        T, n_sets = len(params[0]), 1 if params[1] else 2
        sizes.update(U._eval_sizes(P, R, T, n_sets))
        own_matches = nn_thresh <= 2.0  # a distance of exactly 2 fails the matcher's strict test
        if own_matches:
            sizes["ev_nmatch"] = P * 4
    offs, total = {}, 0
    for k, n in sizes.items():
        offs[k] = total
        total += (n + 255) // 256 * 256
    stage = torch.empty((total,), dtype=torch.uint8, device=dev)
    region = lambda k, dtype, shape: stage[offs[k]:offs[k] + sizes[k]].view(dtype).view(shape)
    d_all = region("desc", torch.float32, (2 * P, 256, kmax))
    matches = region("matches", torch.float64, (P, 3, R))
    nmatch = region("nmatch", torch.int32, (P,))
    # 3. descriptors at the first min(count, kmax) points of every image (zeros after them)
    cap = pts.shape[2]
    for h, d in enumerate((desc, desc_warp)):
        call("ssp_sample_desc_batch", ptr(_lib.f32c(d.detach(), dev)), ptr(pts[h * P:]), cap, ptr(counts_dev[h * P:]), kmax,
             P, 256, Hc, Wc, 8, ptr(d_all[h * P:]), st)
    # 4. + 5. operand planes and the matcher
    planes = U._pack_planes(d_all)
    U._nn_match_planes(planes[:, :P], planes[:, P:], counts_dev[:P], counts_dev[P:], kmax, nn_thresh, matches, nmatch)
    region("pts", torch.float64, (2 * P, 3, kmax)).copy_(pts[:, :, :kmax])
    if homographies is not None:
        ev_matches, ev_nmatch = matches, nmatch
        if own_matches:
            ev_matches = torch.empty((P, 3, R), dtype=torch.float64, device=dev)
            ev_nmatch = region("ev_nmatch", torch.int32, (P,))
            U._nn_match_planes(planes[:, :P], planes[:, P:], counts_dev[:P], counts_dev[P:], kmax, float("inf"), ev_matches,
                               ev_nmatch)
        U._eval_launch(region("pts", torch.float64, (2 * P, 3, kmax)), kmax, counts_dev, P, ev_matches, ev_nmatch, Hs,
                       shape_eval, params, region)
    # 6. the read-back (host sync 2), into page-locked memory: a pageable copy of the descriptors runs at a fraction of the
    # link's rate, and torch's pinned-memory cache reuses the block once the previous call's results are released
    host = torch.empty((total,), dtype=torch.uint8, pin_memory=True)
    host.copy_(stage)
    host = host.numpy()
    view = lambda k, dtype, shape: host[offs[k]:offs[k] + sizes[k]].view(dtype).reshape(shape)
    hp, hd = view("pts", np.float64, (2 * P, 3, kmax)), view("desc", np.float32, (2 * P, 256, kmax))
    hm, hn = view("matches", np.float64, (P, 3, R)), view("nmatch", np.int32, (P,))
    out = []
    for p in range(P):
        k1, k2 = cnt[p], cnt[P + p]
        out.append({"pts": hp[p, :, :k1] if k1 else np.zeros((3, 0)),
                    "desc": hd[p, :, :k1] if k1 else np.zeros((256, 0)),
                    "warped_pts": hp[P + p, :, :k2] if k2 else np.zeros((3, 0)),
                    "warped_desc": hd[P + p, :, :k2] if k2 else np.zeros((256, 0)),
                    "matches": hm[p, :, :hn[p]] if hn[p] else np.zeros((3, 0))})
    if homographies is not None:
        nm = view("ev_nmatch", np.int32, (P,)) if own_matches else hn
        _attach_metrics(out, U._eval_results(view, nm, P, R, T, n_sets))
    return out


def _attach_metrics(results, m):
    """results[p]["metrics"] = pair p's entries of an evaluate_pairs dict."""
    for p, r in enumerate(results):
        r["metrics"] = {k: (v[p] if k == "inliers" else v[p].copy() if v[p].ndim else v[p].item()) for k, v in m.items()}


@torch.no_grad()
def collate_warped_pair(img, pnts_list, homographies=None, erosion_radius=3, bilinear=True, sampler=None,
                        **homography_params):
    """The warped half of a training batch, built on the device from the unwarped images and their keypoints -- what
    datasets/Coco.py:341-392 does per sample in the DataLoader workers (inv_warp_image, warpLabels, compute_valid_mask):
    img [B,1,H,W], pnts_list = B arrays [P,2] (x, y), homographies [B,3,3] (normalised coordinates, already inverted as in
    Coco.py:345).  Returns the batch keys of the reference: warped_img, warped_labels, warped_res [B,2,H,W],
    warped_labels_bi, warped_valid_mask [B,1,H,W], homographies, inv_homographies.  (Photometric augmentation and the
    gaussian label blur are imgaug calls and stay where they are.)
    sampler (a homography.HomographySampler) instead of homographies: the batch's homographies are drawn on the device with
    homography_params (sample_homography_np's keywords, e.g. the config's warped_pair params) and inv_homographies comes
    from the same kernel, with no host round trip."""
    dev = img.device
    B, _, H, W = img.shape
    if (homographies is None) == (sampler is None):
        raise ValueError("collate_warped_pair: pass either homographies or sampler")
    if sampler is not None:
        Hm, Hinv = sampler.sample(B, **homography_params)
    else:
        Hm = torch.as_tensor(homographies, dtype=torch.float32).reshape(B, 3, 3)
        Hinv = torch.inverse(Hm.cpu()).to(dev)  # the reference inverts on the CPU (np.linalg.inv / torch.inverse per sample)
        Hm = Hm.to(dev)
    warped_img = U.inv_warp_image_batch(img, Hinv, device=dev, mode="bilinear")
    lab = U.warp_labels_batch(pnts_list, H, W, Hm, bilinear=bilinear, device=dev)
    mask = U.compute_valid_mask(torch.tensor([H, W]), Hinv, device=dev, erosion_radius=erosion_radius).unsqueeze(1)
    out = {"warped_img": warped_img, "warped_labels": lab["labels"], "warped_res": lab["res"].permute(0, 3, 1, 2).contiguous(),
           "warped_valid_mask": mask, "homographies": Hm, "inv_homographies": Hinv, "warped_pnts": lab["warped_pnts"]}
    if bilinear:
        out["warped_labels_bi"] = lab["labels_bi"]
    return out


@torch.no_grad()
def adaptation_views(img, sampler, num=100, erosion_radius=0, **homography_params):
    """The homography-adaptation branch of the dataset (datasets/Coco.py:258-291) on the device, for I source images at
    once: img [I,1,H,W], sampler a homography.HomographySampler, homography_params sample_homography_np's keywords (the
    export config's homography_adaptation.homographies.params).  Draws I*num homographies, the first of every image the
    identity, warps num bilinear views of each image by inv_homographies and builds their valid masks
    (compute_valid_mask with erosion_radius, the config's valid_border_margin).  No host synchronisation.

    Returns the sample keys of the reference: image [I,num,H,W], valid_mask [I,num,H,W], homographies [I,num,3,3],
    inv_homographies [I,num,3,3].  export.py:284-287 swaps the two names when it reads a sample (the aggregation warps the
    detections back with `homographies`), so the heads' logits semi [I,num,65,H/8,W/8] of out["image"] go to
    adaptation_step(semi, out["homographies"], out["valid_mask"], binary_mask=True)."""
    _lib.require_cuda(img)
    I, C, H, W = img.shape
    if C != 1:
        raise ValueError("adaptation_views: img must be [I, 1, H, W], got %s" % (tuple(img.shape),))
    num = int(num)
    Hm, Hinv = sampler.sample(I * num, group=num, **homography_params)
    views = img.expand(I, num, H, W).reshape(I * num, 1, H, W)  # img.repeat(N, 1, 1, 1) of Coco.py:280
    image = U.inv_warp_image_batch(views, Hinv, device=img.device, mode="bilinear")
    valid = U.compute_valid_mask(torch.tensor([H, W]), Hinv, device=img.device, erosion_radius=erosion_radius)
    return {"image": image.reshape(I, num, H, W), "valid_mask": valid.reshape(I, num, H, W),
            "homographies": Hm.reshape(I, num, 3, 3), "inv_homographies": Hinv.reshape(I, num, 3, 3)}


class GraphedLossStep(object):
    """loss_step forward + backward captured once into a CUDA graph and replayed (the step is a chain of ~25 short
    kernels; replay removes the per-launch host cost).  Inputs are copied into static buffers; outputs (loss
    scalars and the four gradients) live in static buffers that the next replay overwrites.
    With descriptor_loss="sparse" the sampler launch is part of the graph: every replay draws new lists, the first replay
    draws what an eager step from the sampler's state at construction would (the warm-up steps restore that state), and
    the outputs hold the last replay's lists as "lists" = (ia, ib, M)."""

    IN_KEYS = ("semi", "semi_warp", "desc", "desc_warp", "labels_2D", "warped_labels", "mask_2D", "mask_warp_2D", "mat_H")
    SEM_KEYS = ("sem_pred", "sem_warp_pred", "sem", "warped_sem")  # optional: SSp configuration

    def __init__(self, example, overlap=True, loss_keys=None, **kw):
        """loss_keys: the outputs of loss_step whose sum is differentiated (needs fused=False), e.g. the reference's
        multi-task weighting at unit weights: ("loss_det", "loss_det_warp", "positive_dist", "negative_dist")
        (Train_model_heatmap_all.py:355-359).  Default: the uniform-weighting total `loss`."""
        self.kw = kw
        self.loss_keys = loss_keys
        self.semantic = "sem_pred" in example
        if self.semantic:
            self.IN_KEYS = self.IN_KEYS + self.SEM_KEYS
        self.static = {k: example[k].detach().clone() for k in self.IN_KEYS}
        sampler = kw.get("sampler") if kw.get("descriptor_loss") == "sparse" else None
        state = sampler.get_state() if sampler is not None else None
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self._run()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        if sampler is not None:
            sampler.set_state(state)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = self._run()

    def _run(self):
        s = self.static
        names = ("semi", "semi_warp", "desc", "desc_warp") + (("sem_pred", "sem_warp_pred") if self.semantic else ())
        leaves = [s[k].detach().requires_grad_(True) for k in names]
        kw = dict(self.kw)
        if self.semantic:
            kw.update(sem_pred=leaves[4], sem=s["sem"], sem_warp_pred=leaves[5], warped_sem=s["warped_sem"])
        out = loss_step(leaves[0], leaves[1], leaves[2], leaves[3], s["labels_2D"], s["warped_labels"], s["mask_2D"],
                        s["mask_warp_2D"], s["mat_H"], **kw)
        if getattr(self, "_one", None) is None:  # static dL/dloss = 1: no ones_like fill inside the captured step
            self._one = torch.ones_like(out["loss"])
        total = out["loss"]
        if self.loss_keys:
            total = sum(out[k] for k in self.loss_keys[1:]) + out[self.loss_keys[0]]
        total.backward(gradient=self._one)
        res = {k: v.detach() for k, v in out.items()}
        res["grads"] = [l.grad for l in leaves]
        if kw.get("descriptor_loss") == "sparse":
            res["lists"] = kw["sampler"].last
        return res

    def load(self, inputs, non_blocking=True):
        for k in self.IN_KEYS:
            self.static[k].copy_(inputs[k], non_blocking=non_blocking)

    def replay(self):
        self.graph.replay()
        return self.out

    def __call__(self, inputs):
        self.load(inputs)
        return self.replay()
