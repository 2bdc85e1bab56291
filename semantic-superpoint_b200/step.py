"""The two hot loops of the reference, expressed over the kernels (no backbone: heads' outputs come in).

loss_step          = Train_model_heatmap_all.train_val_sample lines 295-365 (detector loss x2 + descriptor loss,
                     optionally the two semantic cross entropies of the SSp configuration)
adaptation_step    = export.export_detector_homoAdapt_gpu lines 304-323 (flatten -> aggregate -> NMS -> top-k)
Both are free of host synchronisation except the final keypoint read-back of adaptation_step.
"""
import torch

from . import utils as U


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
def adaptation_step(semi, inv_homographies, mask_2D, conf_thresh=0.015, nms_dist=4, top_k=600, binary_mask=False):
    """semi [I,N,65,Hc,Wc] (or [N,65,Hc,Wc]), inv_homographies [I,N,3,3], mask_2D [I,N,H,W] -> list of [K,3] arrays
    (x, y, prob), K <= top_k, per source image.
    mask_2D is the stack of valid masks of the warped views; binary_mask=True promises a 0/1 mask (compute_valid_mask's output,
    what the export path always passes): the mask is folded into the flattened heatmap as its sign and the aggregation gathers
    one array instead of two (bit-identical results; a non-binary mask then yields NaN heatmaps)."""
    if semi.dim() == 4:
        semi, inv_homographies = semi.unsqueeze(0), inv_homographies.reshape(1, -1, 3, 3)
        mask_2D = mask_2D.reshape(1, semi.shape[1], mask_2D.shape[-2], mask_2D.shape[-1])
    I, N, C, Hc, Wc = semi.shape
    if binary_mask:
        agg = U.combine_from_logits_batch(semi, inv_homographies, mask_2D)
    else:
        heat = U.flattenDetection(semi.reshape(I * N, C, Hc, Wc)).reshape(I, N, Hc * 8, Wc * 8)
        agg = U.combine_heatmap_batch(heat, inv_homographies, mask_2D)
    pts = U.heatmap_to_pts_batch(agg, conf_thresh, nms_dist, top_k=top_k)
    return [p.transpose() for p in pts]


@torch.no_grad()
def collate_warped_pair(img, pnts_list, homographies, erosion_radius=3, bilinear=True):
    """The warped half of a training batch, built on the device from the unwarped images and their keypoints -- what
    datasets/Coco.py:341-392 does per sample in the DataLoader workers (inv_warp_image, warpLabels, compute_valid_mask):
    img [B,1,H,W], pnts_list = B arrays [P,2] (x, y), homographies [B,3,3] (normalised coordinates, already inverted as in
    Coco.py:345).  Returns the batch keys of the reference: warped_img, warped_labels, warped_res [B,2,H,W],
    warped_labels_bi, warped_valid_mask [B,1,H,W], homographies, inv_homographies.  (Photometric augmentation and the
    gaussian label blur are imgaug calls and stay where they are.)"""
    dev = img.device
    B, _, H, W = img.shape
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
