"""Host-side mirror of the reference's geometry / loss / NMS function library.

Same names, argument order, defaults, kwargs-swallowing and return conventions as
Gabriel-SGama/Semantic-SuperPoint `utils/utils.py` (+ `Train_model_heatmap_all.detector_loss`,
`Train_model_frontend_all.getMasks`, `export.combine_heatmap`), so that binding these over the reference
module attributes (see dropin.py) makes `train_val_sample` / `export_detector_homoAdapt_gpu` run on the
CUDA kernels.  Every function computes on a CUDA device through the C ABI (include/ssp_b200.h); there is
no CPU path.  Results are returned on the device the reference would have returned them on.
"""
import numpy as np
import torch

from . import _lib
from ._lib import call, f32c, ptr, stream_of
from .losses import DescriptorLossFn, DetectorLossPairFn, LazyPairMask, SemanticLossFn, get_descriptor_engine

__all__ = [
    "warp_points", "filter_points", "warp_points_filter", "warp_keypoints", "inv_warp_image_batch", "inv_warp_image",
    "compute_valid_mask", "ellipse_kernel", "labels2Dto3D", "getMasks", "detector_loss", "flattenDetection",
    "combine_heatmap", "getPtsFromHeatmap", "nms_fast", "box_nms", "soft_argmax_points", "descriptor_loss", "normPts",
    "denormPts", "homography_scaling_torch", "homography_scaling", "warpLabels", "warp_labels_batch",
]

_grid_cache = {}
_stencil_cache = {}


def _cuda_device(device, *tensors):
    """Device the kernels run on: a CUDA input wins, then a CUDA `device` argument, then the current GPU."""
    for t in tensors:
        if isinstance(t, torch.Tensor) and t.is_cuda:
            return t.device
    d = torch.device(device) if device is not None else torch.device("cpu")
    if d.type == "cuda":
        return torch.device("cuda", torch.cuda.current_device()) if d.index is None else d
    if not torch.cuda.is_available():
        raise RuntimeError("ssp_b200 has no CPU path: a CUDA device (sm_100a) is required")
    return torch.device("cuda", torch.cuda.current_device())


def _out_device(device, dev_cuda, *tensors):
    """Where the reference would leave the result: on `device` unless the inputs already live on a GPU."""
    for t in tensors:
        if isinstance(t, torch.Tensor) and t.is_cuda:
            return t.device
    d = torch.device(device) if device is not None else torch.device("cpu")
    return dev_cuda if d.type == "cuda" else d


def _linspace_grid(n, dev):
    """torch.linspace(-1, 1, n) evaluated on the CPU exactly like the reference (utils/utils.py:375)."""
    key = (n, str(dev))
    g = _grid_cache.get(key)
    if g is None:
        g = torch.linspace(-1, 1, n).to(dev)
        _grid_cache[key] = g
    return g


# ------------------------------------------------------------------------------------------------
# a1 / a10  point warps
# ------------------------------------------------------------------------------------------------
def _no_grad_inputs(name, *tensors):
    """The reference's versions of these are chains of differentiable torch ops; the kernels are forward-only (nothing in the
    reference back-propagates through them: they sit on the data / label side).  Refuse instead of silently cutting a graph."""
    if torch.is_grad_enabled():
        for t in tensors:
            if isinstance(t, torch.Tensor) and t.requires_grad:
                raise RuntimeError("ssp_b200.%s is forward-only (no autograd); detach() the input or call under torch.no_grad()" % name)


def warp_points(points, homographies, device="cpu"):
    """reference: utils/utils.py:315-343.  points [P,2] (x,y), homographies [3,3] or [B,3,3] -> [P,2] / [B,P,2]."""
    _no_grad_inputs("warp_points", points, homographies)
    no_batches = homographies.dim() == 2
    dev = _cuda_device(device, points, homographies)
    out_dev = _out_device(device, dev, points, homographies)
    Hm = f32c(homographies.reshape(-1, 3, 3), dev)
    pts = f32c(points, dev)
    if pts.dim() != 2 or pts.shape[1] != 2:
        raise RuntimeError("warp_points: points must be [P, 2], got %s" % (tuple(points.shape),))
    B, P = Hm.shape[0], pts.shape[0]
    out = torch.empty((B, P, 2), dtype=torch.float32, device=dev)
    if P > 0:
        call("ssp_warp_points_mask", ptr(pts), P, ptr(Hm), B, 0.0, 0.0, ptr(out), None, stream_of(out))
    out = out.to(out_dev)
    return out[0, :, :] if no_batches else out


def warp_points_filter(points, homographies, shape, device="cpu"):
    """Fused warp_points + filter_points mask (data_tools.warpLabels / repeatability use them back to back).

    Returns (warped [B,P,2] or [P,2], keep bool same leading shape) with keep = 0 <= p <= shape-1 (inclusive),
    shape = (W, H) for (x, y) points -- utils/utils.py:303-311.
    """
    no_batches = homographies.dim() == 2
    dev = _cuda_device(device, points, homographies)
    out_dev = _out_device(device, dev, points, homographies)
    Hm = f32c(homographies.reshape(-1, 3, 3), dev)
    pts = f32c(points, dev)
    B, P = Hm.shape[0], pts.shape[0]
    out = torch.empty((B, P, 2), dtype=torch.float32, device=dev)
    keep = torch.zeros((B, P), dtype=torch.uint8, device=dev)
    sx, sy = float(shape[0]), float(shape[1])
    if P > 0:
        call("ssp_warp_points_mask", ptr(pts), P, ptr(Hm), B, sx, sy, ptr(out), ptr(keep), stream_of(out))
    out, keep = out.to(out_dev), keep.to(out_dev).bool()
    return (out[0], keep[0]) if no_batches else (out, keep)


def filter_points(points, shape, return_mask=False):
    """reference: utils/utils.py:303-311.  Keeps points with 0 <= p <= shape-1 in every coordinate."""
    dev = _cuda_device(None, points)
    pts = f32c(points, dev)
    flat = pts.reshape(-1, 2)
    eye = torch.eye(3, dtype=torch.float32, device=dev).unsqueeze(0)
    shp = shape.float()
    out = torch.empty((1, flat.shape[0], 2), dtype=torch.float32, device=dev)
    keep = torch.zeros((1, flat.shape[0]), dtype=torch.uint8, device=dev)
    if flat.shape[0] > 0:
        call("ssp_warp_points_mask", ptr(flat), flat.shape[0], ptr(eye), 1, float(shp[0]), float(shp[1]), ptr(out),
             ptr(keep), stream_of(out))
    mask = keep.bool().reshape(pts.shape[:-1]).to(points.device)
    pf = points.float()
    if return_mask:
        return pf[mask], mask
    return pf[mask]


def warp_keypoints(keypoints, H, shape=None):
    """float64 pixel-coordinate warp of the evaluation side (evaluations/detector_evaluation.py:139-191).

    keypoints: numpy [K,2] (x,y); H numpy [3,3].  Returns warped [K,2] float64 and, if shape=(H,W) is given,
    also the in-bounds mask 0 <= x < W, 0 <= y < H (strict upper bound, as filter_keypoints).
    """
    dev = _cuda_device("cuda")
    kp = torch.as_tensor(np.ascontiguousarray(keypoints[:, :2], dtype=np.float64)).to(dev)
    Hm = torch.as_tensor(np.ascontiguousarray(H, dtype=np.float64)).to(dev)
    K = kp.shape[0]
    out = torch.empty((K, 2), dtype=torch.float64, device=dev)
    keep = torch.zeros((K,), dtype=torch.uint8, device=dev)
    Hh, W = (shape if shape is not None else (np.inf, np.inf))
    if K > 0:
        call("ssp_warp_keypoints_f64", ptr(kp), K, ptr(Hm), float(W), float(Hh), ptr(out), ptr(keep), stream_of(out))
    out_np = out.cpu().numpy()
    if shape is None:
        return out_np
    return out_np, keep.cpu().numpy().astype(bool)


def homography_scaling_torch(homography, H, W):
    """reference: utils/utils.py:297-300 (pixel <-> normalised coordinates; divides by W, H -- not W-1, H-1)."""
    trans = torch.tensor([[2.0 / W, 0.0, -1], [0.0, 2.0 / H, -1], [0.0, 0.0, 1.0]])
    return trans.inverse() @ homography @ trans


def homography_scaling(homography, H, W):
    """reference: utils/utils.py:291-294."""
    trans = np.array([[2.0 / W, 0.0, -1], [0.0, 2.0 / H, -1], [0.0, 0.0, 1.0]])
    return np.linalg.inv(trans) @ homography @ trans


def normPts(pts, shape):
    """reference: utils/utils.py:745-755."""
    return pts / shape * 2 - 1


def denormPts(pts, shape):
    """reference: utils/utils.py:758-768."""
    return (pts + 1) * shape / 2


# ------------------------------------------------------------------------------------------------
# a2 / a3  image warps
# ------------------------------------------------------------------------------------------------
def inv_warp_image_batch(img, mat_homo_inv, device="cpu", mode="bilinear"):
    """reference: utils/utils.py:347-385.  img [B,C,H,W] (2-D/3-D viewed as [1,1,H,W]), H^-1 [B,3,3] / [3,3]."""
    _no_grad_inputs("inv_warp_image_batch", img, mat_homo_inv)
    if img.dim() == 2 or img.dim() == 3:
        img = img.view(1, 1, img.shape[0], img.shape[1])
    if mat_homo_inv.dim() == 2:
        mat_homo_inv = mat_homo_inv.view(1, 3, 3)
    if mode not in ("bilinear", "nearest"):
        raise ValueError("inv_warp_image_batch: mode must be 'bilinear' or 'nearest', got %r" % (mode,))
    dev = _cuda_device(device, img, mat_homo_inv)
    out_dev = _out_device(device, dev, img)
    x = f32c(img, dev)
    Hm = f32c(mat_homo_inv, dev)
    B, C, H, W = x.shape
    if Hm.shape[0] != B:
        raise RuntimeError("inv_warp_image_batch: %d images but %d homographies" % (B, Hm.shape[0]))
    out = torch.empty_like(x)
    call("ssp_inv_warp_image", ptr(x), B, C, H, W, ptr(Hm), ptr(_linspace_grid(W, dev)), ptr(_linspace_grid(H, dev)),
         0 if mode == "bilinear" else 1, ptr(out), stream_of(out))
    return out.to(out_dev)


def inv_warp_image(img, mat_homo_inv, device="cpu", mode="bilinear"):
    """reference: utils/utils.py:388-405 (squeeze wrapper)."""
    return inv_warp_image_batch(img, mat_homo_inv, device, mode).squeeze()


def ellipse_kernel(erosion_radius):
    """cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (2r, 2r)) restated (OpenCV morph.dispatch.cpp): row i spans
    columns [c - dx, c + dx] with dx = round(c * sqrt((r^2 - dy^2) / r^2)), r = c = ksize // 2.  Anchor = (r, r)."""
    k = int(erosion_radius) * 2
    r = c = k // 2
    inv_r2 = 1.0 / (r * r) if r else 0.0
    ker = np.zeros((k, k), dtype=np.uint8)
    for i in range(k):
        dy = i - r
        if abs(dy) <= r:
            dx = int(np.rint(c * np.sqrt((r * r - dy * dy) * inv_r2)))
            ker[i, max(c - dx, 0):min(c + dx + 1, k)] = 1
    return ker


def compute_valid_mask(image_shape, inv_homography, device="cpu", erosion_radius=0, kernel=None):
    """reference: utils/utils.py:715-742.  Nearest warp of ones + erosion, fused in one kernel (no host trip).

    `kernel` (optional, numpy uint8 [kh,kw], anchor at (kw//2, kh//2)) overrides the ellipse structuring element.
    """
    if inv_homography.dim() == 2:
        inv_homography = inv_homography.view(-1, 3, 3)
    dev = _cuda_device(device, inv_homography)
    out_dev = _out_device(device, dev)
    Hm = f32c(inv_homography, dev)
    B = Hm.shape[0]
    H, W = int(image_shape[0]), int(image_shape[1])
    out = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    kern_t, kh, kw = None, 0, 0
    if kernel is None and erosion_radius > 0:
        key = ("ellipse", int(erosion_radius), str(dev))  # device copy of the structuring element, made once
        if key not in _stencil_cache:
            k = ellipse_kernel(erosion_radius)
            _stencil_cache[key] = (torch.from_numpy(k).to(dev), k.shape)
        kern_t, (kh, kw) = _stencil_cache[key]
    elif kernel is not None and kernel.size > 0:
        kernel = np.ascontiguousarray(kernel, dtype=np.uint8)
        kh, kw = kernel.shape
        kern_t = torch.from_numpy(kernel).to(dev)
    call("ssp_valid_mask", B, H, W, ptr(Hm), ptr(_linspace_grid(W, dev)), ptr(_linspace_grid(H, dev)), ptr(kern_t),
         kh, kw, kw // 2, kh // 2, ptr(out), stream_of(out))
    return out.to(out_dev)


# ------------------------------------------------------------------------------------------------
# a4  detector labels / loss
# ------------------------------------------------------------------------------------------------
def _check_cell(cell_size):
    if int(cell_size) != 8:
        raise ValueError("cell_size must be 8 (the reference hard-codes SpaceToDepth(8), utils/utils.py:422)")


def labels2Dto3D(labels, cell_size, add_dustbin=True):
    """reference: utils/utils.py:408-440.  [B,1,H,W] -> [B,65,H/8,W/8] (64 channels without dustbin)."""
    _check_cell(cell_size)
    dev = _cuda_device(None, labels)
    x = f32c(labels, dev)
    B, C, H, W = x.shape
    if C != 1:
        raise RuntimeError("labels2Dto3D: expected [B,1,H,W], got %s" % (tuple(labels.shape),))
    out = torch.empty((B, 65 if add_dustbin else 64, H // 8, W // 8), dtype=torch.float32, device=dev)
    call("ssp_labels2d_to_3d", ptr(x), B, H, W, 1 if add_dustbin else 0, ptr(out), stream_of(out))
    return out.to(labels.device) if not labels.is_cuda else out


def getMasks(mask_2D, cell_size, device="cpu"):
    """reference: Train_model_frontend_all.py:373-386.  [B,1,H,W] -> [B,H/8,W/8] product over each cell."""
    _check_cell(cell_size)
    dev = _cuda_device(device, mask_2D)
    out_dev = _out_device(device, dev, mask_2D)
    x = f32c(mask_2D, dev)
    B, C, H, W = x.shape
    out = torch.empty((B, H // 8, W // 8), dtype=torch.float32, device=dev)
    call("ssp_cell_mask", ptr(x), B, H, W, ptr(out), stream_of(out))
    return out.to(out_dev)


def detector_loss(input, target, mask=None, loss_type="softmax", dist_group=None):
    """reference: Train_model_heatmap_all.py:155-179.  BCE over softmax(65) probabilities, masked mean."""
    if loss_type == "l2":
        return torch.nn.functional.mse_loss(input, target, reduction="mean")
    if loss_type != "softmax":
        raise ValueError("detector_loss: loss_type must be 'softmax' or 'l2'")
    _lib.require_cuda(input)
    if mask is None:
        mask = torch.ones((input.shape[0],) + tuple(input.shape[2:]), device=input.device)
    return DetectorLossPairFn.apply(input, target, mask, None, None, None, False, dist_group)


def detector_loss_2d(semi, labels_2D, mask_2D, dist_group=None):
    """Fused labels2Dto3D(add_dustbin=True) + getMasks + detector_loss from the 2-D maps (one kernel)."""
    _lib.require_cuda(semi)
    return DetectorLossPairFn.apply(semi, labels_2D, mask_2D, None, None, None, True, dist_group)


def detector_loss_pair_2d(semi, labels_2D, mask_2D, semi_warp, warped_labels, mask_warp_2D, dist_group=None):
    """Both detector losses of a training pair from the 2-D maps in one launch each way.
    Returns (loss_det, loss_det_warp, mask_3D_flattened of the warped mask [B,Hc,Wc])."""
    _lib.require_cuda(semi, semi_warp)
    return DetectorLossPairFn.apply(semi, labels_2D, mask_2D, semi_warp, warped_labels, mask_warp_2D, True, dist_group)


def sem_loss(pred, label, device="cpu", ignore_index=133, dist_group=None):
    """reference: Train_model_heatmap_all.py:181-193 (method sem_loss(self, pred, label, device)):
    nn.CrossEntropyLoss(ignore_index=133)(pred, label).

    pred [B,C,H,W] (what the unmodified model returns) or the head output BEFORE the model's final F.interpolate,
    [B,C,H/8,W/8] (models/SuperPointNet_gauss2_ssmall.py:86-90): then the x8 bilinear upsample is fused into the loss and
    the [B,133,H,W] logits are never materialised.  label [B,H,W] integer."""
    _lib.require_cuda(pred)
    return SemanticLossFn.apply(pred, label, int(ignore_index), dist_group)


# ------------------------------------------------------------------------------------------------
# a6 / a7  heatmaps
# ------------------------------------------------------------------------------------------------
def flattenDetection(semi, tensor=False):
    """reference: utils/utils.py:515-560.  [B,65,Hc,Wc] -> [B,1,8Hc,8Wc]; [65,Hc,Wc] -> [1,8Hc,8Wc]."""
    # forward-only: the reference's trainers call this on logits that require grad (Train_model_frontend_all.py:668,
    # Train_model_heatmap_all.py:371) but only to log / extract points -- nothing back-propagates through it, so the result
    # is a detached tensor rather than an error.
    semi = semi.detach()
    batch = semi.dim() == 4
    dev = _cuda_device(None, semi)
    x = f32c(semi if batch else semi.unsqueeze(0), dev)
    N, C, Hc, Wc = x.shape
    if C != 65:
        raise RuntimeError("flattenDetection: expected 65 channels, got %d" % C)
    heat = torch.empty((N, 1, Hc * 8, Wc * 8), dtype=torch.float32, device=dev)
    call("ssp_flatten_detection", ptr(x), N, Hc, Wc, ptr(heat), stream_of(heat))
    if not semi.is_cuda:
        heat = heat.to(semi.device)
    return heat if batch else heat.squeeze(0)


def combine_heatmap(heatmap, inv_homographies, mask_2D, device="cpu"):
    """reference: export.py:49-60.  heatmap, mask_2D [N,1,H,W]; inv_homographies [1,N,3,3] -> [1,H,W]."""
    dev = _cuda_device(device, heatmap, mask_2D)
    out_dev = _out_device(device, dev, heatmap)
    h = f32c(heatmap, dev)
    m = f32c(mask_2D, dev)
    Hm = f32c(inv_homographies[0, :, :, :], dev)
    N, C, H, W = h.shape
    if C != 1 or m.shape != h.shape or Hm.shape[0] != N:
        raise RuntimeError("combine_heatmap: expected heatmap/mask [N,1,H,W] and homographies [1,N,3,3]")
    return combine_heatmap_batch(h.view(1, N, H, W), Hm[None], m.view(1, N, H, W)).to(out_dev)


def combine_heatmap_batch(heatmap, inv_homographies, mask_2D):
    """Batched export form: heatmap/mask [I,N,H,W], inv_homographies [I,N,3,3] -> [I,H,W] in one launch."""
    dev = _cuda_device("cuda", heatmap)
    h, Hm, m = f32c(heatmap, dev), f32c(inv_homographies, dev), f32c(mask_2D, dev)
    I, N, H, W = h.shape
    out = torch.empty((I, H, W), dtype=torch.float32, device=dev)
    call("ssp_combine_heatmap", ptr(h), ptr(m), ptr(Hm), I, N, H, W, ptr(_linspace_grid(W, dev)), ptr(_linspace_grid(H, dev)),
         ptr(out), stream_of(out))
    return out


def combine_from_logits_batch(semi, inv_homographies, mask_2D):
    """flattenDetection + combine_heatmap for the batched export path when the valid masks are 0/1 images (what
    compute_valid_mask returns): semi [I,N,65,Hc,Wc], inv_homographies [I,N,3,3], mask_2D [I,N,H,W] -> [I,H,W].
    The mask is folded into the flattened heatmap as its sign (csrc/detector.cu: flatten_detection_masked), so the aggregation
    gathers one array per tap instead of two: results bit-identical to flattenDetection + combine_heatmap_batch; a mask value
    other than 0 / 1 turns the output into NaN."""
    dev = _cuda_device("cuda", semi)
    x, Hm, m = f32c(semi, dev), f32c(inv_homographies, dev), f32c(mask_2D, dev)
    I, N, C, Hc, Wc = x.shape
    if C != 65:
        raise RuntimeError("combine_from_logits_batch: expected 65 channels, got %d" % C)
    H, W = Hc * 8, Wc * 8
    if tuple(m.shape[-2:]) != (H, W) or m.numel() != I * N * H * W:
        raise RuntimeError("combine_from_logits_batch: mask_2D must be [I,N,%d,%d], got %s" % (H, W, tuple(mask_2D.shape)))
    st = stream_of(x)
    heat = torch.empty((I, N, H, W), dtype=torch.float32, device=dev)
    flag = torch.zeros((1,), dtype=torch.int32, device=dev)
    call("ssp_flatten_detection_masked", ptr(x), ptr(m), I * N, Hc, Wc, ptr(heat), ptr(flag), st)
    out = torch.empty((I, H, W), dtype=torch.float32, device=dev)
    xs, ys = _linspace_grid(W, dev), _linspace_grid(H, dev)
    call("ssp_combine_heatmap_signed", ptr(heat), ptr(Hm), I, N, H, W, ptr(xs), ptr(ys), ptr(flag), ptr(out), st)
    return out


# ------------------------------------------------------------------------------------------------
# a8 / a9  keypoint extraction
# ------------------------------------------------------------------------------------------------


def _cheb_stencil(R, dev):
    key = ("cheb", R, str(dev))
    s = _stencil_cache.get(key)
    if s is None:
        s = torch.ones(((2 * R + 1) ** 2,), dtype=torch.uint8, device=dev)
        _stencil_cache[key] = s
    return s


def _iou_stencil(size, iou, dev):
    """Offsets (dy,dx) whose size x size boxes overlap with IoU > iou, evaluated in float32 like
    torchvision.ops.nms (inter / (area_a + area_b - inter) > thr)."""
    key = ("iou", float(size), float(iou), str(dev))
    s = _stencil_cache.get(key)
    if s is None:
        R = max(int(np.ceil(size)) - 1, 0)
        d = np.abs(np.arange(-R, R + 1, dtype=np.float32))
        sz = np.float32(size)
        w = np.maximum(sz - d, np.float32(0))
        inter = w[:, None] * w[None, :]
        area = sz * sz
        ovr = inter / (area + area - inter)
        st = (ovr > np.float32(iou)).astype(np.uint8)
        s = (torch.from_numpy(st.reshape(-1).copy()).to(dev), R)
        _stencil_cache[key] = s
    return s


def _nms_ws(I, H, W, capacity, dev):
    nbytes = _lib.load().ssp_nms_ws_bytes(I, H, W, capacity)
    return torch.empty((nbytes,), dtype=torch.uint8, device=dev), nbytes


def _nms_batch(x, conf_thresh, nms_dist, border_remove=4, capacity=None):
    """Device part of getPtsFromHeatmap for a stack x [I,H,W] of fp32 CUDA heatmaps: one ssp_nms_fast call, whose sync also
    reads the per-image counts.  Returns (pts [I,3,capacity] float64 on the device, confidence-descending; host list of
    the counts; the same counts on the device as an int32 [I] view of the NMS workspace)."""
    I, H, W = x.shape
    R = int(nms_dist)
    if capacity is None:
        capacity = (H // (R + 1) + 1) * (W // (R + 1) + 1)  # kept points are > R apart in Chebyshev distance
    pts = torch.empty((I, 3, capacity), dtype=torch.float64, device=x.device)
    counts = (_lib._c.c_int * I)()
    ws, nbytes = _nms_ws(I, H, W, capacity, x.device)
    call("ssp_nms_fast", ptr(x), I, H, W, float(conf_thresh), R, ptr(_cheb_stencil(R, x.device)), int(border_remove),
         capacity, ptr(pts), counts, ptr(ws), nbytes, stream_of(x))
    off = _lib.load().ssp_nms_ws_counts_offset(I, H, W)
    return pts, list(counts), ws[off:off + 4 * I].view(torch.int32)


def heatmap_to_pts_batch(heat, conf_thresh, nms_dist, border_remove=4, capacity=None, top_k=None, subpixel=False,
                         patch_size=5):
    """getPtsFromHeatmap for a stack [I,H,W] of CUDA heatmaps in one call.  Returns a list of [3,K] float64 arrays.
    top_k: only the top_k most confident points of every image are copied back (the list is confidence-descending, so this is
    what the export's `pts[:top_k]` keeps, export.py:317-323).
    subpixel: x and y of the points that are copied back are refined by soft_argmax_points(heat, pts, patch_size) on the
    device before the read-back (export.py:309-314); each point is refined on its own, so refining only the top_k is the
    reference's refine-then-truncate."""
    dev = _cuda_device("cuda", heat)
    x = f32c(heat, dev)
    I, H, W = x.shape
    pts, counts, counts_dev = _nms_batch(x, conf_thresh, nms_dist, border_remove, capacity)
    cnt = [min(c, top_k) for c in counts] if top_k else counts
    kmax = max(cnt) if I else 0
    if subpixel and kmax:
        # per-image counts straight from the NMS workspace: no copy, no sync
        call("ssp_soft_argmax_points", ptr(x), I, H, W, ptr(pts), pts.shape[2], ptr(counts_dev), kmax, int(patch_size),
             stream_of(x))
    host = pts[:, :, :kmax].cpu().numpy() if kmax else np.zeros((I, 3, 0))
    return [host[i, :, :cnt[i]] for i in range(I)]


def getPtsFromHeatmap(heatmap, conf_thresh, nms_dist):
    """reference: utils/utils.py:581-609 (twin models/model_wrap.py:266-293).

    heatmap: numpy (or torch) [H,W].  Returns numpy float64 [3,K] rows (x, y, conf), confidence-descending,
    after greedy Chebyshev-radius NMS and removal of the 4-pixel border; empty -> zeros((3,0)).
    """
    if isinstance(heatmap, np.ndarray):
        if heatmap.dtype != np.float32:
            # the reference compares in the array's own dtype; fp64 heatmaps are not produced by any call site
            heatmap = heatmap.astype(np.float32)
        t = torch.from_numpy(np.ascontiguousarray(heatmap))
    else:
        t = heatmap.detach()
    dev = _cuda_device("cuda", t)
    out = heatmap_to_pts_batch(t.to(dev).reshape(1, t.shape[-2], t.shape[-1]), conf_thresh, nms_dist)[0]
    return out if out.shape[1] else np.zeros((3, 0))


def soft_argmax_points(heatmap, pts, patch_size=5):
    """reference: models/model_wrap.py:212-248 (SuperPointFrontend_torch.soft_argmax_points(self, pts, patch_size=5), which
    reads the heatmap from self.heatmap), with utils/losses.py's extract_patch_from_points, norm_patches, do_log and the
    soft arg-max of torchgeometry's SpatialSoftArgmax2d(normalized_coordinates=False).

    heatmap: torch (any device) or numpy, squeezed to [H,W].  pts: numpy float64 [3,K] (x, y, conf) or a one-element list of
    it.  Returns a one-element list holding the refined [3,K] float64 array: x and y moved to the soft arg-max of the
    patch_size x patch_size patch around (int(x), int(y)) (zeros outside the image), conf unchanged.  K = 0 -> [zeros((3,0))]
    (the reference crashes in np.stack)."""
    if isinstance(pts, (list, tuple)):
        pts = pts[0]
    p = np.ascontiguousarray(pts, dtype=np.float64)  # the kernel reads rows x, y of a row-major [3,K]
    if p.ndim != 2 or p.shape[0] != 3:
        raise RuntimeError("soft_argmax_points: pts must be [3, K] (x, y, conf), got %s" % (p.shape,))
    K = p.shape[1]
    if K == 0:
        return [np.zeros((3, 0))]
    if isinstance(heatmap, np.ndarray):
        heatmap = torch.from_numpy(np.ascontiguousarray(heatmap, dtype=np.float32))
    dev = _cuda_device("cuda", heatmap)
    h = f32c(heatmap.detach().squeeze(), dev)
    if h.dim() != 2:
        raise RuntimeError("soft_argmax_points: heatmap must squeeze to [H, W], got %s" % (tuple(heatmap.shape),))
    H, W = h.shape
    pd = torch.from_numpy(p).to(dev)
    counts = torch.tensor([K], dtype=torch.int32).to(dev)
    call("ssp_soft_argmax_points", ptr(h), 1, H, W, ptr(pd), K, ptr(counts), K, int(patch_size), stream_of(pd))
    return [pd.cpu().numpy()]


def nms_fast(in_corners, H, W, dist_thresh):
    """reference: utils/utils.py:653-712 (twin models/model_wrap.py:129-192).

    in_corners: numpy [3,N] (x, y, conf).  Returns (corners [3,K] sorted by confidence, indices [K])."""
    in_corners = np.asarray(in_corners)
    n = in_corners.shape[1]
    if n == 0:
        return np.zeros((3, 0)).astype(int), np.zeros(0).astype(int)
    inds1 = np.argsort(-in_corners[2, :], kind="stable")
    corners = in_corners[:, inds1]
    rc = corners[:2, :].round().astype(int)
    if n == 1:
        return np.vstack((rc, in_corners[2])).reshape(3, 1), np.zeros((1)).astype(int)
    dev = _cuda_device("cuda")
    grid = np.full((H, W), np.nan, dtype=np.float32)
    inds = np.zeros((H, W), dtype=np.int64)
    # first visit (highest confidence) decides the NMS; the index map keeps the last writer, as the reference.  The
    # priority handed to the device is the point's RANK in the reference's own fp64 ordering (exact in fp32 for
    # n < 2^24), not the confidence: two confidences that differ only beyond fp32 still order the way the reference does.
    assert n < (1 << 24)
    grid[rc[1, ::-1], rc[0, ::-1]] = -np.arange(n - 1, -1, -1, dtype=np.float32)
    inds[rc[1], rc[0]] = np.arange(n)
    heat = torch.from_numpy(grid).to(dev).reshape(1, H, W)
    R = int(dist_thresh)
    capacity = min(n, (H // (R + 1) + 1) * (W // (R + 1) + 1))
    pts = torch.empty((1, 3, capacity), dtype=torch.float64, device=dev)
    counts = (_lib._c.c_int * 1)()
    ws, nbytes = _nms_ws(1, H, W, capacity, dev)
    call("ssp_nms_fast", ptr(heat), 1, H, W, float("-inf"), R, ptr(_cheb_stencil(R, dev)), 0, capacity, ptr(pts),
         counts, ptr(ws), nbytes, stream_of(heat))
    K = counts[0]
    kept = pts[0, :, :K].cpu().numpy()
    # emit in the reference's order: argsort(-values) (stable) over the row-major survivors
    ky, kx = kept[1].astype(int), kept[0].astype(int)
    order = np.lexsort((kx, ky))  # row-major
    ky, kx = ky[order], kx[order]
    inds_keep = inds[ky, kx]
    out = corners[:, inds_keep]
    inds2 = np.argsort(-out[-1, :], kind="stable")
    return out[:, inds2], inds1[inds_keep[inds2]]


def box_nms(prob, size, iou=0.1, min_prob=0.01, keep_top_k=0):
    """reference: utils/utils.py:612-650.  IoU-NMS of size x size boxes centred on every pixel with
    prob > min_prob; survivors keep their score, everything else is 0.  keep_top_k == 0 raises
    NotImplementedError exactly like the reference (its only live branch needs keep_top_k != 0)."""
    if keep_top_k == 0:
        raise NotImplementedError
    _lib.require_cuda(prob)
    x = f32c(prob, prob.device)
    H, W = x.shape
    stencil, R = _iou_stencil(size, iou, x.device)
    out = torch.empty_like(x)
    ws, nbytes = _nms_ws(1, H, W, 1, x.device)
    call("ssp_box_nms", ptr(x), 1, H, W, float(min_prob), R, ptr(stencil), ptr(out), ptr(ws), nbytes, stream_of(x))
    return out


# ------------------------------------------------------------------------------------------------
# a5  dense descriptor loss
# ------------------------------------------------------------------------------------------------
def descriptor_loss(descriptors, descriptors_warped, homographies, mask_valid=None, cell_size=8, lamda_d=250,
                    device="cpu", descriptor_dist=4, **config):
    """reference: utils/utils.py:779-893.

    Returns (loss_desc, mask, pos_sum, neg_sum); all three scalars are differentiable w.r.t. both descriptor
    tensors.  `mask` is the [B,Hc,Wc,Hc,Wc] correspondence mask as a lazy object (materialised on first use,
    the reference's only caller never reads it).  Unknown keyword arguments are swallowed like the reference
    does (its YAML key `lambda_d` never reaches `lamda_d`).  Engine: config key `engine` or
    losses.set_descriptor_engine(): "bf16x3" (default, fp32-grade), "bf16" (fast) or "fp32" (CUDA cores).
    """
    _lib.require_cuda(descriptors, descriptors_warped)
    dev = descriptors.device
    if homographies.dim() == 2:
        homographies = homographies.unsqueeze(0)
    B, Dch, Hc, Wc = descriptors.shape
    Hm = f32c(homographies, dev)
    if Hm.shape[0] != B:
        raise RuntimeError("descriptor_loss: %d pairs but %d homographies" % (B, Hm.shape[0]))
    mv = None
    if mask_valid is not None:
        mv = f32c(mask_valid, dev).reshape(B, -1)
        if mv.shape[1] != Hc * Wc:
            raise RuntimeError("descriptor_loss: mask_valid must be [B,1,Hc,Wc]")
    engine = config.get("engine", None) or get_descriptor_engine()
    out = DescriptorLossFn.apply(descriptors, descriptors_warped, Hm, mv, int(cell_size), float(lamda_d),
                                 float(descriptor_dist), engine, config.get("dist_group", None),
                                 config.get("debug_S", None))
    loss, pos_sum, neg_sum, wpts = out
    mask = LazyPairMask(wpts, B, Hc, Wc, int(cell_size), float(descriptor_dist))
    return loss, mask, pos_sum, neg_sum


# ------------------------------------------------------------------------------------------------
# 8f rank 3: sparse descriptors (export_descriptor / evaluation, the step after NMS)
# ------------------------------------------------------------------------------------------------
def sample_desc_from_points(coarse_desc, pts, cell=8):
    """reference: models/model_wrap.py:295-313 (SuperPointFrontend_torch.sample_desc_from_points(self, coarse_desc, pts)).

    coarse_desc [1,D,Hc,Wc] tensor, pts numpy [3,K] (x, y, conf) -> numpy float32 [D,K], bilinear samples of the coarse
    map at the keypoints (grid_sample align_corners=True), L2-normalised per point; K = 0 -> zeros((D,0))."""
    D = int(coarse_desc.shape[1])
    pts = np.asarray(pts)
    K = int(pts.shape[1])
    if K == 0:
        return np.zeros((D, 0))
    dev = _cuda_device("cuda", coarse_desc)
    cd = f32c(coarse_desc.detach(), dev)
    if cd.dim() != 4 or cd.shape[0] != 1:
        raise RuntimeError("sample_desc_from_points: coarse_desc must be [1,D,Hc,Wc], got %s" % (tuple(coarse_desc.shape),))
    p = torch.from_numpy(np.ascontiguousarray(pts, dtype=np.float64)).to(dev)
    out = torch.empty((D, K), dtype=torch.float32, device=dev)
    count = torch.full((1,), K, dtype=torch.int32, device=dev)
    call("ssp_sample_desc_batch", ptr(cd), ptr(p), K, ptr(count), K, 1, D, int(cd.shape[2]), int(cd.shape[3]), int(cell),
         ptr(out), stream_of(out))
    return out.cpu().numpy()


def nn_match_two_way(desc1, desc2, nn_thresh):
    """reference: models/model_wrap.py:451-494 (PointTracker.nn_match_two_way(self, desc1, desc2, nn_thresh)).

    desc1 [D,K1], desc2 [D,K2] unit descriptors (numpy or tensors) -> numpy float64 [3,L] rows (index in 1, index in 2,
    distance) of the mutual nearest neighbours closer than nn_thresh, in increasing index-1 order."""
    if desc1.shape[0] != desc2.shape[0]:
        raise AssertionError("nn_match_two_way: descriptor dimensions differ")
    K1, K2 = int(desc1.shape[1]), int(desc2.shape[1])
    if K1 == 0 or K2 == 0:
        return np.zeros((3, 0))
    if nn_thresh < 0.0:
        raise ValueError("'nn_thresh' should be non-negative")
    dev = _cuda_device("cuda", *[d for d in (desc1, desc2) if isinstance(d, torch.Tensor)])
    t = lambda d: f32c(d.detach() if isinstance(d, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(d, dtype=np.float32)), dev)
    a, b = t(desc1), t(desc2)
    best = torch.empty((K1 + K2,), dtype=torch.int64, device=dev)
    call("ssp_nn_match", ptr(a), ptr(b), int(a.shape[0]), K1, K2, ptr(best[:K1]), ptr(best[K1:]), stream_of(a))
    keys = best.cpu().numpy().view(np.uint64)
    idx = (keys[:K1] & np.uint64(0xFFFFFFFF)).astype(np.int64)
    scores = (keys[:K1] >> np.uint64(32)).astype(np.uint32).view(np.float32).astype(np.float64)
    idx2 = (keys[K1:] & np.uint64(0xFFFFFFFF)).astype(np.int64)
    keep = np.logical_and(scores < nn_thresh, np.arange(K1) == idx2[idx])     # model_wrap.py:476-481
    matches = np.zeros((3, int(keep.sum())))
    matches[0, :] = np.arange(K1)[keep]
    matches[1, :] = idx[keep]
    matches[2, :] = scores[keep]
    return matches


def _pack_planes(desc):
    """[I,256,K] fp32 CUDA descriptors -> the matcher's bf16 hi / lo planes [2,I,R,256] (R = ceil(K/256)*256, zero rows
    past K) from one ssp_desc_pack launch; [0] is hi, [1] is lo (above hi in memory, as the tensor maps need)."""
    I, D, K = desc.shape
    R = (K + 255) // 256 * 256
    planes = torch.empty((2, I, R, D), dtype=torch.bfloat16, device=desc.device)
    call("ssp_desc_pack", ptr(desc), None, I, D, K, ptr(planes[0]), ptr(planes[1]), stream_of(desc))
    return planes


def _nn_match_planes(planes1, planes2, counts1, counts2, limit, nn_thresh, matches, nmatch):
    """ssp_nn_match_batch on planes [2,P,R,256] from _pack_planes: pair p matches its first min(counts[p], limit) points of
    each set.  matches [P,3,R1] float64 and nmatch [P] int32 are device outputs."""
    P, R1, R2 = planes1.shape[1], planes1.shape[2], planes2.shape[2]
    nbytes = _lib.load().ssp_nn_match_batch_ws_bytes(P, R1, R2)
    ws = torch.empty((nbytes // 8,), dtype=torch.int64, device=planes1.device)
    call("ssp_nn_match_batch", ptr(planes1[0]), ptr(planes1[1]), R1, ptr(planes2[0]), ptr(planes2[1]), R2, ptr(counts1),
         ptr(counts2), int(limit), P, float(nn_thresh), ptr(matches), ptr(nmatch), ptr(ws), nbytes, stream_of(matches))


def _check_nn_thresh(nn_thresh):
    if not nn_thresh >= 0.0:
        raise ValueError("'nn_thresh' should be non-negative")


def nn_match_two_way_batch(desc1, desc2, nn_thresh, counts1=None, counts2=None):
    """nn_match_two_way for P pairs at once, on the tensor cores.

    desc1 [P,256,K1], desc2 [P,256,K2] unit descriptors (CUDA tensors); counts1 / counts2 (optional, length P: sequences or
    integer tensors): pair p uses its first counts[p] columns (capped at K), the rest are ignored.  Returns P numpy float64
    [3,L] arrays (index in 1, index in 2, distance) of the mutual nearest neighbours closer than nn_thresh, in increasing
    index-1 order.  Products are fp32-grade (bf16 hi / lo split, three MMA passes); the threshold is compared in fp32."""
    _check_nn_thresh(nn_thresh)
    if desc1.dim() != 3 or desc2.dim() != 3 or desc1.shape[0] != desc2.shape[0]:
        raise ValueError("nn_match_two_way_batch: expected desc1 [P,256,K1] and desc2 [P,256,K2]")
    if desc1.shape[1] != 256 or desc2.shape[1] != 256:
        raise ValueError("nn_match_two_way_batch: the tensor-core matcher takes 256-dimensional descriptors")
    _lib.require_cuda(desc1, desc2)
    P, K1, K2 = int(desc1.shape[0]), int(desc1.shape[2]), int(desc2.shape[2])
    if P == 0 or K1 == 0 or K2 == 0:
        return [np.zeros((3, 0)) for _ in range(P)]
    dev = desc1.device

    def cnt(c, K):
        if c is None:
            return torch.full((P,), K, dtype=torch.int32, device=dev)
        c = torch.as_tensor(c).to(device=dev, dtype=torch.int32).reshape(-1)
        if c.numel() != P:
            raise ValueError("nn_match_two_way_batch: %d counts for %d pairs" % (c.numel(), P))
        return c.clamp(min=0, max=K)

    c1, c2 = cnt(counts1, K1), cnt(counts2, K2)
    p1, p2 = _pack_planes(f32c(desc1.detach(), dev)), _pack_planes(f32c(desc2.detach(), dev))
    matches = torch.empty((P, 3, p1.shape[2]), dtype=torch.float64, device=dev)
    nmatch = torch.empty((P,), dtype=torch.int32, device=dev)
    _nn_match_planes(p1, p2, c1, c2, max(K1, K2), nn_thresh, matches, nmatch)
    m, n = matches.cpu().numpy(), nmatch.cpu().numpy()
    return [m[p, :, :n[p]] if n[p] else np.zeros((3, 0)) for p in range(P)]


# ------------------------------------------------------------------------------------------------
# 8f rank 4: label warping of the warped training pair (dataset side, moved to the device)
# ------------------------------------------------------------------------------------------------
def warp_labels_batch(pnts_list, H, W, homographies, bilinear=False, device="cuda"):
    """warpLabels for a batch of images in one launch (the GPU-collate form).

    pnts_list: list of B arrays / tensors [P_b, 2] (x, y); homographies [B,3,3] in normalised coordinates.
    Returns dict(labels [B,1,H,W], res [B,H,W,2], warped_pnts = list of [M_b,2] tensors[, labels_bi [B,1,H,W]]), on the device."""
    dev = _cuda_device(device, homographies if isinstance(homographies, torch.Tensor) else None)
    B = len(pnts_list)
    Hn = torch.as_tensor(homographies, dtype=torch.float32).reshape(B, 3, 3).cpu()
    # homography_scaling_torch on the host, op for op as the reference (utils/utils.py:297-300): 3x3 matrices
    Hpix = torch.stack([homography_scaling_torch(Hn[b], H, W) for b in range(B)]).to(dev).contiguous()
    counts_h = [int(len(p)) for p in pnts_list]
    Pmax = max(max(counts_h), 1)
    pts = torch.zeros((B, Pmax, 2), dtype=torch.float32)
    for b, p in enumerate(pnts_list):
        if counts_h[b]:
            pts[b, :counts_h[b]] = torch.as_tensor(np.asarray(p)[:, :2] if not isinstance(p, torch.Tensor) else p[:, :2].cpu(),
                                                   dtype=torch.float32)
    pts = pts.to(dev)
    counts = torch.tensor(counts_h, dtype=torch.int32, device=dev)
    labels = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
    res = torch.empty((B, H, W, 2), dtype=torch.float32, device=dev)
    lbi = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev) if bilinear else None
    warped = torch.empty((B, Pmax, 2), dtype=torch.float32, device=dev)
    kept = torch.empty((B,), dtype=torch.int32, device=dev)
    nbytes = _lib.load().ssp_warp_labels_ws_bytes(B, H, W)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    call("ssp_warp_labels", ptr(pts), ptr(counts), B, Pmax, int(H), int(W), ptr(Hpix), 1 if bilinear else 0, ptr(labels),
         ptr(res), ptr(lbi), ptr(warped), ptr(kept), ptr(ws), nbytes, stream_of(labels))
    kept_h = kept.cpu().tolist()  # the reference returns the filtered point list: its length is data dependent (one sync)
    out = {"labels": labels, "res": res, "warped_pnts": [warped[b, :kept_h[b]] for b in range(B)]}
    if bilinear:
        out["labels_bi"] = lbi
    return out


def warpLabels(pnts, H, W, homography, bilinear=False):
    """reference: datasets/data_tools.py:37-63 (same signature and dict of results: labels [1,H,W], res [H,W,2], warped_pnts
    [M,2] and, with bilinear=True, labels_bi [1,H,W]); results are returned on the CPU like the reference's."""
    o = warp_labels_batch([pnts], H, W, torch.as_tensor(homography, dtype=torch.float32).reshape(1, 3, 3), bilinear)
    out = {"labels": o["labels"][0].cpu(), "res": o["res"][0].cpu(), "warped_pnts": o["warped_pnts"][0].cpu()}
    if bilinear:
        out["labels_bi"] = o["labels_bi"][0].cpu()
    return out


# ------------------------------------------------------------------------------------------------
# evaluation of exported image pairs (evaluation.py:86-499 of the reference lineage)
# ------------------------------------------------------------------------------------------------
RANSAC_HYPOTHESES = 2000   # cv2.findHomography(RANSAC)'s maxIters, every hypothesis evaluated
RANSAC_THRESH = 3.0        # its ransacReprojThreshold
RANSAC_MAX_MATCHES = 8192  # matches per RANSAC problem (include/ssp_b200.h); all-points HPatches pairs hold ~6.2 k


def _eval_params(keep_k_points=1000, distance_thresh=3, correctness_thresh=(1, 3, 5), map_nn_thresh=1.2,
                 map_inliers="ransac", seed=0):
    """Validated evaluation settings (evaluate_pairs' keywords): (thresholds, map_gt flag, keep_k, distance_thresh,
    map_nn_thresh, seed)."""
    thr = tuple(float(t) for t in np.atleast_1d(correctness_thresh))
    if not 1 <= len(thr) <= 8:
        raise ValueError("correctness_thresh: 1 to 8 thresholds, got %d" % len(thr))
    if map_inliers not in ("ransac", "gt"):
        raise ValueError("map_inliers must be 'ransac' or 'gt', got %r" % (map_inliers,))
    if int(keep_k_points) < 1 or not distance_thresh >= 0 or not map_nn_thresh >= 0:
        raise ValueError("keep_k_points must be positive, distance_thresh and map_nn_thresh non-negative")
    return thr, int(map_inliers == "gt"), int(keep_k_points), float(distance_thresh), float(map_nn_thresh), int(seed)


def _homography_pairs(homographies, P):
    """[P,2,9] float64 host array: each pair's pixel homography and its inverse (np.linalg.inv, as evaluation.py)."""
    Hm = np.asarray(homographies, dtype=np.float64).reshape(-1, 3, 3)
    if Hm.shape[0] != P:
        raise ValueError("%d homographies for %d pairs" % (Hm.shape[0], P))
    return np.stack([Hm.reshape(P, 9), np.linalg.inv(Hm).reshape(P, 9)], axis=1)


def _eval_sizes(P, R, T, n_sets):
    """Byte sizes of the device results of _eval_launch (P pairs, match lists R long)."""
    n = n_sets * P
    return {"ev_rep": P * 2 * 8, "ev_met": P * (3 + T) * 8, "ev_H": n * 9 * 8, "ev_ninl": n * 4, "ev_mask": n * R}


def _eval_launch(pts, kmax, counts, P, matches, nmatch, Hs, shape, params, region):
    """The evaluation kernels on device buffers: pts [2P,3,kmax] float64 (image 1 then image 2 of every pair), counts [2P]
    int32 (each capped at kmax), matches [P,3,R] / nmatch [P] the cross-check matches, Hs [P,2,9] float64.  region(key, dtype,
    shape) gives the output buffers named by _eval_sizes."""
    thr, map_gt, keep_k, dthr, nn, seed = params
    R = matches.shape[2]
    n_sets = 1 if map_gt else 2
    st = stream_of(pts)
    H, W = int(shape[0]), int(shape[1])
    p1, p2, c1, c2 = ptr(pts), ptr(pts[P:]), ptr(counts), ptr(counts[P:])
    call("ssp_eval_repeatability", p1, kmax, c1, p2, kmax, c2, kmax, P, ptr(Hs), H, W, keep_k, dthr,
         ptr(region("ev_rep", torch.float64, (P, 2))), st)
    nbytes = _lib.load().ssp_ransac_homography_ws_bytes(n_sets * P, RANSAC_HYPOTHESES)
    ws = torch.empty((nbytes // 8,), dtype=torch.float64, device=pts.device)
    Hest, ninl = region("ev_H", torch.float64, (n_sets * P, 9)), region("ev_ninl", torch.int32, (n_sets * P,))
    mask = region("ev_mask", torch.uint8, (n_sets * P, R))
    best = torch.empty((n_sets * P,), dtype=torch.int32, device=pts.device)
    call("ssp_ransac_homography", p1, kmax, p2, kmax, ptr(matches), ptr(nmatch), R, P, n_sets, nn, RANSAC_HYPOTHESES,
         RANSAC_THRESH, int(seed) & (2 ** 64 - 1), ptr(Hest), ptr(ninl), ptr(mask), ptr(best), None, None,
         ptr(ws), nbytes, st)
    call("ssp_eval_match_metrics", p1, kmax, c1, p2, kmax, c2, kmax, P, ptr(Hs), H, W, ptr(matches), ptr(nmatch), R, nn,
         ptr(Hest), ptr(ninl), ptr(mask), map_gt, (_lib._c.c_double * len(thr))(*thr), len(thr),
         ptr(region("ev_met", torch.float64, (P, 3 + len(thr)))), st)


def _eval_results(view, nm, P, R, T, n_sets):
    """evaluate_pairs' result dict from the host copies of _eval_launch's outputs (view(key, dtype, shape)); nm [P] holds
    the number of cross-check matches of every pair."""
    rep, met = view("ev_rep", np.float64, (P, 2)), view("ev_met", np.float64, (P, 3 + T))
    mask = view("ev_mask", np.uint8, (n_sets * P, R))
    return {"repeatability": rep[:, 0].copy(), "localization_err": rep[:, 1].copy(), "mean_dist": met[:, 0].copy(),
            "correctness": met[:, 3:] > 0.5, "matching_score": met[:, 1].copy(), "ap": met[:, 2].copy(),
            "homography": view("ev_H", np.float64, (n_sets * P, 9))[:P].reshape(P, 3, 3).copy(),
            "inliers": [mask[p, :nm[p]].astype(bool) for p in range(P)]}


def _as_columns(pts, desc, name, p):
    """One image's points [3,K] float64 and descriptors [256,K] float32 from match_step's layout ([3,K], [256,K]) or the
    exported npz files' ([K,3], [K,256])."""
    pts, desc = np.asarray(pts), np.asarray(desc)
    if pts.ndim == 2 and desc.ndim == 2:
        if pts.shape[0] == 3 and desc.shape == (256, pts.shape[1]):
            return pts.astype(np.float64), desc.astype(np.float32)
        if pts.shape[1] == 3 and desc.shape == (pts.shape[0], 256):
            return pts.T.astype(np.float64), desc.T.astype(np.float32)
    raise ValueError("evaluate_pairs: pair %d: %s %s and descriptors %s are neither [3,K] / [256,K] nor [K,3] / [K,256]"
                     % (p, name, tuple(pts.shape), tuple(desc.shape)))


@torch.no_grad()
def evaluate_pairs(pts, warped_pts, desc, warped_desc, homographies, shape, keep_k_points=1000, distance_thresh=3,
                   correctness_thresh=(1, 3, 5), map_nn_thresh=1.2, map_inliers="ransac", seed=0):
    """The metrics of evaluation.py for P exported image pairs, on the device in one pass.

    pts / warped_pts: P arrays [3,K] (x, y, conf) as match_step returns them, or [K,3] as the exported npz files hold them;
    desc / warped_desc: P arrays [256,K] (or [K,256]); homographies [P,3,3] float64, pixel coordinates, image 1 -> image 2;
    shape = (H, W).  Up to RANSAC_MAX_MATCHES points per image.  Per pair:
      repeatability, localization_err   compute_repeatability(pts, warped_pts, H, shape, keep_k_points, distance_thresh)
                                        (detector_evaluation.py), the golden-pinned definition; its select_k_best uses
                                        numpy's default (unstable) argsort, whose order among equal confidences is
                                        unspecified, so where confidences tie at the keep_k cut this keeps the tied points
                                        a stable sort would (the later ones) and may pick other points than the reference
      homography [3,3], inliers         RANSAC on the cross-check matches (mutual L2 nearest neighbours, no threshold, as
                                        BFMatcher(NORM_L2, crossCheck=True)): RANSAC_HYPOTHESES hypotheses from `seed`,
                                        RANSAC_THRESH px, refit by the normalised DLT on the best hypothesis's inliers
                                        (OpenCV's LM refinement is not run); NaN and no inliers without an estimate
      mean_dist, correctness [T]        mean corner distance of the estimate from H, and mean_dist <= each threshold
      matching_score                    2 * inliers / (K1 + K2'), K2' = warped points whose truncated back-warp lies inside
      ap                                average_precision_score of the matches closer than map_nn_thresh, score = -distance,
                                        labelled by a second RANSAC on them ("ransac", evaluation.py's inliers_method 'cv')
                                        or by ||H p1 - p2|| < 3 ("gt")
    Everything but repeatability is restated from the evaluation code this project forked (its inliers_method 'cv',
    nn_thresh 1.2, top_K 1000, rep_thd 3, the truncation in warpLabels, corners from the image shape), not pinned by a
    fixture of the reference; a detail that turns out to differ is a default to change.  Descriptor matching runs on the
    tensor cores (fp32-grade dots), so near-tied nearest neighbours may resolve differently from an fp32 BLAS matcher.
    Returns a dict of per-pair numpy arrays (averaging over pairs is left to the caller)."""
    params = _eval_params(keep_k_points, distance_thresh, correctness_thresh, map_nn_thresh, map_inliers, seed)
    P = len(pts)
    if P == 0 or not (len(warped_pts) == len(desc) == len(warped_desc) == P):
        raise ValueError("evaluate_pairs: pts, warped_pts, desc and warped_desc must be P > 0 arrays each")
    cols = [_as_columns(pts[p], desc[p], "pts", p) for p in range(P)] + \
           [_as_columns(warped_pts[p], warped_desc[p], "warped_pts", p) for p in range(P)]
    counts = np.array([c[0].shape[1] for c in cols], dtype=np.int32)
    kmax = max(int(counts.max()), 1)
    if kmax > RANSAC_MAX_MATCHES:
        raise ValueError("evaluate_pairs: %d points in one image, at most %d are supported" % (kmax, RANSAC_MAX_MATCHES))
    Hs = _homography_pairs(homographies, P)
    dev = _cuda_device("cuda")
    # one upload of every input from one page-locked buffer
    up = {"pts": (np.float64, (2 * P, 3, kmax)), "desc": (np.float32, (2 * P, 256, kmax)), "counts": (np.int32, (2 * P,)),
          "Hs": (np.float64, (P, 2, 9))}
    offs, total = {}, 0
    for k, (dt, shp) in up.items():
        offs[k] = total
        total += (int(np.prod(shp)) * np.dtype(dt).itemsize + 255) // 256 * 256
    host = torch.zeros((total,), dtype=torch.uint8, pin_memory=True)
    hv = lambda k: host.numpy()[offs[k]:offs[k] + int(np.prod(up[k][1])) * np.dtype(up[k][0]).itemsize].view(
        up[k][0]).reshape(up[k][1])
    hp, hd = hv("pts"), hv("desc")
    for i, (pp, dd) in enumerate(cols):
        hp[i, :, :pp.shape[1]] = pp
        hd[i, :, :dd.shape[1]] = dd
    hv("counts")[:] = counts
    hv("Hs")[:] = Hs
    buf = host.to(dev, non_blocking=True)
    dv = lambda k, dtype: buf[offs[k]:offs[k] + int(np.prod(up[k][1])) * np.dtype(up[k][0]).itemsize].view(dtype).view(
        up[k][1])
    d_pts, d_desc, d_cnt, d_H = dv("pts", torch.float64), dv("desc", torch.float32), dv("counts", torch.int32), dv(
        "Hs", torch.float64)
    planes = _pack_planes(d_desc)
    R = planes.shape[2]
    matches = torch.empty((P, 3, R), dtype=torch.float64, device=dev)
    T, n_sets = len(params[0]), 1 if params[1] else 2
    sizes = dict(_eval_sizes(P, R, T, n_sets), nmatch=P * 4)
    ooffs, ototal = {}, 0
    for k, n in sizes.items():
        ooffs[k] = ototal
        ototal += (n + 255) // 256 * 256
    stage = torch.empty((ototal,), dtype=torch.uint8, device=dev)
    region = lambda k, dtype, shape: stage[ooffs[k]:ooffs[k] + sizes[k]].view(dtype).view(shape)
    nmatch = region("nmatch", torch.int32, (P,))
    _nn_match_planes(planes[:, :P], planes[:, P:], d_cnt[:P], d_cnt[P:], kmax, float("inf"), matches, nmatch)
    _eval_launch(d_pts, kmax, d_cnt, P, matches, nmatch, d_H, shape, params, region)
    out = torch.empty((ototal,), dtype=torch.uint8, pin_memory=True)
    out.copy_(stage)
    out = out.numpy()
    view = lambda k, dtype, shp: out[ooffs[k]:ooffs[k] + sizes[k]].view(dtype).reshape(shp)
    return _eval_results(view, view("nmatch", np.int32, (P,)), P, R, T, n_sets)
