"""CPU ORACLE for the homography-warp correspondence path -- TEST INFRASTRUCTURE, NOT PRODUCT.

A numpy restatement of the reference algorithms (Gabriel-SGama/Semantic-SuperPoint), each function citing
the reference file:line it follows.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import this module; the product package (semantic-superpoint_b200/) never does.

Pinning: the reference ships no golden vectors or assertions for this path (SURVEY 4, 8c), so this oracle is
pinned against outputs of the LIVE reference functions, generated in the authoring container by
tests/golden/make_golden.py (which imports /root/reference) and committed as tests/golden/*.npz;
tests/test_oracle_golden.py replays them.  Third-party arithmetic on the path that is restated here:
torch 2.11 (F.grid_sample bilinear/nearest zeros-padding align_corners=True, softmax, BCELoss with the
-100 log clamp, torch.norm), torchvision 0.26 ops.nms, opencv 4.13 getStructuringElement(MORPH_ELLIPSE) +
erode (reference pins opencv-python 3.4.2.16).  The only torch call kept is torch.linspace for the
sampling-grid table (the reference builds it with a CPU torch.linspace, utils/utils.py:375, whose rounding
differs by 1 ulp from the textbook formula).
"""
import numpy as np

f32 = np.float32


# ------------------------------------------------------------------------------------------------
# warps
# ------------------------------------------------------------------------------------------------
def linspace_grid(n):
    import torch
    return torch.linspace(-1, 1, n).numpy().copy()


def warp_points(points, homographies):
    """utils/utils.py:315-343.  points [P,2] (x,y); homographies [3,3] or [B,3,3] -> [P,2] or [B,P,2] (fp32)."""
    H = np.asarray(homographies, dtype=f32)
    no_batches = H.ndim == 2
    H = H.reshape(-1, 3, 3)
    p = np.concatenate([np.asarray(points, dtype=f32), np.ones((len(points), 1), f32)], axis=1)  # [P,3]
    w = np.einsum("bij,pj->bpi", H, p).astype(f32)
    out = (w[:, :, :2] / w[:, :, 2:]).astype(f32)
    return out[0] if no_batches else out


def filter_points(points, shape, return_mask=False):
    """utils/utils.py:303-311.  0 <= p <= shape-1 in every coordinate (inclusive)."""
    points = np.asarray(points, dtype=f32)
    shape = np.asarray(shape, dtype=f32)
    mask = np.all((points >= 0) & (points <= shape - 1), axis=-1)
    return (points[mask], mask) if return_mask else points[mask]


def warp_keypoints_f64(keypoints, H):
    """evaluations/detector_evaluation.py:139-150: float64 [x,y,1] H^T / z in pixel coordinates."""
    kp = np.asarray(keypoints, dtype=np.float64)[:, :2]
    hom = np.concatenate([kp, np.ones((kp.shape[0], 1))], axis=1)
    w = hom @ np.asarray(H, dtype=np.float64).T
    return w[:, :2] / w[:, 2:]


def keep_in_bounds_f64(points, shape):
    """evaluations/detector_evaluation.py:160-191: 0 <= x < W and 0 <= y < H (strict upper bound). shape=(H,W)."""
    return (points[:, 0] >= 0) & (points[:, 0] < shape[1]) & (points[:, 1] >= 0) & (points[:, 1] < shape[0])


def compute_repeatability(prob, warped_prob, H, shape, keep_k_points=300, distance_thresh=3, warp_and_keep=None):
    """evaluations/detector_evaluation.py:152-283 restated.  prob / warped_prob [K,3] (x, y, confidence) in the two
    images, H the pixel homography, shape = (H, W).  warp_and_keep(points[K,2], Hmat, shape) -> (warped [K,2], keep [K])
    defaults to the float64 oracle (warp_keypoints_f64 + keep_in_bounds_f64); tests plug the CUDA path in here.
    Returns (repeatability, localization_err)."""
    if warp_and_keep is None:
        def warp_and_keep(p, Hm, shp):
            w = warp_keypoints_f64(p, Hm)
            return w, keep_in_bounds_f64(w, shp)
    prob = np.array(prob, dtype=np.float64)
    warped_prob = np.array(warped_prob, dtype=np.float64)
    # keep_true_keypoints: detections of the warped image whose back-warp lies inside the image (:172-189)
    _, keep = warp_and_keep(warped_prob[:, :2], np.linalg.inv(H), shape)
    wk = warped_prob[keep]
    # true warps of the detections of the first image, filtered to the image (:232-238)
    tw, keep = warp_and_keep(prob[:, :2], H, shape)
    twk = np.concatenate([tw, prob[:, 2:]], axis=1)[keep]

    def select_k_best(points, k):  # :191-201
        s = points[points[:, 2].argsort(), :2]
        return s[-min(k, points.shape[0]):, :]

    wk, twk = select_k_best(wk, keep_k_points), select_k_best(twk, keep_k_points)
    N1, N2 = twk.shape[0], wk.shape[0]
    norm = np.linalg.norm(twk[:, None, :] - wk[None, :, :], axis=2)
    count1 = count2 = 0
    e1 = e2 = None
    if N2 != 0:
        m1 = norm.min(axis=1)
        count1 = int((m1 <= distance_thresh).sum())
        e1 = m1[m1 <= distance_thresh]
    if N1 != 0:
        m2 = norm.min(axis=0)
        count2 = int((m2 <= distance_thresh).sum())
        e2 = m2[m2 <= distance_thresh]
    rep = (count1 + count2) / (N1 + N2) if N1 + N2 > 0 else 0
    loc = -1
    if count1 + count2 > 0:
        loc = 0
        if e1 is not None:
            loc += e1.sum() / (count1 + count2)
        if e2 is not None:
            loc += e2.sum() / (count1 + count2)
    else:
        rep = 0
    return rep, loc


def _unnormalize(coord, size):
    # ATen grid_sampler_unnormalize, align_corners=True: ((coord + 1) / 2) * (size - 1)
    return ((coord + f32(1)) / f32(2)) * f32(size - 1)


def grid_sample(img, grid, mode):
    """torch F.grid_sample(img [B,C,H,W], grid [B,Ho,Wo,2] (x,y), mode, padding zeros, align_corners=True)."""
    img = np.asarray(img, dtype=f32)
    B, C, H, W = img.shape
    ix = _unnormalize(grid[..., 0].astype(f32), W)
    iy = _unnormalize(grid[..., 1].astype(f32), H)
    out = np.zeros((B, C) + ix.shape[1:], dtype=f32)
    bidx = np.arange(B)[:, None, None]
    if mode == "nearest":
        rx, ry = np.rint(ix), np.rint(iy)  # std::nearbyint = round half to even
        ok = (rx >= 0) & (rx < W) & (ry >= 0) & (ry < H)
        xi = np.where(ok, rx, 0).astype(np.int64)
        yi = np.where(ok, ry, 0).astype(np.int64)
        for c in range(C):
            out[:, c] = np.where(ok, img[bidx, c, yi, xi], f32(0))
        return out
    x0, y0 = np.floor(ix), np.floor(iy)
    x1, y1 = x0 + 1, y0 + 1
    wts = [((x1 - ix) * (y1 - iy), x0, y0), ((ix - x0) * (y1 - iy), x1, y0),
           ((x1 - ix) * (iy - y0), x0, y1), ((ix - x0) * (iy - y0), x1, y1)]
    for wgt, xx, yy in wts:
        ok = (xx >= 0) & (xx < W) & (yy >= 0) & (yy < H)
        xi = np.where(ok, xx, 0).astype(np.int64)
        yi = np.where(ok, yy, 0).astype(np.int64)
        for c in range(C):
            out[:, c] += np.where(ok, img[bidx, c, yi, xi] * wgt.astype(f32), f32(0))
    return out


def inv_warp_image_batch(img, mat_homo_inv, mode="bilinear"):
    """utils/utils.py:347-385."""
    img = np.asarray(img, dtype=f32)
    if img.ndim in (2, 3):
        img = img.reshape(1, 1, img.shape[0], img.shape[1])
    Hm = np.asarray(mat_homo_inv, dtype=f32).reshape(-1, 3, 3)
    B, C, H, W = img.shape
    xs, ys = linspace_grid(W), linspace_grid(H)
    gx, gy = np.meshgrid(xs, ys)  # [H,W] each, (x,y) at pixel (row,col)
    pts = np.stack([gx.reshape(-1), gy.reshape(-1)], axis=1)
    src = warp_points(pts, Hm).reshape(B, H, W, 2)
    return grid_sample(img, src, mode)


def sample_coords_f64(image_shape, mat_homo_inv):
    """Source pixel coordinates (ix, iy) [B,H,W] of inv_warp_image_batch in float64: used by tests to show that a
    nearest-mode pixel that differs between two fp32 implementations sits on a half-pixel rounding tie."""
    H, W = int(image_shape[0]), int(image_shape[1])
    Hm = np.asarray(mat_homo_inv, dtype=np.float64).reshape(-1, 3, 3)
    gx, gy = np.meshgrid(linspace_grid(W).astype(np.float64), linspace_grid(H).astype(np.float64))
    p = np.stack([gx.reshape(-1), gy.reshape(-1), np.ones(H * W)], axis=0)  # [3, HW]
    w = Hm @ p  # [B,3,HW]
    nx, ny = w[:, 0] / w[:, 2], w[:, 1] / w[:, 2]
    ix = (nx + 1.0) / 2.0 * (W - 1)
    iy = (ny + 1.0) / 2.0 * (H - 1)
    return ix.reshape(-1, H, W), iy.reshape(-1, H, W)


def ellipse_kernel(radius):
    """cv2.getStructuringElement(MORPH_ELLIPSE, (2r,2r)) (opencv modules/imgproc/src/morph.dispatch.cpp)."""
    k = int(radius) * 2
    r = c = k // 2
    inv_r2 = 1.0 / (r * r) if r else 0.0
    ker = np.zeros((k, k), np.uint8)
    for i in range(k):
        dy = i - r
        if abs(dy) <= r:
            dx = int(np.rint(c * np.sqrt((r * r - dy * dy) * inv_r2)))
            ker[i, max(c - dx, 0):min(c + dx + 1, k)] = 1
    return ker


def erode(mask, kernel):
    """cv2.erode(mask, kernel): min over the kernel footprint, anchor (kw//2, kh//2), out-of-image taps ignored."""
    H, W = mask.shape
    kh, kw = kernel.shape
    ay, ax = kh // 2, kw // 2
    out = np.ones_like(mask)
    for ky in range(kh):
        for kx in range(kw):
            if not kernel[ky, kx]:
                continue
            dy, dx = ky - ay, kx - ax
            sh = np.ones_like(mask)
            ys0, ys1 = max(0, -dy), min(H, H - dy)
            xs0, xs1 = max(0, -dx), min(W, W - dx)
            sh[ys0:ys1, xs0:xs1] = mask[ys0 + dy:ys1 + dy, xs0 + dx:xs1 + dx]
            out = np.minimum(out, sh)
    return out


def compute_valid_mask(image_shape, inv_homography, erosion_radius=0):
    """utils/utils.py:715-742."""
    Hm = np.asarray(inv_homography, dtype=f32).reshape(-1, 3, 3)
    B = Hm.shape[0]
    H, W = int(image_shape[0]), int(image_shape[1])
    mask = inv_warp_image_batch(np.ones((B, 1, H, W), f32), Hm, mode="nearest").reshape(B, H, W)
    if erosion_radius > 0:
        ker = ellipse_kernel(erosion_radius)
        for i in range(B):
            mask[i] = erode(mask[i], ker)
    return mask


# ------------------------------------------------------------------------------------------------
# detector labels / loss / heatmap
# ------------------------------------------------------------------------------------------------
def space_to_depth(x, bs=8):
    """utils/d2s.py:27-44 == pixel_unshuffle: channel = dy*bs + dx."""
    B, C, H, W = x.shape
    assert C == 1
    y = x.reshape(B, H // bs, bs, W // bs, bs).transpose(0, 2, 4, 1, 3)
    return y.reshape(B, bs * bs, H // bs, W // bs)


def depth_to_space(x, bs=8):
    """utils/d2s.py:8-25 == pixel_shuffle."""
    B, C, Hc, Wc = x.shape
    y = x.reshape(B, bs, bs, Hc, Wc).transpose(0, 3, 1, 4, 2)
    return y.reshape(B, 1, Hc * bs, Wc * bs)


def labels2Dto3D(labels, cell_size=8, add_dustbin=True):
    """utils/utils.py:408-440."""
    lab = space_to_depth(np.asarray(labels, dtype=f32), cell_size)
    if add_dustbin:
        dust = f32(1) - lab.sum(axis=1, dtype=f32)
        dust[dust < 1.0] = 0
        lab = np.concatenate([lab, dust[:, None]], axis=1)
        dn = lab.sum(axis=1, dtype=f32)
        lab = lab / dn[:, None]
    return lab.astype(f32)


def getMasks(mask_2D, cell_size=8):
    """Train_model_frontend_all.py:373-386."""
    return np.prod(space_to_depth(np.asarray(mask_2D, dtype=f32), cell_size), axis=1, dtype=f32)


def softmax(x, axis):
    m = x.max(axis=axis, keepdims=True)
    e = np.exp(x - m)
    return e / e.sum(axis=axis, keepdims=True)


def detector_loss(semi, target, mask, grad=False):
    """Train_model_heatmap_all.py:155-179 (softmax branch): BCE over softmax probabilities, masked mean.
    Computed in float64 from the fp32 inputs; with grad=True also returns dLoss/dsemi (BCELoss backward uses
    (p - t) / max(p (1 - p), 1e-12), softmax backward p * (g - sum p g))."""
    x = np.asarray(semi, dtype=np.float64)
    t = np.asarray(target, dtype=np.float64)
    m = np.asarray(mask, dtype=np.float64)
    p = softmax(x, 1)
    with np.errstate(divide="ignore"):
        bce = -(t * np.maximum(np.log(p), -100) + (1 - t) * np.maximum(np.log(1 - p), -100))
    den = m.sum() + 1e-5
    loss = (bce.sum(axis=1) * m).sum() / den
    if not grad:
        return f32(loss)
    dp = (m / den)[:, None] * (p - t) / np.maximum(p * (1 - p), 1e-12)
    dx = p * (dp - (p * dp).sum(axis=1, keepdims=True))
    return f32(loss), dx.astype(f32)


def flattenDetection(semi):
    """utils/utils.py:515-560: softmax(65) -> drop dustbin -> depth_to_space(8).  [B,65,Hc,Wc] -> [B,1,H,W]."""
    semi = np.asarray(semi, dtype=f32)
    batch = semi.ndim == 4
    if not batch:
        semi = semi[None]
    dense = softmax(semi, 1).astype(f32)
    heat = depth_to_space(dense[:, :-1])
    return heat if batch else heat[0]


def combine_heatmap(heatmap, inv_homographies, mask_2D):
    """export.py:49-60.  heatmap/mask [N,1,H,W], inv_homographies [1,N,3,3] -> [1,H,W]."""
    heatmap = np.asarray(heatmap, dtype=f32) * np.asarray(mask_2D, dtype=f32)
    Hm = np.asarray(inv_homographies, dtype=f32)[0]
    h = inv_warp_image_batch(heatmap, Hm, mode="bilinear").sum(axis=0, dtype=f32)
    m = inv_warp_image_batch(mask_2D, Hm, mode="bilinear").sum(axis=0, dtype=f32)
    with np.errstate(divide="ignore", invalid="ignore"):
        return h / m


# ------------------------------------------------------------------------------------------------
# keypoints
# ------------------------------------------------------------------------------------------------
def nms_fast(in_corners, H, W, dist_thresh):
    """utils/utils.py:653-712, with numpy's unstable default argsort replaced by kind='stable' so that ties
    have a defined order (the reference leaves it undefined)."""
    grid = np.zeros((H, W), dtype=int)
    inds = np.zeros((H, W), dtype=int)
    inds1 = np.argsort(-in_corners[2, :], kind="stable")
    corners = in_corners[:, inds1]
    rcorners = corners[:2, :].round().astype(int)
    if rcorners.shape[1] == 0:
        return np.zeros((3, 0)).astype(int), np.zeros(0).astype(int)
    if rcorners.shape[1] == 1:
        return np.vstack((rcorners, in_corners[2])).reshape(3, 1), np.zeros((1)).astype(int)
    grid[rcorners[1], rcorners[0]] = 1
    inds[rcorners[1], rcorners[0]] = np.arange(rcorners.shape[1])
    pad = dist_thresh
    grid = np.pad(grid, ((pad, pad), (pad, pad)), mode="constant")
    for i in range(rcorners.shape[1]):
        x, y = rcorners[0, i] + pad, rcorners[1, i] + pad
        if grid[y, x] == 1:
            grid[y - pad:y + pad + 1, x - pad:x + pad + 1] = 0
            grid[y, x] = -1
    keepy, keepx = np.where(grid == -1)
    keepy, keepx = keepy - pad, keepx - pad
    inds_keep = inds[keepy, keepx]
    out = corners[:, inds_keep]
    inds2 = np.argsort(-out[-1, :], kind="stable")
    return out[:, inds2], inds1[inds_keep[inds2]]


def getPtsFromHeatmap(heatmap, conf_thresh, nms_dist, border_remove=4):
    """utils/utils.py:581-609 (stable sorts).  Returns float64 [3,K]: x, y, conf, confidence-descending."""
    H, W = heatmap.shape
    ys, xs = np.where(heatmap >= conf_thresh)
    if len(ys) == 0:
        return np.zeros((3, 0))
    pts = np.zeros((3, len(ys)))
    pts[0, :], pts[1, :], pts[2, :] = xs, ys, heatmap[ys, xs]
    pts, _ = nms_fast(pts, H, W, dist_thresh=nms_dist)
    inds = np.argsort(pts[2, :], kind="stable")
    pts = pts[:, inds[::-1]]
    b = border_remove
    rm = (pts[0, :] < b) | (pts[0, :] >= (W - b)) | (pts[1, :] < b) | (pts[1, :] >= (H - b))
    return pts[:, ~rm]


def box_nms(prob, size, iou=0.1, min_prob=0.01):
    """utils/utils.py:612-650 with torchvision.ops.nms restated: greedy in descending score (stable), a box is
    dropped when its IoU with an already kept box exceeds `iou` (fp32 arithmetic like torchvision)."""
    prob = np.asarray(prob, dtype=f32)
    ys, xs = np.nonzero(prob > f32(min_prob))
    out = np.zeros_like(prob)
    if len(ys) == 0:
        return out
    half = f32(size / 2.0)
    pts = np.stack([ys, xs], axis=1).astype(f32)
    boxes = np.concatenate([pts - half, pts + half], axis=1)
    scores = prob[ys, xs]
    order = np.argsort(-scores, kind="stable")
    area = (boxes[:, 2] - boxes[:, 0]) * (boxes[:, 3] - boxes[:, 1])
    alive = np.ones(len(order), bool)
    for ii, i in enumerate(order):
        if not alive[i]:
            continue
        rest = order[ii + 1:]
        rest = rest[alive[rest]]
        if len(rest) == 0:
            break
        w = np.maximum(f32(0), np.minimum(boxes[i, 2], boxes[rest, 2]) - np.maximum(boxes[i, 0], boxes[rest, 0]))
        h = np.maximum(f32(0), np.minimum(boxes[i, 3], boxes[rest, 3]) - np.maximum(boxes[i, 1], boxes[rest, 1]))
        inter = (w * h).astype(f32)
        ovr = inter / (area[i] + area[rest] - inter)
        alive[rest[ovr > f32(iou)]] = False
    keep = np.array([i for i in order if alive[i]], dtype=int)
    out[ys[keep], xs[keep]] = scores[keep]
    return out


# ------------------------------------------------------------------------------------------------
# descriptor loss
# ------------------------------------------------------------------------------------------------
def descriptor_pair_mask(homographies, Hc, Wc, cell_size=8, descriptor_dist=4):
    """utils/utils.py:824-860: warped cell centres and the [B,Nc,Nc] correspondence mask (fp32 op order)."""
    Hm = np.asarray(homographies, dtype=f32).reshape(-1, 3, 3)
    Hpx, Wpx = f32(Hc * cell_size), f32(Wc * cell_size)
    kk, ll = np.meshgrid(np.arange(Hc), np.arange(Wc), indexing="ij")
    cy = (kk.reshape(-1) * cell_size + cell_size // 2).astype(f32)
    cx = (ll.reshape(-1) * cell_size + cell_size // 2).astype(f32)
    ny = cy / Hpx * f32(2) - f32(1)  # normPts divides by H, W
    nx = cx / Wpx * f32(2) - f32(1)
    w = warp_points(np.stack([nx, ny], 1), Hm)  # [B,Nc,2] (x,y)
    wx = (w[..., 0] + f32(1)) * Wpx / f32(2)
    wy = (w[..., 1] + f32(1)) * Hpx / f32(2)
    dy = cy[None, None, :] - wy[:, :, None]
    dx = cx[None, None, :] - wx[:, :, None]
    dist = np.sqrt((dy * dy + dx * dx).astype(f32)).astype(f32)
    return (dist <= f32(descriptor_dist)).astype(f32), np.stack([wx, wy], -1)


def descriptor_loss(descriptors, descriptors_warped, homographies, mask_valid=None, cell_size=8, lamda_d=250,
                    descriptor_dist=4, grad=None, return_mask=False, chunk=1024):
    """utils/utils.py:779-893 restated with a chunked matmul for the all-pairs dot product (the reference
    materialises [B,Hc,Wc,Hc,Wc,256]).  Sums in float64.  grad = (g_loss, g_pos, g_neg) additionally returns
    d/d descriptors and d/d descriptors_warped of  g_loss*loss + g_pos*pos_sum + g_neg*neg_sum."""
    D = np.asarray(descriptors, dtype=f32)
    Dw = np.asarray(descriptors_warped, dtype=f32)
    B, Dch, Hc, Wc = D.shape
    Nc = Hc * Wc
    mask, _ = descriptor_pair_mask(homographies, Hc, Wc, cell_size, descriptor_dist)
    mv = np.ones((B, Nc), f32) if mask_valid is None else np.asarray(mask_valid, dtype=f32).reshape(B, Nc)
    norm = f32(B) * (mv.sum(dtype=f32) + f32(1)) * f32(Hc) * f32(Wc)
    A = D.reshape(B, Dch, Nc).transpose(0, 2, 1)  # [B,Nc,D]
    Bm = Dw.reshape(B, Dch, Nc)                   # [B,D,Nc]
    s_loss = s_pos = s_neg = 0.0
    if grad is not None:
        gl, gp, gn = [float(g) for g in grad]
        dD = np.zeros((B, Nc, Dch), np.float64)
        dDw = np.zeros((B, Dch, Nc), np.float64)
    for b in range(B):
        for r0 in range(0, Nc, chunk):
            r1 = min(Nc, r0 + chunk)
            dot = A[b, r0:r1] @ Bm[b]  # [r,Nc]
            m = mask[b, r0:r1]
            pos = np.maximum(f32(1.0) - dot, f32(0))
            neg = np.maximum(dot - f32(0.2), f32(0))
            lp = f32(lamda_d) * m * pos
            ln = (f32(1) - m) * neg
            s_loss += float(((lp + ln) * mv[b][None, :]).sum(dtype=np.float64))
            s_pos += float(lp.sum(dtype=np.float64))
            s_neg += float(ln.sum(dtype=np.float64))
            if grad is not None:
                x_p, x_n = f32(1.0) - dot, dot - f32(0.2)
                ip = np.where(x_p > 0, 1.0, np.where(x_p == 0, 0.5, 0.0))  # torch.max(a, 0-tensor) ties split
                inn = np.where(x_n > 0, 1.0, np.where(x_n == 0, 0.5, 0.0))
                wl = gl * mv[b][None, :].astype(np.float64)
                G = (-(lamda_d * m) * ip * (wl + gp) + (1.0 - m) * inn * (wl + gn)) / float(norm)
                dD[b, r0:r1] += G @ Bm[b].T.astype(np.float64)
                dDw[b] += A[b, r0:r1].T.astype(np.float64) @ G
    out = [f32(s_loss / float(norm)), f32(s_pos / float(norm)), f32(s_neg / float(norm))]
    res = (out[0], mask.reshape(B, Hc, Wc, Hc, Wc) if return_mask else None, out[1], out[2])
    if grad is not None:
        gD = dD.transpose(0, 2, 1).reshape(B, Dch, Hc, Wc).astype(f32)
        gDw = dDw.reshape(B, Dch, Hc, Wc).astype(f32)
        return res + (gD, gDw)
    return res


def loss_step(semi, semi_warp, desc, desc_warp, labels_2D, warped_labels, mask_2D, mask_warp_2D, mat_H, lamda_d=250,
              descriptor_dist=4, lambda_loss=1.0, weighting="uniform"):
    """Train_model_heatmap_all.py:295-365: detector_loss of both images (:155-179, targets labels2Dto3D, masks
    getMasks(mask_2D) / getMasks(mask_warp_2D)), descriptor_loss with mask_valid = getMasks(mask_warp_2D), then the total
      weighting="uniform":    loss_det + loss_det_warp + lambda_loss * loss_desc   (:361-365)
      weighting="multi_task": loss_det + loss_det_warp + positive_dist + negative_dist (:355-359 at unit weights)
    and its gradients with respect to the four head outputs.  Returns a dict of the six fp32 scalars (loss, loss_det,
    loss_det_warp, loss_desc, positive_dist, negative_dist) and "grads" = (d semi, d semi_warp, d desc, d desc_warp)."""
    if weighting not in ("uniform", "multi_task"):
        raise ValueError("weighting must be 'uniform' or 'multi_task'")
    m3, mw3 = getMasks(mask_2D), getMasks(mask_warp_2D)
    l_det, d_semi = detector_loss(semi, labels2Dto3D(labels_2D), m3, grad=True)
    l_detw, d_semiw = detector_loss(semi_warp, labels2Dto3D(warped_labels), mw3, grad=True)
    g = (float(lambda_loss), 0.0, 0.0) if weighting == "uniform" else (0.0, 1.0, 1.0)
    l_desc, _, pos, neg, d_desc, d_descw = descriptor_loss(desc, desc_warp, mat_H, mw3[:, None], lamda_d=lamda_d,
                                                           descriptor_dist=descriptor_dist, grad=g)
    if weighting == "uniform":
        total = float(l_det) + float(l_detw) + float(lambda_loss) * float(l_desc)
    else:
        total = float(l_det) + float(l_detw) + float(pos) + float(neg)
    return {"loss": f32(total), "loss_det": l_det, "loss_det_warp": l_detw, "loss_desc": l_desc, "positive_dist": pos,
            "negative_dist": neg, "grads": (d_semi, d_semiw, d_desc, d_descw)}


def descriptor_boundary_slack(descriptors, descriptors_warped, homographies, mask_valid=None, cell_size=8, lamda_d=250,
                              descriptor_dist=4, eps=1e-3, per_term=False):
    """Largest change of (loss, pos_sum, neg_sum) if every pair whose centre distance lies within `eps` of
    descriptor_dist flipped its mask bit (the mask is a step function of fp32 coordinates ~1e3 in magnitude, so
    1-ulp differences in the warp arithmetic flip such pairs; each flip moves the numerator by up to lamda_d).
    per_term=True returns the bound of each of the three scalars: (loss, pos_sum, neg_sum)."""
    D = np.asarray(descriptors, dtype=f32)
    Dw = np.asarray(descriptors_warped, dtype=f32)
    B, Dch, Hc, Wc = D.shape
    Nc = Hc * Wc
    _, w = descriptor_pair_mask(homographies, Hc, Wc, cell_size, descriptor_dist)
    kk, ll = np.meshgrid(np.arange(Hc), np.arange(Wc), indexing="ij")
    cy = (kk.reshape(-1) * cell_size + cell_size // 2).astype(np.float64)
    cx = (ll.reshape(-1) * cell_size + cell_size // 2).astype(np.float64)
    mv = np.ones((B, Nc), f32) if mask_valid is None else np.asarray(mask_valid, dtype=f32).reshape(B, Nc)
    norm = float(B) * (float(mv.sum()) + 1.0) * Hc * Wc
    s_pos = s_neg = 0.0
    for b in range(B):
        d = np.sqrt((cy[None, :] - w[b, :, 1:2].astype(np.float64)) ** 2 + (cx[None, :] - w[b, :, 0:1].astype(np.float64)) ** 2)
        rr, cc = np.nonzero(np.abs(d - descriptor_dist) < eps)
        for r, c in zip(rr, cc):
            dot = float(D[b].reshape(Dch, Nc)[:, r].astype(np.float64) @ Dw[b].reshape(Dch, Nc)[:, c].astype(np.float64))
            s_pos += lamda_d * max(1.0 - dot, 0.0)
            s_neg += max(dot - 0.2, 0.0)
    if per_term:
        return (s_pos + s_neg) / norm, s_pos / norm, s_neg / norm
    return (s_pos + s_neg) / norm


def descriptor_unstable_cells(descriptors, descriptors_warped, homographies, cell_size=8, descriptor_dist=4, eps_dot=1e-5,
                              eps_px=1e-3, chunk=1024):
    """Rows / columns whose GRADIENT is not a continuous function of the inputs at this point, so that two correct
    implementations may differ there by a whole descriptor: cells touching a pair whose dot product lies within eps_dot of a
    hinge margin (0.2 / 1.0) or whose centre distance lies within eps_px of descriptor_dist.  Returns two bool [B,Nc]
    arrays (rows = cells of `descriptors`, cols = cells of `descriptors_warped`).  Chunked float64, any size."""
    D = np.asarray(descriptors, dtype=np.float64)
    Dw = np.asarray(descriptors_warped, dtype=np.float64)
    B, Dch, Hc, Wc = D.shape
    Nc = Hc * Wc
    _, w = descriptor_pair_mask(homographies, Hc, Wc, cell_size, descriptor_dist)
    kk, ll = np.meshgrid(np.arange(Hc), np.arange(Wc), indexing="ij")
    cy = (kk.reshape(-1) * cell_size + cell_size // 2).astype(np.float64)
    cx = (ll.reshape(-1) * cell_size + cell_size // 2).astype(np.float64)
    rows = np.zeros((B, Nc), bool)
    cols = np.zeros((B, Nc), bool)
    for b in range(B):
        A = D[b].reshape(Dch, Nc).T
        Bm = Dw[b].reshape(Dch, Nc)
        for r0 in range(0, Nc, chunk):
            r1 = min(Nc, r0 + chunk)
            dot = A[r0:r1] @ Bm
            d = np.sqrt((cy[None, :] - w[b, r0:r1, 1:2].astype(np.float64)) ** 2 + (cx[None, :] - w[b, r0:r1, 0:1].astype(np.float64)) ** 2)
            pos = d <= descriptor_dist + eps_px
            near = (np.abs(d - descriptor_dist) < eps_px) | (~pos & (np.abs(dot - 0.2) < eps_dot)) | (pos & ((np.abs(dot - 1.0) < eps_dot) | (np.abs(dot - 0.2) < eps_dot)))
            rows[b, r0:r1] |= near.any(axis=1)
            cols[b] |= near.any(axis=0)
    return rows, cols


def descriptor_dots(descriptors, descriptors_warped):
    """float64 all-pairs dot products [B,Nc,Nc] (used by tests to locate hinge kinks)."""
    D = np.asarray(descriptors, dtype=np.float64)
    Dw = np.asarray(descriptors_warped, dtype=np.float64)
    B, Dch = D.shape[:2]
    return np.einsum("bdi,bdj->bij", D.reshape(B, Dch, -1), Dw.reshape(B, Dch, -1))


# ------------------------------------------------------------------------------------------------
# semantic head: x8 bilinear upsample + cross entropy  (SURVEY 8f rank 1)
# ------------------------------------------------------------------------------------------------
def _upsample_axis(n_in, n_out):
    """F.interpolate(mode="bilinear", align_corners=False) source indices / weights along one axis
    (torch area_pixel_compute_source_index: src = (dst + 0.5) * in/out - 0.5, clamped below at 0)."""
    scale = f32(n_in) / f32(n_out)
    src = np.maximum((np.arange(n_out, dtype=f32) + f32(0.5)) * scale - f32(0.5), f32(0))
    i0 = np.minimum(src.astype(np.int64), n_in - 1)
    i1 = np.minimum(i0 + 1, n_in - 1)
    lam = (src - i0.astype(f32)).astype(np.float64)
    return i0, i1, lam


def upsample_bilinear(x, out_hw):
    """models/SuperPointNet_gauss2_ssmall.py:90  F.interpolate(sem, x_hw, mode="bilinear", align_corners=False).
    x [B,C,h,w] -> [B,C,H,W] (float64)."""
    x = np.asarray(x, dtype=np.float64)
    H, W = out_hw
    y0, y1, ly = _upsample_axis(x.shape[2], H)
    x0, x1, lx = _upsample_axis(x.shape[3], W)
    rows = x[:, :, y0, :] * (1 - ly)[None, None, :, None] + x[:, :, y1, :] * ly[None, None, :, None]
    return rows[:, :, :, x0] * (1 - lx) + rows[:, :, :, x1] * lx


def upsample_bilinear_adjoint(g, in_hw):
    """Transpose of upsample_bilinear: gradient [B,C,H,W] -> [B,C,h,w]."""
    g = np.asarray(g, dtype=np.float64)
    B, C, H, W = g.shape
    h, w = in_hw
    y0, y1, ly = _upsample_axis(h, H)
    x0, x1, lx = _upsample_axis(w, W)
    cols = np.zeros((B, C, H, w))
    np.add.at(cols, (slice(None), slice(None), slice(None), x0), g * (1 - lx))
    np.add.at(cols, (slice(None), slice(None), slice(None), x1), g * lx)
    out = np.zeros((B, C, h, w))
    np.add.at(out, (slice(None), slice(None), y0, slice(None)), cols * (1 - ly)[None, None, :, None])
    np.add.at(out, (slice(None), slice(None), y1, slice(None)), cols * ly[None, None, :, None])
    return out


def sem_loss(pred, label, ignore_index=133, grad=False, gout=1.0):
    """Train_model_heatmap_all.py:181-193  nn.CrossEntropyLoss(ignore_index=133)(pred [B,C,H,W], label [B,H,W]):
    mean over the non-ignored pixels of -log_softmax(pred)[label]; nothing counted -> NaN (gradient 0).
    If pred's spatial size differs from label's it is first upsampled like the model's last line does
    (SuperPointNet_gauss2_ssmall.py:90) and the gradient is returned with respect to the low-res logits."""
    pred = np.asarray(pred, dtype=np.float64)
    label = np.asarray(label).astype(np.int64)
    lowres = pred.shape[2:] != label.shape[1:]
    full = upsample_bilinear(pred, label.shape[1:]) if lowres else pred
    m = full.max(axis=1, keepdims=True)
    lse = m[:, 0] + np.log(np.exp(full - m).sum(axis=1))
    valid = label != ignore_index
    safe = np.where(valid, label, 0)
    picked = np.take_along_axis(full, safe[:, None], axis=1)[:, 0]
    n = int(valid.sum())
    with np.errstate(invalid="ignore", divide="ignore"):
        loss = f32(np.where(valid, lse - picked, 0.0).sum() / n) if n else f32(np.nan)
    if not grad:
        return loss
    g = np.exp(full - lse[:, None])
    np.put_along_axis(g, safe[:, None], np.take_along_axis(g, safe[:, None], axis=1) - 1.0, axis=1)
    g = g * valid[:, None] * (gout / n if n else 0.0)
    if lowres:
        g = upsample_bilinear_adjoint(g, pred.shape[2:])
    return loss, g.astype(f32)


# ------------------------------------------------------------------------------------------------
# sparse descriptors: sampling at keypoints + two-way nearest-neighbour matching  (SURVEY 8f rank 3)
# ------------------------------------------------------------------------------------------------
def sample_desc_from_points(coarse_desc, pts, cell=8):
    """models/model_wrap.py:295-313.  coarse_desc [1,D,Hc,Wc], pts [3,K] (x, y, conf) -> float32 [D,K]."""
    coarse_desc = np.asarray(coarse_desc, dtype=f32)
    D, Hc, Wc = coarse_desc.shape[1:]
    H, W = Hc * cell, Wc * cell
    pts = np.asarray(pts)
    if pts.shape[1] == 0:
        return np.zeros((D, 0))
    samp = pts[:2, :].astype(np.float64).copy()
    samp[0, :] = samp[0, :] / (float(W) / 2.0) - 1.0
    samp[1, :] = samp[1, :] / (float(H) / 2.0) - 1.0
    grid = samp.T.astype(f32).reshape(1, 1, -1, 2)
    desc = grid_sample(coarse_desc, grid, "bilinear").reshape(D, -1)
    with np.errstate(invalid="ignore", divide="ignore"):
        return (desc / np.linalg.norm(desc, axis=0)[np.newaxis, :]).astype(f32)


def nn_match_two_way(desc1, desc2, nn_thresh):
    """models/model_wrap.py:451-494.  [D,K1], [D,K2] -> float64 [3,L] (index 1, index 2, distance)."""
    assert desc1.shape[0] == desc2.shape[0]
    if desc1.shape[1] == 0 or desc2.shape[1] == 0:
        return np.zeros((3, 0))
    if nn_thresh < 0.0:
        raise ValueError("'nn_thresh' should be non-negative")
    dmat = np.dot(desc1.T, desc2)
    dmat = np.sqrt(2 - 2 * np.clip(dmat, -1, 1))
    idx = np.argmin(dmat, axis=1)
    scores = dmat[np.arange(dmat.shape[0]), idx]
    keep = scores < nn_thresh
    idx2 = np.argmin(dmat, axis=0)
    keep = np.logical_and(keep, np.arange(len(idx)) == idx2[idx])
    matches = np.zeros((3, int(keep.sum())))
    matches[0, :] = np.arange(desc1.shape[1])[keep]
    matches[1, :] = idx[keep]
    matches[2, :] = scores[keep]
    return matches


# ------------------------------------------------------------------------------------------------
# label warping of the dataset side  (SURVEY 8f rank 4; oracle only so far -- no CUDA counterpart yet)
# ------------------------------------------------------------------------------------------------
def homography_scaling(homography, H, W):
    """utils/utils.py:291-300: normalised -> pixel coordinates, T^-1 . H . T with T = [[2/W,0,-1],[0,2/H,-1],[0,0,1]] (fp32)."""
    trans = np.array([[2.0 / W, 0.0, -1], [0.0, 2.0 / H, -1], [0.0, 0.0, 1.0]], dtype=f32)
    return (np.linalg.inv(trans).astype(f32) @ np.asarray(homography, f32) @ trans).astype(f32)


def _scatter_last_wins(H, W, pts, values, channels=None):
    """datasets/data_tools.py:19-23: out[round(y), round(x)] = value; sequential index_put, the last duplicate wins."""
    out = np.zeros((H, W) if channels is None else (H, W, channels), dtype=f32)
    q = np.round(np.asarray(pts, dtype=f32)).astype(np.int64)  # torch.round = half to even, like np.round
    for i in range(q.shape[0]):
        out[q[i, 1], q[i, 0]] = values if np.isscalar(values) else values[i]
    return out


def warp_labels(pnts, H, W, homography, bilinear=False):
    """datasets/data_tools.py:37-63 warpLabels (+ :6-34 for labels_bi).  pnts [P,2] (x, y), truncated to integers;
    homography [3,3] in normalised coordinates.  Returns dict(labels [1,H,W], res [H,W,2], warped_pnts [M,2]
    [, labels_bi [1,H,W]])."""
    pnts = np.trunc(np.asarray(pnts, dtype=np.float64)).astype(np.int64)
    warped = warp_points(pnts[:, :2].astype(f32), homography_scaling(homography, H, W))
    outs = {}
    if bilinear:
        base = np.trunc(warped).astype(f32)                                   # .long() truncates toward zero
        ext = np.concatenate([base, base + np.array([0, 1], f32), base + np.array([1, 0], f32), base + 1], axis=0)
        rx, ry = warped[:, 0] - base[:, 0], warped[:, 1] - base[:, 1]
        wts = np.concatenate([(1 - rx) * (1 - ry), (1 - rx) * ry, rx * (1 - ry), rx * ry]).astype(f32)
        ext_f, keep = filter_points(ext, [W, H], return_mask=True)
        outs["labels_bi"] = _scatter_last_wins(H, W, ext_f, wts[keep])[None]
    warped = filter_points(warped, [W, H])
    outs["labels"] = _scatter_last_wins(H, W, warped, 1.0)[None]
    outs["res"] = _scatter_last_wins(H, W, warped, (warped - np.round(warped)).astype(f32), channels=2)
    outs["warped_pnts"] = warped
    return outs


# ------------------------------------------------------------------------------------------------
# 8f rank 2: sparse descriptor loss, evaluation half (the sampled index lists are inputs)
# ------------------------------------------------------------------------------------------------
def sparse_descriptor_loss(descriptors, descriptors_warped, matches_a, matches_b, non_matches_a, non_matches_b, lamda_d=250,
                           grad=None):
    """utils/loss_functions/sparse_loss.py:65-284 with pixelwise_contrastive_loss.py:140-265 (dist="cos", method="1d"), given
    the index lists the reference samples: [B,K] matches and [B,K*n] non-matches (cell index u + v*Wc in each image).
      match_b = 1/K sum max(1 - dot, 0);  nonmatch_b = sum max(dot - 0.2, 0) / (#nonzero + 1);  loss_b = lamda_d match_b + nonmatch_b
    Returns the batch means (loss, match, nonmatch); grad = (g_loss, g_match, g_nonmatch) adds d/d descriptors, d/d descriptors_warped
    (torch.clamp passes the gradient at the bound; the hard-negative count is a constant)."""
    D = np.asarray(descriptors, dtype=np.float64)
    Dw = np.asarray(descriptors_warped, dtype=np.float64)
    B, Dch, Hc, Wc = D.shape
    Nc = Hc * Wc
    A, Bm = D.reshape(B, Dch, Nc), Dw.reshape(B, Dch, Nc)
    ma, mb, na, nb = (np.asarray(x, dtype=np.int64) for x in (matches_a, matches_b, non_matches_a, non_matches_b))
    K = ma.shape[1]
    loss, match, non = [], [], []
    if grad is not None:
        gl, gm, gn = (float(g) for g in grad)
        dD, dDw = np.zeros_like(A), np.zeros_like(Bm)
    for b in range(B):
        dm = (A[b][:, ma[b]] * Bm[b][:, mb[b]]).sum(0).astype(f32)
        dn = (A[b][:, na[b]] * Bm[b][:, nb[b]]).sum(0).astype(f32)
        tm = np.maximum(f32(1.0) - dm, f32(0))
        tn = np.maximum(dn - f32(0.2), f32(0))
        hard = int(np.count_nonzero(tn))
        m_b = f32(1.0 / K) * tm.sum(dtype=f32)
        n_b = tn.sum(dtype=f32) / f32(hard + 1)
        match.append(m_b); non.append(n_b); loss.append(f32(lamda_d) * m_b + n_b)
        if grad is not None:
            cm = np.where(f32(1.0) - dm >= 0, -(gl * lamda_d + gm) / (K * B), 0.0)
            cn = np.where(dn - f32(0.2) >= 0, (gl + gn) / ((hard + 1) * B), 0.0)
            np.add.at(dD[b].T, ma[b], (cm[None, :] * Bm[b][:, mb[b]]).T)
            np.add.at(dDw[b].T, mb[b], (cm[None, :] * A[b][:, ma[b]]).T)
            np.add.at(dD[b].T, na[b], (cn[None, :] * Bm[b][:, nb[b]]).T)
            np.add.at(dDw[b].T, nb[b], (cn[None, :] * A[b][:, na[b]]).T)
    out = (f32(np.mean(np.array(loss, f32))), f32(np.mean(np.array(match, f32))), f32(np.mean(np.array(non, f32))))
    if grad is not None:
        return out + (dD.reshape(D.shape).astype(f32), dDw.reshape(D.shape).astype(f32))
    return out
