"""Sparse descriptor loss behind the reference's names (SURVEY 8f rank 2).

reference: utils/loss_functions/sparse_loss.py:65-284 -- `descriptor_loss_sparse(descriptors, descriptors_warped, homographies,
...)` for one image and `batch_descriptor_loss_sparse` (returns `(loss, None, pos, neg)` like the dense loss, so it slots into
Train_model_heatmap_all.py:333-347 unchanged).

The reference draws its correspondences on the HOST with numpy / torch CPU random numbers; `sample_correspondences` makes the
same calls in the same order (np.random.permutation [+ np.random.choice], torch.rand, torch.rand, torch.randn), so under the
same RNG state it returns the reference's own index lists (tests pin this against fixtures of the live reference).  The
lists go to the device once per batch; the loss and its gradient are CUDA kernels (csrc/sparse.cu).

DeviceSampler draws lists with the same distribution on the device (ssp_sparse_sample) from a seed and a launch counter held
in device memory: no host RNG call and no host synchronisation, so the whole sparse step can be captured into a CUDA graph
whose replays draw fresh lists.  Its draws are not the reference's RNG stream; batch_descriptor_loss_sparse uses it only
when it is passed one.
"""
from collections import namedtuple

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import _lib
from ._lib import call, f32c, ptr, stream_of
from .losses import grad_vector
from .rng import DeviceRng

CHECK_EMPTY_IMAGES = False  # DeviceSampler.sample raises when an image had no candidate (costs a host sync per call)


def scale_homography_torch(H, shape, shift=(-1, -1), dtype=torch.float32):
    """reference: utils/homographies.py:270-276 (normalised -> cell-grid coordinates of a [height, width] grid)."""
    height, width = shape[0], shape[1]
    trans = torch.tensor([[2.0 / width, 0.0, shift[0]], [0.0, 2.0 / height, shift[1]], [0.0, 0.0, 1.0]], dtype=dtype)
    return torch.inverse(trans) @ H @ trans


def sample_correspondences(homography, Hc, Wc, num_matching_attempts=1000, num_masked_non_matches_per_match=10):
    """The sampling half of descriptor_loss_sparse (sparse_loss.py:170-255 + correspondence_finder.py:191-320), on the CPU like
    the reference.  Returns int64 tensors (matches_a [K], matches_b [K], non_matches_a [K*n], non_matches_b [K*n]) of cell
    indices u + v * Wc."""
    K, nper = int(num_matching_attempts), int(num_masked_non_matches_per_match)
    vv, uu = torch.meshgrid(torch.arange(Hc), torch.arange(Wc), indexing="ij")
    uv_a = torch.stack((uu.reshape(-1), vv.reshape(-1)), dim=1).float()          # all cells, (x, y), row-major
    Hcell = scale_homography_torch(homography.float().cpu(), (Hc, Wc), shift=(-1, -1))
    pts = torch.cat((uv_a, torch.ones((uv_a.shape[0], 1))), dim=1)               # warp_points, utils/utils.py:315-343
    w = (Hcell.view(1, 3, 3).view(3, 3) @ pts.transpose(0, 1)).view(1, 3, -1).transpose(2, 1)
    uv_b = (w[:, :, :2] / w[:, :, 2:])[0]
    uv_b.round_()
    keep = ((uv_b >= 0) & (uv_b <= torch.tensor([Wc, Hc]).float() - 1)).all(dim=1)  # filter_points, inclusive bounds
    uv_b, uv_a = uv_b[keep], uv_a[keep]
    M = int(uv_b.shape[0])
    if M == 0:
        raise RuntimeError("descriptor_loss_sparse: the homography maps no cell into the image")
    choice = np.random.permutation(M)                                              # crop_or_pad_choice(shuffle=True)
    if M >= K:
        choice = choice[:K]
    else:
        choice = np.concatenate([choice, np.random.choice(choice, K - M, replace=True)])
    choice = torch.as_tensor(choice, dtype=torch.int64)
    uv_a, uv_b = uv_a[choice], uv_b[choice]
    matches_a = (uv_a[:, 0] + uv_a[:, 1] * Wc).long()
    matches_b = (uv_b[:, 0] + uv_b[:, 1] * Wc).long()
    # non-matches: uniform pixels of image b.  The reference then means to push away the samples that fall within one pixel of
    # the true match, but its mask of "ones" is built with zeros_like (correspondence_finder.py:268-275), so the perturbation
    # is identically zero and a non-match may coincide with the match -- reproduced as is.  The random numbers of the
    # perturbation are still drawn (they advance the RNG stream the next image samples from).
    n = K * nper
    r2 = torch.rand(2, n)
    nu = torch.floor(r2[0] * Wc).long().float()
    nv = torch.floor(r2[1] * Hc).long().float()
    torch.rand(n)
    torch.randn(n)
    non_a = uv_a[:, 0:1].repeat(1, nper).reshape(-1) + uv_a[:, 1:2].repeat(1, nper).reshape(-1) * Wc
    non_b = nu + nv * Wc
    return matches_a, matches_b, non_a.long(), non_b.long()


class DeviceSampler(DeviceRng):
    """Correspondence lists of the sparse loss drawn on the device (ssp_sparse_sample, csrc/sparse.cu): per image, the cells
    whose warp lands in the image are the candidates; K matches are a random K-subset of them (or all of them plus draws
    with replacement when there are fewer than K), and every match gets n non-matches at uniform cells.

    The random numbers are Philox4x32-10 keyed by (seed, image, launch counter), with the state handling of rng.DeviceRng:
    eager calls and graph replays draw fresh lists without the host, and get_state() / set_state() reproduce a sequence bit
    for bit.  An image whose homography maps no cell into the image turns
    the loss into NaN and counts in a device flag (empty_images(); CHECK_EMPTY_IMAGES raises on it).  Grids up to 8192
    cells (one block of 1024 threads x 8 cells per image: 30x40, 60x80 and KITTI's 47x155 fit); larger ones are an error."""

    def __init__(self, seed=0, device="cuda"):
        super().__init__(seed, device)  # state[3]: images with M = 0 so far
        self.last = None  # (ia, ib, M) of the last call

    def sample(self, mat_H, Hc, Wc, K=1000, n=10):
        """mat_H [B,3,3] (normalised coordinates) -> ia, ib int32 [B, K + K*n] (cell indices u + v*Wc into the descriptors
        and the warped descriptors, the K matches first) and M int32 [B], the candidate count of every image."""
        Hm = f32c(mat_H.detach().reshape(-1, 3, 3), self.device)
        B, K, n = Hm.shape[0], int(K), int(n)
        ia = torch.empty((B, K + K * n), dtype=torch.int32, device=self.device)
        ib = torch.empty_like(ia)
        M = torch.empty((B,), dtype=torch.int32, device=self.device)
        call("ssp_sparse_sample", ptr(Hm), B, int(Hc), int(Wc), K, n, ptr(self.state), ptr(ia), ptr(ib), ptr(M), stream_of(Hm))
        self.last = (ia, ib, M)
        if CHECK_EMPTY_IMAGES and int(self.state[3]) != 0:  # host sync: debugging / tests only (the NaN loss is the signal)
            n_empty = int(self.state[3])
            self.state[3] = 0
            raise RuntimeError("DeviceSampler: the homography maps no cell into the image (%d images)" % n_empty)
        return ia, ib, M

    def empty_images(self):
        """Images that had no candidate since the sampler was created (host sync)."""
        return int(self.state[3])


# What sparse_backward needs of sparse_forward: saved = (Dt, Dwt, ia, ib, dots, stats), out3 = [loss, match, nonmatch]
SparseState = namedtuple("SparseState", "saved out3 dims K Kn lamda")


def sparse_forward(D, Dw, ia, ib, K, Kn, lamda, M=None):
    """SparseDescriptorLossFn's forward -> SparseState."""
    _lib.require_cuda(D, Dw)
    dev = D.device
    Dc, Dwc = f32c(D.detach(), dev), f32c(Dw.detach(), dev)
    B, Dch, Hc, Wc = Dc.shape
    Nc = Hc * Wc
    s = stream_of(Dc)
    Dt = torch.empty((B, Nc, Dch), dtype=torch.float32, device=dev)
    Dwt = torch.empty_like(Dt)
    call("ssp_transpose_batched", ptr(Dc), B, Dch, Nc, ptr(Dt), s)
    call("ssp_transpose_batched", ptr(Dwc), B, Dch, Nc, ptr(Dwt), s)
    dots = torch.empty((B, K + Kn), dtype=torch.float32, device=dev)
    stats = torch.empty((B, 4), dtype=torch.float32, device=dev)
    out3 = torch.empty((3,), dtype=torch.float32, device=dev)
    call("ssp_sparse_desc_loss_fwd", ptr(Dt), ptr(Dwt), ptr(ia), ptr(ib), B, Nc, Dch, K, Kn, float(lamda), 1.0, 0.2,
         ptr(dots), ptr(stats), ptr(out3), s)
    if M is not None:
        call("ssp_sparse_finalize", ptr(M), B, ptr(out3), None, None, 0.0, None, s)
    return SparseState((Dt, Dwt, ia, ib, dots, stats), out3, (B, Dch, Hc, Wc), K, Kn, float(lamda))


def sparse_backward(st, g3):
    """Gradients (dD, dDw) [B,Dch,Hc,Wc] of sparse_forward's loss for g3 = device {dL/dloss, dL/dmatch, dL/dnonmatch}."""
    Dt, Dwt, ia, ib, dots, stats = st.saved
    B, Dch, Hc, Wc = st.dims
    Nc = Hc * Wc
    s = stream_of(Dt)
    dDt = torch.empty_like(Dt)
    dDwt = torch.empty_like(Dwt)
    call("ssp_sparse_desc_loss_bwd", ptr(Dt), ptr(Dwt), ptr(ia), ptr(ib), ptr(dots), ptr(stats), ptr(g3), B, Nc, Dch, st.K,
         st.Kn, st.lamda, 1.0, 0.2, ptr(dDt), ptr(dDwt), s)
    dD = torch.empty((B, Dch, Hc, Wc), dtype=torch.float32, device=Dt.device)
    dDw = torch.empty_like(dD)
    call("ssp_transpose_batched", ptr(dDt), B, Nc, Dch, ptr(dD), s)
    call("ssp_transpose_batched", ptr(dDwt), B, Nc, Dch, ptr(dDw), s)
    return dD, dDw


class SparseDescriptorLossFn(torch.autograd.Function):
    """(loss, match, nonmatch) batch means from descriptors [B,Dch,Hc,Wc] and index lists ia / ib [B, K + Kn] (int32).
    M: the candidate counts of DeviceSampler.sample, or None; a zero count turns the three means into NaN."""

    @staticmethod
    def forward(ctx, D, Dw, ia, ib, K, Kn, lamda, M=None):
        st = sparse_forward(D, Dw, ia, ib, K, Kn, lamda, M)
        ctx.save_for_backward(*st.saved)
        ctx.st = st._replace(saved=None)
        return st.out3[0], st.out3[1], st.out3[2]

    @staticmethod
    @once_differentiable
    def backward(ctx, g_loss, g_match, g_non):
        st = ctx.st._replace(saved=ctx.saved_tensors)
        dD, dDw = sparse_backward(st, grad_vector((g_loss, g_match, g_non), st.out3.device))
        return dD, dDw, None, None, None, None, None, None


def sparse_loss_from_lists(descriptors, descriptors_warped, matches_a, matches_b, non_matches_a, non_matches_b, lamda_d=250):
    """Loss from explicit index lists [B,K] / [B,K*n] (any integer dtype / device).  Returns (loss, match, nonmatch) means."""
    dev = descriptors.device
    ia = torch.cat([torch.as_tensor(matches_a), torch.as_tensor(non_matches_a)], dim=1).to(device=dev, dtype=torch.int32).contiguous()
    ib = torch.cat([torch.as_tensor(matches_b), torch.as_tensor(non_matches_b)], dim=1).to(device=dev, dtype=torch.int32).contiguous()
    K, Kn = int(torch.as_tensor(matches_a).shape[1]), int(torch.as_tensor(non_matches_a).shape[1])
    return SparseDescriptorLossFn.apply(descriptors, descriptors_warped, ia, ib, K, Kn, float(lamda_d))


def batch_descriptor_loss_sparse(descriptors, descriptors_warped, homographies, mask_valid=None, cell_size=8, device="cpu",
                                 descriptor_dist=4, lamda_d=250, num_matching_attempts=1000,
                                 num_masked_non_matches_per_match=10, dist="cos", method="1d", sampler=None, **config):
    """reference: utils/loss_functions/sparse_loss.py:267-284.  Returns (loss, None, positive, negative), batch means.
    sampler=None samples on the host like the reference (its RNG call order); a DeviceSampler samples on the device."""
    if dist != "cos" or method != "1d":
        raise NotImplementedError("descriptor_loss_sparse: only dist='cos', method='1d' (what every shipped config uses)")
    _lib.require_cuda(descriptors, descriptors_warped)
    B, _, Hc, Wc = descriptors.shape
    if sampler is not None:
        K = int(num_matching_attempts)
        ia, ib, M = sampler.sample(homographies, Hc, Wc, K, num_masked_non_matches_per_match)
        loss, pos, neg = SparseDescriptorLossFn.apply(descriptors, descriptors_warped, ia, ib, K, ia.shape[1] - K,
                                                      float(lamda_d), M)
        return loss, None, pos, neg
    lists = [sample_correspondences(homographies[i].detach().float().cpu(), Hc, Wc, num_matching_attempts,
                                    num_masked_non_matches_per_match) for i in range(B)]
    ma, mb, na, nb = (torch.stack([l[j] for l in lists]) for j in range(4))
    loss, pos, neg = sparse_loss_from_lists(descriptors, descriptors_warped, ma, mb, na, nb, lamda_d)
    return loss, None, pos, neg


def descriptor_loss_sparse(descriptors, descriptors_warped, homographies, mask_valid=None, cell_size=8, device="cpu",
                           descriptor_dist=4, lamda_d=250, num_matching_attempts=1000, num_masked_non_matches_per_match=10,
                           dist="cos", method="1d", **config):
    """reference: utils/loss_functions/sparse_loss.py:65-262, one image: descriptors [D,Hc,Wc], homographies [3,3].
    Returns (loss, match_loss, non_match_loss)."""
    loss, _, pos, neg = batch_descriptor_loss_sparse(descriptors.unsqueeze(0), descriptors_warped.unsqueeze(0),
                                                     homographies.reshape(1, 3, 3), mask_valid, cell_size, device,
                                                     descriptor_dist, lamda_d, num_matching_attempts,
                                                     num_masked_non_matches_per_match, dist, method, **config)
    return loss, pos, neg
