"""autograd.Functions that drive the detector-loss and dense descriptor-loss kernels through the C ABI.

reference: Train_model_heatmap_all.py:155-179 (detector_loss), utils/utils.py:779-893 (descriptor_loss).
Multi-GPU (SURVEY 8e): both losses use GLOBAL-batch normalisers, so with `dist_group` set the local
numerators / mask sums are exchanged by ONE peer-memory kernel (dist.LossExchange, csrc/exchange.cu) that rewrites
the loss scalars and normalisers in place, stream ordered, before the forward returns; the backward kernels
scale by the global normaliser.
"""
import contextlib
import functools
from collections import namedtuple

import torch
from torch.autograd.function import once_differentiable

from . import _lib
from ._lib import call, f32c, ptr, stream_of

_ENGINES = ("bf16x3", "bf16", "fp32")
_engine = "bf16x3"
CHECK_LIST_OVERFLOW = False  # tests turn this on (costs a host sync per call)


def set_descriptor_engine(name):
    """'bf16x3' (tcgen05, hi/lo split, fp32-grade), 'bf16' (tcgen05 single pass) or 'fp32' (CUDA cores)."""
    global _engine
    if name not in _ENGINES:
        raise ValueError("descriptor engine must be one of %s" % (_ENGINES,))
    _engine = name


def get_descriptor_engine():
    return _engine


_side_streams = {}


class _Fork(object):
    """`with _Fork(dev):` runs the body on a per-device side stream, ordered after everything queued so far on the
    current stream; .join() makes the current stream wait for it.  Buffers are allocated on the current stream before
    the fork and stay referenced until after the join, so the caching allocator never recycles them early."""

    def __init__(self, dev):
        self.cur = torch.cuda.current_stream(dev)
        key = (dev.index, self.cur.cuda_stream)
        if key not in _side_streams:
            _side_streams[key] = torch.cuda.Stream(device=dev)
        self.side = _side_streams[key]
        self.ctx = None

    def __enter__(self):
        self.side.wait_stream(self.cur)
        self.ctx = torch.cuda.stream(self.side)
        self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        self.ctx.__exit__(*exc)
        return False

    def join(self):
        self.cur.wait_stream(self.side)


# ------------------------------------------------------------------------------------------------
class SemanticLossFn(torch.autograd.Function):
    """Cross entropy of the semantic head with ignore_index (Train_model_heatmap_all.py:181-193).

    pred [B,C,H,W] at the label resolution -> streaming softmax-CE kernels.
    pred [B,C,H/8,W/8] (the head output before the model's F.interpolate, SuperPointNet_gauss2_ssmall.py:90) -> the x8
    bilinear upsample is fused into the loss and its backward; the full-resolution logits never exist.
    With dist_group the mean runs over the counted pixels of the GLOBAL batch (sum and count are all-reduced)."""

    @staticmethod
    def forward(ctx, pred, label, ignore_index, dist_group=None):
        _lib.require_cuda(pred)
        dev = pred.device
        x = f32c(pred.detach(), dev)
        lab = label.detach().to(device=dev, dtype=torch.int64).contiguous()
        if x.dim() != 4 or lab.dim() != 3 or lab.shape[0] != x.shape[0]:
            raise RuntimeError("sem_loss: expected pred [B,C,h,w] and label [B,H,W], got %s and %s"
                               % (tuple(pred.shape), tuple(label.shape)))
        B, C, h, w = x.shape
        H, W = lab.shape[1:]
        up = (h, w) != (H, W)
        if up and (H != 8 * h or W != 8 * w):
            raise RuntimeError("sem_loss: pred %dx%d must match the label size %dx%d or be exactly 1/8 of it" % (h, w, H, W))
        out3 = torch.empty((3,), dtype=torch.float32, device=dev)
        nbytes = _lib.load().ssp_sem_ce_ws_bytes(B, C, H, W, 1 if up else 0)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        need_grad = ctx.needs_input_grad[0]
        if up:
            gsum = torch.empty_like(x) if need_grad else None
            call("ssp_sem_ce_up8", ptr(x), ptr(lab), B, C, h, w, int(ignore_index), ptr(gsum), ptr(out3), ptr(ws), nbytes,
                 stream_of(x))
            ctx.saved = (gsum,)
        else:
            lse2 = torch.empty((B, H, W), dtype=torch.float32, device=dev)
            call("ssp_sem_ce_fwd", ptr(x), ptr(lab), B, C, H, W, int(ignore_index), ptr(lse2), ptr(out3), ptr(ws), nbytes,
                 stream_of(x))
            ctx.saved = (x, lab, lse2)
        ctx.up, ctx.shape, ctx.ignore = up, (B, C, h, w), int(ignore_index)
        ctx.out3 = out3  # attribute, see DetectorLossPairFn
        if dist_group is not None:
            from .dist import get_exchange
            get_exchange(dist_group).run(sem0=out3)
        return out3[0]

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        B, C, h, w = ctx.shape
        out3 = ctx.out3
        g = f32c(gout.reshape(1), out3.device)
        if ctx.up:
            (gsum,) = ctx.saved
            d = torch.empty_like(gsum)
            call("ssp_sem_ce_up8_bwd", ptr(gsum), ptr(out3), ptr(g), B, C, h, w, ptr(d), stream_of(d))
        else:
            x, lab, lse2 = ctx.saved
            d = torch.empty_like(x)
            call("ssp_sem_ce_bwd", ptr(x), ptr(lab), ptr(lse2), B, C, h, w, ctx.ignore, ptr(out3), ptr(g), ptr(d),
                 stream_of(d))
        return d, None, None, None


def grad_vector(grads, dev):
    """The upstream gradients of a node's scalar outputs as one contiguous fp32 device vector, zero where none came."""
    zero = torch.zeros((), dtype=torch.float32, device=dev)
    return torch.stack([(g if g is not None else zero).reshape(()).to(torch.float32) for g in grads]).contiguous()


@functools.lru_cache(maxsize=None)
def _lam3_vector(lam, dev):
    """The device vector [lam, 0, 0]: g * it is the gradient vector of a descriptor loss weighted by lam."""
    return torch.tensor([lam, 0.0, 0.0], dtype=torch.float32, device=dev)


# ------------------------------------------------------------------------------------------------
# saved = fp32 (x0, t0, m0, x1, t1, m1), the last three None for one loss; out [n,3]: a triple per image
DetPair = namedtuple("DetPair", "saved out fused2d")


def det_pair_forward(semi, target, mask, semi_w, target_w, mask_w, fused2d):
    """One detector loss (semi_w None) or both of a pair in one launch -> (DetPair, getMasks() of the warped mask
    [B,Hc,Wc], None for one loss)."""
    _lib.require_cuda(semi, semi_w)
    dev = semi.device
    pair = semi_w is not None
    n = 2 if pair else 1
    fc = lambda a: f32c(a.detach(), dev)
    x0, t0, m0 = fc(semi), fc(target), fc(mask)
    x1, t1, m1 = (fc(semi_w), fc(target_w), fc(mask_w)) if pair else (None, None, None)
    B, C, Hc, Wc = x0.shape
    if C != 65 or (pair and x1.shape != x0.shape):
        raise RuntimeError("detector_loss: logits must be [B,65,Hc,Wc], the same shape for both images of a pair")
    n2d = B * Hc * Wc * 64
    for t, m in ((t0, m0), (t1, m1))[:n]:
        ok = (t.numel() == n2d and m.numel() == n2d) if fused2d else (t.shape == x0.shape and m.numel() == B * Hc * Wc)
        if not ok:
            raise RuntimeError("detector_loss: target / mask shapes do not match the logits")
    out = torch.empty((n, 3), dtype=torch.float32, device=dev)
    cellmask = torch.empty((B, Hc, Wc), dtype=torch.float32, device=dev) if pair else None
    per = (_lib.load().ssp_detector_loss_ws_bytes(B, Hc, Wc) + 15) // 16 * 16
    ws = torch.empty((n * per,), dtype=torch.uint8, device=dev)
    call("ssp_detector_loss_fwd_pair", ptr(x0), ptr(t0), ptr(m0), ptr(x1), ptr(t1), ptr(m1), B, Hc, Wc,
         1 if fused2d else 0, ptr(out[0]), ptr(out[1]) if pair else None, ptr(cellmask), ptr(ws), n * per, stream_of(x0))
    return DetPair((x0, t0, m0, x1, t1, m1), out, fused2d), cellmask


def det_pair_backward(st, g0, g1=None):
    """(d semi, d semi_w) for upstream gradients g0, g1: 1-element device tensors (the fused step passes one twice).
    One loss: g1 and d semi_w are None."""
    x0, t0, m0, x1, t1, m1 = st.saved
    pair = x1 is not None
    B, C, Hc, Wc = x0.shape
    d0, d1 = torch.empty_like(x0), (torch.empty_like(x1) if pair else None)
    call("ssp_detector_loss_bwd_pair", ptr(x0), ptr(t0), ptr(m0), ptr(x1), ptr(t1), ptr(m1), B, Hc, Wc,
         1 if st.fused2d else 0, ptr(st.out[0]), ptr(st.out[1]) if pair else None, ptr(g0), ptr(g1), ptr(d0), ptr(d1),
         stream_of(x0))
    return d0, d1


class DetectorLossPairFn(torch.autograd.Function):
    """loss = sum_cells mask * sum_c BCE(softmax(semi)_c, target_c) / (sum mask + 1e-5) of one image (semi_w None) or of
    both images of a training pair (image, warped image), in ONE launch each way.

    fused2d=False: target [B,65,Hc,Wc], mask [B,Hc,Wc]  (reference signature)
    fused2d=True : target = labels_2D [B,1,H,W], mask = mask_2D [B,1,H,W] (labels2Dto3D + getMasks fused)
    Returns loss for one image; (loss, loss_warp, cell_mask_warp) for a pair, where cell_mask_warp = getMasks() of the
    warped mask is a by-product (it is the descriptor loss's mask_valid)."""

    @staticmethod
    def forward(ctx, semi, target, mask, semi_w, target_w, mask_w, fused2d, dist_group=None):
        pair = semi_w is not None
        st, cellmask = det_pair_forward(semi, target, mask, semi_w, target_w, mask_w, fused2d)
        ctx.save_for_backward(*st.saved)
        ctx.st = st._replace(saved=None)  # out is an attribute, not a saved tensor (the exchange rewrites it in place)
        if dist_group is not None:
            from .dist import get_exchange
            get_exchange(dist_group).run(det0=st.out[0], det1=st.out[1] if pair else None)
        if not pair:
            return st.out[0, 0]
        ctx.mark_non_differentiable(cellmask)
        return st.out[0, 0], st.out[1, 0], cellmask

    @staticmethod
    @once_differentiable
    def backward(ctx, g0, g1=None, _gm=None):
        st = ctx.st._replace(saved=ctx.saved_tensors)
        g = grad_vector((g0, g1)[:len(st.out)], st.out.device)
        d0, d1 = det_pair_backward(st, *g.split(1))
        return d0, None, None, d1, None, None, None, None


# ------------------------------------------------------------------------------------------------
_MPOS, _MNEG = 1.0, 0.2  # hinge margins, hard-coded in the reference (utils/utils.py:817-818)


def _nc_pad(nc):
    return (nc + 255) // 256 * 256


# What desc_backward needs of desc_forward: saved = (Dc, Dwc, mv_pad, bitsR, bitsC, lists_i, lists_f, Ahi, Alo, Bhi, Blo), None
# where the engine or need_grad has none; out8 = [loss, pos, neg, norm, num_loss, num_pos, num_neg, sum(mask_valid)].
DescState = namedtuple("DescState", "saved out8 dims lamda engine fold")


def desc_forward(D, Dw, Hm, *, mask_valid=None, mask_2d=None, cell, lamda, dist, engine, need_grad, fold, debug_S=None):
    """The dense descriptor loss up to desc_finalize -> (DescState, partial sums for desc_finalize, wpts [B,Ncp,2]).
    mask_valid [B,Hc*Wc] or mask_2d [B,1,8Hc,8Wc] (getMasks fused into the geometry kernel).  fold (tensor-core engines with
    need_grad): the mask is folded into the indicator words and the backward needs no pack pass.  Exact only for a 0/1 mask
    and g_neg = 0; a non-binary mask poisons the normaliser with NaN in the geometry kernel (loud, no sync)."""
    lib = _lib.load()
    dev = D.device
    Dc = f32c(D.detach(), dev)
    Dwc = f32c(Dw.detach(), dev)
    if Dc.shape != Dwc.shape:
        raise RuntimeError("descriptor_loss: descriptor shapes differ")
    B, Dch, Hc, Wc = Dc.shape
    Nc = Hc * Wc
    Ncp = _nc_pad(Nc)
    s = stream_of(Dc)
    if engine not in _ENGINES:
        raise ValueError("descriptor engine must be one of %s" % (_ENGINES,))
    if Dch != 256:
        engine = "fp32"  # the tcgen05 kernels are specialised for 256 channels
    split = engine == "bf16x3"
    fold = bool(fold and need_grad and engine != "fp32")

    wpts = torch.empty((B, Ncp, 2), dtype=torch.float32, device=dev)
    mv_pad = torch.empty((B, Ncp), dtype=torch.float32, device=dev)
    mvbits = torch.empty((B, Ncp // 32), dtype=torch.int32, device=dev) if fold else None
    nmv = lib.ssp_desc_geometry_nblocks(B, Nc)
    mv_part = torch.empty((nmv,), dtype=torch.float64, device=dev)

    # sparse positive pairs: exact dots, partial sums, pair lists for the backward
    maxp = lib.ssp_desc_maxp()
    npos = lib.ssp_desc_pos_planes_nblocks(B, Nc) if split else lib.ssp_desc_pos_nblocks(B, Nc)
    pos_part = torch.empty((npos, 4), dtype=torch.float64, device=dev)
    lists_i = torch.empty((3, B, Ncp, maxp), dtype=torch.int32, device=dev)   # rowcol, colrow, (colcnt in [2,:,:,0])
    lists_f = torch.empty((2, B, Ncp, maxp), dtype=torch.float32, device=dev)  # rowdot, coldot
    rowcol, colrow, colcnt = lists_i[0], lists_i[1], lists_i[2].view(-1)[: B * Ncp + 1]
    rowdot, coldot = lists_f[0], lists_f[1]
    overflow = colcnt[B * Ncp:]  # pairs that did not fit a list: desc_finalize turns a non-zero count into NaN
    bitsR = bitsC = None
    if need_grad:
        bitsR = torch.empty((B, Ncp // 32, Ncp), dtype=torch.int32, device=dev)
        bitsC = torch.empty((B, Ncp // 32, Ncp), dtype=torch.int32, device=dev)
    Ahi = Alo = Bhi = Blo = None
    # every buffer of the forward is allocated before the fork (see _Fork)
    if engine == "fp32":
        nneg = lib.ssp_desc_dense_simt_nblocks(B, Nc)
    else:
        nneg = lib.ssp_desc_dense_tc_nblocks(B, Nc)
        # hi (and lo) planes of one tensor in ONE allocation, lo above hi: the backward's TMA box spans both planes
        PA = torch.empty((2 if split else 1, B, Ncp, Dch), dtype=torch.bfloat16, device=dev)
        PB = torch.empty_like(PA)
        Ahi, Alo = PA[0], (PA[1] if split else None)
        Bhi, Blo = PB[0], (PB[1] if split else None)
    neg_part = torch.empty((nneg, 2), dtype=torch.float64, device=dev)
    out8 = torch.empty((8,), dtype=torch.float32, device=dev)
    # geometry (warped cell centres, mask) and, on the tensor-core engines, the operand pack in one launch (independent work):
    # every positive-pair kernel needs the warped points.  The fp32 engine packs nothing (hi planes NULL).
    call("ssp_desc_pack2_geometry", ptr(Dc), ptr(Dwc), B, Dch, Hc, Wc, ptr(Ahi), ptr(Alo), ptr(Bhi), ptr(Blo), ptr(Hm),
         ptr(mask_valid), ptr(mask_2d), cell, ptr(wpts), ptr(mv_pad), ptr(mv_part), ptr(mvbits), s)
    if split:
        # bf16x3: the positive pairs read the packed hi/lo planes (2 x 512 contiguous bytes per cell instead of 256
        # strided channels), so they run right after the pack, in front of the tensor-core kernel
        call("ssp_desc_pos_fwd_planes", ptr(Ahi), ptr(Alo), ptr(Bhi), ptr(Blo), ptr(wpts), ptr(mv_pad), B, Hc, Wc, cell,
             dist, lamda, _MPOS, _MNEG, ptr(pos_part), ptr(rowcol), ptr(rowdot), ptr(colcnt), ptr(colrow), ptr(coldot), s)
        # bitsC (the column-orientation indicator words) is only read by the backward GEMM: it is transposed from bitsR by
        # extra blocks of the backward's coefficient launch, not here
        call("ssp_desc_dense_fwd_tc", ptr(Ahi), ptr(Alo), ptr(Bhi), ptr(Blo), ptr(mv_pad), ptr(mvbits), B, Hc, Wc, _MNEG,
             ptr(neg_part), ptr(bitsR), ptr(debug_S), s)
    else:
        # the HBM-bound exact positive-pair kernel overlaps the GEMM kernel
        with _Fork(dev) as fork:
            call("ssp_desc_pos_fwd", ptr(Dc), ptr(Dwc), ptr(wpts), ptr(mv_pad), B, Hc, Wc, Dch, cell, dist, lamda, _MPOS,
                 _MNEG, ptr(pos_part), ptr(rowcol), ptr(rowdot), ptr(colcnt), ptr(colrow), ptr(coldot), stream_of(Dc))
        if engine == "fp32":
            call("ssp_desc_dense_fwd_simt", ptr(Dc), ptr(Dwc), ptr(mv_pad), B, Hc, Wc, Dch, _MNEG, ptr(neg_part),
                 ptr(bitsR), ptr(bitsC), ptr(debug_S), s)
        else:
            call("ssp_desc_dense_fwd_tc", ptr(Ahi), None, ptr(Bhi), None, ptr(mv_pad), ptr(mvbits), B, Hc, Wc, _MNEG,
                 ptr(neg_part), ptr(bitsR), ptr(debug_S), s)
        fork.join()
    st = DescState((Dc, Dwc, mv_pad, bitsR, bitsC, lists_i, lists_f, Ahi, Alo, Bhi, Blo), out8, (B, Dch, Hc, Wc), lamda,
                   engine, fold)
    return st, (pos_part, npos, neg_part, nneg, mv_part, nmv, overflow), wpts


def desc_finalize(st, parts, det_out=None, lambda_loss=0.0, total=None):
    """ssp_desc_finalize: reduces the partial sums of desc_forward into st.out8 (a positive pair that did not fit the lists
    turns the loss into NaN).  With det_out ([2,3], det_pair_forward's out) it also writes the fused step's total
    det_out[0,0] + det_out[1,0] + lambda_loss * loss_desc into total [1]."""
    pos_part, npos, neg_part, nneg, mv_part, nmv, overflow = parts
    B, _, Hc, Wc = st.dims
    call("ssp_desc_finalize", ptr(pos_part), npos, ptr(neg_part), nneg, ptr(mv_part), nmv, B, Hc, Wc, ptr(overflow),
         ptr(st.out8), ptr(None if det_out is None else det_out[0]), ptr(None if det_out is None else det_out[1]),
         float(lambda_loss), ptr(total), stream_of(pos_part))
    if CHECK_LIST_OVERFLOW and int(overflow[0]) != 0:  # host sync: debugging / tests only (the NaN above is the product signal)
        raise RuntimeError("descriptor_loss: %d positive pairs overflowed the sparse lists" % int(overflow[0]))


def desc_backward(st, g3, gscale=1.0, gmode=0, det=None):
    """(dD, dDw) for g3 = device {dL/dloss, dL/dpos, dL/dneg} (gmode 0) or, folded mask only, the fused step's upstream
    gradient scaled by gscale in the coefficient kernel (gmode 1).  det = (DetPair, g, d0, d1), folded mask only: the
    detector-pair backward for g into d0 / d1 rides in the coefficient launch."""
    if det is not None and not st.fold:
        raise ValueError("desc_backward: the detector backward merges only into the folded-mask backward")
    Dc, Dwc, mv_pad, bitsR, bitsC, lists_i, lists_f, Ahi, Alo, Bhi, Blo = st.saved
    out8, lamda, fold = st.out8, st.lamda, st.fold
    B, Dch, Hc, Wc = st.dims
    dev = Dc.device
    Nc = Hc * Wc
    Ncp = _nc_pad(Nc)
    s = stream_of(Dc)
    tc_engine = st.engine != "fp32"
    split = st.engine == "bf16x3"
    # alpha[b,c] = (g_loss * mv[c] + g_neg) / norm: coefficient of the negative hinge of column c; srow = alpha at mv = 1
    # (row scale of the folded backward).  Folded: both come out of the coefficient kernel below.
    alpha = torch.empty((B, Ncp), dtype=torch.float32, device=dev)
    srow = torch.empty((B, Ncp), dtype=torch.float32, device=dev) if fold else None
    if not fold:
        call("ssp_desc_alpha", ptr(mv_pad), ptr(g3), ptr(out8), B, Ncp, ptr(alpha), s)
    rowcol, colrow, colcnt = lists_i[0], lists_i[1], lists_i[2]
    rowdot, coldot = lists_f[0], lists_f[1]
    coefs = torch.empty((2,) + tuple(rowdot.shape), dtype=torch.float32, device=dev)
    colrow_sorted = torch.empty_like(colrow)  # the saved lists stay as the forward wrote them (retain_graph safe)
    dD = torch.empty_like(Dc)
    dDw = torch.empty_like(Dwc)
    if tc_engine and not fold:
        PS = torch.empty((2 if split else 1, B, Ncp, Dch), dtype=torch.bfloat16, device=dev)
        Shi, Slo = PS[0], (PS[1] if split else None)
    # dD [b,:,r] = sum_c I[r,c] alpha[c] Dw[b,:,c] + sum_n rowcoef[r,n] Dw[b,:,rowcol[r,n]]
    # dDw[b,:,c] = alpha[c] sum_r I[r,c] D[b,:,r]  + sum_n colcoef[c,n] D [b,:,colrow[c,n]]
    # tensor-core engines: both GEMMs run in ONE persistent launch, the positive pairs are applied inside the GEMM
    # epilogues (dedicated epilogue warps hide the gathers behind the next item's main loop);
    # fp32 engine: one streaming apply kernel after the GEMMs.
    # stream plan:  [pos_coef]  ||  [pack(alpha * Dw), unless folded]  ->  GEMM pair
    # folded: bitsR / bitsC already exclude the columns with mask_valid = 0, dD = srow * (I' @ Dw) on the forward planes
    if det is not None:
        # fused step: the detector-loss backward of both images rides in the same launch (heterogeneous blocks)
        dst, dg, d0, d1 = det
        x0, t0, m0, x1, t1, m1 = dst.saved
        call("ssp_step_bwd_prologue", ptr(x0), ptr(t0), ptr(m0), ptr(x1), ptr(t1), ptr(m1), B, Hc, Wc, ptr(dst.out[0]),
             ptr(dst.out[1]), ptr(dg), ptr(d0), ptr(d1),
             ptr(rowcol), ptr(rowdot), ptr(colcnt), ptr(colrow), ptr(coldot), ptr(bitsR), ptr(mv_pad), ptr(g3), gscale,
             gmode, ptr(out8), lamda, _MPOS, ptr(coefs[0]), ptr(colrow_sorted), ptr(coefs[1]), ptr(alpha), ptr(srow),
             ptr(bitsC), s)
    else:
        # folded, the coefficient launch also writes alpha and srow; on the tensor-core engines it transposes bitsR into
        # bitsC (fp32: the forward wrote it).  Unfolded, it runs on a side stream next to alpha and the pack.
        side = contextlib.nullcontext() if fold else _Fork(dev)
        with side:
            call("ssp_desc_pos_coef", ptr(rowcol), ptr(rowdot), ptr(colcnt), ptr(colrow), ptr(coldot), ptr(bitsR),
                 ptr(mv_pad), ptr(g3), gscale, gmode, ptr(out8), B, Ncp, lamda, _MPOS, ptr(coefs[0]), ptr(colrow_sorted),
                 ptr(coefs[1]), ptr(alpha) if fold else None, ptr(srow), ptr(bitsC) if tc_engine else None,
                 Nc if tc_engine else 0, stream_of(Dc))
    if not fold:
        if not tc_engine:
            call("ssp_desc_bits_gemm_simt", ptr(bitsR), ptr(Dwc), ptr(alpha), None, B, Dch, Nc, ptr(dD), s)
            call("ssp_desc_bits_gemm_simt", ptr(bitsC), ptr(Dc), None, ptr(alpha), B, Dch, Nc, ptr(dDw), s)
            side.join()
            call("ssp_desc_pos_apply", ptr(rowcol), ptr(coefs[0]), ptr(colrow_sorted), ptr(coefs[1]), ptr(Dc), ptr(Dwc), B, Dch,
                 Nc, ptr(dD), ptr(dDw), s)
            return dD, dDw
        call("ssp_desc_pack", ptr(Dwc), ptr(alpha), B, Dch, Nc, ptr(Shi), ptr(Slo), s)
        side.join()
    # the dD GEMM reads the forward planes of Dw (rows scaled by srow) when folded, the packed alpha * Dw otherwise; the
    # positive-pair partners come from the packed planes of the forward (Dw for dD, D for dDw)
    Whi, Wlo = (Bhi, Blo) if fold else (Shi, Slo)
    call("ssp_desc_bits_gemm_tc_pair",
         ptr(bitsR), ptr(Whi), ptr(Wlo), ptr(srow), ptr(rowcol), ptr(coefs[0]), ptr(Bhi), ptr(Blo), ptr(dD),
         ptr(bitsC), ptr(Ahi), ptr(Alo), ptr(alpha), ptr(colrow_sorted), ptr(coefs[1]), ptr(Ahi), ptr(Alo), ptr(dDw),
         B, Nc, s)
    return dD, dDw


class DescriptorLossFn(torch.autograd.Function):
    """Dense descriptor hinge loss.  Returns (loss_desc, pos_sum, neg_sum, wpts); the three scalars are
    differentiable w.r.t. descriptors and descriptors_warped, wpts (warped cell centres) is not."""

    @staticmethod
    def forward(ctx, D, Dw, Hm, mv, cell, lamda, dist, engine, dist_group=None, debug_S=None):
        need_grad = bool(ctx.needs_input_grad[0] or ctx.needs_input_grad[1])
        st, parts, wpts = desc_forward(D, Dw, Hm, mask_valid=mv, cell=cell, lamda=lamda, dist=dist, engine=engine,
                                       need_grad=need_grad, fold=False, debug_S=debug_S)
        desc_finalize(st, parts)
        if dist_group is not None:
            from .dist import get_exchange
            B, _, Hc, Wc = st.dims
            get_exchange(dist_group).run(desc8=st.out8, B_local=B, Hc=Hc, Wc=Wc)
        if need_grad:
            ctx.save_for_backward(*st.saved)
        ctx.st = st._replace(saved=None)  # out8 is an attribute, see DetectorLossPairFn
        ctx.mark_non_differentiable(wpts)
        return st.out8[0], st.out8[1], st.out8[2], wpts

    @staticmethod
    @once_differentiable
    def backward(ctx, g_loss, g_pos, g_neg, _g_wpts):
        st = ctx.st._replace(saved=ctx.saved_tensors)
        dD, dDw = desc_backward(st, grad_vector((g_loss, g_pos, g_neg), st.out8.device))
        return dD, dDw, None, None, None, None, None, None, None, None


# ------------------------------------------------------------------------------------------------
class LossStepFn(torch.autograd.Function):
    """The whole loss step (Train_model_heatmap_all.py:295-365, uniform weighting) as ONE autograd node:
    loss = loss_det + loss_det_warp + lambda_loss * loss_desc.  Same kernels as DetectorLossPairFn + DescriptorLossFn;
    what disappears is the dozen 2-microsecond torch kernels (scalar mul / add, ones_like, zeros, stack) that autograd
    needs to route three scalars through two nodes -- 7 % of a 0.45 ms step.
    Returns (loss, loss_det, loss_det_warp, loss_desc, pos, neg); only `loss` is differentiable."""

    @staticmethod
    def forward(ctx, semi, labels_2D, mask_2D, semi_w, warped_labels, mask_warp_2D, desc, desc_w, Hm, lamda_d, dist,
                lambda_loss, engine, dist_group=None):
        B, _, Hc, Wc = semi.shape
        dev = semi.device
        # The two detector losses (HBM-bound, + their one-block finalize) run on a forked stream next to the first half of
        # the descriptor chain (geometry -> pack -> positive pairs: a mix of HBM- and latency-bound kernels): nothing there
        # needs them except the cell mask of the warped valid mask, which the geometry kernel computes itself (getMasks fused
        # in).  The streams join in front of desc_finalize, which reads both detector triples for the step total.
        fork = _Fork(dev)
        with fork:
            det, _ = det_pair_forward(semi, labels_2D, mask_2D, semi_w, warped_labels, mask_warp_2D, True)
        mw = f32c(mask_warp_2D.detach(), dev)
        if mw.numel() != B * Hc * Wc * 64:
            raise RuntimeError("loss_step: mask_warp_2D must be [B,1,%d,%d]" % (Hc * 8, Wc * 8))
        want_desc = bool(ctx.needs_input_grad[6] or ctx.needs_input_grad[7])
        total = torch.empty((1,), dtype=torch.float32, device=dev)
        # fold=True (measured: 0.339 -> 0.330 ms per step): g_neg = 0 holds because only `loss` is differentiable, and a
        # non-binary mask turns the loss into NaN.  A soft mask belongs on fused=False, whose descriptor_loss packs
        # alpha * Dw into its own planes.
        st, parts, _wpts = desc_forward(desc, desc_w, Hm, mask_2d=mw, cell=8, lamda=lamda_d, dist=dist, engine=engine,
                                        need_grad=want_desc, fold=True)
        fork.join()
        desc_finalize(st, parts, det.out, lambda_loss, total)
        if dist_group is not None:
            # multi-GPU: ONE exchange kernel turns the three local results into global-batch values in place (the scalars
            # below are views of det.out / st.out8) and rewrites the weighted total; the backward kernels read the global
            # normalisers from the same buffers
            from .dist import get_exchange
            get_exchange(dist_group).run(det0=det.out[0], det1=det.out[1], desc8=st.out8, B_local=B, Hc=Hc, Wc=Wc,
                                         lambda_loss=lambda_loss, total=total)
        ctx.det, ctx.desc, ctx.lambda_loss = det, (st if want_desc else None), float(lambda_loss)
        outs = (det.out[0, 0], det.out[1, 0], st.out8[0], st.out8[1], st.out8[2])
        ctx.mark_non_differentiable(*outs)
        ctx.set_materialize_grads(False)  # no zero-filled gradient tensors for the five logging outputs
        return (total[0],) + outs

    @staticmethod
    @once_differentiable
    def backward(ctx, g, *_unused):
        if g is None:
            return (None,) * 14
        g = f32c(g.reshape(1), g.device)
        det, desc, lam = ctx.det, ctx.desc, ctx.lambda_loss
        d0 = d1 = dD = dDw = None
        want_det = ctx.needs_input_grad[0] or ctx.needs_input_grad[3]
        # folded mask: one launch runs the detector backward and the descriptor backward's coefficient / transpose blocks
        merged = want_det and desc is not None and desc.fold
        if merged:
            d0, d1 = torch.empty_like(det.saved[0]), torch.empty_like(det.saved[3])
        elif want_det:
            d0, d1 = det_pair_backward(det, g, g)
        if desc is not None:
            if desc.fold:  # the coefficient kernel scales g by lambda_loss itself: no torch kernel here
                dD, dDw = desc_backward(desc, g, lam, 1, det=(det, g, d0, d1) if merged else None)
            else:
                dD, dDw = desc_backward(desc, g * _lam3_vector(lam, g.device))
        return d0, None, None, d1, None, None, dD, dDw, None, None, None, None, None, None


class SparseLossStepFn(torch.autograd.Function):
    """The loss step of the shipped configs (sparse_loss.enable) as ONE autograd node: both detector losses plus the sparse
    descriptor loss on device-sampled lists ia / ib [B, K + Kn] with candidate counts M,
    loss = loss_det + loss_det_warp + lambda_loss * loss_desc (Train_model_heatmap_all.py:333-365, uniform weighting).
    Returns (loss, loss_det, loss_det_warp, loss_desc, pos, neg); only `loss` is differentiable.  The total is formed by
    ssp_sparse_finalize, which also turns it into NaN when an image had no candidate."""

    @staticmethod
    def forward(ctx, semi, labels_2D, mask_2D, semi_w, warped_labels, mask_warp_2D, desc, desc_w, ia, ib, M, K, lamda_d,
                lambda_loss):
        from .sparse import sparse_forward
        det, _ = det_pair_forward(semi, labels_2D, mask_2D, semi_w, warped_labels, mask_warp_2D, True)
        sp = sparse_forward(desc, desc_w, ia, ib, K, ia.shape[1] - K, lamda_d)
        total = torch.empty((1,), dtype=torch.float32, device=semi.device)
        call("ssp_sparse_finalize", ptr(M), M.shape[0], ptr(sp.out3), ptr(det.out[0]), ptr(det.out[1]), float(lambda_loss),
             ptr(total), stream_of(total))
        ctx.det, ctx.sparse, ctx.lambda_loss = det, sp, float(lambda_loss)
        outs = (det.out[0, 0], det.out[1, 0], sp.out3[0], sp.out3[1], sp.out3[2])
        ctx.mark_non_differentiable(*outs)
        ctx.set_materialize_grads(False)
        return (total[0],) + outs

    @staticmethod
    @once_differentiable
    def backward(ctx, g, *_unused):
        from .sparse import sparse_backward
        if g is None:
            return (None,) * 14
        g = f32c(g.reshape(1), g.device)
        d0 = d1 = dD = dDw = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[3]:
            d0, d1 = det_pair_backward(ctx.det, g, g)
        if ctx.needs_input_grad[6] or ctx.needs_input_grad[7]:
            dD, dDw = sparse_backward(ctx.sparse, g * _lam3_vector(ctx.lambda_loss, g.device))
        return d0, None, None, d1, None, None, dD, dDw, None, None, None, None, None, None


# ------------------------------------------------------------------------------------------------
class LazyPairMask(object):
    """The [B,Hc,Wc,Hc,Wc] float correspondence mask of descriptor_loss (utils/utils.py:854-860), built only
    when somebody looks at it: the reference's single caller never does, and at B=32 it is 184 MB."""

    def __init__(self, wpts, B, Hc, Wc, cell, dist):
        self._wpts, self._geom, self._t = wpts, (B, Hc, Wc, cell, dist), None

    @property
    def shape(self):
        B, Hc, Wc, _, _ = self._geom
        return torch.Size((B, Hc, Wc, Hc, Wc))

    def materialize(self):
        if self._t is None:
            B, Hc, Wc, cell, dist = self._geom
            m = torch.empty((B, Hc * Wc, Hc * Wc), dtype=torch.float32, device=self._wpts.device)
            call("ssp_desc_pair_mask", ptr(self._wpts), B, Hc, Wc, cell, dist, ptr(m), stream_of(m))
            self._t = m.view(B, Hc, Wc, Hc, Wc)
        return self._t

    def __getattr__(self, name):  # anything else behaves like the tensor
        return getattr(self.materialize(), name)

    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        conv = lambda a: a.materialize() if isinstance(a, LazyPairMask) else a
        return func(*[conv(a) for a in args], **{k: conv(v) for k, v in (kwargs or {}).items()})
