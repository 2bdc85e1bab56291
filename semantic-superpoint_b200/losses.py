"""autograd.Functions that drive the detector-loss and dense descriptor-loss kernels through the C ABI.

reference: Train_model_heatmap_all.py:155-179 (detector_loss), utils/utils.py:779-893 (descriptor_loss).
Multi-GPU (SURVEY 8e): both losses use GLOBAL-batch normalisers, so with `dist_group` set the local
numerators / mask sums are exchanged by ONE peer-memory kernel (dist.LossExchange, csrc/exchange.cu) that rewrites
the loss scalars and normalisers in place, stream ordered, before the forward returns; the backward kernels
scale by the global normaliser.
"""
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
_SAME = object()  # marker: "second gradient == first gradient" (no stack / cat kernels)


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
class DetectorLossFn(torch.autograd.Function):
    """loss = sum_cells mask * sum_c BCE(softmax(semi)_c, target_c) / (sum mask + 1e-5)

    fused2d=False: target [B,65,Hc,Wc], mask [B,Hc,Wc]  (reference signature)
    fused2d=True : target = labels_2D [B,1,H,W], mask = mask_2D [B,1,H,W] (labels2Dto3D + getMasks fused)
    """

    @staticmethod
    def forward(ctx, semi, target, mask, fused2d, dist_group=None):
        _lib.require_cuda(semi)
        dev = semi.device
        x = f32c(semi.detach(), dev)
        t = f32c(target.detach(), dev)
        m = f32c(mask.detach(), dev)
        B, C, Hc, Wc = x.shape
        if C != 65:
            raise RuntimeError("detector_loss: input must have 65 channels, got %d" % C)
        if fused2d:
            if t.numel() != B * Hc * Wc * 64 or m.numel() != B * Hc * Wc * 64:
                raise RuntimeError("detector_loss_2d: labels_2D / mask_2D must be [B,1,8Hc,8Wc]")
        else:
            if t.shape != x.shape or m.numel() != B * Hc * Wc:
                raise RuntimeError("detector_loss: target must be [B,65,Hc,Wc] and mask [B,Hc,Wc]")
        out3 = torch.empty((3,), dtype=torch.float32, device=dev)
        nbytes = _lib.load().ssp_detector_loss_ws_bytes(B, Hc, Wc)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        call("ssp_detector_loss_fwd", ptr(x), ptr(t), ptr(m), B, Hc, Wc, 1 if fused2d else 0, ptr(out3), ptr(ws),
             nbytes, stream_of(x))
        ctx.save_for_backward(x, t, m)
        ctx.out3 = out3  # attribute, not a saved tensor (the exchange rewrites it in place)
        ctx.fused2d = fused2d
        if dist_group is not None:
            from .dist import globalize_detector
            globalize_detector(out3, dist_group)
        return out3[0]

    @staticmethod
    @once_differentiable
    def backward(ctx, gout):
        x, t, m = ctx.saved_tensors
        out3 = ctx.out3
        B, C, Hc, Wc = x.shape
        g = f32c(gout.reshape(1), x.device)
        dsemi = torch.empty_like(x)
        call("ssp_detector_loss_bwd", ptr(x), ptr(t), ptr(m), B, Hc, Wc, 1 if ctx.fused2d else 0, ptr(out3), ptr(g),
             ptr(dsemi), stream_of(x))
        return dsemi, None, None, None, None


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
        ctx.out3 = out3  # attribute, see DetectorLossFn
        if dist_group is not None:
            from .dist import globalize_semantic
            globalize_semantic(out3, dist_group)
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


class DetectorLossPairFn(torch.autograd.Function):
    """Both detector losses of a training pair (image, warped image) in ONE launch each way, plus getMasks() of the
    warped mask as a by-product (it is the descriptor loss's mask_valid).  Returns (loss, loss_warp, cell_mask_warp)."""

    @staticmethod
    def forward(ctx, semi, target, mask, semi_w, target_w, mask_w, fused2d, dist_group=None):
        _lib.require_cuda(semi, semi_w)
        dev = semi.device
        x0, t0, m0 = f32c(semi.detach(), dev), f32c(target.detach(), dev), f32c(mask.detach(), dev)
        x1, t1, m1 = f32c(semi_w.detach(), dev), f32c(target_w.detach(), dev), f32c(mask_w.detach(), dev)
        B, C, Hc, Wc = x0.shape
        if C != 65 or x1.shape != x0.shape:
            raise RuntimeError("detector_loss: inputs must be two [B,65,Hc,Wc] tensors of the same shape")
        n2d = B * Hc * Wc * 64
        for t, m in ((t0, m0), (t1, m1)):
            ok = (t.numel() == n2d and m.numel() == n2d) if fused2d else (t.shape == x0.shape and m.numel() == B * Hc * Wc)
            if not ok:
                raise RuntimeError("detector_loss: target / mask shapes do not match the logits")
        out = torch.empty((2, 3), dtype=torch.float32, device=dev)
        cellmask = torch.empty((B, Hc, Wc), dtype=torch.float32, device=dev)
        per = (_lib.load().ssp_detector_loss_ws_bytes(B, Hc, Wc) + 15) // 16 * 16
        ws = torch.empty((2 * per,), dtype=torch.uint8, device=dev)
        call("ssp_detector_loss_fwd_pair", ptr(x0), ptr(t0), ptr(m0), ptr(x1), ptr(t1), ptr(m1), B, Hc, Wc,
             1 if fused2d else 0, ptr(out[0]), ptr(out[1]), ptr(cellmask), ptr(ws), 2 * per, stream_of(x0))
        ctx.save_for_backward(x0, t0, m0, x1, t1, m1)
        ctx.out = out  # see DetectorLossFn
        ctx.fused2d = fused2d
        ctx.mark_non_differentiable(cellmask)
        if dist_group is not None:
            from .dist import get_exchange
            get_exchange(dist_group).run(det0=out[0], det1=out[1])
        return out[0, 0], out[1, 0], cellmask

    @staticmethod
    @once_differentiable
    def backward(ctx, g0, g1, _gm):
        x0, t0, m0, x1, t1, m1 = ctx.saved_tensors
        out = ctx.out
        B, C, Hc, Wc = x0.shape
        dev = x0.device
        if g1 is _SAME:  # fused step: both losses share one upstream gradient scalar
            g = f32c(g0.reshape(1), dev).expand(2)
        else:
            zero = torch.zeros((), dtype=torch.float32, device=dev)
            g = torch.stack([(a if a is not None else zero).reshape(()).to(torch.float32) for a in (g0, g1)]).contiguous()
        d0, d1 = torch.empty_like(x0), torch.empty_like(x1)
        call("ssp_detector_loss_bwd_pair", ptr(x0), ptr(t0), ptr(m0), ptr(x1), ptr(t1), ptr(m1), B, Hc, Wc,
             1 if ctx.fused2d else 0, ptr(out[0]), ptr(out[1]), ptr(g[0:1]), ptr(g[1:2]) if g1 is not _SAME else ptr(g[0:1]),
             ptr(d0), ptr(d1), stream_of(x0))
        return d0, None, None, d1, None, None, None, None


# ------------------------------------------------------------------------------------------------
def _nc_pad(nc):
    return (nc + 255) // 256 * 256


class DescriptorLossFn(torch.autograd.Function):
    """Dense descriptor hinge loss.  Returns (loss_desc, pos_sum, neg_sum, wpts); the three scalars are
    differentiable w.r.t. descriptors and descriptors_warped, wpts (warped cell centres) is not."""

    @staticmethod
    def forward(ctx, D, Dw, Hm, mv, cell, lamda, dist, engine, dist_group=None, debug_S=None, fold_alpha=False, step_total=None):
        # step_total (LossStepFn only): (det_out [2,3], lambda_loss, total [1]) -- the finalize kernel also writes the weighted
        # sum of the fused step, so no torch add / mul kernels are needed for it
        lib = _lib.load()
        dev = D.device
        Dc = f32c(D.detach(), dev)
        Dwc = f32c(Dw.detach(), dev)
        if Dc.shape != Dwc.shape:
            raise RuntimeError("descriptor_loss: descriptor shapes differ")
        B, Dch, Hc, Wc = Dc.shape
        Nc = Hc * Wc
        Ncp = _nc_pad(Nc)
        st = stream_of(Dc)
        mpos, mneg = 1.0, 0.2  # hard-coded in the reference (utils/utils.py:817-818)
        if engine not in _ENGINES:
            raise ValueError("descriptor engine must be one of %s" % (_ENGINES,))
        if Dch != 256:
            engine = "fp32"  # the tcgen05 kernels are specialised for 256 channels
        need_grad = bool(ctx.needs_input_grad[0] or ctx.needs_input_grad[1])
        split = engine == "bf16x3"
        # "fold": the (binary) mask is folded into the indicator words, the dD GEMM runs on the forward planes of Dw and
        # the backward needs no pack pass.  Exact only for a 0/1 mask and g_neg = 0 (LossStepFn guarantees the latter);
        # a non-binary mask poisons the normaliser with NaN in the geometry kernel (loud, no sync).
        fold_alpha = bool(fold_alpha and need_grad and engine != "fp32")

        wpts = torch.empty((B, Ncp, 2), dtype=torch.float32, device=dev)
        mv_pad = torch.empty((B, Ncp), dtype=torch.float32, device=dev)
        mvbits = torch.empty((B, Ncp // 32), dtype=torch.int32, device=dev) if fold_alpha else None
        nmv = lib.ssp_desc_geometry_nblocks(B, Nc)
        mv_part = torch.empty((nmv,), dtype=torch.float64, device=dev)
        mask2d = None
        if isinstance(mv, tuple):  # ("2d", mask [B,1,8Hc,8Wc]): LossStepFn -- getMasks is fused into the geometry kernel
            mask2d, mv = mv[1], None
        geom_args = (ptr(Hm), ptr(mv), ptr(mask2d), cell, ptr(wpts), ptr(mv_pad), ptr(mv_part), ptr(mvbits))
        if engine == "fp32":
            call("ssp_desc_geometry", geom_args[0], geom_args[1], geom_args[2], B, Hc, Wc, *geom_args[3:], st)
        # tensor-core engines: the geometry blocks ride in the operand pack's launch (independent work, one launch instead of two)

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
        planes = None
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
        if split:
            # bf16x3: the positive pairs read the packed hi/lo planes (2 x 512 contiguous bytes per cell instead of 256
            # strided channels), so they run right after the pack, in front of the tensor-core kernel
            call("ssp_desc_pack2_geometry", ptr(Dc), ptr(Dwc), B, Dch, Hc, Wc, ptr(Ahi), ptr(Alo), ptr(Bhi), ptr(Blo), *geom_args, st)
            call("ssp_desc_pos_fwd_planes", ptr(Ahi), ptr(Alo), ptr(Bhi), ptr(Blo), ptr(wpts), ptr(mv_pad), B, Hc, Wc, cell,
                 dist, lamda, mpos, mneg, ptr(pos_part), ptr(rowcol), ptr(rowdot), ptr(colcnt), ptr(colrow), ptr(coldot), st)
            # bitsC (the column-orientation indicator words) is only read by the backward GEMM: it is transposed from bitsR by
            # extra blocks of the backward's coefficient launch, not here
            call("ssp_desc_dense_fwd_tc", ptr(Ahi), ptr(Alo), ptr(Bhi), ptr(Blo), ptr(mv_pad), ptr(mvbits), B, Hc, Wc, mneg,
                 ptr(neg_part), ptr(bitsR), None, ptr(debug_S), st)
            planes = (Ahi, Alo, Bhi, Blo)
        else:
            # the HBM-bound exact positive-pair kernel overlaps the pack + tensor-core kernels
            if engine != "fp32":  # single-pass bf16: pack + geometry first (the positive-pair kernel needs the warped points)
                call("ssp_desc_pack2_geometry", ptr(Dc), ptr(Dwc), B, Dch, Hc, Wc, ptr(Ahi), None, ptr(Bhi), None, *geom_args, st)
            with _Fork(dev) as fork:
                call("ssp_desc_pos_fwd", ptr(Dc), ptr(Dwc), ptr(wpts), ptr(mv_pad), B, Hc, Wc, Dch, cell, dist, lamda, mpos,
                     mneg, ptr(pos_part), ptr(rowcol), ptr(rowdot), ptr(colcnt), ptr(colrow), ptr(coldot), stream_of(Dc))
            if engine == "fp32":
                call("ssp_desc_dense_fwd_simt", ptr(Dc), ptr(Dwc), ptr(mv_pad), B, Hc, Wc, Dch, mneg, ptr(neg_part),
                     ptr(bitsR), ptr(bitsC), ptr(debug_S), st)
            else:
                call("ssp_desc_dense_fwd_tc", ptr(Ahi), None, ptr(Bhi), None, ptr(mv_pad), ptr(mvbits), B, Hc, Wc, mneg,
                     ptr(neg_part), ptr(bitsR), None, ptr(debug_S), st)
                planes = (Ahi, None, Bhi, None)
            fork.join()

        if step_total is not None:
            det_out, lam_loss, total = step_total[:3]
            if len(step_total) > 3 and step_total[3] is not None:
                step_total[3].join()  # the detector losses ran on a forked stream (LossStepFn)
            call("ssp_desc_finalize", ptr(pos_part), npos, ptr(neg_part), nneg, ptr(mv_part), nmv, B, Hc, Wc, ptr(overflow),
                 ptr(out8), ptr(det_out[0]), ptr(det_out[1]), float(lam_loss), ptr(total), st)
        else:
            call("ssp_desc_finalize", ptr(pos_part), npos, ptr(neg_part), nneg, ptr(mv_part), nmv, B, Hc, Wc, ptr(overflow),
                 ptr(out8), None, None, 0.0, None, st)
        if CHECK_LIST_OVERFLOW and int(overflow[0]) != 0:  # host sync: debugging / tests only (the NaN above is the product signal)
            raise RuntimeError("descriptor_loss: %d positive pairs overflowed the sparse lists" % int(overflow[0]))
        if dist_group is not None:
            from .dist import globalize_descriptor
            globalize_descriptor(out8, B, Hc, Wc, dist_group)

        if need_grad:
            ctx.save_for_backward(Dc, Dwc, mv_pad, bitsR, bitsC, lists_i, lists_f,
                                  *([p for p in planes if p is not None] if planes else []))
            ctx.out8 = out8  # see DetectorLossFn
        ctx.meta = (B, Dch, Hc, Wc, cell, lamda, dist, mpos, engine, planes is not None and planes[1] is not None)
        ctx.fold_alpha = fold_alpha
        ctx.mark_non_differentiable(wpts)
        return out8[0], out8[1], out8[2], wpts

    @staticmethod
    @once_differentiable
    def backward(ctx, g_loss, g_pos, g_neg, _g_wpts):
        saved = ctx.saved_tensors
        Dc, Dwc, mv_pad, bitsR, bitsC, lists_i, lists_f = saved[:7]
        out8 = ctx.out8
        B, Dch, Hc, Wc, cell, lamda, dist, mpos, engine, split = ctx.meta
        dev = Dc.device
        Nc = Hc * Wc
        Ncp = _nc_pad(Nc)
        st = stream_of(Dc)
        tc_engine = engine != "fp32"
        fold = tc_engine and getattr(ctx, "fold_alpha", False)
        gscale, gmode = 1.0, 0
        if g_pos is _SAME:  # fused step: g_loss is the upstream gradient of the step total (one element), to be scaled by lambda_loss
            lam = float(getattr(ctx, "gscale", 1.0))
            if fold:
                g3, gscale, gmode = g_loss, lam, 1  # the coefficient kernel applies the scale itself: no torch kernel here
            else:
                key = (dev.index, lam)
                if key not in _lam3:
                    _lam3[key] = torch.tensor([lam, 0.0, 0.0], dtype=torch.float32, device=dev)
                g3 = g_loss * _lam3[key]
        else:
            zero = torch.zeros((), dtype=torch.float32, device=dev)
            g3 = torch.stack([(g if g is not None else zero).reshape(()).to(torch.float32) for g in (g_loss, g_pos, g_neg)])
            g3 = g3.contiguous()
        # alpha[b,c] = (g_loss * mv[c] + g_neg) / norm: coefficient of the negative hinge of column c; srow = alpha at mv = 1
        # (row scale of the folded backward).  Folded: both come out of the coefficient kernel below.
        alpha = torch.empty((B, Ncp), dtype=torch.float32, device=dev)
        srow = torch.empty((B, Ncp), dtype=torch.float32, device=dev) if fold else None
        if not fold:
            call("ssp_desc_alpha", ptr(mv_pad), ptr(g3), ptr(out8), B, Ncp, ptr(alpha), None, st)
        rowcol, colrow, colcnt = lists_i[0], lists_i[1], lists_i[2]
        rowdot, coldot = lists_f[0], lists_f[1]
        coefs = torch.empty((2,) + tuple(rowdot.shape), dtype=torch.float32, device=dev)
        colrow_sorted = torch.empty_like(colrow)  # the saved lists stay as the forward wrote them (retain_graph safe)
        dD = torch.empty_like(Dc)
        dDw = torch.empty_like(Dwc)
        if tc_engine:
            if split:
                Ahi, Alo, Bhi, Blo = saved[7:11]
            else:
                (Ahi, Bhi), Alo, Blo = saved[7:9], None, None
            if not fold:
                PS = torch.empty((2 if split else 1, B, Ncp, Dch), dtype=torch.bfloat16, device=dev)
                Shi, Slo = PS[0], (PS[1] if split else None)
        # dD [b,:,r] = sum_c I[r,c] alpha[c] Dw[b,:,c] + sum_n rowcoef[r,n] Dw[b,:,rowcol[r,n]]
        # dDw[b,:,c] = alpha[c] sum_r I[r,c] D[b,:,r]  + sum_n colcoef[c,n] D [b,:,colrow[c,n]]
        # tensor-core engines: both GEMMs run in ONE persistent launch, the positive pairs are applied inside the GEMM
        # epilogues (dedicated epilogue warps hide the gathers behind the next item's main loop);
        # fp32 engine: one streaming apply kernel after the GEMMs.
        # stream plan:  [pos_coef]  ||  [pack(alpha * Dw), unless folded]  ->  GEMM pair
        if fold:
            # bitsR / bitsC already exclude the columns with mask_valid = 0: dD = s * (I' @ Dw) on the forward planes, s = g_loss / norm
            det_job = getattr(ctx, "det_job", None)
            if det_job is not None:
                # fused step: the detector-loss backward of both images rides in the same launch (heterogeneous blocks)
                x0, t0, m0, x1, t1, m1, dout, dg, d0, d1 = det_job
                call("ssp_step_bwd_prologue", ptr(x0), ptr(t0), ptr(m0), ptr(x1), ptr(t1), ptr(m1), B, Hc, Wc, ptr(dout[0]),
                     ptr(dout[1]), ptr(dg), ptr(d0), ptr(d1),
                     ptr(rowcol), ptr(rowdot), ptr(colcnt), ptr(colrow), ptr(coldot), ptr(bitsR), ptr(mv_pad), ptr(g3), gscale,
                     gmode, ptr(out8), lamda, mpos, ptr(coefs[0]), ptr(colrow_sorted), ptr(coefs[1]), ptr(alpha), ptr(srow),
                     ptr(bitsC), st)
            else:
                call("ssp_desc_pos_coef", ptr(rowcol), ptr(rowdot), ptr(colcnt), ptr(colrow), ptr(coldot), ptr(bitsR),
                     ptr(mv_pad), ptr(g3), gscale, gmode, ptr(out8), B, Ncp, lamda, mpos, ptr(coefs[0]), ptr(colrow_sorted),
                     ptr(coefs[1]), ptr(alpha), ptr(srow), ptr(bitsC), Nc, st)
            call("ssp_desc_bits_gemm_tc_pair",
                 ptr(bitsR), ptr(Bhi), ptr(Blo), ptr(srow), ptr(rowcol), ptr(coefs[0]), ptr(Bhi), ptr(Blo), ptr(dD),
                 ptr(bitsC), ptr(Ahi), ptr(Alo), ptr(alpha), ptr(colrow_sorted), ptr(coefs[1]), ptr(Ahi), ptr(Alo), ptr(dDw),
                 B, Nc, st)
        elif tc_engine:
            with _Fork(dev) as f1:
                call("ssp_desc_pos_coef", ptr(rowcol), ptr(rowdot), ptr(colcnt), ptr(colrow), ptr(coldot), ptr(bitsR),
                     ptr(mv_pad), ptr(g3), gscale, gmode, ptr(out8), B, Ncp, lamda, mpos, ptr(coefs[0]), ptr(colrow_sorted),
                     ptr(coefs[1]), None, None, ptr(bitsC), Nc, stream_of(Dc))
            call("ssp_desc_pack", ptr(Dwc), ptr(alpha), B, Dch, Nc, ptr(Shi), ptr(Slo), st)
            f1.join()
            # positive-pair partners from the packed planes of the forward (Dw for dD, D for dDw)
            call("ssp_desc_bits_gemm_tc_pair",
                 ptr(bitsR), ptr(Shi), ptr(Slo), None, ptr(rowcol), ptr(coefs[0]), ptr(Bhi), ptr(Blo), ptr(dD),
                 ptr(bitsC), ptr(Ahi), ptr(Alo), ptr(alpha), ptr(colrow_sorted), ptr(coefs[1]), ptr(Ahi), ptr(Alo), ptr(dDw),
                 B, Nc, st)
        else:
            with _Fork(dev) as f1:
                call("ssp_desc_pos_coef", ptr(rowcol), ptr(rowdot), ptr(colcnt), ptr(colrow), ptr(coldot), ptr(bitsR),
                     ptr(mv_pad), ptr(g3), gscale, gmode, ptr(out8), B, Ncp, lamda, mpos, ptr(coefs[0]), ptr(colrow_sorted),
                     ptr(coefs[1]), None, None, None, 0, stream_of(Dc))
            call("ssp_desc_bits_gemm_simt", ptr(bitsR), ptr(Dwc), ptr(alpha), None, None, None, None, B, Dch, Nc, ptr(dD), st)
            call("ssp_desc_bits_gemm_simt", ptr(bitsC), ptr(Dc), None, ptr(alpha), None, None, None, B, Dch, Nc, ptr(dDw), st)
            f1.join()
            call("ssp_desc_pos_apply", ptr(rowcol), ptr(coefs[0]), ptr(colrow_sorted), ptr(coefs[1]), ptr(Dc), ptr(Dwc), B, Dch, Nc, 0,
                 ptr(dD), ptr(dDw), st)
        return dD, dDw, None, None, None, None, None, None, None, None, None, None


# ------------------------------------------------------------------------------------------------
class _Ctx(object):
    """Stand-in for the autograd context so LossStepFn can run the bodies of the two Functions above."""

    def __init__(self, needs):
        self.needs_input_grad = needs
        self.saved_tensors = ()

    def save_for_backward(self, *tensors):
        self.saved_tensors = tensors

    def mark_non_differentiable(self, *tensors):
        pass


_lam3 = {}


class LossStepFn(torch.autograd.Function):
    """The whole loss step (Train_model_heatmap_all.py:295-365, uniform weighting) as ONE autograd node:
    loss = loss_det + loss_det_warp + lambda_loss * loss_desc.  Same kernels as DetectorLossPairFn + DescriptorLossFn;
    what disappears is the dozen 2-microsecond torch kernels (scalar mul / add, ones_like, zeros, stack) that autograd
    needs to route three scalars through two nodes -- 7 % of a 0.45 ms step.
    Returns (loss, loss_det, loss_det_warp, loss_desc, pos, neg); only `loss` is differentiable."""

    @staticmethod
    def forward(ctx, semi, labels_2D, mask_2D, semi_w, warped_labels, mask_warp_2D, desc, desc_w, Hm, lamda_d, dist,
                lambda_loss, engine, dist_group=None):
        c1 = _Ctx((ctx.needs_input_grad[0], False, False, ctx.needs_input_grad[3], False, False, False, False))
        B, _, Hc, Wc = semi.shape
        dev = semi.device
        # The two detector losses (HBM-bound, + their one-block finalize) run on a forked stream next to the first half of
        # the descriptor chain (geometry -> pack -> positive pairs: a mix of HBM- and latency-bound kernels): nothing there
        # needs them except the cell mask of the warped valid mask, which the geometry kernel computes itself (getMasks fused
        # in).  The streams join in front of desc_finalize, which reads both detector triples for the step total.
        fork = _Fork(dev)
        with fork:
            l0, l1, _cm = DetectorLossPairFn.forward(c1, semi, labels_2D, mask_2D, semi_w, warped_labels, mask_warp_2D, True)
        mw = f32c(mask_warp_2D.detach(), dev)
        if mw.numel() != B * Hc * Wc * 64:
            raise RuntimeError("loss_step: mask_warp_2D must be [B,1,%d,%d]" % (Hc * 8, Wc * 8))
        c2 = _Ctx((ctx.needs_input_grad[6], ctx.needs_input_grad[7]) + (False,) * 8)
        total = torch.empty((1,), dtype=torch.float32, device=dev)
        # fold_alpha=True: the cell mask is folded into the indicator words of the tensor-core engines, so the backward needs
        # no pack pass (measured: 0.339 -> 0.330 ms per step).  Fold requires a binary mask and g_neg = 0; the latter holds
        # because only `loss` is differentiable, and a non-binary mask turns the loss into NaN.  A soft mask belongs on
        # fused=False, whose descriptor_loss packs alpha * Dw into its own planes.
        ld, pos, neg, _wpts = DescriptorLossFn.forward(c2, desc, desc_w, Hm, ("2d", mw), 8, lamda_d, dist, engine,
                                                       None, None, True, (c1.out, lambda_loss, total, fork))
        if dist_group is not None:
            # multi-GPU: ONE exchange kernel turns the three local results into global-batch values in place (the scalars
            # above are views of c1.out / c2.out8) and rewrites the weighted total; the backward kernels read the global
            # normalisers from the same buffers
            from .dist import get_exchange
            get_exchange(dist_group).run(det0=c1.out[0], det1=c1.out[1], desc8=c2.out8, B_local=B, Hc=Hc, Wc=Wc,
                                         lambda_loss=lambda_loss, total=total)
        loss = total[0]
        ctx.c1, ctx.c2, ctx.lambda_loss = c1, c2, float(lambda_loss)
        ctx.mark_non_differentiable(l0, l1, ld, pos, neg)
        ctx.set_materialize_grads(False)  # no zero-filled gradient tensors for the five logging outputs
        return loss, l0, l1, ld, pos, neg

    @staticmethod
    @once_differentiable
    def backward(ctx, g, *_unused):
        if g is None:
            return (None,) * 14
        dev = g.device
        g = f32c(g.reshape(1), dev)
        d0 = d1 = dD = dDw = None
        want_det = ctx.needs_input_grad[0] or ctx.needs_input_grad[3]
        want_desc = ctx.needs_input_grad[6] or ctx.needs_input_grad[7]
        c2 = ctx.c2
        c2.det_job = None
        merged = (want_det and want_desc and getattr(c2, "fold_alpha", False) and c2.meta[8] != "fp32" and ctx.c1.fused2d)
        if merged:
            # one launch for the detector backward and the descriptor backward's coefficient / transpose blocks
            x0, t0, m0, x1, t1, m1 = ctx.c1.saved_tensors
            d0, d1 = torch.empty_like(x0), torch.empty_like(x1)
            c2.det_job = (x0, t0, m0, x1, t1, m1, ctx.c1.out, g, d0, d1)
        elif want_det:
            d0, _, _, d1 = DetectorLossPairFn.backward(ctx.c1, g, _SAME, None)[:4]
        if want_desc:
            c2.gscale = ctx.lambda_loss
            dD, dDw = DescriptorLossFn.backward(c2, g, _SAME, None, None)[:2]
            c2.det_job = None
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
        from .sparse import SparseDescriptorLossFn
        c1 = _Ctx((ctx.needs_input_grad[0], False, False, ctx.needs_input_grad[3], False, False, False, False))
        l0, l1, _cm = DetectorLossPairFn.forward(c1, semi, labels_2D, mask_2D, semi_w, warped_labels, mask_warp_2D, True)
        c2 = _Ctx((ctx.needs_input_grad[6], ctx.needs_input_grad[7]) + (False,) * 6)
        ld, pos, neg = SparseDescriptorLossFn.forward(c2, desc, desc_w, ia, ib, K, ia.shape[1] - K, lamda_d)
        total = torch.empty((1,), dtype=torch.float32, device=semi.device)
        call("ssp_sparse_finalize", ptr(M), M.shape[0], ptr(c2.out3), ptr(c1.out[0]), ptr(c1.out[1]), float(lambda_loss),
             ptr(total), stream_of(total))
        ctx.c1, ctx.c2, ctx.lambda_loss = c1, c2, float(lambda_loss)
        ctx.mark_non_differentiable(l0, l1, ld, pos, neg)
        ctx.set_materialize_grads(False)
        return total[0], l0, l1, ld, pos, neg

    @staticmethod
    @once_differentiable
    def backward(ctx, g, *_unused):
        from .sparse import sparse_loss_backward
        if g is None:
            return (None,) * 14
        dev = g.device
        g = f32c(g.reshape(1), dev)
        d0 = d1 = dD = dDw = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[3]:
            d0, _, _, d1 = DetectorLossPairFn.backward(ctx.c1, g, _SAME, None)[:4]
        if ctx.needs_input_grad[6] or ctx.needs_input_grad[7]:
            key = (dev.index, ctx.lambda_loss)
            if key not in _lam3:
                _lam3[key] = torch.tensor([ctx.lambda_loss, 0.0, 0.0], dtype=torch.float32, device=dev)
            dD, dDw = sparse_loss_backward(ctx.c2, g * _lam3[key])
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
