"""Micro-benchmark of the tcgen05 kernels in isolation (CUDA events, 20 launches each, warm L2)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from ssp_b200 import _lib, synth
from ssp_b200._lib import call, ptr, stream_of

B, Hc, Wc, Dch = 32, 30, 40, 256
Nc, Ncp = Hc * Wc, 1280
dev = "cuda"
lib = _lib.load()
D = torch.from_numpy(synth.unit_descriptors(B, Dch, Hc, Wc, 1, smooth=0.3)).to(dev)
Dw = torch.from_numpy(synth.unit_descriptors(B, Dch, Hc, Wc, 2, smooth=0.3)).to(dev)
mv = torch.ones((B, Ncp), device=dev)
PA = torch.empty((2, B, Ncp, Dch), dtype=torch.bfloat16, device=dev)  # hi, lo planes of D (lo above hi)
PB = torch.empty_like(PA)                                             # hi, lo planes of Dw
st = stream_of(D)
call("ssp_desc_pack", ptr(D), None, B, Dch, Nc, ptr(PA[0]), ptr(PA[1]), st)
call("ssp_desc_pack", ptr(Dw), None, B, Dch, Nc, ptr(PB[0]), ptr(PB[1]), st)
nneg = lib.ssp_desc_dense_tc_nblocks(B, Nc)
part = torch.empty((nneg, 2), dtype=torch.float64, device=dev)
bitsR = torch.empty((B, Ncp // 32, Ncp), dtype=torch.int32, device=dev)
bitsC = torch.empty_like(bitsR)
out = torch.empty((B, Dch, Nc), device=dev)
out2 = torch.empty((B, Dch, Nc), device=dev)
maxp = lib.ssp_desc_maxp()
plist = torch.full((B, Ncp, maxp), -1, dtype=torch.int32, device=dev)
plist[:, :Nc, 0] = torch.arange(Nc, device=dev, dtype=torch.int32)[None]
pcoef = torch.ones((B, Ncp, maxp), device=dev)


def fwd(bits=True, split=True):
    call("ssp_desc_dense_fwd_tc", ptr(PA[0]), ptr(PA[1]) if split else None, ptr(PB[0]), ptr(PB[1]) if split else None, ptr(mv), None,
         B, Hc, Wc, 0.2, ptr(part), ptr(bitsR) if bits else None, None, st)


def transpose_bits():
    """bitsC from bitsR the way the backward makes it: the transpose blocks of the coefficient launch (empty pair lists)."""
    nolist = torch.full((B, Ncp, maxp), -1, dtype=torch.int32, device=dev)
    zi, zf = torch.zeros((B, Ncp), dtype=torch.int32, device=dev), torch.zeros((B, Ncp, maxp), device=dev)
    g3, out8 = torch.zeros(3, device=dev), torch.ones(8, device=dev)
    coef, srt = torch.empty((2, B, Ncp, maxp), device=dev), torch.empty_like(nolist)
    call("ssp_desc_pos_coef", ptr(nolist), ptr(zf), ptr(zi), ptr(nolist), ptr(zf), ptr(bitsR), ptr(mv), ptr(g3), 1.0, 0,
         ptr(out8), B, Ncp, 1.0, 1.0, ptr(coef[0]), ptr(srt), ptr(coef[1]), None, None, ptr(bitsC), Nc, st)


def bwd2(pos=True, split=True):
    lo = (lambda t: ptr(t[1])) if split else (lambda t: None)
    pl, pc = (ptr(plist), ptr(pcoef)) if pos else (None, None)
    call("ssp_desc_bits_gemm_tc_pair", ptr(bitsR), ptr(PB[0]), lo(PB), None, pl, pc, ptr(PB[0]), lo(PB), ptr(out),
         ptr(bitsC), ptr(PA[0]), lo(PA), ptr(mv), pl, pc, ptr(PA[0]), lo(PA), ptr(out2), B, Nc, st)


def timeit(name, fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    print("%-44s %8.1f us" % (name, 1e3 * e0.elapsed_time(e1) / n), flush=True)


timeit("fwd x3 bits", lambda: fwd())
timeit("fwd x3 nobits", lambda: fwd(bits=False))
timeit("fwd x1 bits", lambda: fwd(split=False))
fwd()
transpose_bits()
timeit("bwd pair x3 + pos", lambda: bwd2())
timeit("bwd pair x3 no pos", lambda: bwd2(pos=False))
timeit("bwd pair x1 + pos", lambda: bwd2(split=False))
timeit("bwd pair x1 no pos", lambda: bwd2(pos=False, split=False))
