"""world_size-2 gloo test of the only exchange step on the path: the global-batch normalisers of both losses
(SURVEY 8e).  The two ranks hold 3 and 2 of the 5 pairs (uneven shards: the batch size is part of the exchanged
payload); after the exchange every rank must report the loss the oracle computes on the whole batch.  On CPU the
exchange runs its torch.distributed form (one all-reduce); the peer-memory kernel is covered by the -m gpu tests."""
import os
import socket

import numpy as np
import torch
import torch.multiprocessing as mp

from oracle import ssp_oracle as O
from ssp_b200 import synth

B, HC, WC, DCH = 5, 6, 8, 32


def _inputs():
    rng = np.random.default_rng(3)
    Hs = np.stack([np.linalg.inv(synth.sample_homography(rng)) for _ in range(B)]).astype(np.float32)
    D = synth.unit_descriptors(B, DCH, HC, WC, 1, smooth=0.4)
    Dw = synth.unit_descriptors(B, DCH, HC, WC, 2, smooth=0.4)
    mv = (synth.uniform((B, 1, HC, WC), 3) < 0.7).astype(np.float32)
    semi = synth.pseudo_normal((B, 65, HC, WC), 4)
    lab = O.labels2Dto3D(synth.keypoint_labels(B, HC * 8, WC * 8, 5, p=0.02))
    m3 = (synth.uniform((B, HC, WC), 6) < 0.8).astype(np.float32)
    return Hs, D, Dw, mv, semi, lab, m3


def _sem_inputs():
    rng = np.random.default_rng(8)
    lab = rng.integers(0, 134, (B, HC * 8, WC * 8))
    lab[0, :20] = 133  # uneven counts across the two shards
    return synth.pseudo_normal((B, 133, HC, WC), 9) * 2, lab


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    if torch.cuda.is_available():
        # with a CUDA device the default exchange is the peer-memory kernel (covered by the -m gpu tests); this test
        # drives the torch.distributed form with CPU tensors
        os.environ["SSP_EXCHANGE"] = "allreduce"
    import torch.distributed as tdist
    from ssp_b200.dist import (LossExchange, get_exchange, globalize_descriptor, globalize_detector, globalize_semantic,
                               init_from_env, shard_range)
    init_from_env(backend="gloo")
    assert get_exchange(True).backend == "allreduce"  # CPU tensors / gloo: the torch.distributed form of the exchange
    Hs, D, Dw, mv, semi, lab, m3 = _inputs()
    lo, hi = shard_range(B, rank, world)   # B = 5 over 2 ranks: shards of 3 and 2 pairs (uneven on purpose)
    # local shard through the oracle -> the raw sums the kernels would emit (out8 / out3 layouts)
    l, _, p, n = O.descriptor_loss(D[lo:hi], Dw[lo:hi], Hs[lo:hi], mv[lo:hi])
    norm = np.float32(hi - lo) * (mv[lo:hi].sum() + 1) * HC * WC
    out8 = torch.tensor([l, p, n, norm, l * norm, p * norm, n * norm, mv[lo:hi].sum()], dtype=torch.float32)
    globalize_descriptor(out8, hi - lo, HC, WC, True)
    ld = O.detector_loss(semi[lo:hi], lab[lo:hi], m3[lo:hi])
    den = np.float32(m3[lo:hi].sum() + 1e-5)
    out3 = torch.tensor([ld, ld * den, den], dtype=torch.float32)
    globalize_detector(out3, True)
    # the fused step exchanges everything in ONE call: same numbers
    out8d = torch.tensor([l, p, n, norm, l * norm, p * norm, n * norm, mv[lo:hi].sum()], dtype=torch.float32)
    out3d = torch.tensor([ld, ld * den, den], dtype=torch.float32)
    out3e = out3d.clone()
    LossExchange(True).run(det0=out3d, det1=out3e, desc8=out8d, B_local=hi - lo, Hc=HC, Wc=WC)
    assert torch.equal(out8d, out8) and torch.equal(out3d, out3) and torch.equal(out3e, out3)
    # semantic cross entropy: mean over the counted pixels of the global batch
    sl, slab = _sem_inputs()
    ls = O.sem_loss(sl[lo:hi], slab[lo:hi])
    cnt = np.float32((slab[lo:hi] != 133).sum())
    outs = torch.tensor([ls, ls * cnt, cnt], dtype=torch.float32)
    globalize_semantic(outs, True)
    q.put((rank, out8.numpy().copy(), out3.numpy().copy(), outs.numpy().copy()))
    tdist.barrier()
    tdist.destroy_process_group()


def test_global_normalisers_world2():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted(q.get(timeout=120) for _ in range(2))
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    Hs, D, Dw, mv, semi, lab, m3 = _inputs()
    l, _, p, n = O.descriptor_loss(D, Dw, Hs, mv)
    ld = O.detector_loss(semi, lab, m3)
    sl, slab = _sem_inputs()
    for rank, out8, out3, outs in res:
        np.testing.assert_allclose(outs[0], O.sem_loss(sl, slab), rtol=1e-5)
        np.testing.assert_allclose(outs[2], (slab != 133).sum())
        np.testing.assert_allclose(out8[:3], [l, p, n], rtol=1e-5)
        np.testing.assert_allclose(out8[3], B * (mv.sum() + 1) * HC * WC, rtol=1e-6)
        np.testing.assert_allclose(out3[0], ld, rtol=1e-5)
    np.testing.assert_array_equal(res[0][1], res[1][1])  # identical on both ranks
