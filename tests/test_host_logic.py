"""Host-side logic that needs no GPU: structuring elements, NMS stencils, input generators, drop-in binding,
loud failure without CUDA."""
import hashlib
import types

import numpy as np
import pytest
import torch

import ssp_b200 as S
from ssp_b200 import synth


def test_ellipse_kernel_matches_opencv(golden):
    g = golden("valid_mask")
    for r in range(1, 9):
        assert np.array_equal(S.ellipse_kernel(r), g["ellipse_%d" % r])
    assert S.ellipse_kernel(3).tolist() == [[0, 0, 0, 1, 0, 0], [0, 1, 1, 1, 1, 1], [1] * 6, [1] * 6, [1] * 6, [0, 1, 1, 1, 1, 1]]


def test_box_nms_stencil_size4():
    """SURVEY 8a-a9: with size=4, IoU>0.1 suppresses exactly these |dx|,|dy| offsets."""
    from ssp_b200.utils import _iou_stencil
    st, R = _iou_stencil(4, 0.1, "cpu")
    assert R == 3
    st = st.numpy().reshape(7, 7)
    want = {(0, 1), (0, 2), (0, 3), (1, 0), (1, 1), (1, 2), (1, 3), (2, 0), (2, 1), (2, 2), (3, 0), (3, 1), (0, 0)}
    got = {(abs(dx), abs(dy)) for dy in range(-3, 4) for dx in range(-3, 4) if st[dy + 3, dx + 3]}
    assert got == want


def test_synth_is_bit_reproducible():
    h = hashlib.sha256(synth.uniform((1000,), 7).tobytes()).hexdigest()
    assert h == hashlib.sha256(synth.uniform((1000,), 7).tobytes()).hexdigest()
    u = synth.uniform((4096,), 1)
    assert 0.0 <= u.min() and u.max() < 1.0 and abs(u.mean() - 0.5) < 0.02
    assert float(u[0]) == pytest.approx(float(synth.uniform((1,), 1)[0]))
    d = synth.unit_descriptors(2, 256, 3, 4, 5)
    np.testing.assert_allclose((d.astype(np.float64) ** 2).sum(1), 1.0, atol=1e-6)
    hm = synth.unique_heatmap(24, 32, 3)
    assert len(np.unique(hm)) == 24 * 32
    Hm = synth.sample_homography(np.random.default_rng(0))
    assert Hm.shape == (3, 3) and abs(Hm[2, 2] - 1.0) < 0.2 and abs(np.linalg.det(Hm)) > 0.1


def test_dropin_binds_and_restores():
    fake = types.ModuleType("fake_utils")
    fake.descriptor_loss = lambda *a, **k: "ref"
    fake.warp_points = lambda *a, **k: "ref"

    class Trainer:
        def detector_loss(self, *a, **k):
            return "ref"

    bound = S.dropin.install(utils_module=fake, trainer_class=Trainer)
    assert fake.descriptor_loss is S.utils.descriptor_loss and fake.labels2Dto3D is S.utils.labels2Dto3D
    assert any(b.endswith("detector_loss") for b in bound)
    # dataset-side names: ours in the main process, the reference's own function inside a DataLoader worker (no CUDA there)
    assert fake.warp_points.__wrapped__ is S.utils.warp_points
    import torch.utils.data as tud
    orig_info = tud.get_worker_info
    tud.get_worker_info = lambda: object()
    try:
        assert fake.warp_points(torch.zeros(4, 2), torch.eye(3)) == "ref"
    finally:
        tud.get_worker_info = orig_info
    sparse_mod = types.ModuleType("fake_sparse")
    sparse_mod.batch_descriptor_loss_sparse = lambda *a, **k: "ref"
    bound = S.dropin.install(utils_module=fake, sparse_module=sparse_mod)
    assert sparse_mod.batch_descriptor_loss_sparse is S.sparse.batch_descriptor_loss_sparse
    S.dropin.uninstall()
    assert fake.descriptor_loss() == "ref" and Trainer().detector_loss() == "ref" and fake.warp_points() == "ref"
    assert sparse_mod.batch_descriptor_loss_sparse() == "ref"

    # method twins of the inference front-end and the tracker (models/model_wrap.py)
    class Frontend:
        def sample_desc_from_points(self, coarse_desc, pts):
            return "ref"

    class Tracker:
        def nn_match_two_way(self, desc1, desc2, nn_thresh):
            return "ref"

    saved = (Frontend.sample_desc_from_points, Tracker.nn_match_two_way)
    bound = S.dropin.install(utils_module=fake, frontend_class=Frontend, tracker_class=Tracker)
    assert any(b.endswith("sample_desc_from_points") for b in bound) and any(b.endswith("nn_match_two_way") for b in bound)
    assert (Frontend.sample_desc_from_points, Tracker.nn_match_two_way) != saved
    S.dropin.uninstall()
    assert (Frontend.sample_desc_from_points, Tracker.nn_match_two_way) == saved


def test_signatures_mirror_reference():
    import inspect
    sig = inspect.signature(S.descriptor_loss)
    assert list(sig.parameters)[:8] == ["descriptors", "descriptors_warped", "homographies", "mask_valid", "cell_size",
                                        "lamda_d", "device", "descriptor_dist"]
    assert sig.parameters["lamda_d"].default == 250 and sig.parameters["descriptor_dist"].default == 4
    assert any(p.kind == p.VAR_KEYWORD for p in sig.parameters.values())  # **config swallows lambda_d=800
    assert list(inspect.signature(S.inv_warp_image_batch).parameters)[:4] == ["img", "mat_homo_inv", "device", "mode"]
    assert list(inspect.signature(S.warp_points).parameters) == ["points", "homographies", "device"]
    assert list(inspect.signature(S.getPtsFromHeatmap).parameters) == ["heatmap", "conf_thresh", "nms_dist"]
    assert list(inspect.signature(S.box_nms).parameters) == ["prob", "size", "iou", "min_prob", "keep_top_k"]
    assert list(inspect.signature(S.compute_valid_mask).parameters)[:4] == ["image_shape", "inv_homography", "device", "erosion_radius"]
    # Train_model_heatmap_all.sem_loss(self, pred, label, device="cpu")
    sem = inspect.signature(S.utils.sem_loss)
    assert list(sem.parameters)[:3] == ["pred", "label", "device"] and sem.parameters["device"].default == "cpu"
    assert sem.parameters["ignore_index"].default == 133


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_cuda():
    with pytest.raises(RuntimeError, match="no CPU path"):
        S.warp_points(torch.zeros(4, 2), torch.eye(3))
    with pytest.raises(RuntimeError, match="no CPU path"):
        S.descriptor_loss(torch.zeros(1, 256, 4, 4), torch.zeros(1, 256, 4, 4), torch.eye(3)[None])
    with pytest.raises(RuntimeError, match="no CPU path"):
        S.detector_loss(torch.zeros(1, 65, 4, 4), torch.zeros(1, 65, 4, 4), torch.ones(1, 4, 4))
    with pytest.raises(NotImplementedError):
        S.box_nms(torch.zeros(8, 8), 4)


def test_shard_range_covers_everything():
    from ssp_b200.dist import shard_range
    for n in (0, 1, 7, 8, 100):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1


def test_orchestration_call_sequences(monkeypatch):
    """The host side of the loss step with the C library faked out (every entry point recorded, nothing computed): the
    Python orchestration -- buffer shapes, autograd plumbing, engine dispatch, fused / unfused / semantic / sparse variants,
    partial gradients -- runs on a CPU-only box and issues the documented kernel sequence (DESIGN 4.3)."""
    from ssp_b200 import _lib, losses, sparse, step, utils
    calls = []
    for m in (_lib, losses, sparse, utils):
        monkeypatch.setattr(m, "call", lambda name, *a: calls.append(name))
        monkeypatch.setattr(m, "stream_of", lambda t: None)
    monkeypatch.setattr(_lib, "require_cuda", lambda *t: None)
    monkeypatch.setattr(utils, "_cuda_device", lambda device, *t: torch.device("cpu"))

    class NoFork(object):
        def __init__(self, dev):
            pass

        def __enter__(self):
            return self

        def __exit__(self, *exc):
            return False

        def join(self):
            pass

    monkeypatch.setattr(losses, "_Fork", NoFork)
    monkeypatch.setattr(losses, "CHECK_LIST_OVERFLOW", False)  # reads a device counter the fake library never writes
    B, Hc, Wc = 2, 6, 8
    leaf = lambda *shape: torch.randn(*shape).requires_grad_()
    semi, semi_w, D, Dw = leaf(B, 65, Hc, Wc), leaf(B, 65, Hc, Wc), leaf(B, 256, Hc, Wc), leaf(B, 256, Hc, Wc)
    lab, m, H = torch.zeros(B, 1, Hc * 8, Wc * 8), torch.ones(B, 1, Hc * 8, Wc * 8), torch.eye(3).repeat(B, 1, 1)

    def run(loss_keys=("loss",), grad_on=(semi, semi_w, D, Dw), **kw):
        del calls[:]
        for t in (semi, semi_w, D, Dw):
            t.grad = None
            t.requires_grad_(any(t is g for g in grad_on))
        out = step.loss_step(semi, semi_w, D, Dw, lab, lab, m, m, H, **kw)
        sum(out[k] for k in loss_keys).backward()
        for t in (semi, semi_w, D, Dw):
            assert (t.grad is not None) == any(t is g for g in grad_on)
            t.requires_grad_()
        return list(calls)

    fwd = ["ssp_detector_loss_fwd_pair", "ssp_desc_pack2_geometry", "ssp_desc_pos_fwd_planes",
           "ssp_desc_dense_fwd_tc", "ssp_desc_finalize"]
    # one-node fused step: the mask is folded into the indicator words, no pack pass in the backward, both GEMMs in one launch
    # backward of the one-node fused step: detector backward + coefficient / alpha / transpose blocks in ONE launch, then both GEMMs
    assert run() == fwd + ["ssp_step_bwd_prologue", "ssp_desc_bits_gemm_tc_pair"]
    # one side of the step differentiated: no merged launch
    assert run(grad_on=(D, Dw)) == fwd + ["ssp_desc_pos_coef", "ssp_desc_bits_gemm_tc_pair"]
    assert run(grad_on=(semi, semi_w)) == fwd + ["ssp_detector_loss_bwd_pair"]
    # separately differentiable components (reference multi_task_loss weighting): general mask path with the pack pass
    bwd_desc = ["ssp_desc_alpha", "ssp_desc_pos_coef", "ssp_desc_pack", "ssp_desc_bits_gemm_tc_pair"]
    unfused = run(fused=False)
    assert unfused[:5] == fwd and sorted(unfused[5:]) == sorted(bwd_desc + ["ssp_detector_loss_bwd_pair"])
    multi = run(fused=False, loss_keys=("loss_det", "loss_det_warp", "positive_dist", "negative_dist"))
    assert multi[:5] == fwd and sorted(multi[5:]) == sorted(bwd_desc + ["ssp_detector_loss_bwd_pair"])
    assert run(fused=False, grad_on=(D, Dw), loss_keys=("positive_dist", "negative_dist")) == fwd + bwd_desc
    assert [c for c in run(engine="fp32") if "_desc_" in c] == [
        "ssp_desc_geometry", "ssp_desc_pos_fwd", "ssp_desc_dense_fwd_simt", "ssp_desc_finalize", "ssp_desc_alpha",
        "ssp_desc_pos_coef", "ssp_desc_bits_gemm_simt", "ssp_desc_bits_gemm_simt", "ssp_desc_pos_apply"]
    assert "ssp_desc_pos_fwd" in run(engine="bf16") and "ssp_desc_pos_fwd_planes" not in run(engine="bf16")
    sp, sl = leaf(B, 133, Hc, Wc), torch.randint(0, 134, (B, Hc * 8, Wc * 8))
    sem = run(sem_pred=sp, sem=sl, sem_warp_pred=sp, warped_sem=sl)
    assert sem.count("ssp_sem_ce_up8") == 2 and sem.count("ssp_sem_ce_up8_bwd") == 2      # 1/8-resolution logits: fused upsample
    full = leaf(B, 133, Hc * 8, Wc * 8)
    sem = run(sem_pred=full, sem=sl, sem_warp_pred=full, warped_sem=sl)
    assert sem.count("ssp_sem_ce_fwd") == 2 and sem.count("ssp_sem_ce_bwd") == 2          # full-resolution logits
    with pytest.raises(RuntimeError, match="1/8"):
        utils.sem_loss(leaf(B, 133, Hc * 4, Wc * 4), sl)

    # the sparse step on device-sampled lists (a stand-in sampler: the real one refuses a CPU device)
    sampler = object.__new__(sparse.DeviceSampler)
    sampler.device, sampler.state, sampler.last = torch.device("cpu"), torch.zeros(4, dtype=torch.int64), None
    sk = dict(descriptor_loss="sparse", sampler=sampler, num_matching_attempts=7, num_masked_non_matches_per_match=3)
    sfwd = ["ssp_sparse_sample", "ssp_detector_loss_fwd_pair", "ssp_transpose_batched", "ssp_transpose_batched",
            "ssp_sparse_desc_loss_fwd", "ssp_sparse_finalize"]
    sbwd = ["ssp_sparse_desc_loss_bwd", "ssp_transpose_batched", "ssp_transpose_batched"]
    assert run(**sk) == sfwd + ["ssp_detector_loss_bwd_pair"] + sbwd
    assert run(grad_on=(D, Dw), **sk) == sfwd + sbwd
    unfused = run(fused=False, **sk)
    assert unfused[:6] == sfwd and sorted(unfused[6:]) == sorted(sbwd + ["ssp_detector_loss_bwd_pair"])
    assert sampler.last[0].shape == (B, 7 * 4)

    # the descriptors saved for the backward are still checked by autograd for in-place modification
    Dn = D * 1.0
    loss, _mask, _pos, _neg = utils.descriptor_loss(Dn, Dw, H)
    Dn.add_(1.0)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        loss.backward()
