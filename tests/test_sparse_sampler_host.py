"""The device correspondence sampler of the sparse loss, the parts that need no GPU: the candidate oracle
(sparse_oracle.sparse_candidates) pinned against the live reference's sampled lists and against the product's host sampler,
argument checks of the new C-ABI entry points, and the errors of the sparse loss step that come before any launch."""
import ctypes

import numpy as np
import pytest
import torch

from sparse_oracle import sparse_candidates

TIE_EPS = 1e-3  # cells whose warp lies this close to a rounding tie may round either way in another operation order


def seeded_homographies(n, seed):
    from ssp_b200 import synth
    rng = np.random.default_rng(seed)
    return np.stack([np.linalg.inv(synth.sample_homography(rng)) for _ in range(n)]).astype(np.float32)


def test_candidates_contain_reference_matches(golden):
    """Every (matches_a, matches_b) pair the live reference sampled (tests/golden/sparse_loss.npz, 30x40 cells) is a
    candidate of sparse_candidates, and the distinct sampled pairs of the padded image are all its candidates."""
    g = golden("sparse_loss")
    for i in range(g["H"].shape[0]):
        c = sparse_candidates(g["H"][i], 30, 40)
        assert c["a"].size > 0 and np.array_equal(c["a"], np.sort(c["a"]))
        assert np.array_equal(c["b_all"][c["a"]], c["b"])
        got = c["b_all"][g["matches_a"][i]]
        off = np.unique(g["matches_a"][i][got != g["matches_b"][i]])
        # image 1 has one cell 2e-6 from a tie that the reference's torch matmul rounds the other way
        assert np.all(c["tie"][off] < TIE_EPS) and off.size <= 1, (i, off, c["tie"][off])
        if len(np.unique(g["matches_a"][i])) < 1000:  # M < K: every candidate was drawn
            assert np.array_equal(np.unique(g["matches_a"][i]), c["a"]), i


@pytest.mark.parametrize("Hc,Wc", [(30, 40), (47, 155), (60, 80), (7, 9)])
def test_candidates_equal_host_sampler(Hc, Wc):
    """On seeded homographies the oracle's candidate set equals the one sparse.sample_correspondences (the torch CPU lines
    sparse.py:32-40) keeps: with K above the cell count every candidate is drawn at least once."""
    from ssp_b200 import sparse
    Hs = seeded_homographies(6, 100 + Hc)
    Hs[0] = np.diag([0.3, 0.3, 1.0]).astype(np.float32)  # a shrink: many cells map onto few
    np.random.seed(7)
    torch.manual_seed(7)
    for i, H in enumerate(Hs):
        c = sparse_candidates(H, Hc, Wc)
        ma, mb, _, _ = sparse.sample_correspondences(torch.from_numpy(H), Hc, Wc, Hc * Wc + 1, 0)
        host = {(int(a), int(b)) for a, b in zip(ma.numpy(), mb.numpy())}
        ours = set(zip(c["a"].tolist(), c["b"].tolist()))
        diff = {a for a, _ in host ^ ours}
        assert all(c["tie"][a] < TIE_EPS for a in diff), (i, sorted(diff)[:10])
        assert len(diff) <= 2, (i, len(diff))
        assert np.all(c["bound"][c["a"]] >= c["tie"][c["a"]] - 1e-6)  # a bound of the kept region is a rounding tie


def test_candidates_empty_and_identity():
    c = sparse_candidates(np.eye(3, dtype=np.float32), 30, 40)
    assert np.array_equal(c["a"], np.arange(1200)) and np.array_equal(c["b"], np.arange(1200))
    far = np.array([[1, 0, 5.0], [0, 1, 5.0], [0, 0, 1]], np.float32)  # shifted by 2.5 image widths
    c = sparse_candidates(far, 30, 40)
    assert c["a"].size == 0 and np.all(c["b_all"] == -1)


def test_sample_argument_errors_without_gpu():
    """ssp_sparse_sample and ssp_sparse_finalize validate their arguments before any CUDA call."""
    from ssp_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(16)
    assert lib.ssp_sparse_sample(None, 1, 30, 40, 1000, 10, p, p, p, p, None) < 0
    assert b"null pointer" in lib.ssp_last_error()
    assert lib.ssp_sparse_sample(p, 1, 30, 40, 1000, 10, p, None, p, p, None) < 0
    assert b"null pointer" in lib.ssp_last_error()
    for K, n in ((0, 10), (-3, 10), (1000, -1)):
        assert lib.ssp_sparse_sample(p, 1, 30, 40, K, n, p, p, p, p, None) < 0
        assert b"K > 0 and n >= 0" in lib.ssp_last_error()
    assert lib.ssp_sparse_sample(p, 1, 64, 129, 1000, 10, p, p, p, p, None) < 0  # 8256 cells
    assert b"exceed the supported 8192 cells" in lib.ssp_last_error()
    assert lib.ssp_sparse_sample(p, 0, 30, 40, 1000, 10, p, p, p, p, None) < 0
    assert b"bad sizes" in lib.ssp_last_error()
    assert lib.ssp_sparse_finalize(p, 1, None, None, None, 1.0, None, None) < 0
    assert lib.ssp_sparse_finalize(p, 1, p, None, None, 1.0, p, None) < 0  # a total needs both detector triples
    assert b"null pointer" in lib.ssp_last_error()


def test_sparse_loss_step_errors_before_any_launch():
    import ssp_b200 as S
    x = torch.zeros(1)
    args = (x,) * 9
    with pytest.raises(NotImplementedError, match="one GPU"):
        S.step.loss_step(*args, descriptor_loss="sparse", dist_group=object())
    with pytest.raises(ValueError, match="DeviceSampler"):
        S.step.loss_step(*args, descriptor_loss="sparse")
    with pytest.raises(ValueError, match="'dense' or 'sparse'"):
        S.step.loss_step(*args, descriptor_loss="pixelwise")
    with pytest.raises(RuntimeError, match="CUDA device"):
        S.sparse.DeviceSampler(0, "cpu")
