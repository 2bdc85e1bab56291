"""The homography sampler, the parts that need no GPU: the oracle (homography_oracle.sample_homography_np) reproduces the
homographies the live reference drew for the golden fixtures, and the argument checks of ssp_sample_homography and
HomographySampler come before any launch."""
import ctypes

import numpy as np
import pytest
import torch

import homography_oracle as HO

# (fixture, key, draws, np.random seed, 0 = homographies / 1 = inv_homographies, identity first): tests/golden/make_golden.py
GOLDEN_DRAWS = [("warp_points", "H", 3, 1, 0, False), ("inv_warp", "Hinv", 3, 2, 1, False),
                ("valid_mask", "Hinv5", 5, 3, 1, False), ("valid_mask", "Hinv2", 2, 4, 1, False),
                ("combine", "Hwarp", 7, 5, 0, True), ("desc_small", "H", 2, 6, 0, False), ("desc_30x40", "H", 1, 7, 0, False),
                ("warp_labels", "H", 2, 9, 0, False)]


@pytest.mark.parametrize("fixture,key,n,seed,which,identity_first", GOLDEN_DRAWS)
def test_oracle_reproduces_reference_draws(golden, fixture, key, n, seed, which, identity_first):
    want = golden(fixture)[key]
    got = HO.dataset_homographies(n, seed, identity_first=identity_first)[which]
    assert got.dtype == want.dtype and np.array_equal(got, want)


def test_oracle_reproduces_sparse_loss_draws(golden):
    """sparse_loss.npz: rows 0 and 2 are reference draws under seed 17 (row 1 was replaced by a zoom in the fixture)."""
    want = golden("sparse_loss")["H"]
    got = HO.dataset_homographies(3, 17)[0]
    assert np.array_equal(got[[0, 2]], want[[0, 2]])


def test_oracle_vectorised_draws_are_homographies():
    """n > 1 draws each quantity as an array: shapes, and the corners recovered from the inverse are the sampled ones."""
    np.random.seed(0)
    H = HO.sample_homography_np(n=50, **HO.WARP_PARAMS)
    assert H.shape == (50, 3, 3) and np.all(H[:, 2, 2] == 1)
    c = HO.corners(np.linalg.inv(H))
    assert np.all(np.isfinite(c)) and np.abs(c - 0.5).max() < 1.5


def test_sample_argument_errors_without_gpu():
    from ssp_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(16)
    ok = (5, 25, 0.2, 0.2, 0.2, 0.85, 1.57)

    def run(B=4, flags=15, args=ok, group=0, state=p, out=p):
        return lib.ssp_sample_homography(B, flags, *args, group, state, out, p, None)

    assert run(state=None) < 0 and b"null pointer" in lib.ssp_last_error()
    assert run(out=None) < 0 and b"null pointer" in lib.ssp_last_error()
    for B, group in ((0, 0), (-1, 0), (4, -1)):
        assert run(B=B, group=group) < 0 and b"bad sizes" in lib.ssp_last_error()
    assert run(flags=16) < 0 and b"unknown flag bits" in lib.ssp_last_error()
    assert run(args=(0,) + ok[1:]) < 0 and b"n_scales > 0" in lib.ssp_last_error()
    assert run(args=ok[:1] + (0,) + ok[2:]) < 0 and b"n_angles > 0" in lib.ssp_last_error()
    for pr in (0.0, 1.5, float("nan")):
        assert run(args=ok[:5] + (pr, 1.57)) < 0 and b"patch_ratio" in lib.ssp_last_error()
    for sa in (0.0, -0.1, float("inf")):
        assert run(args=ok[:2] + (sa,) + ok[3:]) < 0 and b"scaling amplitude" in lib.ssp_last_error()
    assert run(args=ok[:3] + (0.0,) + ok[4:]) < 0 and b"perspective amplitudes" in lib.ssp_last_error()
    assert run(args=ok[:4] + (float("nan"),) + ok[5:]) < 0 and b"perspective amplitudes" in lib.ssp_last_error()
    assert run(args=ok[:6] + (float("inf"),)) < 0 and b"max_angle" in lib.ssp_last_error()
    # a disabled component's parameters are not looked at
    assert run(flags=8, args=(0, 0, 0.0, 0.0, 0.0, 0.85, float("nan")), state=None) < 0
    assert b"null pointer" in lib.ssp_last_error()


def test_sampler_errors_before_any_launch():
    import ssp_b200 as S
    with pytest.raises(RuntimeError, match="CUDA device"):
        S.HomographySampler(0, "cpu")
    s = S.homography.HomographySampler.__new__(S.homography.HomographySampler)  # no device state: nothing may launch
    with pytest.raises(NotImplementedError, match="allow_artifacts"):
        s.sample(4)
    with pytest.raises(NotImplementedError, match="translation_overflow"):
        s.sample(4, allow_artifacts=True, translation_overflow=0.1)
    with pytest.raises(NotImplementedError, match="shape"):
        s.sample(4, allow_artifacts=True, shape=[240, 320])
    with pytest.raises(ValueError, match="either homographies or sampler"):
        S.step.collate_warped_pair(torch.zeros((1, 1, 16, 16)), [np.zeros((0, 2))])
