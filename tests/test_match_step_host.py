"""Argument checks of the batched descriptor export (step.match_step, utils.nn_match_two_way_batch) and of its two C-ABI
entry points: they run before any CUDA call, so they hold on a machine without a GPU."""
import ctypes

import pytest
import torch

import ssp_b200 as S
from ssp_b200 import _lib

P1 = ctypes.c_void_p(256)  # any non-null, aligned address: the checks fail before it is dereferenced


def _err():
    return _lib.load().ssp_last_error()


def test_sample_desc_batch_argument_errors():
    lib = _lib.load()
    assert lib.ssp_sample_desc_batch(None, P1, 8, P1, 4, 2, 256, 4, 4, 8, P1, None) < 0
    assert b"null pointer" in _err()
    assert lib.ssp_sample_desc_batch(P1, P1, 8, None, 4, 2, 256, 4, 4, 8, P1, None) < 0  # counts are required
    assert b"null pointer" in _err()
    for bad in ((8, 0, 2), (8, 4, 0), (3, 4, 2)):  # limit <= 0, I <= 0, limit > capacity
        cap, limit, I = bad
        assert lib.ssp_sample_desc_batch(P1, P1, cap, P1, limit, I, 256, 4, 4, 8, P1, None) < 0
        assert b"bad sizes" in _err()


def _nn(**kw):
    a = dict(hi1=P1, lo1=P1, R1=256, hi2=P1, lo2=P1, R2=512, c1=P1, c2=P1, limit=300, P=2, thr=0.7, m=P1, n=P1, ws=P1,
             nbytes=_lib.load().ssp_nn_match_batch_ws_bytes(2, 256, 512))
    a.update(kw)
    return _lib.load().ssp_nn_match_batch(a["hi1"], a["lo1"], a["R1"], a["hi2"], a["lo2"], a["R2"], a["c1"], a["c2"],
                                          a["limit"], a["P"], a["thr"], a["m"], a["n"], a["ws"], a["nbytes"], None)


def test_nn_match_batch_argument_errors():
    lib = _lib.load()
    assert lib.ssp_nn_match_batch_ws_bytes(2, 256, 512) == 2 * (256 + 512) * 8
    for k in ("hi1", "lo2", "c1", "c2", "m", "n", "ws"):
        assert _nn(**{k: None}) < 0, k
        assert b"null pointer" in _err()
    for k, v in (("P", 0), ("R1", 0), ("R2", -256), ("limit", 0)):
        assert _nn(**{k: v}) < 0, k
        assert b"bad sizes" in _err()
    for k, v in (("R1", 300), ("R2", 128)):
        assert _nn(**{k: v}) < 0, k
        assert b"multiples of 256" in _err()
    assert _nn(nbytes=100) < 0
    assert b"workspace too small" in _err()
    assert _nn(thr=-0.1) < 0 and _nn(thr=float("nan")) < 0
    assert b"non-negative" in _err()


def test_match_step_argument_errors():
    semi = torch.zeros((2, 65, 4, 6))
    desc = torch.zeros((2, 256, 4, 6))
    with pytest.raises(ValueError, match="non-negative"):
        S.step.match_step(semi, desc, semi, desc, nn_thresh=-0.5)
    with pytest.raises(ValueError, match="256"):
        S.step.match_step(semi, desc[:, :128], semi, desc[:, :128])
    with pytest.raises(ValueError, match="65"):
        S.step.match_step(semi[:, :64], desc, semi[:, :64], desc)
    with pytest.raises(RuntimeError, match="no CPU path"):
        S.step.match_step(semi, desc, semi, desc)


def test_nn_match_two_way_batch_argument_errors():
    d = torch.zeros((3, 256, 10))
    with pytest.raises(ValueError, match="non-negative"):
        S.utils.nn_match_two_way_batch(d, d, -1.0)
    with pytest.raises(ValueError, match="256"):
        S.utils.nn_match_two_way_batch(d[:, :64], d[:, :64], 0.7)
    with pytest.raises(ValueError):
        S.utils.nn_match_two_way_batch(d, d[:2], 0.7)
    with pytest.raises(RuntimeError, match="no CPU path"):
        S.utils.nn_match_two_way_batch(d, d, 0.7)
