"""ctypes binding of lib/libssp_b200.so (include/ssp_b200.h).

The product path has no fallback: if the library is missing it is built with nvcc, and if that fails (or a
tensor is not on a CUDA device) the call raises.  Nothing here imports oracle/.
"""
import ctypes
import os
import threading

import torch

from . import build as _build

_c = ctypes
_P = _c.c_void_p
_I = _c.c_int
_F = _c.c_float
_D = _c.c_double
_Z = _c.c_size_t

# name -> (restype, argtypes); mirrors include/ssp_b200.h one to one (tests/test_abi.py checks this)
SIGNATURES = {
    "ssp_version": (_I, []),
    "ssp_last_error": (_c.c_char_p, []),
    "ssp_warp_points_mask": (_I, [_P, _I, _P, _I, _F, _F, _P, _P, _P]),
    "ssp_warp_keypoints_f64": (_I, [_P, _I, _P, _D, _D, _P, _P, _P]),
    "ssp_inv_warp_image": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _I, _P, _P]),
    "ssp_valid_mask": (_I, [_I, _I, _I, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "ssp_labels2d_to_3d": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "ssp_cell_mask": (_I, [_P, _I, _I, _I, _P, _P]),
    "ssp_detector_loss_ws_bytes": (_Z, [_I, _I, _I]),
    "ssp_detector_loss_fwd_pair": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "ssp_detector_loss_bwd_pair": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "ssp_flatten_detection": (_I, [_P, _I, _I, _I, _P, _P]),
    "ssp_flatten_detection_masked": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "ssp_combine_heatmap": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "ssp_combine_heatmap_signed": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "ssp_nms_ws_bytes": (_Z, [_I, _I, _I, _I]),
    "ssp_nms_ws_counts_offset": (_Z, [_I, _I, _I]),
    "ssp_nms_fast": (_I, [_P, _I, _I, _I, _F, _I, _P, _I, _I, _P, _P, _P, _Z, _P]),
    "ssp_soft_argmax_points": (_I, [_P, _I, _I, _I, _P, _I, _P, _I, _I, _P]),
    "ssp_box_nms": (_I, [_P, _I, _I, _I, _F, _I, _P, _P, _P, _Z, _P]),
    "ssp_desc_geometry_nblocks": (_I, [_I, _I]),
    "ssp_desc_pos_nblocks": (_I, [_I, _I]),
    "ssp_desc_maxp": (_I, []),
    "ssp_desc_pos_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _F, _F, _F, _P, _P, _P, _P, _P, _P, _P]),
    "ssp_desc_pos_planes_nblocks": (_I, [_I, _I]),
    "ssp_desc_pos_fwd_planes": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _F, _F, _F, _P, _P, _P, _P, _P, _P, _P]),
    "ssp_desc_dense_simt_nblocks": (_I, [_I, _I]),
    "ssp_desc_dense_fwd_simt": (_I, [_P, _P, _P, _I, _I, _I, _I, _F, _P, _P, _P, _P, _P]),
    "ssp_desc_pack": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "ssp_desc_pack2_geometry": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P]),
    "ssp_desc_dense_tc_nblocks": (_I, [_I, _I]),
    "ssp_desc_dense_fwd_tc": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P, _P, _P, _P]),
    "ssp_desc_finalize": (_I, [_P, _I, _P, _I, _P, _I, _I, _I, _I, _P, _P, _P, _P, _F, _P, _P]),
    "ssp_desc_pair_mask": (_I, [_P, _I, _I, _I, _I, _F, _P, _P]),
    "ssp_desc_alpha": (_I, [_P, _P, _P, _I, _I, _P, _P]),
    "ssp_desc_pos_coef": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _F, _I, _P, _I, _I, _F, _F, _P, _P, _P, _P, _P, _P, _I, _P]),
    "ssp_step_bwd_prologue": (_I, [_P] * 6 + [_I] * 3 + [_P] * 5 + [_P] * 8 + [_F, _I, _P, _F, _F] + [_P] * 7),
    "ssp_desc_pos_apply": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _P]),
    "ssp_desc_bits_gemm_simt": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _P]),
    "ssp_desc_bits_gemm_tc_pair": (_I, [_P] * 18 + [_I, _I, _P]),
    "ssp_sem_ce_ws_bytes": (_Z, [_I, _I, _I, _I, _I]),
    "ssp_sem_ce_fwd": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _Z, _P]),
    "ssp_sem_ce_bwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "ssp_sem_ce_up8": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _Z, _P]),
    "ssp_sem_ce_up8_bwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "ssp_nn_match": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "ssp_sample_desc_batch": (_I, [_P, _P, _I, _P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "ssp_nn_match_batch_ws_bytes": (_Z, [_I, _I, _I]),
    "ssp_nn_match_batch": (_I, [_P, _P, _I, _P, _P, _I, _P, _P, _I, _I, _F, _P, _P, _P, _Z, _P]),
    "ssp_transpose_batched": (_I, [_P, _I, _I, _I, _P, _P]),
    "ssp_sparse_desc_loss_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _F, _F, _P, _P, _P, _P]),
    "ssp_sparse_desc_loss_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _F, _F, _P, _P, _P]),
    "ssp_sparse_sample": (_I, [_P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "ssp_sparse_finalize": (_I, [_P, _I, _P, _P, _P, _F, _P, _P]),
    "ssp_sample_homography": (_I, [_I, _I, _I, _I, _D, _D, _D, _D, _D, _I, _P, _P, _P, _P]),
    "ssp_warp_labels_ws_bytes": (_Z, [_I, _I, _I]),
    "ssp_warp_labels": (_I, [_P, _P, _I, _I, _I, _I, _P, _I, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "ssp_ransac_homography_ws_bytes": (_Z, [_I, _I]),
    "ssp_ransac_homography": (_I, [_P, _I, _P, _I, _P, _P, _I, _I, _I, _D, _I, _D, _c.c_ulonglong] + [_P] * 7 + [_Z, _P]),
    "ssp_eval_repeatability": (_I, [_P, _I, _P, _P, _I, _P, _I, _I, _P, _I, _I, _I, _D, _P, _P]),
    "ssp_eval_match_metrics": (_I, [_P, _I, _P, _P, _I, _P, _I, _I, _P, _I, _I, _P, _P, _I, _D, _P, _P, _P, _I, _P, _I, _P,
                                    _P]),
    "ssp_debug_trace": (_I, [_P]),
    "ssp_debug_trace_cap": (_I, []),
    "ssp_xchg_max_ranks": (_I, []),
    "ssp_xchg_alloc": (_I, [_c.POINTER(_P), _P]),
    "ssp_xchg_open": (_I, [_P, _c.POINTER(_P)]),
    "ssp_xchg_close": (_I, [_P]),
    "ssp_xchg_free": (_I, [_P]),
    "ssp_xchg_status": (_I, [_P, _P]),
    "ssp_loss_exchange": (_I, [_c.POINTER(_P), _I, _I, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P, _D, _P]),
}

_lib = None
_lock = threading.Lock()
launch_count = 0  # kernels-launching C-ABI calls made through this module (bench.py reports it)


def lib_path():
    return _build.LIB_PATH


def load(build_if_missing=True):
    """Load (building first if needed) the shared library and declare every prototype."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB_PATH
        if not os.path.exists(path):
            if not build_if_missing:
                raise RuntimeError("libssp_b200.so is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
            _build.build_library()
        lib = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError = header / library mismatch, fail loudly
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return _lib


def check(rc, what):
    if rc != 0:
        msg = load().ssp_last_error()
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else ""))


# kernels launched per entry point (memsets / copies not counted); the NMS drivers launch init + >= 2 rounds +
# compact + rank, counted at their minimum
KERNELS_PER_CALL = {"ssp_nms_fast": 5, "ssp_box_nms": 4, "ssp_detector_loss_fwd_pair": 2, "ssp_sem_ce_fwd": 2,
                    "ssp_sem_ce_up8": 2, "ssp_nn_match_batch": 2,
                    "ssp_ransac_homography": 2}
kernel_count = 0
_prof = None


def profile_begin():
    """Start bracketing every entry point with CUDA events on the launching (current) stream."""
    global _prof
    _prof = {}


def profile_end():
    """Stop profiling; returns {entry point: (calls, total milliseconds)}."""
    global _prof
    torch.cuda.synchronize()
    out = {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in _prof.items()}
    _prof = None
    return out


def check_arity(name, args):
    """Raise TypeError unless args fits the entry point's SIGNATURES entry.  ctypes rejects too few arguments but passes
    surplus ones on silently: a call site not updated after a parameter was removed would run with its arguments shifted
    by one slot (its stream dropped as the surplus) and no error anywhere."""
    want = len(SIGNATURES[name][1])
    if len(args) != want:
        raise TypeError("%s takes %d arguments, got %d" % (name, want, len(args)))


def call(name, *args):
    """Invoke an int-returning entry point and raise RuntimeError(ssp_last_error()) on failure."""
    global launch_count, kernel_count
    check_arity(name, args)
    launch_count += 1
    kernel_count += KERNELS_PER_CALL.get(name, 1)
    fn = getattr(load(), name)
    if _prof is None:
        check(fn(*args), name)
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = fn(*args)
    e1.record()
    _prof.setdefault(name, []).append((e0, e1))
    check(rc, name)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else _c.c_void_p(t.data_ptr())


def stream_of(t):
    return _c.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "ssp_b200 has no CPU path: got a %s tensor; move inputs to a CUDA device (sm_100a)" % t.device
            )


def f32c(t, device=None):
    """fp32, contiguous, 16-byte aligned view/copy of t (optionally moved to `device`)."""
    if device is not None and t.device != torch.device(device):
        t = t.to(device)
    if t.dtype != torch.float32:
        t = t.float()
    t = t.contiguous()
    if t.data_ptr() % 16:
        t = t.clone()
    return t
