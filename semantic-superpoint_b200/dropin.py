"""Bind the CUDA path over the reference's own callables (SURVEY 8b: the boundary is a set of Python names).

    import sys; sys.path.insert(0, "/path/to/Semantic-SuperPoint")
    import ssp_b200; ssp_b200.dropin.install()
    # from here on `from utils.utils import descriptor_loss` (Train_model_heatmap_all.py:133), labels2Dto3D
    # (:278), inv_warp_image_batch (export.py:40), getPtsFromHeatmap (:698) ... resolve to the sm_100a kernels.

Most reference call sites import late (inside the function body), so patching module attributes before the
first training / export step covers them; `export.py:40` imports at module import, hence `install()` must run
before `import export`.  `install()` returns the list of names it bound; `uninstall()` restores the originals.
"""
import importlib
import sys

from . import utils as _u

# reference attribute -> replacement.
# TRAINER_NAMES are called from the training / export process itself.  DATASET_NAMES are the ones the reference datasets capture
# in `init_var` and call from `__getitem__` (datasets/Coco.py:99-111, Coco_sem.py:120-123, SyntheticDataset_gaussian.py:181,
# data_tools.py:38-40), i.e. inside forked DataLoader workers, where CUDA cannot be initialised: they are bound to wrappers that
# run the CUDA kernel in the main process and hand the call back to the saved reference function inside a worker, so `install()` is safe with `workers_train > 0`.
TRAINER_NAMES = ["labels2Dto3D", "flattenDetection", "getPtsFromHeatmap", "nms_fast", "box_nms", "descriptor_loss", "normPts",
                 "denormPts", "homography_scaling_torch"]
DATASET_NAMES = ["warp_points", "filter_points", "inv_warp_image_batch", "inv_warp_image", "compute_valid_mask"]
UTILS_NAMES = DATASET_NAMES + TRAINER_NAMES
_saved = []


def _in_worker():
    """True inside a DataLoader worker process -- the one place the reference's own CPU function is handed the call back
    (a forked worker cannot create a CUDA context).  Everywhere else the CUDA path runs, and fails loudly without a GPU."""
    import torch.utils.data as tud
    return tud.get_worker_info() is not None


def _worker_safe(ours, theirs):
    """`ours` in the main process, the reference's own CPU function inside DataLoader workers."""
    if theirs is None:
        return ours

    def f(*a, **k):
        return theirs(*a, **k) if _in_worker() else ours(*a, **k)

    f.__name__ = getattr(ours, "__name__", "f")
    f.__doc__ = ours.__doc__
    f.__wrapped__ = ours
    return f


def _bind(obj, name, fn, bound):
    if hasattr(obj, name):
        _saved.append((obj, name, getattr(obj, name)))
    setattr(obj, name, fn)
    bound.append("%s.%s" % (getattr(obj, "__name__", type(obj).__name__), name))


def install(utils_module=None, trainer_class=None, frontend_class=None, export_module=None, tracker_class=None,
            sparse_module=None, data_tools_module=None):
    """Patch `utils.utils` (imported from sys.path unless given) and, when passed, the trainer class
    (`Train_model_heatmap_all`: detector_loss, getMasks, sem_loss), the inference front-end class
    (`SuperPointFrontend_torch`: getPtsFromHeatmap, nms_fast, sample_desc_from_points, soft_argmax_points), the tracker class
    (`PointTracker`: nn_match_two_way), the `export` module (combine_heatmap), `utils.loss_functions.sparse_loss`
    (batch_descriptor_loss_sparse / descriptor_loss_sparse) and `datasets.data_tools` (warpLabels)."""
    bound = []
    if utils_module is None:
        utils_module = importlib.import_module("utils.utils")
    for n in TRAINER_NAMES:
        _bind(utils_module, n, getattr(_u, n), bound)
    for n in DATASET_NAMES:
        _bind(utils_module, n, _worker_safe(getattr(_u, n), getattr(utils_module, n, None)), bound)
    if trainer_class is not None:
        _bind(trainer_class, "detector_loss",
              lambda self, input, target, mask=None, loss_type="softmax": _u.detector_loss(input, target, mask, loss_type), bound)
        _bind(trainer_class, "getMasks",
              lambda self, mask_2D, cell_size, device="cpu": _u.getMasks(mask_2D, cell_size, device), bound)
        _bind(trainer_class, "sem_loss", lambda self, pred, label, device="cpu": _u.sem_loss(pred, label, device), bound)
    if frontend_class is not None:
        _bind(frontend_class, "getPtsFromHeatmap",
              lambda self, heatmap: _u.getPtsFromHeatmap(heatmap, self.conf_thresh, self.nms_dist), bound)
        _bind(frontend_class, "nms_fast",
              lambda self, in_corners, H, W, dist_thresh: _u.nms_fast(in_corners, H, W, dist_thresh), bound)
        _bind(frontend_class, "sample_desc_from_points",
              lambda self, coarse_desc, pts: _u.sample_desc_from_points(coarse_desc, pts, self.cell), bound)

        def _soft_argmax(self, pts, patch_size=5):
            # the reference also keeps its log-patches in self.patches (debug only); that attribute is not produced
            self.pts_subpixel = _u.soft_argmax_points(self.heatmap, pts, patch_size)
            return self.pts_subpixel.copy()

        _bind(frontend_class, "soft_argmax_points", _soft_argmax, bound)
    if tracker_class is not None:  # models/model_wrap.py PointTracker

        def _nn(self, desc1, desc2, nn_thresh):
            self.mscores = _u.nn_match_two_way(desc1, desc2, nn_thresh)   # the reference keeps the matches here too
            return self.mscores

        _bind(tracker_class, "nn_match_two_way", _nn, bound)
    if sparse_module is None:
        sparse_module = sys.modules.get("utils.loss_functions.sparse_loss")
    if sparse_module is not None:
        from . import sparse as _sp
        _bind(sparse_module, "batch_descriptor_loss_sparse", _sp.batch_descriptor_loss_sparse, bound)
        _bind(sparse_module, "descriptor_loss_sparse", _sp.descriptor_loss_sparse, bound)
    if data_tools_module is None:
        data_tools_module = sys.modules.get("datasets.data_tools")
    if data_tools_module is not None:
        _bind(data_tools_module, "warpLabels", _worker_safe(_u.warpLabels, getattr(data_tools_module, "warpLabels", None)), bound)
    if export_module is None:
        export_module = sys.modules.get("export")
    if export_module is not None:
        _bind(export_module, "combine_heatmap", _u.combine_heatmap, bound)
        _bind(export_module, "inv_warp_image_batch", _u.inv_warp_image_batch, bound)
    return bound


def uninstall():
    while _saved:
        obj, name, fn = _saved.pop()
        setattr(obj, name, fn)
