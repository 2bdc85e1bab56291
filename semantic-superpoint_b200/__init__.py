"""ssp_b200 -- B200-native (sm_100a) homography-warp correspondence path of Semantic-SuperPoint.

Import as `import ssp_b200` (the repo-root shim maps that name onto this directory).  The public surface
mirrors the reference's function library (utils.py), see dropin.install() for binding it over the
reference's own `utils.utils` module.
"""
from . import _lib, build  # noqa: F401
from .losses import get_descriptor_engine, set_descriptor_engine  # noqa: F401
from .utils import *  # noqa: F401,F403
from .utils import combine_heatmap_batch, detector_loss_2d, detector_loss_pair_2d, heatmap_to_pts_batch, warp_labels_batch  # noqa: F401
from . import dist, dropin, homography, sparse, step, synth  # noqa: F401
from .homography import HomographySampler  # noqa: F401
from .sparse import batch_descriptor_loss_sparse, descriptor_loss_sparse  # noqa: F401

__version__ = "0.1.0"
