"""tfrpn -- B200-native (sm_100a) drop-in for the box hot path of FurkanOM/tf-rpn.

Mirrors the reference's module layout: ``tfrpn.utils.bbox_utils`` and ``tfrpn.utils.train_utils``
export the reference's function names and signatures (utils/bbox_utils.py, utils/train_utils.py)
and run on hand-written CUDA kernels in libtfrpn_cuda.so through the C ABI of include/tfrpn.h.
There is no CPU implementation in this package.
"""
from . import _lib  # noqa: F401
from .utils import bbox_utils, data_utils, train_utils  # noqa: F401
from .proposals import generate_proposals, predict_top_boxes  # noqa: F401
from .pipeline import HostPipeline, prefetching_rpn_generator  # noqa: F401
from .evaluation import DetectionMAP, ProposalRecall, detection_map, proposal_recall  # noqa: F401
from .roi_targets import RoiTargets, roi_target_cfg, roi_targets  # noqa: F401

__version__ = "0.1.0"
