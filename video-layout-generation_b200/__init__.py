"""video-layout-generation_b200: B200-native flow-guided warp + per-pixel losses (fwd/bwd).

Hand-written sm_100a CUDA kernels behind a C ABI (include/vlg_b200.h, libvlg_b200.so), with the
reference's Python call signatures on top.  Import as `vlg_b200` (see vlg_b200.py at the repo
root; the directory name carries a hyphen).
"""
from . import _build, _cabi  # noqa: F401
from ._cabi import VlgError, launch_count  # noqa: F401
from .graphs import CapturedStep  # noqa: F401
from .losses import (CombinedLoss, CrossEntropyLoss, GradientLoss, L1Loss, PixelLosses,  # noqa: F401
                     SsimLoss, WarpLoss)
from .metrics import IoUResult, LayoutIoU  # noqa: F401
from .ops import (CITYSCAPES_PALETTE, WarpLossConfig, colorize, confusion_matrix, empty_nhwc, ingest, one_hot_layout,  # noqa: F401
                  pixel_losses, prepare_frames, rollout, to_nhwc, warp, warp_labels, warp_loss, warp_loss_labels)

__version__ = "2.0"
