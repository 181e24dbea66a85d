"""brainmagick_b200: B200-native (sm_100a) drop-in for brainmagick's contrastive training step --
`SimpleConv` (bm/models/simpleconv.py) and `ClipLoss` (bm/losses.py) behind the reference's module surface -- and for the
callers either side of it: batch preparation (`norm`: bm/norm.py), the DeepMel feature model (`features`:
bm/models/features.py) and the retrieval evaluation (`retrieval`: scripts/run_eval_probs.py, bm/wer.py)."""
import os as _os

import torch as _torch

# The training step keeps ~7 CUDA streams busy per process (main, weight-gradient side stream, candidate gather, NCCL, input
# copies).  With the driver's default of 8 hardware work queues, streams alias and a spinning symmetric-memory barrier kernel
# can sit in front of an NCCL kernel: 20-50 ms stalls every few steps at N = 2 (profiles/README.md).  More queues remove
# them; the variable only takes effect before the CUDA context exists and an explicit user setting is left alone.
if "CUDA_DEVICE_MAX_CONNECTIONS" not in _os.environ and not _torch.cuda.is_initialized():
    _os.environ["CUDA_DEVICE_MAX_CONNECTIONS"] = "32"

from .simpleconv import SimpleConv  # noqa: F401,E402
from .losses import ClipLoss, L1Loss, L2Loss  # noqa: F401,E402
from .common import ChannelMerger, ConvSequence, FourierEmb, PositionGetter, SubjectLayers  # noqa: F401
from .features import DeepMel  # noqa: F401
from .norm import BatchScaler, ScaleReject  # noqa: F401

__all__ = ["SimpleConv", "ClipLoss", "L1Loss", "L2Loss", "ChannelMerger", "ConvSequence", "FourierEmb", "PositionGetter",
           "SubjectLayers", "DeepMel", "BatchScaler", "ScaleReject"]
