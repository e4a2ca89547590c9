"""tf_raft_b200 -- B200-native (sm_100a) RAFT forward/update hot path behind the Python API of
daigo0927/tf-raft: `CorrBlock`, `BasicUpdateBlock` / `SmallUpdateBlock`, `RAFT` / `SmallRAFT`.

Compute lives in libraft_b200.so (hand-written CUDA, C ABI in include/raft_b200.h); PyTorch supplies
device memory, streams, CUDA graphs and torch.distributed.  No CPU fallback.
"""
from . import _lib
from .layers.corr import CorrBlock, bilinear_sampler, coords_grid, tfa_sampler, upflow8
from .layers.extractor import BasicEncoder, SmallEncoder
from .layers.update import BasicUpdateBlock, SmallUpdateBlock
from .losses import EndPointError, end_point_error, sequence_loss
from .model import RAFT, SmallRAFT
from .checkpoint import load_tf_checkpoint, read_tf_checkpoint, write_tf_checkpoint
from .preprocess import CropOrPadder, pad_to_multiple, resize_with_crop_or_pad
from .video import VideoFlow, forward_interpolate
from .train import AdamW, CyclicalLearningRate, first_cycle_scaler, inverse_scaler
from . import datasets

__all__ = ['CorrBlock', 'bilinear_sampler', 'coords_grid', 'tfa_sampler', 'upflow8', 'BasicEncoder', 'SmallEncoder',
           'BasicUpdateBlock', 'SmallUpdateBlock', 'RAFT', 'SmallRAFT', 'sequence_loss', 'end_point_error',
           'resize_with_crop_or_pad', 'CropOrPadder', 'pad_to_multiple', 'load_tf_checkpoint', 'read_tf_checkpoint',
           'write_tf_checkpoint', 'VideoFlow', 'forward_interpolate']
