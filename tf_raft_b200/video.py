"""Video inference: each frame encoded once, each pair optionally warm-started from the previous one.

`forward_interpolate(flow)` is the original RAFT's warm start (core/utils/utils.py there): the low-resolution
flow of one pair is forward-splatted and every grid point takes the flow of the nearest kept sample.  It is one
call into libraft_b200.so (raft_b200_forward_interpolate, exact brute-force nearest neighbour, DESIGN.md).

`VideoFlow(model)` runs a RAFT / SmallRAFT over B videos in lockstep.  Pairwise calls `model([f[t-1], f[t]])`
run the feature encoder on every interior frame twice; the stream keeps the previous frame's feature map and
raw context-encoder output, so each call encodes only the new frames.  The rest of the pair (correlation
pyramid, context split, iteration loop) is the model's own code, so without warm start a stream output is
bit-identical to `model([f[t-1], f[t]], training=False, last_only=True)[-1]`.
"""
import torch

from . import _lib
from .layers.corr import coords_grid
from .model import _check_image_size


def forward_interpolate(flow, *, as_coords=False):
    """flow (B, h, w, 2) float32 on the GPU -> (B, h, w, 2): the warm-start flow for the next pair.

    Sample (x, y) lands at (x + fx, y + fy); it is kept iff it lands strictly inside (0, w) x (0, h).  Each grid
    point takes the flow of the nearest kept sample (squared distance in fp64, ties to the lowest row-major
    index); an image that keeps no sample gives zeros.  `as_coords=True` returns coords_grid + that flow, the
    `coords1` the forward loop starts from.  Cost is O((h*w)^2) per image."""
    flow = _lib.f32c(flow)
    if flow.dim() != 4 or flow.shape[-1] != 2:
        raise ValueError(f'flow must be (B, h, w, 2); got {tuple(flow.shape)}')
    b, h, w, _ = flow.shape
    out = torch.empty_like(flow)
    with torch.cuda.device(flow.device):
        _lib.check(_lib.lib().raft_b200_forward_interpolate(_lib.ptr(flow), b, h, w, int(bool(as_coords)),
                                                            _lib.ptr(out), _lib.stream()), 'forward_interpolate')
    return out


class VideoFlow:
    """`vf = VideoFlow(model, warm_start=True)`; `vf(frames)` with frames (B, H, W, 3) in 0..255 on the GPU: frame t
    of B independent videos that advance in lockstep.

    The first call (and the first after `reset()`) encodes the frames and returns None.  Every later call returns
    the final full-resolution flow (B, H, W, 2) from the previous frames to these -- what `predict_step` returns --
    and sets `flow_low` (B, H/8, W/8, 2).  With `warm_start` the loop of each pair after the first starts from
    `forward_interpolate(flow_low)` of the pair before.  Runs eagerly whatever `model.use_graph` says; the
    iteration count is `model.iters_pred`.  A change of frame shape needs `reset()` first."""

    def __init__(self, model, warm_start=True):
        self.model = model
        self.warm_start = bool(warm_start)
        self.reset()

    def reset(self):
        """Forget the previous frames: the next call starts new videos."""
        self._shape = None
        self._fmap = None
        self._cnet = None
        self.flow_low = None

    def __call__(self, frames):
        m = self.model
        frames = _lib.f32c(frames)
        if frames.dim() != 4 or frames.shape[-1] != 3:
            raise ValueError(f'frames must be (B, H, W, 3); got {tuple(frames.shape)}')
        shape = tuple(frames.shape)
        if self._shape is not None and shape != self._shape:
            raise ValueError(f'frame shape changed from {self._shape} to {shape}; call reset() before a new video')
        bs, H, W, _ = shape
        _check_image_size(H, W)
        m._sync_trained_params()
        # model.py:70-82 on the new frames only; the raw cnet output waits for the pair in which they are image1
        fmap = m.fnet(frames, training=False, raw_image=True)
        cnet = m.cnet(frames, training=False, raw_image=True)
        fmap1, cnet1 = self._fmap, self._cnet
        self._shape, self._fmap, self._cnet = shape, fmap, cnet
        if fmap1 is None:
            return None
        net, inp = m._split_context(cnet1)                 # per pair: the loop updates net in place
        if self.warm_start and self.flow_low is not None:
            coords1 = forward_interpolate(self.flow_low, as_coords=True)
        else:
            coords1 = coords_grid(bs, H // 8, W // 8, m.device)
        preds = m._decode(fmap1, fmap, net, inp, coords1, False, True)
        self.flow_low = coords1 - coords_grid(bs, H // 8, W // 8, m.device)
        return preds[-1]
