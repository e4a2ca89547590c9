"""RAFT / SmallRAFT -- host-side mirror of tf_raft/model.py.

`RAFT(drop_rate=0, iters=12, iters_pred=24)([image1, image2], training)` returns the list of
`iters` (training) or `iters_pred` (inference) flow predictions (B, H, W, 2), like the reference
(model.py:68-109 / 190-226).  The whole iteration loop (lookup -> update block -> coords += delta ->
upsample) is ONE call into libraft_b200.so (raft_b200_forward_loop); the correlation pyramid is
another (raft_b200_corr_pyramid_build).  Optionally the loop is replayed from a CUDA graph.
"""
from collections import OrderedDict

import torch

from . import _lib
from .layers.corr import CorrBlock, coords_grid, upflow8
from .layers.extractor import BasicEncoder, SmallEncoder
from .layers.update import BasicUpdateBlock, SmallUpdateBlock
from .losses import end_point_error, sequence_loss


def _check_image_size(H, W):
    if H % 8 or W % 8:
        raise ValueError(f'image height and width must be multiples of 8 (got {H}x{W}); the reference fails in '
                         'update.py:146 for other sizes -- crop-or-pad first (datasets/dataset.py:323-334)')


class RAFT:
    _variant = _lib.VARIANT_BASIC

    def __init__(self, drop_rate=0, iters=12, iters_pred=24, *, precision=None, device='cuda', seed=None,
                 use_graph=False, encoder_backend=None, **kwargs):
        self.hidden_dim = 128
        self.context_dim = 128
        self.corr_levels = 4
        self.corr_radius = 4
        self.drop_rate = drop_rate
        self.iters = iters
        self.iters_pred = iters_pred
        self.precision = _lib.resolve_precision(precision)
        self.device = torch.device(device)
        self.use_graph = use_graph
        self.encoder_backend = encoder_backend
        self._build_layers(seed)
        self._graphs = {}
        self.flow_metrics = None
        self.optimizer = None
        self._trainer = None
        self._params_stale = False

    def _encoder_backend(self):
        # the all-FFMA reference configuration keeps cuDNN IEEE-fp32 encoders; the product path is native
        return self.encoder_backend or ('native' if self.precision == _lib.PREC_F16X2 else 'torch')

    def _build_layers(self, seed):
        s = 0 if seed is None else seed
        self.fnet = BasicEncoder(output_dim=256, norm_type='instance', drop_rate=self.drop_rate, device=self.device,
                                 seed=s, backend=self._encoder_backend())
        self.cnet = BasicEncoder(output_dim=self.hidden_dim + self.context_dim, norm_type='batch',
                                 drop_rate=self.drop_rate, device=self.device, seed=s + 1, backend=self._encoder_backend())
        self.update_block = BasicUpdateBlock(filters=self.hidden_dim, precision=self.precision, device=self.device,
                                             seed=s + 2)

    # -- parameters ---------------------------------------------------------------------------
    def load_params(self, params):
        """`{'fnet.conv1.kernel': ..., 'cnet....', 'update_block.encoder.convc1.kernel': ...}` (NumPy or torch)."""
        self.fnet.load_params(params, 'fnet.')
        self.cnet.load_params(params, 'cnet.')
        self.update_block.load_params(params, 'update_block.')
        self._graphs.clear()
        self._trainer = None                               # a training state built on the old values is void
        self._params_stale = False

    def state_dict(self):
        self._sync_trained_params()
        out = OrderedDict()
        out.update(self.fnet.state_dict('fnet.'))
        out.update(self.cnet.state_dict('cnet.'))
        out.update(self.update_block.state_dict('update_block.'))
        return out

    # -- reference helpers ----------------------------------------------------------------------
    def initialize_flow(self, image):
        """model.py:32-37: coords0 = coords1 = coords_grid(B, H//8, W//8)."""
        bs, h, w, _ = image.shape
        return coords_grid(bs, h // 8, w // 8, self.device), coords_grid(bs, h // 8, w // 8, self.device)

    def upsample_flow(self, flow, mask):
        """model.py:39-66: convex 8x upsampling."""
        flow, mask = _lib.f32c(flow), _lib.f32c(mask)
        b, h, w, _ = flow.shape
        if tuple(mask.shape) != (b, h, w, 576):
            raise ValueError(f'mask: expected {(b, h, w, 576)}, got {tuple(mask.shape)}')
        out = torch.empty((b, 8 * h, 8 * w, 2), dtype=torch.float32, device=flow.device)
        with torch.cuda.device(flow.device):
            _lib.check(_lib.lib().raft_b200_upsample_convex(_lib.ptr(flow), _lib.ptr(mask), b, h, w, _lib.ptr(out),
                                                            _lib.stream()), 'upsample_convex')
        return out

    # -- forward ----------------------------------------------------------------------------------
    def _encode(self, image1, image2, training):
        # model.py:70-71 (2*(x/255)-1) happens inside the encoders' first load (raw_image=True)
        fmap1, fmap2 = self.fnet([image1, image2], training=training, raw_image=True)     # :74
        cnet = self.cnet(image1, training=training, raw_image=True)                       # :82
        net, inp = self._split_context(cnet)
        return fmap1, fmap2, net, inp

    def _split_context(self, cnet):
        """model.py:84-86: net = tanh(cnet[..., :hidden]), inp = relu(cnet[..., hidden:]) into fresh buffers."""
        b, h, w, _ = cnet.shape
        net = torch.empty((b, h, w, self.hidden_dim), dtype=torch.float32, device=cnet.device)
        inp = torch.empty((b, h, w, self.context_dim), dtype=torch.float32, device=cnet.device)
        with torch.cuda.device(cnet.device):
            _lib.check(_lib.lib().raft_b200_context_split(_lib.ptr(cnet), b * h * w, self.hidden_dim,
                                                          self.context_dim, _lib.ptr(net), _lib.ptr(inp),
                                                          _lib.stream()), 'context_split')
        return net, inp

    def _loop(self, corr_block, net, inp, coords1, flow_ups, b, h, w):
        ub = self.update_block
        ws = ub.workspace(b, h, w)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().raft_b200_forward_loop(
                self._variant, _lib.ptr(ub.prepared()), _lib.ptr_array(corr_block.corr_pyramid), self.corr_levels,
                self.corr_radius, _lib.ptr(net), _lib.ptr(inp), _lib.ptr(coords1), _lib.ptr_array(flow_ups),
                len(flow_ups), b, h, w, _lib.ptr(ws), ws.numel(), self.precision, _lib.stream()), 'forward_loop')

    def __call__(self, inputs, training, *, last_only=False, flow_init=None):
        """inputs = [image1, image2], each (B, H, W, 3) float in 0..255 on the GPU.

        `training` is required, as in the reference (model.py:68).  `last_only=True` (keyword-only
        extra) computes just the final prediction -- what predict_step returns (model.py:166).
        `flow_init` (keyword-only extra): a (B, H/8, W/8, 2) float32 flow on the model's device; the loop then
        starts from coords1 = coords_grid + flow_init instead of coords_grid (the original RAFT's warm start
        for video, see `forward_interpolate` / `VideoFlow`).
        With `use_graph=True` the whole forward of a given input shape is captured once into a CUDA graph
        and replayed; the returned tensors are then static buffers that the next call overwrites."""
        image1, image2 = inputs
        image1, image2 = _lib.f32c(image1), _lib.f32c(image2)
        if flow_init is not None:
            flow_init = self._check_flow_init(flow_init, image1.shape)
        self._sync_trained_params()
        if self.use_graph and not training:
            return self._graph_call(image1, image2, last_only, flow_init)
        return self._forward(image1, image2, training, last_only, flow_init)

    def _check_flow_init(self, flow_init, image_shape):
        if not isinstance(flow_init, torch.Tensor):
            raise ValueError(f'flow_init must be a torch tensor, got {type(flow_init).__name__}')
        dev = self.device
        if dev.type == 'cuda' and dev.index is None:
            dev = torch.device('cuda', torch.cuda.current_device())
        if flow_init.device != dev:
            raise ValueError(f'flow_init must be on the model\'s device {dev}, got {flow_init.device}')
        bs, H, W, _ = image_shape
        want = (bs, H // 8, W // 8, 2)
        if tuple(flow_init.shape) != want:
            raise ValueError(f'flow_init: expected shape {want} for {H}x{W} images, got {tuple(flow_init.shape)}')
        if flow_init.dtype != torch.float32:
            raise ValueError(f'flow_init must be float32, got {flow_init.dtype}')
        return flow_init.contiguous()

    def _graph_call(self, image1, image2, last_only, flow_init=None):
        key = (tuple(image1.shape), bool(last_only), flow_init is not None)
        entry = self._graphs.get(key)
        if entry is None:
            s1, s2 = image1.clone(), image2.clone()
            sf = None if flow_init is None else flow_init.clone()
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):                      # warm-up: allocations, attributes, weight packing
                for _ in range(2):
                    self._forward(s1, s2, False, last_only, sf)
            torch.cuda.current_stream(self.device).wait_stream(side)
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                outs = self._forward(s1, s2, False, last_only, sf)
            # The captured kernels hold raw addresses of the encoder / update-block workspaces; those caches keep one
            # shape at a time, so the graph entry owns references to the buffers it was captured with.
            keep = [list(m._ws.values()) for m in (self.fnet, self.cnet, self.update_block)]
            entry = (graph, s1, s2, sf, outs, self._last, keep)
            self._graphs[key] = entry
        graph, s1, s2, sf, outs, last, _keep = entry
        s1.copy_(image1, non_blocking=True)
        s2.copy_(image2, non_blocking=True)
        if sf is not None:
            sf.copy_(flow_init, non_blocking=True)
        graph.replay()
        self._last = last
        return outs

    def _forward(self, image1, image2, training, last_only, flow_init=None):
        bs, H, W, _ = image1.shape
        _check_image_size(H, W)
        fmap1, fmap2, net, inp = self._encode(image1, image2, training)
        coords1 = coords_grid(bs, H // 8, W // 8, self.device)                # :89
        if flow_init is not None:
            coords1.add_(flow_init)
        return self._decode(fmap1, fmap2, net, inp, coords1, training, last_only)

    def _decode(self, fmap1, fmap2, net, inp, coords1, training, last_only):
        """Everything after the encoders: the correlation pyramid of (fmap1, fmap2) and the iteration loop from
        `coords1` (updated in place), with `net` / `inp` the split context of image1."""
        bs, h, w, _ = coords1.shape
        H, W = 8 * h, 8 * w
        iters = self.iters if training else self.iters_pred                  # model.py:92
        corr_block = CorrBlock(fmap1, fmap2, num_levels=self.corr_levels, radius=self.corr_radius,
                               precision=self.precision)                      # :77-79
        preds = [torch.empty((bs, H, W, 2), dtype=torch.float32, device=self.device)
                 if (not last_only or i == iters - 1) else None for i in range(iters)]
        if iters:
            self._loop(corr_block, net, inp, coords1, preds, bs, h, w)        # :93-106
        self._last = dict(net=net, coords1=coords1, corr_block=corr_block)
        return [p for p in preds if p is not None] if last_only else preds

    call = __call__

    # -- keras-style steps (model.py:111-170) ---------------------------------------------------
    def compile(self, optimizer=None, clip_norm=None, loss=sequence_loss, epe=end_point_error, **kwargs):
        self.optimizer = optimizer
        self.clip_norm = clip_norm
        self.loss = loss
        self.epe = epe
        self.flow_metrics = OrderedDict((k, [0.0, 0]) for k in ('loss', 'epe', 'u1', 'u3', 'u5'))

    def _metric_update(self, key, value):
        m = self.flow_metrics[key]
        m[0] += float(value)
        m[1] += 1

    def _metric_results(self):
        return {k: (s / n if n else 0.0) for k, (s, n) in self.flow_metrics.items()}

    def train_step(self, data):
        """model.py:126-144: forward with training=True under autograd, sequence loss, clip_by_global_norm,
        optimizer.apply_gradients, metrics.  data = (image1, image2, flow_gt, valid) on the GPU.  Under an initialised
        torch.distributed process group the gradients are all-reduced (one flat NCCL call) and the context encoder's
        BatchNorm statistics are taken over the global batch (tf_raft_b200/train.py)."""
        from .train import AdamW, Trainer
        if self.flow_metrics is None or getattr(self, 'optimizer', None) is None:
            raise RuntimeError('compile(optimizer=..., clip_norm=...) before train_step, as in train_chairs.py:92-98')
        if not isinstance(self.optimizer, AdamW):
            raise TypeError('optimizer must be tf_raft_b200.train.AdamW (tfa.optimizers.AdamW semantics)')
        if self._trainer is None:
            self._trainer = Trainer(self)
        loss, info = self._trainer.step(data, self.optimizer, self.clip_norm, self.loss, self.epe)
        self._params_stale = True                      # the layers' own copies are refreshed on the next inference call
        self._metric_update('loss', loss)
        for k in ('epe', 'u1', 'u3', 'u5'):
            self._metric_update(k, info[k])
        return self._metric_results()

    def _sync_trained_params(self):
        if self._trainer is not None and self._params_stale:
            trainer = self._trainer
            self.load_params(trainer.params())         # copies into the layers, drops prepared blobs and graphs
            self._trainer = trainer
            self._params_stale = False

    def test_step(self, data):
        """model.py:146-159."""
        if self.flow_metrics is None:
            self.compile()
        image1, image2, flow, valid = data
        preds = self([image1, image2], training=False, last_only=True)
        info = self.epe([flow, valid], preds[-1])
        for k in ('epe', 'u1', 'u3', 'u5'):
            self._metric_update(k, info[k])
        return self._metric_results()

    def predict_step(self, data):
        """model.py:161-166: only the finest prediction."""
        image1, image2, *_ = data
        return self([image1, image2], training=False, last_only=True)[-1]

    def reset_metrics(self):
        if self.flow_metrics is not None:
            for m in self.flow_metrics.values():
                m[0], m[1] = 0.0, 0


class SmallRAFT(RAFT):
    _variant = _lib.VARIANT_SMALL

    def _build_layers(self, seed):
        self.hidden_dim = 96
        self.context_dim = 64
        self.corr_levels = 4
        self.corr_radius = 3
        s = 0 if seed is None else seed
        self.fnet = SmallEncoder(output_dim=128, norm_type='instance', drop_rate=self.drop_rate, device=self.device,
                                 seed=s, backend=self._encoder_backend())
        self.cnet = SmallEncoder(output_dim=self.hidden_dim + self.context_dim, norm_type=None,
                                 drop_rate=self.drop_rate, device=self.device, seed=s + 1, backend=self._encoder_backend())
        self.update_block = SmallUpdateBlock(filters=self.hidden_dim, precision=self.precision, device=self.device,
                                             seed=s + 2)

    def upsample_flow(self, flow, mask=None):
        """SmallRAFT upsamples with upflow8 (model.py:223)."""
        return upflow8(flow)
