"""CPU references for video inference (test infrastructure).

`forward_interpolate`: NumPy fp64 brute force with exactly the semantics of raft_b200_forward_interpolate
(include/raft_b200.h): sample (x, y) lands at (x + fx, y + fy) and is kept iff strictly inside (0, w) x (0, h);
each grid point takes the flow of the kept sample with the least d2 = ((qx-x)-fx)^2 + ((qy-y)-fy)^2, every
operation a separately rounded fp64 NumPy op; ties go to the first index (argmin); no kept sample -> zeros.

`forward`: `oracle.raft_torch.forward` with the loop started from coords_grid + flow_init, built from the same
oracle layers.
"""
import numpy as np
import torch

from oracle import raft_torch as rt

CHUNK = 512                         # queries per block: 512 x 7168 fp64 = 29 MB at 56x128


def nearest(flow_img):
    """flow_img (h, w, 2) -> (idx, d2 best, d2 second best) per grid point, row-major; idx = -1 if nothing is kept."""
    h, w, _ = flow_img.shape
    n = h * w
    gy, gx = np.meshgrid(np.arange(h, dtype=np.float64), np.arange(w, dtype=np.float64), indexing='ij')
    x, y = gx.reshape(n), gy.reshape(n)
    fx = flow_img[..., 0].reshape(n).astype(np.float64)
    fy = flow_img[..., 1].reshape(n).astype(np.float64)
    with np.errstate(invalid='ignore'):
        px, py = x + fx, y + fy
        kept = (px > 0) & (px < w) & (py > 0) & (py < h)
    idx = np.full(n, -1, dtype=np.int64)
    best = np.full(n, np.inf)
    second = np.full(n, np.inf)
    if not kept.any():
        return idx, best, second
    ks = np.nonzero(kept)[0]
    kx, ky, kfx, kfy = x[ks], y[ks], fx[ks], fy[ks]
    for q0 in range(0, n, CHUNK):
        qx, qy = x[q0:q0 + CHUNK, None], y[q0:q0 + CHUNK, None]
        dx = (qx - kx[None]) - kfx[None]
        dy = (qy - ky[None]) - kfy[None]
        d2 = dx * dx + dy * dy
        j = np.argmin(d2, axis=1)
        rows = np.arange(d2.shape[0])
        idx[q0:q0 + CHUNK] = ks[j]
        best[q0:q0 + CHUNK] = d2[rows, j]
        if d2.shape[1] > 1:
            d2[rows, j] = np.inf
            second[q0:q0 + CHUNK] = d2.min(axis=1)
    return idx, best, second


def forward_interpolate(flow, as_coords=False):
    """flow (B, h, w, 2) float32 -> (B, h, w, 2) float32."""
    flow = np.ascontiguousarray(flow, dtype=np.float32)
    b, h, w, _ = flow.shape
    out = np.zeros_like(flow)
    for i in range(b):
        idx = nearest(flow[i])[0]
        got = idx >= 0
        o = out[i].reshape(h * w, 2)
        o[got] = flow[i].reshape(h * w, 2)[idx[got]]
    if as_coords:
        gy, gx = np.meshgrid(np.arange(h, dtype=np.float32), np.arange(w, dtype=np.float32), indexing='ij')
        out = np.stack([gx, gy], axis=-1)[None] + out            # fp32 add
    return out


def forward(params, image1, image2, variant='raft', iters=12, flow_init=None, dtype=torch.float32):
    """rt.forward (model.py:68-109 / 190-226) with coords1 = coords_grid + flow_init (B, H/8, W/8, 2)."""
    cfg = rt.VARIANTS[variant]
    ops = rt.Ops(params, dtype)
    x1 = 2 * (rt._t(image1, dtype) / 255.0) - 1.0
    x2 = 2 * (rt._t(image2, dtype) / 255.0) - 1.0
    bs, H, W, _ = x1.shape
    both = torch.cat([x1, x2], dim=0).permute(0, 3, 1, 2)
    fm = rt.encoder(ops, both, 'fnet', cfg['fnorm'], False).permute(0, 2, 3, 1)
    corr_block = rt.CorrBlock(fm[:bs].contiguous(), fm[bs:].contiguous(), cfg['levels'], cfg['radius'])
    cnet = rt.encoder(ops, x1.permute(0, 3, 1, 2), 'cnet', cfg['cnorm'], False)
    net = torch.tanh(cnet[:, :cfg['hidden']])
    inp = torch.relu(cnet[:, cfg['hidden']:])
    coords0 = rt.coords_grid(bs, H // 8, W // 8, dtype)
    coords1 = coords0.clone() if flow_init is None else coords0 + rt._t(flow_init, dtype)
    block = rt.basic_update_block if variant == 'raft' else rt.small_update_block
    preds = []
    for _ in range(iters):
        corr = corr_block.retrieve(coords1)
        flow = coords1 - coords0
        net, mask, delta = block(ops, net, inp, corr.permute(0, 3, 1, 2), flow.permute(0, 3, 1, 2))
        coords1 = coords1 + delta.permute(0, 2, 3, 1)
        if variant == 'raft':
            preds.append(rt.upsample_flow(coords1 - coords0, mask.permute(0, 2, 3, 1)))
        else:
            preds.append(rt.upflow8(coords1 - coords0))
    return preds
