"""Video inference: the forward_interpolate warm start (kernel against the NumPy fp64 brute force, bit for bit),
RAFT's `flow_init`, and the `VideoFlow` stream against the pairwise calls it replaces."""
import ctypes

import numpy as np
import pytest
import torch

import cases
import warm_start_ref as ref
from oracle import raft_torch as rt, weights

gpu = pytest.mark.gpu
F32 = np.float32


def random_flow(b, h, w, seed, scale=2.5, out_frac=0.2):
    """Seeded flows of a few pixels; about `out_frac` of the samples are sent far outside the image."""
    rng = np.random.default_rng(seed)
    f = rng.uniform(-scale, scale, (b, h, w, 2)).astype(F32)
    away = rng.random((b, h, w)) < out_frac
    f[away] += rng.choice(np.array([-1, 1], F32), (int(away.sum()), 2)) * F32(10 * max(h, w))
    return f


def smooth_flow(b, h, w, seed, amp=3.0):
    rng = np.random.default_rng(seed)
    gy, gx = np.meshgrid(np.arange(h) / h, np.arange(w) / w, indexing='ij')
    out = np.empty((b, h, w, 2), F32)
    for i in range(b):
        for c in range(2):
            p = rng.uniform(0, 2 * np.pi, 2)
            out[i, ..., c] = amp * np.sin(2 * np.pi * gx + p[0]) * np.cos(2 * np.pi * gy + p[1])
    return out


def grid(b, h, w):
    gy, gx = np.meshgrid(np.arange(h, dtype=F32), np.arange(w, dtype=F32), indexing='ij')
    return np.tile(np.stack([gx, gy], axis=-1)[None], (b, 1, 1, 1))


# --------------------------------------------------------------------------------------------- CPU: the reference
@pytest.mark.parametrize('h,w', [(13, 29), (56, 128)])
def test_reference_forward_interpolate_vs_scipy_griddata(h, w):
    """The fp64 brute force picks what scipy's nearest-neighbour griddata picks, up to near-ties: where the best and
    second-best d2 differ by more than 1e-9*max(1, d2) the values are equal, elsewhere scipy's pick is a kept sample
    within that margin of the minimum."""
    interpolate = pytest.importorskip('scipy.interpolate')
    flow = random_flow(2, h, w, seed=h * w)
    want = ref.forward_interpolate(flow)
    gy, gx = np.meshgrid(np.arange(h), np.arange(w), indexing='ij')
    qx, qy = gx.reshape(-1).astype(np.float64), gy.reshape(-1).astype(np.float64)
    for i in range(flow.shape[0]):
        fx = flow[i, ..., 0].reshape(-1).astype(np.float64)
        fy = flow[i, ..., 1].reshape(-1).astype(np.float64)
        px, py = qx + fx, qy + fy
        kept = (px > 0) & (px < w) & (py > 0) & (py < h)
        assert 0.6 < kept.mean() < 0.9
        got = interpolate.griddata((px[kept], py[kept]), flow[i].reshape(-1, 2)[kept], (qx, qy), method='nearest')
        _, best, second = ref.nearest(flow[i])
        margin = 1e-9 * np.maximum(1.0, best)
        clear = second - best > margin
        assert clear.mean() > 0.9
        np.testing.assert_array_equal(got[clear], want[i].reshape(-1, 2)[clear])
        kf = flow[i].reshape(-1, 2)[kept]
        for q in np.nonzero(~clear)[0]:
            d2 = ((qx[q] - qx[kept]) - fx[kept]) ** 2 + ((qy[q] - qy[kept]) - fy[kept]) ** 2
            near = d2 <= best[q] + margin[q]
            assert (kf[near] == got[q]).all(axis=1).any(), f'query {q}: scipy picked a sample that is not nearest'


def test_reference_forward_interpolate_edge_cases():
    """Strict bounds, NaN never kept, ties to the first index, an image with no kept sample gives zeros."""
    h, w = 3, 4
    f = np.zeros((2, h, w, 2), F32)
    f[0] = 0.5                                               # every sample lands half a pixel off: exact ties
    f[0, 0, 0] = [-0.0, 0.5]                                 # lands on x = 0: dropped
    f[0, 1, 1] = [np.nan, 0.5]
    f[1] = 100.0                                             # nothing kept
    out = ref.forward_interpolate(f)
    np.testing.assert_array_equal(out[1], 0)
    idx, best, second = ref.nearest(f[0])
    assert idx[0] == 1 and best[0] == second[0] == 2.5       # q(0,0): samples (1,0) and (0,1) tie; (0,0) dropped
    assert 5 not in idx                                      # the NaN sample
    np.testing.assert_array_equal(ref.forward_interpolate(f, as_coords=True)[1], grid(1, h, w)[0])


def test_reference_forward_without_flow_init_is_the_oracle():
    p = weights.init_params('small', 5, bias_scale=0.05, norm_jitter=0.1)
    im1, im2 = cases.images(1, 64, 64, 3, 4)
    want = rt.forward(p, im1, im2, 'small', 2)
    got = ref.forward(p, im1, im2, 'small', 2)
    assert all(torch.equal(a, b) for a, b in zip(got, want))


def test_forward_interpolate_host_side_argument_errors():
    from tf_raft_b200 import build, _lib
    build.build()
    L = _lib.lib()
    fake = ctypes.c_void_p(1 << 20)
    assert L.raft_b200_forward_interpolate(None, 1, 8, 8, 0, fake, None) == -1
    assert L.raft_b200_forward_interpolate(fake, 1, 8, 8, 0, None, None) == -1
    assert L.raft_b200_forward_interpolate(fake, 0, 8, 8, 0, ctypes.c_void_p(1 << 24), None) == -2
    assert L.raft_b200_forward_interpolate(fake, 1, 0, 8, 1, ctypes.c_void_p(1 << 24), None) == -2
    assert L.raft_b200_forward_interpolate(fake, 1, 8, -1, 0, ctypes.c_void_p(1 << 24), None) == -2
    assert L.raft_b200_forward_interpolate(fake, 70000, 8, 8, 0, ctypes.c_void_p(1 << 30), None) == -2
    assert L.raft_b200_forward_interpolate(fake, 1, 8, 8, 0, fake, None) == -1                      # out == flow
    assert L.raft_b200_forward_interpolate(fake, 1, 8, 8, 0, ctypes.c_void_p((1 << 20) + 256), None) == -1  # overlap
    assert L.raft_b200_forward_interpolate(fake, 1, 8, 8, 0, ctypes.c_void_p((1 << 20) - 256), None) == -1


# --------------------------------------------------------------------------------------------- GPU
def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope='module')
def T():
    import tf_raft_b200
    from tf_raft_b200 import _lib
    assert _lib.lib().raft_b200_device_ok(torch.cuda.current_device()) == 0, 'needs an sm_100 GPU'
    return tf_raft_b200


def _flow_cases():
    tie = np.full((2, 13, 29, 2), 0.5, F32)                  # constant half-pixel flow: exact ties everywhere
    tie[1] = -0.5
    nan = random_flow(1, 13, 29, seed=9)
    nan[0, ::5, ::3] = np.nan
    nan[0, 2, :, 0] = -np.arange(29, dtype=F32)              # lands exactly on x = 0: dropped
    return {'random_3x13x29': random_flow(3, 13, 29, seed=1), 'random_2x56x128': random_flow(2, 56, 128, seed=2),
            'half_pixel_ties': tie, 'half_pixel_ties_56x128': np.full((1, 56, 128, 2), 0.5, F32),
            'nan_and_borders': nan}


@gpu
@pytest.mark.parametrize('name', list(_flow_cases()))
def test_forward_interpolate_kernel_bitwise_vs_reference(T, name):
    flow = _flow_cases()[name]
    got = T.forward_interpolate(dev(flow))
    np.testing.assert_array_equal(got.cpu().numpy(), ref.forward_interpolate(flow))
    coords = T.forward_interpolate(dev(flow), as_coords=True)
    b, h, w, _ = flow.shape
    assert torch.equal(coords, T.coords_grid(b, h, w, 'cuda') + got)
    np.testing.assert_array_equal(coords.cpu().numpy(), ref.forward_interpolate(flow, as_coords=True))


@gpu
def test_forward_interpolate_all_samples_outside(T):
    flow = np.full((2, 13, 29, 2), 40.0, F32)
    flow[1] = -3.0e38
    assert torch.equal(T.forward_interpolate(dev(flow)), torch.zeros(flow.shape, device='cuda'))
    assert torch.equal(T.forward_interpolate(dev(flow), as_coords=True), T.coords_grid(2, 13, 29, 'cuda'))


def _model(T, variant, iters, params, **kw):
    cls = T.RAFT if variant == 'raft' else T.SmallRAFT
    m = cls(iters=iters, iters_pred=iters, precision='f16x2', **kw)
    m.load_params(params)
    return m


@gpu
@pytest.mark.parametrize('variant', ['raft', 'small'])
def test_zero_flow_init_is_no_flow_init(T, variant):
    """Eager and CUDA-graph: a zero flow_init gives the bits of no flow_init; the graph keys on whether flow_init is
    given and copies its value in on every replay."""
    p = weights.init_params(variant, 3, bias_scale=0.02)
    im1, im2 = cases.images(2, 64, 96, 5, 6)
    a, b = dev(im1), dev(im2)
    zero = torch.zeros((2, 8, 12, 2), device='cuda')
    fi = dev(smooth_flow(2, 8, 12, seed=4))
    eager = _model(T, variant, 3, p)
    want = eager([a, b], training=False)
    warm = [t.clone() for t in eager([a, b], training=False, flow_init=fi)]
    got = eager([a, b], training=False, flow_init=zero)
    assert all(torch.equal(x, y) for x, y in zip(got, want))
    assert not torch.equal(warm[-1], want[-1])
    graph = _model(T, variant, 3, p, use_graph=True)
    for _ in range(2):
        got = graph([a, b], training=False, flow_init=zero)
        assert all(torch.equal(x, y) for x, y in zip(got, want))
        got = graph([a, b], training=False, flow_init=fi)
        assert all(torch.equal(x, y) for x, y in zip(got, warm))
        got = graph([a, b], training=False)
        assert all(torch.equal(x, y) for x, y in zip(got, want))


@gpu
def test_flow_init_argument_errors(T):
    p = weights.init_params('small', 3)
    m = _model(T, 'small', 1, p)
    a = dev(cases.images(1, 64, 96)[0])
    for bad in (torch.zeros((1, 8, 13, 2), device='cuda'), torch.zeros((2, 8, 12, 2), device='cuda'),
                torch.zeros((1, 8, 12, 2)), torch.zeros((1, 8, 12, 2), device='cuda', dtype=torch.float64)):
        with pytest.raises(ValueError):
            m([a, a], training=False, flow_init=bad)


@gpu
@pytest.mark.parametrize('variant,shape,iters', [('raft', (72, 200), 3), ('small', (128, 256), 4)])
def test_warm_started_forward_vs_oracle(T, variant, shape, iters):
    H, W = shape
    p = weights.init_params(variant, 77, bias_scale=0.02, norm_jitter=0.05)
    im1, im2 = cases.images(1, H, W, 11, 12)
    fi = smooth_flow(1, H // 8, W // 8, seed=13)
    want = ref.forward(p, im1, im2, variant, iters, flow_init=fi)
    got = _model(T, variant, iters, p)([dev(im1), dev(im2)], training=False, flow_init=dev(fi))
    for i in range(iters):
        err = float((got[i].cpu() - want[i]).abs().max())
        assert err <= 1e-3, f'{variant} {H}x{W} iteration {i}: max-abs {err}'


def _frames(n, b, H, W, seed=40):
    return [dev(np.random.default_rng(seed + t).uniform(0, 255, (b, H, W, 3)).astype(F32)) for t in range(n)]


@gpu
@pytest.mark.parametrize('shape,iters', [((128, 256), 4), ((448, 1024), 3)])
def test_stream_without_warm_start_is_pairwise(T, shape, iters):
    """Each frame encoded once (B images) gives the bits of the pairwise call (2B images through fnet)."""
    H, W = shape
    p = weights.init_params('raft', 21, bias_scale=0.02, norm_jitter=0.05)
    m = _model(T, 'raft', iters, p)
    frames = _frames(4, 2, H, W)
    vf = T.VideoFlow(m, warm_start=False)
    assert vf(frames[0]) is None
    for t in range(1, 4):
        got = vf(frames[t]).clone()
        assert tuple(got.shape) == (2, H, W, 2) and tuple(vf.flow_low.shape) == (2, H // 8, W // 8, 2)
        want = m([frames[t - 1], frames[t]], training=False, last_only=True)[-1]
        assert torch.equal(got, want), f'pair {t}'


@gpu
@pytest.mark.parametrize('variant', ['raft', 'small'])
def test_stream_with_warm_start_is_the_manual_chain(T, variant):
    H, W, iters = 128, 256, 4
    p = weights.init_params(variant, 22, bias_scale=0.02, norm_jitter=0.05)
    m = _model(T, variant, iters, p)
    frames = _frames(4, 2, H, W, seed=50)
    vf = T.VideoFlow(m)
    assert vf(frames[0]) is None
    outs = [vf(frames[t]).clone() for t in range(1, 4)]
    g = T.coords_grid(2, H // 8, W // 8, 'cuda')
    flow_init = None
    for t in range(1, 4):
        want = m([frames[t - 1], frames[t]], training=False, last_only=True, flow_init=flow_init)[-1]
        assert torch.equal(outs[t - 1], want), f'pair {t}'
        flow_init = T.forward_interpolate(m._last['coords1'] - g)
    assert torch.equal(vf.flow_low, m._last['coords1'] - g)


@gpu
def test_stream_reset_and_shape_change(T):
    p = weights.init_params('small', 23, bias_scale=0.02)
    m = _model(T, 'small', 3, p)
    f = _frames(3, 1, 64, 96, seed=60)
    vf = T.VideoFlow(m)
    vf(f[0])
    vf(f[1])
    vf(f[2])
    vf.reset()
    assert vf(f[1]) is None and vf.flow_low is None
    got = vf(f[0]).clone()
    fresh = T.VideoFlow(m)
    fresh(f[1])
    assert torch.equal(got, fresh(f[0]))
    with pytest.raises(ValueError):
        vf(_frames(1, 1, 64, 104)[0])
    with pytest.raises(ValueError):
        vf(_frames(1, 2, 64, 96)[0])
