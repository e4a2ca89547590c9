"""Video inference on the GPU: the VideoFlow stream against pairwise calls, and the forward_interpolate kernel alone.

    python scripts/video_stream_bench.py --out OUTDIR            # -> OUTDIR/video_stream.json

(a) RAFT at 448x512 x 12 iterations and 448x1024 x 24, batch 4 (four videos in lockstep), seeded weights, 16 seeded
    frames (15 pairs).  Four arms: pairwise eager `model([f[t-1], f[t]], training=False, last_only=True)`, the same
    with `use_graph=True`, `VideoFlow(warm_start=False)` and `VideoFlow(warm_start=True)`.  After one warm-up pass
    per arm, the arms alternate for --rounds rounds; each round times the whole 16-frame sequence with CUDA events
    (the stream's first call, which only encodes frame 0, included) and divides by the 15 pairs.  Median and
    range of pairs/s over the rounds.  Untimed, in the same run: the VideoFlow(warm_start=False) flows are
    torch.equal to the pairwise eager ones.
(b) forward_interpolate_kernel alone, CUDA events over --launches launches at (4, 56, 128) and (1, 136, 240):
    ms per launch, evaluated (query, sample) pairs per second, and the time per image as a share of one pair's
    forward at the same size (the pairwise-graph time of (a) at 448x1024 x 24; a batch-1 eager forward at
    1088x1920 x 24 timed here for the larger size).
The card's name, power limit and max SM clock are read (nvidia-smi, read-only) before any timing.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = [(448, 512, 12), (448, 1024, 24)]
KERNEL_SIZES = [(4, 56, 128), (1, 136, 240)]
B, FRAMES = 4, 16


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else 'unknown'


def timed(fn):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    out = fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end), out


def frames(H, W, seed=100):
    return [torch.from_numpy(np.random.default_rng(seed + t).uniform(0, 255, (B, H, W, 3)).astype(np.float32)).cuda()
            for t in range(FRAMES)]


def workload(T, weights, H, W, iters, rounds):
    p = weights.init_params('raft', 1234)
    eager = T.RAFT(iters=iters, iters_pred=iters, precision='f16x2')
    graph = T.RAFT(iters=iters, iters_pred=iters, precision='f16x2', use_graph=True)
    eager.load_params(p)
    graph.load_params(p)
    f = frames(H, W)

    def pairwise(model):
        return lambda: [model([f[t - 1], f[t]], training=False, last_only=True)[-1] for t in range(1, FRAMES)]

    def stream(warm):
        def run():
            vf = T.VideoFlow(eager, warm_start=warm)
            return [vf(x) for x in f][1:]
        return run

    arms = {'pairwise_eager': pairwise(eager), 'pairwise_graph': pairwise(graph),
            'stream': stream(False), 'stream_warm_start': stream(True)}
    for fn in arms.values():                                       # warm-up: allocations, weight packing, graph capture
        timed(fn)
    ms = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            ms[k].append(timed(fn)[0] / (FRAMES - 1))
    want = [x.clone() for x in arms['pairwise_eager']()]
    got = arms['stream']()
    equal = all(torch.equal(a, b) for a, b in zip(got, want))
    res = dict(H=H, W=W, iters=iters, batch=B, frames=FRAMES, pairs=FRAMES - 1,
               stream_without_warm_start_equals_pairwise_eager=equal, arms={})
    for k, v in ms.items():
        pps = [B * 1e3 / x for x in v]
        res['arms'][k] = dict(ms_per_pair_step=[round(x, 4) for x in v], pairs_per_s_median=round(statistics.median(pps), 2),
                              pairs_per_s_min=round(min(pps), 2), pairs_per_s_max=round(max(pps), 2))
    g = res['arms']['pairwise_graph']['pairs_per_s_median']
    for k in ('stream', 'stream_warm_start'):
        res['arms'][k]['speedup_vs_pairwise_graph'] = round(res['arms'][k]['pairs_per_s_median'] / g, 4)
    del eager, graph, f, want, got
    torch.cuda.empty_cache()
    return res


def pair_forward_ms(T, weights, H, W, iters, reps=5):
    """One batch-1 eager forward (last_only) at H x W, median of `reps` after one warm-up."""
    p = weights.init_params('raft', 1234)
    m = T.RAFT(iters=iters, iters_pred=iters, precision='f16x2')
    m.load_params(p)
    a, b = [torch.from_numpy(np.random.default_rng(s).uniform(0, 255, (1, H, W, 3)).astype(np.float32)).cuda()
            for s in (1, 2)]
    m([a, b], training=False, last_only=True)
    torch.cuda.synchronize()
    t = statistics.median(timed(lambda: m([a, b], training=False, last_only=True))[0] for _ in range(reps))
    del m
    torch.cuda.empty_cache()
    return t


def kernel(T, b, h, w, launches, pair_ms):
    g = torch.Generator(device='cuda')
    g.manual_seed(7)
    flow = (torch.rand((b, h, w, 2), device='cuda', generator=g) - 0.5) * 8
    out = torch.empty_like(flow)
    from tf_raft_b200 import _lib
    L = _lib.lib()

    def launch():
        for _ in range(launches):
            _lib.check(L.raft_b200_forward_interpolate(_lib.ptr(flow), b, h, w, 1, _lib.ptr(out), _lib.stream()))

    for _ in range(10):
        _lib.check(L.raft_b200_forward_interpolate(_lib.ptr(flow), b, h, w, 1, _lib.ptr(out), _lib.stream()))
    torch.cuda.synchronize()
    ms = timed(launch)[0] / launches
    n = h * w
    return dict(B=b, h=h, w=w, input=f'{8 * h}x{8 * w}', launches=launches, ms_per_launch=round(ms, 5),
                evaluated_pairs_per_s=float(f'{b * n * n / (ms * 1e-3):.4g}'),
                pair_forward_ms=round(pair_ms, 4), share_of_one_pair_forward=round(ms / b / pair_ms, 5))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--out', help='directory for video_stream.json')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--launches', type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('video_stream_bench.py needs a CUDA device')
    result = dict(card=card())                                     # before any timing
    import tf_raft_b200 as T
    from oracle import weights
    result['workloads'] = [workload(T, weights, H, W, it, args.rounds) for H, W, it in WORKLOADS]
    sintel = result['workloads'][1]
    pair_ms = {(56, 128): 1e3 / sintel['arms']['pairwise_graph']['pairs_per_s_median'],
               (136, 240): pair_forward_ms(T, weights, 1088, 1920, 24)}
    result['forward_interpolate'] = [kernel(T, b, h, w, args.launches, pair_ms[(h, w)]) for b, h, w in KERNEL_SIZES]
    result['notes'] = ('pairs_per_s over the 15 pairs of a 16-frame batch-4 sequence (first frame encode included for '
                       'the stream); pair_forward_ms at 56x128 = the pairwise-graph time per pair at 448x1024 x 24, '
                       'at 136x240 = one batch-1 eager forward at 1088x1920 x 24')
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'video_stream.json'), 'w') as fh:
            fh.write(text + '\n')


if __name__ == '__main__':
    main()
