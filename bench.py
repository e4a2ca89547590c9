#!/usr/bin/env python
"""Headline benchmark: frame-pairs/sec of the RAFT forward at 448x512, iters_pred=12, batch 4 per GPU
(BASELINE.json `metric`, configs[1]); final-flow max-abs vs the oracle reported beside it.

    python bench.py --gpus N --steps K --warmup W                 # this repo's CUDA path, configs[1]
    python bench.py --config sintel ...                           # configs[2]: 448x1024 (436x1024 padded), iters_pred=24
    python bench.py --config train ...                            # configs[3]: training step 384x512, iters=12
    python bench.py --impl reference --steps K --warmup W         # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                        # also write the last timed step's outputs as DIR/<name>.npy

N > 1 is launched by torchrun (one rank per GPU): the batch axis shards (weak scaling: 4 pairs per GPU); inference has
no data-path collective, the training step all-reduces one flat gradient buffer (NCCL) and the context encoder's
BatchNorm statistics.  Prints ONE JSON line (rank 0).
"""
import argparse
import ctypes
import faulthandler
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import torch  # noqa: E402

CONFIGS = {
    'chairs': dict(H=448, W=512, iters=12, B=4, train=False,
                   workload='RAFT inference, batch 4 per GPU, 448x512, iters_pred=12 (BASELINE.json configs[1])'),
    'sintel': dict(H=448, W=1024, iters=24, B=4, train=False,
                   workload='RAFT inference, batch 4 per GPU (32 over 8 GPUs), 436x1024 crop-or-padded to 448x1024, '
                            'iters_pred=24 (BASELINE.json configs[2])'),
    'train': dict(H=384, W=512, iters=12, B=4, train=True,
                  workload='RAFT training step, batch 4 per GPU (32 over 8 GPUs), synthetic FlyingChairs 384x512, iters=12, '
                           'AdamW + one-cycle LR + global-norm clip, NCCL gradient all-reduce (BASELINE.json configs[3])'),
}
METRIC = 'frame-pairs/sec at 448\u00d7512 iters=12; final-flow max-abs vs ref'        # BASELINE.json's string, verbatim (\u00d7 = multiplication sign)
N_ROTATE = 12            # distinct input batches cycled through: 12 x 2 x 11 MB = 264 MB > 126 MB L2

# Algorithmic work of BasicUpdateBlock per feature-grid pixel (update.py:128-153, SURVEY.md section 8(d))
UPDATE_MAC_PER_PX = 3_118_336
# Tensor-core layers of one BasicUpdateBlock application without the mask head (update.py:143-153): (output columns N of the
# tile, 64-channel K chunks incl. taps) -- convc1, convf1, convc2, convf2, conv, z|r x2, q x2, flow_head.conv1, flow_head.conv2
# (N = 32: the CTA pair's minimum).  Used for the shared-memory traffic of update_mega_kernel (DESIGN.md 3.2).
UPDATE_LAYERS_N_CHUNKS = ((256, 6), (128, 2), (192, 36), (64, 18), (128, 36), (256, 30), (256, 30), (128, 30), (128, 30),
                          (256, 18), (32, 36))
MASK_MAC_PER_PX = 294_912 + 147_456               # mask[0] 3x3 128->256 + mask[2] 1x1 256->576 (update.py:137-141): only
                                                  # executed on iterations whose prediction is upsampled
DUMP_LIMIT_BYTES = 64 << 20


def log(msg):
    """progress on stderr (stdout carries only the JSON line)"""
    print(f'[bench {time.strftime("%H:%M:%S")}] {msg}', file=sys.stderr, flush=True)


def dump_outputs(path, arrays):
    """Write {name: array} as path/<name>.npy: what the last timed step returned to its caller, so that two builds run with
    the same arguments (hence the same seeded inputs) can be compared output for output.  Tensors keep float32, host scalars
    become float64.  The largest output (sintel: 4 x 448 x 1024 x 2 float32, 14.7 MB) is stored whole."""
    import numpy as np
    out = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a, dtype=np.float64)
        out[name] = a.astype(np.float64 if a.dtype == np.float64 else np.float32, copy=False)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f'--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES} byte limit')
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + '.npy'), a)
    log(f'outputs of the last timed step written to {path}: ' + ', '.join(f'{k} {tuple(a.shape)}' for k, a in out.items()))


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        d = json.load(open(path))
        return dict(hbm_gbs=float(d['hbm_gbs']), bf16_tflops=float(d.get('bf16_tflops_sustained', d['bf16_tflops'])),
                    bf16_tflops_burst=float(d['bf16_tflops']), source='measured (MEASURED_PEAKS.json)')
    except Exception:
        return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, bf16_tflops_burst=1590.0, source='fallback (B200_PROFILING.md)')


def load_traffic():
    """DRAM bytes per launch of the profiled kernels, extracted from the committed `ncu --set full` captures by
    scripts/ncu_traffic.py (profiles/r02_traffic.json); None when the file is absent."""
    try:
        return json.load(open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')))
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = [r for r in self.rows if len(r) >= 6 and r[0].isdigit()]
        if not rows:
            return None
        sm = sorted(int(r[0]) for r in rows)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith('active') for r in rows)]
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=int(rows[0][1]), reasons=reasons, samples=len(rows))


def oracle_forward_time(cfg, n_pairs, steps, warmup):
    """Time the CPU restatement of the reference forward (oracle/raft_torch.py) on all host cores."""
    import cases
    from oracle import raft_torch as rt, weights
    cores = torch.get_num_threads()      # PyTorch's own intra-op pool size; resizing it after use can stall oneDNN
    p = weights.init_params('raft', 1234)
    im1, im2 = cases.images(n_pairs, cfg['H'], cfg['W'])
    for _ in range(warmup):
        rt.forward(p, im1, im2, 'raft', cfg['iters'])
    t0 = time.perf_counter()
    for _ in range(steps):
        out = rt.forward(p, im1, im2, 'raft', cfg['iters'])
    dt = time.perf_counter() - t0
    return n_pairs * steps / dt, dt / steps, cores, out[-1]


def oracle_train_time(cfg, n_pairs, steps, warmup):
    """One training step (forward, torch.autograd backward, clip, AdamW) of the CPU restatement on all host cores."""
    import cases
    import numpy as np
    from oracle import raft_torch as rt, weights
    cores = torch.get_num_threads()
    p = weights.init_params('raft', 1234)
    frozen = ('moving_mean', 'moving_variance')
    leaves = {k: torch.tensor(v, dtype=torch.float32, requires_grad=not k.endswith(frozen)) for k, v in p.items()}
    names = [k for k, v in leaves.items() if v.requires_grad]
    opt = torch.optim.AdamW([leaves[k] for k in names], lr=1e-4, eps=1e-7, weight_decay=1e-5)
    im1, im2 = cases.images(n_pairs, cfg['H'], cfg['W'])
    gt = torch.from_numpy(np.random.default_rng(3).normal(0, 5, (n_pairs, cfg['H'], cfg['W'], 2)).astype(np.float32))

    def step():
        preds = rt.forward(leaves, im1, im2, 'raft', cfg['iters'], training=True)
        loss = sum(0.8 ** (cfg['iters'] - i - 1) * (q - gt).abs().mean() for i, q in enumerate(preds))
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_([leaves[k] for k in names], 1.0)
        opt.step()
        return loss.detach()
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        loss = step()
    dt = time.perf_counter() - t0
    return n_pairs * steps / dt, dt / steps, cores, loss


def run_reference(args, cfg):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return None
    if cfg['train']:
        pps, sec, cores, loss = oracle_train_time(cfg, 1, args.steps, args.warmup)
        what = 'training step (forward + autograd backward + clip + AdamW)'
        outputs = {'loss': float(loss)}
    else:
        pps, sec, cores, flow = oracle_forward_time(cfg, 1, args.steps, args.warmup)
        what = 'forward'
        outputs = {'flow': flow}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    sample = (f'1 pair per step ({cfg["H"]}x{cfg["W"]}, {cfg["iters"]} iterations, {what}), {args.steps} steps after '
              f'{args.warmup} warm-up')
    return {
        'impl': 'reference', 'metric': METRIC, 'value': pps, 'unit': 'pairs/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': cfg['workload'], 'name': args.config,
                   'sample': 'each step is a bounded sample of that workload: ONE pair of the batch (pairs are independent, '
                             'pairs/s is per pair)',
                   'note': 'reference algorithm restated on PyTorch-CPU (oracle/raft_torch.py): TensorFlow 2.3 is not '
                           'installable in this image, so tf_raft itself cannot run'},
        'cpu_baseline': {'value': pps, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': pps, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }


def run_ours(args, cfg):
    import numpy as np
    import torch.distributed as dist
    import cases
    from oracle import weights
    import tf_raft_b200 as T
    from tf_raft_b200 import _lib, parallel

    H, W, ITERS, B = cfg['H'], cfg['W'], cfg['iters'], cfg['B']
    PX = (H // 8) * (W // 8)
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.gpus > 1 and world == 1:
        raise SystemExit('--gpus N > 1 must be launched with torchrun (one rank per GPU)')
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=device)

    precision = args.precision
    train = cfg['train']
    model = T.RAFT(iters=ITERS, iters_pred=ITERS, precision=precision, device=device, use_graph=not args.no_graph and not train)
    params = weights.init_params('raft', 1234)          # seeded Glorot-uniform (keras defaults), SURVEY 8(d)
    model.load_params(params)

    # synthetic inputs: rotating set of distinct batches, each rank its own seeds (weak scaling)
    n_rot = N_ROTATE if not train else 4
    host = [tuple(torch.from_numpy(a).pin_memory() for a in
                  cases.images(B, H, W, 1000 * rank + 2 * i, 1000 * rank + 2 * i + 1)) for i in range(n_rot)]
    dev_in = [(a.to(device), b.to(device)) for a, b in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        dev_s = e0.elapsed_time(e1) / 1e3
        barrier()
        return parallel.max_over_ranks(dev_s, device), parallel.max_over_ranks(wall, device)

    if train:
        return run_train(args, cfg, model, host, dev_in, timed, barrier, rank, world, local, device)

    last = {}

    def step_resident(i):
        a, b = dev_in[i % n_rot]
        last['flow'] = model([a, b], training=False, last_only=True)[-1]
        return last['flow']

    def step_e2e(i):
        a, b = host[i % n_rot]
        out = model.predict_step((a.to(device, non_blocking=True), b.to(device, non_blocking=True)))
        return out.to('cpu', non_blocking=False)

    log('model and inputs ready; warm-up')
    for i in range(args.warmup):
        step_resident(i)
    torch.cuda.synchronize()
    log('warm-up done; timing device-resident steps')
    # kernels per step: counted on one directly-launched forward (a CUDA-graph replay launches the same kernel
    # nodes without passing through the host-side counter)
    _lib.launch_count_reset()
    model._forward(dev_in[0][0], dev_in[0][1], False, True)
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    dev_s, _ = timed(step_resident, args.steps)
    clocks = sampler.stop() if sampler else None
    # the CUDA graph returns a static buffer that the next replay overwrites: keep the last timed step's flow now
    timed_flow = last['flow'].cpu() if args.dump_outputs and rank == 0 else None
    launches = launches_per_step * args.steps
    value = world * B * args.steps / dev_s

    log(f'resident: {value:.1f} pairs/s; timing end-to-end steps')
    for i in range(min(args.warmup, 2)):
        step_e2e(i)
    if not args.sync_e2e:  # uploads / read-backs overlapped with the neighbouring steps' compute (same copies every step)
        def run_pipelined(steps):
            barrier()
            t0 = time.perf_counter()
            n = 0
            for out in parallel.predict_stream(lambda a, b: model.predict_step((a, b)),
                                               (host[i % n_rot] for i in range(steps)), device, reuse_host_buffers=True):
                n += out.shape[0]
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            assert n == steps * B
            barrier()
            return parallel.max_over_ranks(wall, device)
        run_pipelined(2)
        # wall-clock leg of K steps: host jitter of a shared box moves it by tens of percent from one run to the next
        # (profiles/README.md), so it is run twice and the faster run is reported; both are kept in `e2e.runs_pairs_per_s`
        e2e_walls = [run_pipelined(args.steps), run_pipelined(args.steps)]
        e2e_wall = min(e2e_walls)
    else:
        _, e2e_wall = timed(step_e2e, args.steps)
        e2e_walls = [e2e_wall]
    e2e_value = world * B * args.steps / e2e_wall
    h2d = 2 * B * H * W * 3 * 4
    d2h = B * H * W * 2 * 4

    line = None
    if rank == 0:
        peaks = load_peaks()
        traffic = load_traffic() or {}
        log(f'e2e: {e2e_value:.1f} pairs/s; kernel-level timings')
        # --- kernel-level timing for the roofline objects (rank 0, CUDA events on the launching stream) ---
        a, b = dev_in[0]
        fmap1, fmap2, net, inp = model._encode(a, b, False)
        h, w = H // 8, W // 8

        def ev_time(fn, reps=5):
            fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / 1e3 / reps

        cb = T.CorrBlock(fmap1, fmap2, 4, 4, precision=precision)
        pyr_ptrs = _lib.ptr_array(cb.corr_pyramid)

        def build_corr():           # same buffers every time: times the kernels, not the allocator
            _lib.check(_lib.lib().raft_b200_corr_pyramid_build(
                _lib.ptr(fmap1), _lib.ptr(fmap2), B, h, w, 256, 4, pyr_ptrs, _lib.ptr(cb._ws), cb._ws.numel(),
                cb.precision, _lib.stream()), 'corr_pyramid_build')
        t_corr = ev_time(build_corr)
        # the loop exactly as the timed step runs it (last prediction only), with the library's per-kernel events armed:
        # lookup = the fp16 hi/lo-plane variant the loop uses (it also writes convf1's im2col planes), update = the update-block kernel(s)
        preds = [None] * (ITERS - 1) + [torch.empty((B, H, W, 2), device=device)]
        L = _lib.lib()
        reps, t_lookup, t_update = 3, 0.0, 0.0
        for r in range(reps + 1):
            c1 = T.coords_grid(B, h, w, device)
            net_r = net.clone()
            L.raft_b200_profile_loop(1)
            model._loop(cb, net_r, inp, c1, preds, B, h, w)
            lk, up, n_it = ctypes.c_float(), ctypes.c_float(), ctypes.c_int()
            _lib.check(L.raft_b200_profile_read(ctypes.byref(lk), ctypes.byref(up), ctypes.byref(n_it)), 'profile_read')
            L.raft_b200_profile_loop(0)
            if r > 0:                                 # first pass = warm-up
                t_lookup += lk.value / 1e3 / ITERS / reps
                t_update += up.value / 1e3 / ITERS / reps
        n_upsampled = sum(1 for q in preds if q is not None)      # the timed loop upsamples the last prediction only
        flops_per_launch = 2.0 * ((UPDATE_MAC_PER_PX - MASK_MAC_PER_PX) * ITERS + MASK_MAC_PER_PX * n_upsampled) * PX * B / ITERS
        ach_tflops = flops_per_launch / max(t_update, 1e-9) / 1e12
        corr_bytes_pair = 4 * sum(PX * ((H // 8) >> l) * ((W // 8) >> l) for l in range(4)) + 8 * PX * 256
        lookup_bytes = B * PX * 2904
        # in the loop the lookup launch also writes the im2col planes of the current flow for convf1 (2 planes x 128 channels x
        # 2 bytes per query, + the 8-byte flow it reads): part of that launch's algorithmic traffic, listed separately
        rider_bytes = B * PX * (2 * 128 * 2 + 8)
        corr_bytes = B * corr_bytes_pair + ITERS * (lookup_bytes + rider_bytes)
        ach_gbs = corr_bytes / (t_corr + ITERS * t_lookup) / 1e9
        corr_flops_3pass = 3 * B * 2.0 * 256 * sum(PX * ((H // 8) >> l) * ((W // 8) >> l) for l in range(4))

        if args.quick or world > 1:     # the CPU legs (oracle parity, CPU baseline) belong to the N=1 line only
            parity, max_abs, cpu_pps, cores = {'skipped': '--quick' if args.quick else 'reported at N=1'}, None, None, 0
        else:
            log('parity check of the timed configuration against the oracle')
            # --- parity of the TIMED configuration (CUDA graph, last prediction only, batch 4) against the oracle, pair 0;
            #     a plain (no graph, all predictions) model gives the per-iteration trace ---
            from oracle import raft_torch as rt
            im1, im2 = cases.images(B, H, W, 0, 1)
            want = rt.forward(params, im1[:1], im2[:1], 'raft', ITERS)
            timed_out = step_resident(0).clone()                 # dev_in[0] was generated from seeds (0, 1) on rank 0
            check_model = T.RAFT(iters=ITERS, iters_pred=ITERS, precision=precision, device=device)
            check_model.load_params(params)
            got = check_model([dev_in[0][0][:1], dev_in[0][1][:1]], training=False)
            per_iter = [float((g.cpu() - o).abs().max()) for g, o in zip(got, want)]
            final_err = (timed_out[:1].cpu() - want[-1]).abs()
            max_abs = float(final_err.max())
            within = 0
            while within < ITERS and per_iter[within] <= 1e-3:
                within += 1
            parity = {'max_abs': max_abs, 'median_abs': float(final_err.flatten().median()),
                      'frac_px_within_1e-3': float((final_err <= 1e-3).float().mean()),
                      'checked': 'output of the timed path itself (CUDA graph, last_only, batch 4), pair 0',
                      'timed_path_equals_plain_path': bool(torch.equal(timed_out[:1], got[-1])),
                      'iterations_within_1e-3': within, 'max_abs_per_iteration': per_iter,
                      'flow_magnitude_px': float(want[-1].abs().max()),
                      'note': 'free-running vs the CPU oracle on pair 0; the reference sampler is discontinuous at integer / '
                              'border coordinates (corr.py:45-60), so once one tap crosses, that pixel legitimately diverges '
                              '(DESIGN.md section 4); teacher-forced stage parity is in tests/test_gpu_stages.py'}
            log(f'max-abs {max_abs:.2e}; CPU baseline')
            # --- CPU baseline: the restated reference on the host cores, bounded sample ---
            cpu_pps, cpu_sec, cores, _ = oracle_forward_time(cfg, 1, 3, 1)

        mega_traffic = traffic.get('update_mega_kernel')
        line = {
            'metric': METRIC, 'value': value, 'unit': 'pairs/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': dev_s / args.steps * 1e3, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': cfg['workload'], 'name': args.config, 'global_batch': world * B, 'parallelism': f'dp{world}',
                       'arithmetic': {'f16x2': 'tcgen05 fp16 hi/lo split, 3 passes, fp32 accumulate (fp32-grade)',
                                      'fp32': 'CUDA-core FFMA'}[precision],
                       'encoders': {'f16x2': 'native: the same tcgen05 implicit-GEMM kernel (stride-2 TMA boxes, fused norm affine)',
                                    'fp32': 'cuDNN IEEE fp32 via PyTorch'}[precision],
                       'cuda_graph': not args.no_graph, 'last_only': True,
                       'l2': f'inputs rotate over {n_rot} distinct batches ({n_rot * 2 * B * H * W * 12 / 1e6:.0f} MB) and every step '
                             f'rewrites the {B * corr_bytes_pair / 1e6:.0f} MB correlation pyramid: working set > 126 MB L2'},
            'final_flow_max_abs_vs_oracle': max_abs,
            'parity': parity,
            'e2e': {'value': e2e_value, 'unit': 'pairs/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'runs_pairs_per_s': [world * B * args.steps / t for t in e2e_walls],
                    'api': 'RAFT.predict_step, one synchronous call per step' if args.sync_e2e else
                           'parallel.predict_stream over RAFT.predict_step: pinned host -> device -> host every step, copies '
                           'overlapped with the neighbouring steps (device-timed `value` explains it)'},
            'gpu_launches': int(launches),
            'clocks': clocks,
            'roofline': {'bound': 'tensor',
                         'kernel': 'update_mega_kernel (all tensor-core layers of one update-block application; one launch per '
                                   'iteration)',
                         'achieved': ach_tflops, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s',
                         'frac': ach_tflops / peaks['bf16_tflops'],
                         'traffic': mega_traffic,
                         'algorithmic_flops_per_launch': flops_per_launch, 'ms_per_launch': t_update * 1e3,
                         'peak_source': peaks['source'] + ' (sustained cuBLAS bf16: the kernel runs inside a long step)',
                         'note': 'achieved = algorithmic fp32 FLOPs one launch executes (2*2,675,968 MAC/px; + 2*442,368 MAC/px of '
                                 'mask head on the one upsampled iteration, averaged over the launches) / CUDA-event time per '
                                 'launch measured inside raft_b200_forward_loop; the kernel executes 3 fp16 MMA passes per '
                                 'FLOP, so the tensor pipe is 3x busier than `frac`',
                         'executed_frac': 3 * ach_tflops / peaks['bf16_tflops'],
                         # what the mainloop is measured to sit on (profiles/README.md): per 64-channel chunk a CTA of a pair
                         # receives 32 KB of activations + N/2 weight rows by TMA and its twelve MMAs read 12 x (4 KB + N x 32 B)
                         'shared_memory': (lambda by, pk: {
                             'bytes_per_launch': by, 'achieved_TBps': by / max(t_update, 1e-9) / 1e12, 'peak_TBps': pk / 1e12,
                             'frac': by / max(t_update, 1e-9) / pk,
                             'note': 'TMA writes + tcgen05 operand reads of shared memory per launch (mask head excluded) against '
                                     f'148 SMs x 128 B/clk at the sampled SM clock; a layer has {B * PX // 128} tiles for 148 SMs and '
                                     'the 9 chain layers run one after the other (at 112 tiles: 0.76 of this peak at most)'})(
                             B * PX / 128 * sum(c * (32768 + (n // 2) * 256 + 12 * (4096 + n * 32)) for n, c in UPDATE_LAYERS_N_CHUNKS),
                             148 * 128 * 1e6 * float((clocks or {}).get('sm_mhz') or 1965))},
            'roofline_corr_lookup': {'bound': 'hbm', 'kernel': f'correlation pyramid build + {ITERS} lookups',
                                     'achieved': ach_gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                                     'frac': ach_gbs / peaks['hbm_gbs'],
                                     'traffic': {'lookup': traffic.get('corr_lookup_win_kernel'),
                                                 'correlation': traffic.get('corr_tc_kernel'),
                                                 'lookup_algorithmic_bytes': lookup_bytes,
                                                 'lookup_launch_im2col_rider_bytes': rider_bytes,
                                                 'correlation_algorithmic_bytes': B * corr_bytes_pair},
                                     'ms': {'pyramid_build': t_corr * 1e3, 'lookup': t_lookup * 1e3},
                                     'pyramid_build_alone': {
                                         'hbm_frac': B * corr_bytes_pair / t_corr / 1e9 / peaks['hbm_gbs'],
                                         'tensor_frac_3pass': corr_flops_3pass / t_corr / 1e12 / peaks['bf16_tflops_burst'],
                                         'note': 'the fp32-grade correlation needs 3 fp16 passes, which makes the tensor pipe '
                                                 '(burst cuBLAS peak) its tighter bound; both fractions given'},
                                     'lookup_alone_hbm_frac': (lookup_bytes + rider_bytes) / t_lookup / 1e9 / peaks['hbm_gbs'],
                                     'peak_source': peaks['source']},
            'cpu_baseline': {'value': cpu_pps, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port',
                             'sample': f'1 pair ({H}x{W}, {ITERS} iterations) x 3 steps after 1 warm-up, '
                                       'oracle/raft_torch.py on all host cores'},
        }
    if timed_flow is not None:
        dump_outputs(args.dump_outputs, {'flow': timed_flow})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


def run_train(args, cfg, model, host, dev_in, timed, barrier, rank, world, local, device):
    """configs[3]: the reference's train_step (model.py:126-144) on synthetic FlyingChairs-shaped data."""
    import numpy as np
    import torch.distributed as dist
    from tf_raft_b200 import _lib
    from tf_raft_b200.train import AdamW, CyclicalLearningRate, first_cycle_scaler
    H, W, ITERS, B = cfg['H'], cfg['W'], cfg['iters'], cfg['B']
    n_rot = len(host)
    rng = np.random.default_rng(77 + rank)
    flows = [torch.from_numpy(rng.normal(0, 5, (B, H, W, 2)).astype(np.float32)).pin_memory() for _ in range(n_rot)]
    valid = torch.ones((B, H, W), dtype=torch.bool)
    dev_fl = [f.to(device) for f in flows]
    dev_va = valid.to(device)
    sched = CyclicalLearningRate(1e-4, 2e-4, 1000, scale_fn=first_cycle_scaler)      # train_chairs.py:79-85 (lr 1e-4)
    model.compile(optimizer=AdamW(weight_decay=1e-5, learning_rate=sched), clip_norm=1.0)   # :87-98

    losses = []
    last = {}

    def step_resident(i):
        a, b = dev_in[i % n_rot]
        out = model.train_step((a, b, dev_fl[i % n_rot], dev_va))
        losses.append(out['loss'])
        last['metrics'] = out

    def step_e2e(i):
        a, b = host[i % n_rot]
        out = model.train_step((a.to(device, non_blocking=True), b.to(device, non_blocking=True),
                                flows[i % n_rot].to(device, non_blocking=True), dev_va))
        return out['loss']                      # python float: the loss has been read back from the device

    log('model and inputs ready; warm-up')
    for i in range(args.warmup):
        step_resident(i)
    torch.cuda.synchronize()
    _lib.launch_count_reset()
    step_resident(0)
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    dev_s, _ = timed(step_resident, args.steps)
    clocks = sampler.stop() if sampler else None
    timed_metrics = last['metrics']                # what train_step returned on the last timed step: the running metrics
    value = world * B * args.steps / dev_s
    log(f'resident: {value:.2f} pairs/s; end-to-end steps')
    _, e2e_wall = timed(step_e2e, args.steps)
    e2e_value = world * B * args.steps / e2e_wall
    # cost of the collective: the flat gradient all-reduce alone, timed on the device
    tr = model._trainer
    ar_ms = None
    if world > 1:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(10):
            dist.all_reduce(tr.flat.g)
        e1.record()
        torch.cuda.synchronize()
        ar_ms = e0.elapsed_time(e1) / 10
    line = None
    if rank == 0:
        cpu = None
        if not args.quick and world == 1:
            log('CPU baseline: one oracle training step')
            cpu_pps, _, cores, _ = oracle_train_time(cfg, 1, 1, 0)
            cpu = {'value': cpu_pps, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port',
                   'sample': f'1 pair ({H}x{W}, {ITERS} iterations), one training step of oracle/raft_torch.py under torch.autograd'}
        line = {
            'metric': 'frame-pairs/sec of the training step at 384x512 iters=12 (forward + backward + clip + AdamW)',
            'value': value, 'unit': 'pairs/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': dev_s / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': cfg['workload'], 'name': args.config, 'global_batch': world * B, 'parallelism': f'dp{world}',
                       'collectives': 'one flat fp32 gradient all-reduce per step (NCCL) + all-reduced BatchNorm statistics of the '
                                      'context encoder (forward and backward)',
                       'gradient_bytes': int(tr.flat.g.numel() * 4), 'allreduce_ms': ar_ms,
                       'arithmetic': 'correlation forward: tcgen05 fp16 hi/lo; lookup forward/backward, clip + AdamW: hand-written '
                                     'CUDA; convolutions / norms / gates forward and backward: IEEE-fp32 cuDNN via torch.autograd'},
            'loss_first_last': [losses[0], losses[-1]],
            'e2e': {'value': e2e_value, 'unit': 'pairs/s', 'h2d_bytes_per_step': 2 * B * H * W * 3 * 4 + B * H * W * 2 * 4,
                    'd2h_bytes_per_step': 4, 'api': 'RAFT.train_step (images and ground-truth flow uploaded every step, loss read back)'},
            'gpu_launches': int(launches_per_step * args.steps),
            'clocks': clocks,
            'cpu_baseline': cpu,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, timed_metrics)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='chairs', choices=sorted(CONFIGS),
                    help='chairs = BASELINE.json configs[1] (the headline), sintel = configs[2], train = configs[3]')
    ap.add_argument('--no-graph', action='store_true', help='launch kernels directly instead of replaying a CUDA graph')
    ap.add_argument('--sync-e2e', action='store_true',
                    help='end-to-end leg as one synchronous predict_step per step instead of parallel.predict_stream')
    ap.add_argument('--quick', action='store_true', help='timing only: skip the parity and CPU-baseline legs (A/B runs)')
    ap.add_argument('--precision', default=os.environ.get('RAFT_B200_PRECISION', 'f16x2'), choices=['f16x2', 'fp32'])
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one returned as DIR/<name>.npy (float32 / float64)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    cfg = CONFIGS[args.config]
    # stdout must carry exactly one JSON line: libraries (NCCL prints its version banner there) get stderr instead
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    # torchrun exports OMP_NUM_THREADS=1; the CPU baseline / reference arm should use the host's cores.  Size the
    # intra-op pool once, before its first use (resizing a pool that is already in use stalled oneDNN for minutes).
    torch.set_num_threads(max(1, min(host_cores(), 64)))
    faulthandler.enable()
    faulthandler.dump_traceback_later(600, exit=False)     # a hang leaves stack traces on stderr
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else max(args.warmup, 1)
    line = run_reference(args, cfg) if args.impl == 'reference' else run_ours(args, cfg)
    if line is not None:
        os.write(real_stdout, (json.dumps(line) + '\n').encode())


if __name__ == '__main__':
    main()
