"""A/B of two library builds on the encoders' memory-bound passes: bitwise outputs, per-kernel times, bench steps.

    # on the build machine: cross-compile a git revision's library into the ignored build/ tree
    python scripts/encoder_passes_ab.py --build-base HEAD~1            # -> build/base/libraft_b200.so
    # on the GPU (both libraries travel with the tree)
    python scripts/encoder_passes_ab.py --base build/base/libraft_b200.so --out OUTDIR [--bench-rounds 3]

Each build runs in subprocesses of its own (`_lib` loads one library per process, chosen by RAFT_B200_LIB):
  (a) encoder outputs of both builds compared with torch.equal: fnet and cnet for RAFT and SmallRAFT weights at
      448x512 batch 4 (8 images into fnet), 448x1024 batch 4, the ragged 72x104 batch 3 (raw and already-normalised
      input) and training-mode cnet (batch statistics) at 64x96 batch 2;
  (b) torch.profiler (CUDA activities) over the encoders of one bench step (fnet on 8 images + cnet on 4, 448x512),
      in a run of its own: us per step and achieved GB/s of the stem gather (with `image_norm_kernel`, where a build
      has it), `norm_stats_kernel` and, as a reference point, `norm_apply_kernel`;
  (c) with --bench-rounds R: `bench.py --quick` alternating base / new R times each per configuration, with
      --dump-outputs, comparing every dumped flow with np.array_equal;
and OUTDIR/encoder_passes_ab.json gets all of it with the card name and power limit.
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_LIB = os.path.join(ROOT, 'tf_raft_b200', 'libraft_b200.so')

# (name, variant, which, N, H, W, training, raw_image)
OUTPUT_CASES = []
for _v in ('raft', 'small'):
    OUTPUT_CASES += [(f'{_v}.fnet.448x512', _v, 'fnet', 8, 448, 512, False, True),
                     (f'{_v}.cnet.448x512', _v, 'cnet', 4, 448, 512, False, True),
                     (f'{_v}.fnet.448x1024', _v, 'fnet', 8, 448, 1024, False, True),
                     (f'{_v}.cnet.448x1024', _v, 'cnet', 4, 448, 1024, False, True),
                     (f'{_v}.fnet.72x104', _v, 'fnet', 3, 72, 104, False, True),
                     (f'{_v}.cnet.72x104', _v, 'cnet', 3, 72, 104, False, True),
                     (f'{_v}.fnet.72x104.normalised', _v, 'fnet', 3, 72, 104, False, False)]
OUTPUT_CASES.append(('raft.cnet.64x96.training', 'raft', 'cnet', 2, 64, 96, True, True))


def _encoder(variant, which, seed=99):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from oracle import raft_torch as rt, weights
    from tf_raft_b200.layers.extractor import BasicEncoder, SmallEncoder
    p = weights.init_params(variant, seed, bias_scale=0.05, norm_jitter=0.2)
    cfg = rt.VARIANTS[variant]
    norm = cfg['fnorm'] if which == 'fnet' else cfg['cnorm']
    out_dim = {('raft', 'fnet'): 256, ('raft', 'cnet'): 256, ('small', 'fnet'): 128, ('small', 'cnet'): 160}[(variant, which)]
    enc = (BasicEncoder if variant == 'raft' else SmallEncoder)(output_dim=out_dim, norm_type=norm, backend='native')
    enc.load_params(p, which + '.')
    return enc


def _image(n, h, w, raw, seed):
    import numpy as np
    import torch
    x = torch.from_numpy(np.random.default_rng(seed).uniform(0, 255, (n, h, w, 3)).astype(np.float32))
    if not raw:
        x = 2 * (x / 255.0) - 1.0
    return x.cuda()


def worker_outputs(outdir):
    import torch
    for i, (name, variant, which, n, h, w, training, raw) in enumerate(OUTPUT_CASES):
        enc = _encoder(variant, which)
        y = enc(_image(n, h, w, raw, 40 + i), training=training, raw_image=raw)
        torch.cuda.synchronize()
        torch.save(y.cpu(), os.path.join(outdir, name + '.pt'))


def pass_bytes(variant, n_f, n_c, H, W):
    """Bytes each pass has to move per bench step (fnet on n_f images with instance norm, cnet on n_c images)."""
    c0, cs = (64, (64, 96, 128)) if variant == 'raft' else (32, (32, 64, 96))
    pad64 = lambda c: -(-c // 64) * 64
    h, w = -(-H // 2), -(-W // 2)
    stem = (n_f + n_c) * (H * W * 3 * 4 + h * w * 192 * 2 * 2)     # image read once, hi + lo planes written
    # fnet norms: (pixels, C, skip bytes per pixel, output bytes per pixel)
    norms = [(h * w, c0, 0, pad64(c0) * 4)]
    for k in range(6):
        c, st = cs[k // 2], ((1, 2, 2)[k // 2] if k % 2 == 0 else 1)
        h, w = -(-h // st), -(-w // st)
        norms.append((h * w, c, 0, pad64(c) * 4))                       # norm1 -> hi/lo
        if st != 1:
            norms.append((h * w, c, 0, c * 4))                          # downsample norm -> fp32
        norms.append((h * w, c, c * 4 if st != 1 else pad64(c) * 4, pad64(c) * 4))   # norm2 + skip -> hi/lo
    stats = n_f * sum(p * c * 4 for p, c, _, _ in norms)
    apply = n_f * sum(p * (c * 4 + s + o) for p, c, s, o in norms)
    return {'stem': stem, 'norm_stats_kernel': stats, 'norm_apply_kernel': apply}


def worker_profile(outpath, steps=20):
    import torch
    from torch.profiler import ProfilerActivity, profile
    H, W, B = 448, 512, 4
    fnet, cnet = _encoder('raft', 'fnet'), _encoder('raft', 'cnet')
    im1, im2 = _image(B, H, W, True, 1), _image(B, H, W, True, 2)

    def step():
        fnet([im1, im2], training=False, raw_image=True)
        cnet(im1, training=False, raw_image=True)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
    us = {}
    for ev in prof.key_averages():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            us[ev.key] = us.get(ev.key, 0.0) + ev.device_time_total / steps
    groups = {'stem': ('stem_gather_kernel', 'stem_im2col_kernel', 'image_norm_kernel'),
              'norm_stats_kernel': ('norm_stats_kernel',), 'norm_apply_kernel': ('norm_apply_kernel',)}
    nbytes = pass_bytes('raft', 2 * B, B, H, W)
    res = {}
    for g, names in groups.items():
        parts = {k: v for k, v in us.items() if any(nm in k for nm in names)}
        t = sum(parts.values())
        res[g] = {'us_per_step': t, 'bytes_per_step': nbytes[g], 'GB_per_s': nbytes[g] / t / 1e3 if t else None,
                  'kernels': {k.split('(')[0].replace('void ', '').replace('raft::', ''): v for k, v in parts.items()}}
    # norm_stats_kernel launch by launch (fnet's 15 norms in order), averaged over the profiled steps
    st = [e.time_range.elapsed_us() for e in prof.events()
          if e.device_type == torch.autograd.DeviceType.CUDA and 'norm_stats_kernel' in e.name]
    per = len(st) // steps
    res['norm_stats_kernel']['launch_us'] = [sum(st[k::per]) / steps for k in range(per)] if per else []
    res['all_kernels_us_per_step'] = sum(us.values())
    with open(outpath, 'w') as f:
        json.dump(res, f, indent=1)


def run_worker(lib, mode, target):
    env = dict(os.environ, RAFT_B200_LIB=os.path.abspath(lib))
    subprocess.run([sys.executable, os.path.abspath(__file__), '--worker', mode, '--target', target], env=env, cwd=ROOT,
                   check=True)


def run_bench(lib, config, dump_dir, steps, warmup):
    env = dict(os.environ, RAFT_B200_LIB=os.path.abspath(lib))
    cmd = [sys.executable, 'bench.py', '--gpus', '1', '--quick', '--config', config, '--steps', str(steps),
           '--warmup', str(warmup), '--dump-outputs', dump_dir]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f'bench failed ({lib}, {config}):\n{r.stderr[-3000:]}')
    return json.loads(r.stdout.strip().splitlines()[-1])


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else 'unknown'


def build_base(rev):
    """Cross-compile `rev`'s library (sources from git, flags of tf_raft_b200/build.py) into build/base/."""
    sys.path.insert(0, ROOT)
    from tf_raft_b200 import build as B
    src = tempfile.mkdtemp(prefix='enc_ab_src_')
    try:
        arch = subprocess.run(['git', 'archive', rev, 'tf_raft_b200/csrc', 'include'], cwd=ROOT, capture_output=True,
                              check=True).stdout
        subprocess.run(['tar', '-x', '-C', src], input=arch, check=True)
        out = os.path.join(ROOT, 'build', 'base', 'libraft_b200.so')
        os.makedirs(os.path.dirname(out), exist_ok=True)
        flags = [f for f in B.NVCC_FLAGS if not f.startswith('--use_fast_math')]
        subprocess.run([B._nvcc()] + flags + [os.path.join(src, 'tf_raft_b200', 'csrc', s) for s in B.SOURCES] +
                       ['-o', out], check=True)
        print(out)
    finally:
        shutil.rmtree(src)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--build-base', metavar='REV')
    ap.add_argument('--base', help='library of the base build')
    ap.add_argument('--new', default=NEW_LIB, help='library of the new build (default: the in-tree build)')
    ap.add_argument('--out', help='directory for encoder_passes_ab.json')
    ap.add_argument('--bench-rounds', type=int, default=0)
    ap.add_argument('--bench-configs', default='chairs,sintel')
    ap.add_argument('--bench-steps', type=int, default=20)
    ap.add_argument('--bench-warmup', type=int, default=5)
    ap.add_argument('--worker', choices=['outputs', 'profile'])
    ap.add_argument('--target')
    a = ap.parse_args()
    if a.build_base:
        return build_base(a.build_base)
    if a.worker == 'outputs':
        return worker_outputs(a.target)
    if a.worker == 'profile':
        return worker_profile(a.target)
    if not a.base or not a.out:
        ap.error('--base and --out are required')
    import numpy as np
    import torch
    os.makedirs(a.out, exist_ok=True)
    libs = {'base': a.base, 'new': a.new}
    res = {'card': card(), 'libs': {k: os.path.relpath(os.path.abspath(v), ROOT) for k, v in libs.items()}}
    tmp = tempfile.mkdtemp(prefix='enc_ab_')
    try:
        # (a) bitwise outputs
        for side, lib in libs.items():
            os.makedirs(os.path.join(tmp, side))
            run_worker(lib, 'outputs', os.path.join(tmp, side))
        eq = {}
        for name, *_ in OUTPUT_CASES:
            x, y = (torch.load(os.path.join(tmp, s, name + '.pt')) for s in ('base', 'new'))
            eq[name] = bool(torch.equal(x, y))
            print(f'{name:<32} equal={eq[name]}' + ('' if eq[name] else f'  max-abs {float((x - y).abs().max()):.3e}'))
        res['outputs_equal'] = eq
        # (b) per-kernel times
        res['profile'] = {}
        for side, lib in libs.items():
            path = os.path.join(tmp, f'profile_{side}.json')
            run_worker(lib, 'profile', path)
            res['profile'][side] = json.load(open(path))
            for g in ('stem', 'norm_stats_kernel', 'norm_apply_kernel'):
                d = res['profile'][side][g]
                print(f'{side:<4} {g:<18} {d["us_per_step"]:8.1f} us/step  {d["GB_per_s"] or 0:7.0f} GB/s  {d["kernels"]}')
        # (c) bench steps, alternating, with bitwise flow comparison (a timing of differing outputs means nothing)
        if a.bench_rounds and all(eq.values()):
            res['bench'] = {}
            for config in a.bench_configs.split(','):
                ms = {'base': [], 'new': []}
                flows_equal = True
                for r in range(a.bench_rounds):
                    flows = {}
                    for side, lib in libs.items():
                        d = os.path.join(tmp, f'dump_{config}_{side}_{r}')
                        line = run_bench(lib, config, d, a.bench_steps, a.bench_warmup)
                        ms[side].append(line['ms_per_step'])
                        flows[side] = np.load(os.path.join(d, 'flow.npy'))
                        print(f'bench {config} round {r} {side}: {line["ms_per_step"]:.3f} ms/step, {line["value"]:.1f} pairs/s')
                    flows_equal &= bool(np.array_equal(flows['base'], flows['new']))
                summ = {s: {'ms_per_step': v, 'median': statistics.median(v), 'spread': max(v) - min(v)} for s, v in ms.items()}
                summ['median_delta_ms'] = summ['new']['median'] - summ['base']['median']
                summ['flow_array_equal'] = flows_equal
                res['bench'][config] = summ
                print(f'bench {config}: base median {summ["base"]["median"]:.3f} (spread {summ["base"]["spread"]:.3f}), '
                      f'new median {summ["new"]["median"]:.3f} (spread {summ["new"]["spread"]:.3f}), '
                      f'delta {summ["median_delta_ms"]:+.3f} ms, flows equal {flows_equal}')
    finally:
        shutil.rmtree(tmp)
    res['card_after'] = card()
    with open(os.path.join(a.out, 'encoder_passes_ab.json'), 'w') as f:
        json.dump(res, f, indent=1)
    ok = all(res['outputs_equal'].values()) and all(b['flow_array_equal'] for b in res.get('bench', {}).values())
    print('all outputs bitwise equal' if ok else 'OUTPUTS DIFFER')
    return 0 if ok else 1


if __name__ == '__main__':
    sys.exit(main())
