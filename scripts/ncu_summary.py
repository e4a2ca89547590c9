"""Summarise an `ncu --metrics gpu__time_duration.sum --csv` launch list.

  python scripts/ncu_summary.py launches.csv                  per-kernel totals
  python scripts/ncu_summary.py launches.csv --seq START N    launch sequence (grid, duration) from launch START
  python scripts/ncu_summary.py launches.csv --forward [K]    breakdown of the K-th model forward (default: the last
                                                              one whose lookup grid is the largest, i.e. a full batch):
                                                              before-the-loop vs one loop iteration, encoder conv list
A forward starts at a `stem_gather_kernel` pair (feature + context encoder) and ends before the next one.
"""
import collections, csv, sys


def load(path):
    rows = list(csv.reader(open(path, errors='ignore')))
    hdr, seq = None, []
    for r in rows:
        if 'Kernel Name' in r:
            hdr = r
            continue
        if hdr and len(r) == len(hdr):
            d = dict(zip(hdr, r))
            if d.get('Metric Name') != 'gpu__time_duration.sum':
                continue
            try:
                v = float(d['Metric Value'].replace(',', ''))
            except ValueError:
                continue
            unit = d.get('Metric Unit', 'ns')
            us = v / 1e3 if unit in ('ns', 'nsecond') else v if unit in ('us', 'usecond') else v * 1e3
            seq.append((d['Kernel Name'].replace('void ', '').replace('raft::', '')[:64], d.get('Grid Size', ''), us))
    return seq


def totals(seq):
    agg = collections.defaultdict(lambda: [0, 0.0])
    for k, _, us in seq:
        agg[k][0] += 1
        agg[k][1] += us
    tot = sum(v[1] for v in agg.values())
    for k, (n, t) in sorted(agg.items(), key=lambda kv: -kv[1][1])[:30]:
        print(f'{t/1e3:9.3f} ms {100*t/tot:5.1f}%  n={n:5d}  avg {t/n:8.1f} us  {k}')
    print(f'total {tot/1e3:.3f} ms over {len(seq)} launches')


def forward(seq, which):
    starts = [i for i, (k, _, _) in enumerate(seq) if k.startswith('stem_gather_kernel')]
    fws = []
    for a in range(0, len(starts) - 1, 2):
        end = starts[a + 2] if a + 2 < len(starts) else len(seq)
        fw = seq[starts[a]:end]
        lk = [int(g.strip('()').split(',')[0]) for k, g, _ in fw if k.startswith('corr_lookup')]
        fws.append((fw, lk[0] if lk else 0))
    if not fws:
        sys.exit('no forward found (no stem_gather_kernel launches)')
    if which is None:
        big = max(g for _, g in fws)
        which = max(i for i, (fw, g) in enumerate(fws) if g == big and len(fw) == min(len(f) for f, gg in fws if gg == big))
    fw, grid = fws[which]
    lks = [i for i, (k, _, _) in enumerate(fw) if k.startswith('corr_lookup')]
    pre = fw[:lks[0]] if lks else fw
    print(f'forward {which}: {len(fw)} launches, {sum(u for _, _, u in fw)/1e3:.3f} ms of kernel time, lookup grid {grid}')
    print(f'before the loop: {sum(u for _, _, u in pre)/1e3:.3f} ms in {len(pre)} launches')
    agg = collections.defaultdict(float)
    for k, _, us in pre:
        agg[k[:44]] += us
    for k, t in sorted(agg.items(), key=lambda kv: -kv[1])[:10]:
        print(f'   {t:9.1f} us  {k}')
    print('   tensor-core convolutions before the loop (us/grid): ' +
          ' '.join(f"{us:.0f}/{g.strip('()').split(',')[0]}" for k, g, us in pre if k.startswith('conv_tc_kernel')))
    if len(lks) > 6:
        it = fw[lks[5]:lks[6]]
        print(f'one loop iteration (the 6th): {sum(u for _, _, u in it):.1f} us')
        for k, g, us in it:
            print(f'   {us:7.1f} us  grid {g:>14}  {k[:50]}')


def main():
    seq = load(sys.argv[1])
    if '--forward' in sys.argv:
        i = sys.argv.index('--forward')
        forward(seq, int(sys.argv[i + 1]) if len(sys.argv) > i + 1 else None)
        return
    totals(seq)
    if '--seq' in sys.argv:
        start = int(sys.argv[sys.argv.index('--seq') + 1])
        count = int(sys.argv[sys.argv.index('--seq') + 2])
        for k, g, us in seq[start:start + count]:
            print(f'{us:9.1f} us  grid {g:>16}  {k}')


if __name__ == '__main__':
    main()
