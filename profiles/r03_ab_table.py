"""Tabulate the bench lines written by profiles/r03_bwd_ab.sh: ms_per_step and kernel_ms.blend_bwd of every run, and per
(workload, library) the median and the spread (max - min).
python profiles/r03_ab_table.py OUT_DIR"""
import collections
import glob
import json
import os
import re
import sys


def main(out):
    runs = collections.defaultdict(list)
    for f in sorted(glob.glob(os.path.join(out, 'bench_*_*_*.json'))):
        m = re.match(r'bench_(\w+?)_(old|new|sg)_(\d+)\.json', os.path.basename(f))
        lines = [ln for ln in open(f).read().splitlines() if ln.startswith('{')]
        if not m or not lines:
            print(f'{os.path.basename(f)}: no result line')
            continue
        d = json.loads(lines[-1])
        runs[(m.group(1), m.group(2))].append((int(m.group(3)), d['ms_per_step'], d['kernel_ms']['blend_bwd'],
                                               d.get('clocks', {}).get('sm_mhz')))
    print('| workload | library | run | ms_per_step | blend_bwd ms | SM MHz |')
    print('|---|---|---|---|---|---|')
    for (w, v), rs in sorted(runs.items()):
        for rep, ms, bwd, mhz in sorted(rs):
            print(f'| {w} | {v} | {rep} | {ms:.4f} | {bwd:.4f} | {mhz} |')
    print('\n| workload | library | runs | ms_per_step median (spread) | blend_bwd median (spread) |')
    print('|---|---|---|---|---|')
    for (w, v), rs in sorted(runs.items()):
        ms = sorted(r[1] for r in rs)
        bwd = sorted(r[2] for r in rs)
        print(f'| {w} | {v} | {len(rs)} | {ms[len(ms) // 2]:.4f} ({ms[-1] - ms[0]:.4f}) | '
              f'{bwd[len(bwd) // 2]:.4f} ({bwd[-1] - bwd[0]:.4f}) |')


if __name__ == '__main__':
    main(sys.argv[1])
