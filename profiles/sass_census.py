"""SASS census of the shipped library: which tensor-core / matrix-load / warp-collective / atomic instructions each kernel
contains.  python profiles/sass_census.py > profiles/r02_sass_census.md   (needs cuobjdump and c++filt; no GPU)"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, 'log_b200', '_lib', 'liblog_b200_raster.so')
PATS = collections.OrderedDict([
    ('HMMA (mma.sync tf32)', r'\bHMMA\.'), ('LDSM (ldmatrix)', r'\bLDSM'), ('UTC*MMA / LDTM (tcgen05)', r'UTC\w*MMA|LDTM'),
    ('UBLKCP / UTMA (bulk / tensor copies)', r'UBLKCP|UTMA'), ('REDUX', r'\bREDUX'), ('VOTE', r'\bVOTE'), ('MATCH', r'\bMATCH'),
    ('SHFL', r'\bSHFL'), ('ATOMS / REDS (shared)', r'\bATOMS|\bREDS'), ('ATOMG (returning)', r'\bATOMG'), ('RED (global)', r'\bREDG?\.E\.'),
    ('MUFU.EX2', r'MUFU\.EX2'), ('BAR', r'\bBAR\.'), ('LDG.128', r'LDG\.E\.(\w+\.)*128'), ('STG.128', r'STG\.E\.(\w+\.)*128'),
    ('CCTL (L2 prefetch)', r'\bCCTL')])


def main():
    sass = subprocess.run(['cuobjdump', '-sass', LIB], capture_output=True, text=True, check=True).stdout
    stats, cur = collections.OrderedDict(), None
    for line in sass.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            cur = m.group(1)
            stats[cur] = collections.Counter()
        elif cur and re.search(r'/\*[0-9a-f]{4}\*/', line):
            stats[cur]['instructions'] += 1
            for k, p in PATS.items():
                if re.search(p, line):
                    stats[cur][k] += 1
    print('# SASS census of `liblog_b200_raster.so` (sm_100a), static instruction counts per kernel\n')
    print('`cuobjdump -sass` of the shipped library, grouped by `profiles/sass_census.py`. The tensor-core path is the legacy')
    print('`mma.sync.m16n8k8.tf32` (`HMMA.1688.F32.TF32`) fed by `ldmatrix` (`LDSM`) in `blend_bwd_kernel`; there is no')
    print('`tcgen05` / TMA instruction in the library (the path has no GEMM-shaped stage large enough to own TMEM, DESIGN.md §3).\n')
    print('| kernel | instructions | ' + ' | '.join(PATS) + ' |')
    print('|---|---|' + '---|' * len(PATS))
    for k, c in stats.items():
        name = subprocess.run(['c++filt', k], capture_output=True, text=True).stdout.strip().split('(')[0].replace('void ', '').replace('lgr::', '')
        print(f'| `{name}` | {c["instructions"]} | ' + ' | '.join(str(c[p]) if c[p] else '' for p in PATS) + ' |')


if __name__ == '__main__':
    main()
