"""Compare two `bench.py --dump-outputs` directories file by file.
python profiles/r03_compare_dumps.py OLD_DIR NEW_DIR

Forward outputs must be bit-identical; every other array is reported as the norm-wise relative difference
||new - old|| / ||old|| (float64), which for the gradients should be float-reassociation noise (<= 1e-5)."""
import os
import sys

import numpy as np

FORWARD = ('gaussian_index', 'pixel_index', 'image', 'radii', 'point_id_pixel', 'point_weight_pixel', 'point_weight')


def main(old_dir, new_dir):
    names = sorted(f[:-4] for f in os.listdir(old_dir) if f.endswith('.npy'))
    assert names == sorted(f[:-4] for f in os.listdir(new_dir) if f.endswith('.npy')), 'different file sets'
    bad = False
    for name in names:
        a = np.load(os.path.join(old_dir, name + '.npy')).astype(np.float64)
        b = np.load(os.path.join(new_dir, name + '.npy')).astype(np.float64)
        same = a.shape == b.shape and np.array_equal(a, b, equal_nan=True)
        rel = float(np.linalg.norm(b - a) / max(np.linalg.norm(a), 1e-300)) if a.shape == b.shape else float('inf')
        if name in FORWARD:
            verdict = 'bit-identical' if same else 'DIFFERS'
            bad |= not same
        else:
            verdict = 'ok' if rel <= 1e-5 else 'ABOVE 1e-5'
            bad |= rel > 1e-5
        print(f'{name:22s} shape={str(a.shape):14s} bit-identical={same!s:5s} rel={rel:.3e}  {verdict}')
    print('RESULT:', 'FAIL' if bad else 'PASS')
    return 1 if bad else 0


if __name__ == '__main__':
    sys.exit(main(sys.argv[1], sys.argv[2]))
