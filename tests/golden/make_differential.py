"""Writes tests/golden/differential.npz: the scenarios of tests/test_reference_differential.py run through the oracle
(tests/test_differential_golden.py says why that recording stands for the reference's outputs).

  python tests/golden/make_differential.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from tests.test_differential_golden import ROLLOUTS, gap_follow_action, gap_follow_scans, record  # noqa: E402

if __name__ == '__main__':
    out = {}
    for name in ROLLOUTS:
        out.update(('%s__%s' % (name, k), v) for k, v in record(name).items())
        print(name, len(out[name + '__time']) - 1, 'steps')
    out['gap_follow__actions'] = np.stack([gap_follow_action(s) for s in gap_follow_scans()])
    np.savez_compressed(os.path.join(HERE, 'differential.npz'), **out)
    print('differential.npz', os.path.getsize(os.path.join(HERE, 'differential.npz')) // 1024, 'KiB')
