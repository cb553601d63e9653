#!/usr/bin/env python3
"""Golden outputs of the reference's ``normalize_data`` and ``split_train_val``
(src/utils/normalize_data.py, src/utils/split_train_val.py), produced by EXECUTING both reference
functions unchanged (split_train_val needs scikit-learn) on a fixed synthetic ground-truth mapping.
As in demo4_gen_gt_files.py, split_train_val runs on normalize_data's output, right after it, on the
global ``np.random`` stream seeded with ``np.random.seed(SEED)``.

  python tools/make_golden_gt_files.py <OverlapNet checkout>

Writes tests/golden/gt_files.npz (input mapping, seed, the three outputs); its provenance
(generator, reference version, scikit-learn version) is stored in the file.
"""
import io
import os
import subprocess
import sys
from contextlib import redirect_stdout

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, 'tests', 'golden', 'gt_files.npz')
SEEDS = (0, 7)


def synthetic_mapping(n=20, seed=3):
  """All n*n rows [frame, reference, overlap, yaw bin] of a made-up sequence: overlaps from a skewed
  distribution (most pairs below 0.1, as in a real sequence), bin edges 0.1 .. 0.9 hit exactly, yaw
  bins in [0, 360)."""
  rng = np.random.default_rng(seed)
  m = np.zeros((n * n, 4))
  m[:, 0] = np.repeat(np.arange(n), n)
  m[:, 1] = np.tile(np.arange(n), n)
  m[:, 2] = np.clip(rng.beta(0.5, 2.0, n * n), 0.0, 1.0)
  m[::37, 2] = np.linspace(0.0, 1.0, len(m[::37]))
  m[1:12, 2] = np.arange(11) / 10
  m[:, 3] = rng.integers(0, 360, n * n)
  return m


def ref_version(ref):
  """The checkout's git commit, if it is a git checkout."""
  try:
    return subprocess.run(['git', '-C', ref, 'rev-parse', '--short', 'HEAD'], capture_output=True, text=True,
                          check=True).stdout.strip()
  except (OSError, subprocess.CalledProcessError):
    return 'an OverlapNet checkout'


def main():
  ref = sys.argv[1] if len(sys.argv) > 1 else '.'
  sys.path.insert(0, os.path.join(ref, 'src', 'utils'))
  from normalize_data import normalize_data           # the reference's functions, unmodified
  from split_train_val import split_train_val
  import sklearn
  mapping = synthetic_mapping()
  out = {'mapping': mapping, 'seeds': np.array(SEEDS, np.int64)}
  for seed in SEEDS:
    np.random.seed(seed)
    with redirect_stdout(io.StringIO()):
      norm = normalize_data(mapping)
      train, val = split_train_val(norm)
    out['normalized_seed%d' % seed] = norm
    out['train_seed%d' % seed] = train
    out['validation_seed%d' % seed] = val
  out['generator'] = np.array('tools/make_golden_gt_files.py: normalize_data + split_train_val of %s, scikit-learn %s'
                              % (ref_version(ref), sklearn.__version__))
  np.savez_compressed(OUT, **out)
  print('wrote', OUT, {k: v.shape for k, v in out.items()})


if __name__ == '__main__':
  main()
