#!/usr/bin/env python3
"""Golden shift schedule of rotate_training_data, produced by EXECUTING the reference's own
``ImagePairOverlapOrientationSequence`` (src/two_heads/ImagePairOverlapOrientationSequence.py) here.

keras is not installed, so a stub ``keras.utils`` module provides an empty ``Sequence`` base class; the
reference file is then imported unchanged.  The tiny synthetic dataset has one-row depth images whose
value is the column index, so the shift the reference applied to each RIGHT image reads back from its
first pixel: shift = -x2[i, 0, 0, 0] mod W.  For modes 1 and 2 it records the shifts of a fixed sequence of
``__getitem__`` calls over 10 pairs in batches of 4 (the last batch is short).

  python tools/make_golden_rotation.py <OverlapNet checkout>

Writes tests/golden/rotation_shifts.npz; its provenance (generator, reference version) is stored in the file.
"""
import os
import subprocess
import sys
import tempfile
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, 'tests', 'golden', 'rotation_shifts.npz')
N_PAIRS, BATCH, WIDTH = 10, 4, 900
CALLS = {1: [2, 0, 1, 2, 1, 0], 2: [1, 0, 2, 0, 2, 1, 2, 0]}     # two to three epochs in shuffled orders


def ref_version(ref):
  """The checkout's git commit, if it is a git checkout."""
  try:
    return subprocess.run(['git', '-C', ref, 'rev-parse', '--short', 'HEAD'], capture_output=True, text=True,
                          check=True).stdout.strip()
  except (OSError, subprocess.CalledProcessError):
    return 'an OverlapNet checkout'


def stub_keras():
  keras = types.ModuleType('keras')
  utils = types.ModuleType('keras.utils')

  class Sequence:                                 # keras.utils.Sequence stand-in: a plain base class
    pass

  utils.Sequence = Sequence
  keras.utils = utils
  sys.modules['keras'] = keras
  sys.modules['keras.utils'] = utils


def main():
  ref = sys.argv[1] if len(sys.argv) > 1 else '/root/reference'
  stub_keras()
  sys.path.insert(0, os.path.join(ref, 'src', 'two_heads'))
  from ImagePairOverlapOrientationSequence import ImagePairOverlapOrientationSequence
  out = {'n_pairs': N_PAIRS, 'batch_size': BATCH, 'width': WIDTH}
  with tempfile.TemporaryDirectory() as root:
    os.makedirs(os.path.join(root, '00', 'depth'))
    names = ['%06d' % i for i in range(N_PAIRS)]
    for nm in names:
      np.save(os.path.join(root, '00', 'depth', nm + '.npy'), np.arange(WIDTH, dtype=np.float32)[None, :])
    for mode, calls in CALLS.items():
      seq = ImagePairOverlapOrientationSequence(
          root, names, names[::-1], ['00'] * N_PAIRS, ['00'] * N_PAIRS, np.linspace(0, 1, N_PAIRS),
          np.zeros(N_PAIRS), 360, BATCH, 1, WIDTH, no_channels=1, use_depth=True, use_normals=False,
          rotate_data=mode)
      shifts = []
      for idx in calls:
        (x1, x2), _ = seq[idx]
        assert np.array_equal(x1[:, 0, :, 0], np.tile(np.arange(WIDTH), (len(x1), 1)))   # LEFT never rolled
        shifts.append((-x2[:, 0, 0, 0].astype(np.int64)) % WIDTH)
      out['calls_mode%d' % mode] = np.array(calls, np.int64)
      out['sizes_mode%d' % mode] = np.array([len(s) for s in shifts], np.int64)
      out['shifts_mode%d' % mode] = np.concatenate(shifts)
  out['generator'] = np.array('tools/make_golden_rotation.py: ImagePairOverlapOrientationSequence of %s' % ref_version(ref))
  np.savez(OUT, **out)
  print('wrote', OUT)


if __name__ == '__main__':
  main()
