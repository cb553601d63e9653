#!/usr/bin/env python3
"""Store what the reference-parity tests compare against, so that they run without the reference.

Runs the reference's own ``range_projection`` (src/utils/utils.py, imported unmodified) and reads
its shipped fixtures, then writes

  tests/golden/reference_outputs.json
    synthetic_range   the reference's range image of four seeded full-size synthetic clouds, as
                      its SHA-256 plus the few pixels where it differs from oracle/projection.py
                      (tests/test_oracle_projection.py::test_live_reference_synthetic)
    gt_range_frame2   the reference's range image of the first three ground-truth test clouds in
                      the frame of pose 2, as SHA-256 and filled-pixel count
                      (tests/test_oracle_gt.py::test_live_reference_range_image)
  tests/golden/kitti_semantic_sample.npz
    for each fixture scan, a seeded sample of pixels of the shipped semantic fixture, the shipped
    class-probability rows of the points shown there and the fixture's values at those pixels
    (tests/test_oracle_projection.py::test_live_reference_fixtures_and_semantic); the full .label
    files are 10 MB each.

  python tools/make_golden_reference.py <OverlapNet checkout>
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from make_golden_gt import gt_test_clouds  # noqa: E402
from oracle import gt as G  # noqa: E402
from oracle import projection as P  # noqa: E402
from overlapnet_b200 import synth  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
SEMANTIC_PIXELS = 256


def sha(a):
  return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main(ref):
  sys.path.insert(0, os.path.join(ref, 'src', 'utils'))
  import utils as ref_utils  # the reference's module
  out = {'_generator': 'tools/make_golden_reference.py on numpy %s, reference commit 4188c3a' % np.__version__}

  out['synthetic_range'] = []
  for seed in range(4):
    zeros = 3 * (seed % 2)
    pts = synth.kitti_like_cloud(seed, zero_points=zeros)
    want = ref_utils.range_projection(pts)[0]
    mine = P.range_projection(pts)[0]
    differs = [[int(r), int(c), float(want[r, c])] for r, c in np.argwhere(want != mine)]
    out['synthetic_range'].append({'seed': seed, 'zero_points': zeros, 'points_sha': sha(pts),
                                   'range_sha': sha(want), 'differs': differs})

  clouds, poses = gt_test_clouds(GOLDEN)
  out['gt_range_frame2'] = []
  for c, T in zip(clouds[:3], poses[:3]):
    v = np.linalg.inv(poses[2]).dot(T.dot(G.homogeneous_points(c).T)).T
    want = ref_utils.range_projection(v)[0]
    assert want.dtype == np.float32 and want.shape == (64, 900)
    out['gt_range_frame2'].append({'range_sha': sha(want), 'filled': int((want > 0).sum())})

  sample = {}
  for k, name in enumerate(('000000', '000001')):
    pts = np.fromfile(os.path.join(ref, 'data', 'scans', name + '.bin'), dtype=np.float32).reshape(-1, 4)
    labels = np.fromfile(os.path.join(ref, 'data', 'semantic_probs', name + '.label'), dtype=np.float32).reshape(-1, 20)
    shipped = np.load(os.path.join(ref, 'data', 'preprocess_data_demo', 'semantic', name + '.npy'))
    _, _, _, idx_inf = ref_utils.range_projection(pts, max_range=np.inf)
    sem = np.full((64, 900, 20), -1, dtype=np.float32)                  # gen_semantic_data.py:42-46
    sem[idx_inf >= 0] = labels[idx_inf[idx_inf >= 0]]
    assert np.array_equal(sem, shipped), 'reference semantic fixture mismatch'
    flat = np.sort(np.random.default_rng(200 + k).choice(64 * 900, SEMANTIC_PIXELS, replace=False))
    r, c = np.divmod(flat, 900)
    point_idx = idx_inf[r, c].astype(np.int32)
    sample[name + '_pixels'] = np.stack([r, c], 1).astype(np.int32)
    sample[name + '_point_idx'] = point_idx
    sample[name + '_label_rows'] = labels[point_idx[point_idx >= 0]]
    sample[name + '_semantic'] = shipped[r, c]

  with open(os.path.join(GOLDEN, 'reference_outputs.json'), 'w') as f:
    json.dump(out, f, indent=1)
    f.write('\n')
  np.savez_compressed(os.path.join(GOLDEN, 'kitti_semantic_sample.npz'), **sample)
  print(json.dumps(out, indent=1))


if __name__ == '__main__':
  if len(sys.argv) != 2:
    raise SystemExit(__doc__)
  main(sys.argv[1])
