"""Oracle of the ground-truth overlap / yaw generator vs the golden vectors produced by the
reference's own ``com_overlap_yaw`` (tools/make_golden_gt.py) and ``range_projection``
(tools/make_golden_reference.py)."""
import hashlib
import io
import os
import sys
import tempfile
from contextlib import redirect_stdout

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from make_golden_gt import gt_test_clouds  # noqa: E402
from oracle import gt as G  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


@pytest.fixture(scope='module')
def fixture():
  clouds, poses = gt_test_clouds(GOLDEN)
  gold = np.load(os.path.join(GOLDEN, 'gt_overlap_yaw.npz'))
  assert np.array_equal(gold['poses'], poses)
  return clouds, poses, gold


@pytest.mark.parametrize('frame', [0, 3])
def test_mapping_matches_reference_golden(fixture, frame):
  clouds, poses, gold = fixture
  rows = G.overlap_yaw_mapping(clouds, poses, frame)
  want = gold['mapping_frame%d' % frame]
  assert np.array_equal(rows[:, [0, 1, 3]], want[:, [0, 1, 3]])        # indices and yaw bins: exact
  assert np.array_equal(rows[:, 2], want[:, 2])                        # overlaps: same pixel counts


def test_yaw_bin_precedence():
  # int(-(yaw/pi) * W // 2 + W // 2): floor division binds before the addition (com_overlap_yaw.py:54)
  assert G.yaw_bin(0.0) == 180
  assert G.yaw_bin(np.deg2rad(1.5)) == 178          # floor(-1.5) = -2
  assert G.yaw_bin(np.deg2rad(-1.5)) == 181
  assert G.yaw_bin(np.pi) == 0
  assert G.yaw_bin(-np.pi) == 360                   # the reference's bin range is [0, 360]


def test_range_image_is_float32_of_float64_minimum():
  rng = np.random.default_rng(3)
  v = np.ones((1000, 4))
  v[:, :3] = rng.normal(0, 8, (1000, 3))
  img = G.range_image_f64(v)
  assert img.dtype == np.float32 and img.shape == (64, 900)
  d = np.sqrt((v[:, 0] ** 2 + v[:, 1] ** 2) + v[:, 2] ** 2)
  assert np.float32(d[d < 50].min()) == img[img > 0].min()
  assert np.all(img[img <= 0] == -1)


def test_live_reference_range_image(fixture, reference_outputs):
  """The reference's range_projection of float64 clouds, stored as hashes (tools/make_golden_reference.py)."""
  clouds, poses, _ = fixture
  for c, T, want in zip(clouds[:3], poses[:3], reference_outputs['gt_range_frame2']):
    v = G.homogeneous_points(c)
    v = np.linalg.inv(poses[2]).dot(T.dot(v.T)).T
    img = G.range_image_f64(v)
    assert img.dtype == np.float32 and img.shape == (64, 900)
    assert int((img > 0).sum()) == want['filled']
    assert hashlib.sha256(np.ascontiguousarray(img).tobytes()).hexdigest() == want['range_sha']
