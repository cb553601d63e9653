"""Sequence-wide ground truth on the GPU (ovn_gt_pair_counts, overlapnet_b200.gt.overlap_yaw_sequence)
against the per-frame path it must equal exactly, and the demo-4 training files.

The per-frame path (overlap_yaw_from_clouds: ovn_gt_range_batch + ovn_gt_overlap_count, one frame at
a time) is the reference here: the pair kernel's 32-bit shared-memory image equals the 64-bit global
one bit for bit (DESIGN.md section 11), so every column must agree with np.array_equal."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from make_golden_gt import gt_test_clouds  # noqa: E402
from oracle import gt as G  # noqa: E402

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
MAX_PIXELS = 3            # as tests/test_gpu_gt.py: float64 rounding freedom against the reference's NumPy


def per_frame(clouds, poses, frames):
  from overlapnet_b200.gt import overlap_yaw_from_clouds
  return np.concatenate([overlap_yaw_from_clouds(clouds, poses, f) for f in frames])


@pytest.fixture(scope='module')
def golden():
  clouds, poses = gt_test_clouds(GOLDEN)
  return clouds, poses, np.load(os.path.join(GOLDEN, 'gt_overlap_yaw.npz'))


@pytest.fixture(scope='module')
def trajectory():
  from overlapnet_b200 import synth
  clouds, poses = synth.trajectory_sequence(11, 40, n_points=20000)
  return clouds, poses, per_frame(clouds, poses, range(40))


def test_golden_fixture_equals_per_frame_and_reference(golden):
  from overlapnet_b200.gt import overlap_yaw_sequence
  clouds, poses, gold = golden
  rows = overlap_yaw_sequence(clouds, poses)
  assert rows.dtype == np.float64 and rows.shape == (25, 4)
  assert np.array_equal(rows, per_frame(clouds, poses, range(5)))
  for f in (0, 3):
    want = gold['mapping_frame%d' % f]
    got = rows[5 * f:5 * f + 5]
    assert np.array_equal(got[:, [0, 1, 3]], want[:, [0, 1, 3]])
    valid_num = np.count_nonzero(G.range_image_f64(G.homogeneous_points(clouds[f])) > 0)
    assert np.max(np.abs(got[:, 2] - want[:, 2])) <= MAX_PIXELS / valid_num


def test_trajectory_equals_per_frame_loop(trajectory):
  from overlapnet_b200.gt import cull_mask, overlap_yaw_sequence
  clouds, poses, want = trajectory
  rows = overlap_yaw_sequence(clouds, poses)
  assert np.array_equal(rows, want)
  # the sequence covers every kind of pair
  radius = torch.tensor([np.linalg.norm(c[:, :3].astype(np.float64), axis=1).max() for c in clouds])
  cur_inv = torch.from_numpy(np.stack([np.linalg.inv(p) for p in poses]))
  culled = cull_mask(cur_inv, torch.from_numpy(poses), radius, 50.0).numpy().ravel()
  ov = rows[:, 2]
  assert culled.sum() > 100 and np.all(ov[culled] == 0)
  assert np.count_nonzero(~culled & (ov == 0)) > 20
  assert np.count_nonzero((ov > 0) & (ov < 0.5)) > 20
  assert np.count_nonzero(ov > 0.5) >= 40                      # every frame against itself: 1.0
  # the revisit at the opposite heading overlaps
  assert rows[39, 2] > 0.2 and abs(rows[39, 3] - 180) > 150


def test_trajectory_chunked_and_permuted(trajectory, monkeypatch):
  from overlapnet_b200 import engine
  from overlapnet_b200.gt import overlap_yaw_sequence
  clouds, poses, want = trajectory
  calls = []
  orig = engine.Engine.gt_pair_counts

  def spy(self, batch, pose_ref, pose_cur_inv, cur_ranges, pairs, **kw):
    calls.append((tuple(torch.as_tensor(pose_ref).reshape(-1, 16)[0].cpu().tolist()), batch.n, cur_ranges.shape[0]))
    return orig(self, batch, pose_ref, pose_cur_inv, cur_ranges, pairs, **kw)

  monkeypatch.setattr(engine.Engine, 'gt_pair_counts', spy)
  # 6 current images per chunk, 12 reference scans (320 kB each) per chunk
  rows = overlap_yaw_sequence(clouds, poses, resident_bytes=4 * 6 * 64 * 900 * 4)
  assert np.array_equal(rows, want)
  assert len({c[1] for c in calls}) >= 2 and len(calls) >= 6
  assert len({c[0] for c in calls}) >= 3 and max(c[2] for c in calls) <= 6   # >= 3 reference chunks
  frames = [17, 3, 39, 3, 0, 25, 8]
  rows = overlap_yaw_sequence(clouds, poses, frame_idxs=frames)
  assert np.array_equal(rows, np.concatenate([want[f * 40:(f + 1) * 40] for f in frames]))


def test_zero_valid_current_frame_raises(trajectory):
  from overlapnet_b200.gt import overlap_yaw_from_clouds, overlap_yaw_sequence
  clouds, poses, _ = trajectory
  clouds = list(clouds[:4])
  clouds[2] = np.zeros((0, 4), np.float32)
  with pytest.raises(ZeroDivisionError):
    overlap_yaw_from_clouds(clouds, poses[:4], 2)
  with pytest.raises(ZeroDivisionError):
    overlap_yaw_sequence(clouds, poses[:4])
  # an empty reference scan is fine in both paths
  assert np.array_equal(overlap_yaw_sequence(clouds, poses[:4], [0, 1]), per_frame(clouds, poses[:4], [0, 1]))


def edge_clouds():
  from overlapnet_b200 import synth
  base = synth.kitti_like_cloud(21, n_points=20000)
  far = base.copy()
  far[:, :3] *= 60.0 / np.maximum(np.linalg.norm(far[:, :3], axis=1, keepdims=True), 1e-3)   # all at 60 m
  odd = base.copy()
  odd[:500] = 0.0
  odd[500:600, :3] = np.nan
  odd[600:650, 0] = np.inf
  tied = np.zeros((4000, 4), np.float32)
  tied[:, 0] = np.linspace(10.0, 10.9, 4000, dtype=np.float32)       # one ray: thousands of points per pixel
  tied[:, 1] = 1e-4
  tied = np.concatenate([tied, base[:3000]])
  return [np.zeros((0, 4), np.float32), far, odd, tied, base]


def test_pair_counts_equal_range_plus_count_on_edge_cases(engine_fp32):
  from overlapnet_b200 import synth
  eng = engine_fp32
  clouds = edge_clouds()
  rng = np.random.default_rng(8)
  pose_ref = np.stack([np.eye(4)] + [np.eye(4)] * 3 + [np.eye(4)])
  pose_ref[4, :3, 3] = [0.3, -0.2, 0.05]
  pose_ref[3, :3, 3] = [0.0, 0.0, 0.0]
  curs = [synth.kitti_like_cloud(22, n_points=20000), clouds[3]]
  cur_poses = np.stack([np.eye(4), np.eye(4)])
  cur_poses[0, :3, 3] = rng.normal(0, 0.5, 3)
  cur_inv = np.stack([np.linalg.inv(p) for p in cur_poses])
  cur_img = eng.gt_range(eng.upload_clouds(curs))
  batch = eng.upload_clouds(clouds)
  pairs = np.array([[c, r] for r in range(len(clouds)) for c in range(2)], np.int32)
  got = eng.gt_pair_counts(batch, pose_ref, cur_inv, cur_img, pairs).cpu().numpy()
  eng.check()
  want = []
  for r in range(len(clouds)):
    for c in range(2):
      img = eng.gt_range(batch, pose_ref=pose_ref, pose_cur_inv=cur_inv[c])
      want.append(int(eng.gt_overlap_count(img[r:r + 1], cur_img[c])[0]))
  assert got.tolist() == want
  assert want[0] == want[1] == want[2] == want[3] == 0          # empty scan, everything beyond max_range
  assert want[7] > 0                                            # the tied scan against itself


def test_pair_counts_reject_bad_indices(engine_fp32):
  from overlapnet_b200._cabi import OvnError
  eng = engine_fp32
  clouds = edge_clouds()[3:]
  batch = eng.upload_clouds(clouds)
  cur = eng.gt_range(eng.upload_clouds(clouds[:1]))
  poses = np.stack([np.eye(4)] * 2)
  pairs = np.array([[0, 0], [1, 0], [0, 2], [0, -1], [0, 1]], np.int32)
  got = eng.gt_pair_counts(batch, poses, np.eye(4)[None], cur, pairs).cpu().numpy()
  with pytest.raises(OvnError, match='OVN_ERR_INVALID_ARG'):
    eng.check()
  assert got[1] == got[2] == got[3] == -1 and got[0] > 0 and got[4] > 0
  again = eng.gt_pair_counts(batch, poses, np.eye(4)[None], cur, pairs[[0, 4]]).cpu().numpy()
  eng.check()                                                   # the flag was cleared when reported
  assert again.tolist() == [got[0], got[4]]


def test_pair_counts_image_must_fit_shared_memory():
  from overlapnet_b200._cabi import OvnError
  from overlapnet_b200.engine import Engine
  eng = Engine(precision='fp32', proj_H=128, proj_W=900, max_batch_scans=2, max_batch_pairs=1)
  batch = eng.upload_clouds([np.ones((10, 4), np.float32)])
  cur = torch.zeros((1, 128, 900), device=eng.device)
  with pytest.raises(OvnError, match='OVN_ERR_BAD_CONFIG'):
    eng.gt_pair_counts(batch, np.eye(4)[None], np.eye(4)[None], cur, np.zeros((1, 2), np.int32))
  eng.close()


def write_bins(clouds, folder):
  os.makedirs(folder, exist_ok=True)
  paths = []
  for i, c in enumerate(clouds):
    p = os.path.join(folder, '%06d.bin' % i)
    np.ascontiguousarray(c, np.float32).tofile(p)
    paths.append(p)
  return paths


def test_sequence_reads_each_bin_once(golden, tmp_path, monkeypatch, capsys):
  from overlapnet_b200 import gt
  clouds, poses, _ = golden
  paths = write_bins(clouds, str(tmp_path))
  reads = []
  orig = gt._read_scan
  monkeypatch.setattr(gt, '_read_scan', lambda p: reads.append(p) or orig(p))
  rows = gt.com_overlap_yaw_sequence(paths, poses, frame_idxs=[4, 0, 3])
  assert sorted(reads) == paths
  out = capsys.readouterr().out
  assert 'Start to compute ground truth overlap and yaw ...' in out and 'Finish generating ground_truth_mapping!' in out
  assert np.array_equal(rows, per_frame(clouds, poses, [4, 0, 3]))


def test_demo4_cli_writes_training_files(golden, tmp_path):
  from overlapnet_b200 import gt
  clouds, poses, _ = golden
  write_bins(clouds, str(tmp_path / '07' / 'velodyne'))
  calib = poses[2]                       # any rigid camera-to-LiDAR transform
  cam = np.stack([calib.dot(p).dot(np.linalg.inv(calib)) for p in poses])
  (tmp_path / '07' / 'poses.txt').write_text('\n'.join(' '.join('%.17g' % v for v in p[:3].ravel()) for p in cam))
  (tmp_path / '07' / 'calib.txt').write_text('Tr: ' + ' '.join('%.17g' % v for v in calib[:3].ravel()) + '\n')
  (tmp_path / 'demo.yml').write_text(
      'Demo4:\n  poses_file: "%s"\n  calib_file: "%s"\n  scan_folder: "%s"\n  dst_folder: "%s"\n'
      % (tmp_path / '07' / 'poses.txt', tmp_path / '07' / 'calib.txt', tmp_path / '07' / 'velodyne', tmp_path / '07'))
  np.random.seed(3)
  assert gt.main([str(tmp_path / 'demo.yml'), '--all-pairs', '--seq', '07']) == 0
  d = tmp_path / '07' / 'ground_truth'
  assert sorted(os.listdir(d)) == ['ground_truth_overlap_yaw.npz', 'train_set.npz', 'validation_set.npz']
  lidar = gt.kitti_lidar_poses(str(tmp_path / '07' / 'poses.txt'), str(tmp_path / '07' / 'calib.txt'))
  full = np.load(d / 'ground_truth_overlap_yaw.npz', allow_pickle=True)
  want = gt.overlap_yaw_sequence(clouds, lidar)
  assert np.array_equal(full['overlaps'], want)
  assert full['seq'].shape == (25, 2) and set(full['seq'].ravel()) == {'07'}
  np.random.seed(3)
  n = len(gt.normalize_data(want))
  train = np.load(d / 'train_set.npz', allow_pickle=True)['overlaps']
  val = np.load(d / 'validation_set.npz', allow_pickle=True)['overlaps']
  assert len(train) == n - n // 10 and len(val) == n // 10
