"""Host logic of sequence-wide ground truth (overlapnet_b200.gt): vectorised yaw bins against the
scalar per-row code, the cull bound against float64 NumPy projections, normalize_data /
split_train_val against the reference's outputs, and the training files of the demo-4 flow."""
import os

import numpy as np
import pytest
import torch

from overlapnet_b200 import gt, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def se3(yaw, pitch=0.0, roll=0.0, t=(0.0, 0.0, 0.0)):
  Rz = np.array([[np.cos(yaw), -np.sin(yaw), 0], [np.sin(yaw), np.cos(yaw), 0], [0, 0, 1]])
  Ry = np.array([[np.cos(pitch), 0, np.sin(pitch)], [0, 1, 0], [-np.sin(pitch), 0, np.cos(pitch)]])
  Rx = np.array([[1, 0, 0], [0, np.cos(roll), -np.sin(roll)], [0, np.sin(roll), np.cos(roll)]])
  T = np.eye(4)
  T[:3, :3] = Rz @ Ry @ Rx
  T[:3, 3] = t
  return T


def random_poses(rng, n, spread=1.0):
  return np.stack([se3(*rng.uniform(-np.pi, np.pi, 3) * spread, t=rng.normal(0, 30, 3)) for _ in range(n)])


def structured_poses():
  ps = [np.eye(4), se3(0.0, np.pi / 2), se3(0.0, -np.pi / 2), se3(0.3, np.pi / 2, 0.2), se3(-1.0, -np.pi / 2, 0.4),
        se3(np.pi), se3(-np.pi), se3(0.5, np.pi / 2 - 1e-6), se3(0.5, np.pi / 2 - 5e-3)]
  ps += [se3(np.deg2rad(k)) for k in range(-179, 181)]          # -(yaw/pi)*360 on even integers: floor edges
  ps += [se3(np.deg2rad(k) + 1e-15) for k in range(-179, 181, 7)]
  return np.stack(ps)


def scalar_bins(cur_inv, poses, W=360):
  return np.array([gt._yaw_bin_scalar(cur_inv, p, W) for p in poses], np.int64)


def test_stacked_product_equals_per_row_dot():
  rng = np.random.default_rng(0)
  poses = random_poses(rng, 400)
  cur_inv = np.linalg.inv(poses[17])
  stacked = cur_inv @ poses
  assert np.array_equal(stacked, np.stack([cur_inv.dot(p) for p in poses]))


@pytest.mark.parametrize('W', [360, 900])
def test_yaw_bins_equal_scalar_random(W):
  rng = np.random.default_rng(1)
  poses = random_poses(rng, 320)
  for c in (0, 5, 111):
    cur_inv = np.linalg.inv(poses[c])
    assert np.array_equal(gt.yaw_bins(cur_inv, poses, W), scalar_bins(cur_inv, poses, W))


def test_yaw_bins_equal_scalar_structured():
  poses = structured_poses()
  for cur in (np.eye(4), se3(0.25), se3(np.pi / 2)):
    cur_inv = np.linalg.inv(cur)
    got = gt.yaw_bins(cur_inv, poses)
    assert np.array_equal(got, scalar_bins(cur_inv, poses))
  # both isclose branches and the floor edges were really exercised
  r20 = (np.eye(4) @ poses)[:, 2, 0]
  assert np.any(np.isclose(r20, -1.0, rtol=1e-5, atol=1e-8)) and np.any(np.isclose(r20, 1.0, rtol=1e-5, atol=1e-8))
  assert len(set(gt.yaw_bins(np.eye(4), poses).tolist())) >= 300


def test_yaw_bins_non_finite_pose_raises_like_scalar():
  poses = np.stack([np.eye(4), np.full((4, 4), np.nan)])
  with pytest.raises(ValueError):
    scalar_bins(np.eye(4), poses)
  with pytest.raises(ValueError):
    gt.yaw_bins(np.eye(4), poses)


def kernel_depths(cloud, pose_ref, cur_inv):
  """Depths as the kernel computes them: (x,y,z,1) float64, pose_ref then cur_inv, each row a
  left-to-right sum of separately rounded products, then sqrt(x*x + y*y + z*z) left to right."""
  v = np.ones((cloud.shape[0], 4))
  v[:, :3] = cloud[:, :3].astype(np.float64)
  for M in (pose_ref, cur_inv):
    v = np.stack([((M[i, 0] * v[:, 0] + M[i, 1] * v[:, 1]) + M[i, 2] * v[:, 2]) + M[i, 3] * v[:, 3]
                  for i in range(4)], axis=1)
  return np.sqrt((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2])


def test_cull_bound_is_sound():
  rng = np.random.default_rng(2)
  clouds = [synth.kitti_like_cloud(s, n_points=3000) for s in range(6)]
  clouds[5][:, :3] *= 0.3
  poses = np.concatenate([random_poses(rng, 10, spread=0.2) * 1.0,
                          np.stack([se3(rng.uniform(-np.pi, np.pi), t=(d, 0.0, 0.0)) for d in np.linspace(60, 200, 14)])])
  poses[:, :3, 3] *= rng.uniform(0.5, 6.0, (len(poses), 1))
  radius = torch.tensor([np.linalg.norm(c[:, :3].astype(np.float64), axis=1).max() for c in clouds])
  cur_inv = np.stack([np.linalg.inv(p) for p in poses])
  culled_total = kept_total = 0
  for s, cloud in enumerate(clouds):
    ref = poses[(s * 3) % len(poses)][None].repeat(1, 0)
    mask = gt.cull_mask(torch.from_numpy(cur_inv), torch.from_numpy(ref), radius[s:s + 1], 50.0).numpy()[:, 0]
    for c in np.flatnonzero(mask):
      assert kernel_depths(cloud, ref[0], cur_inv[c]).min() >= 50.0
    for c in np.flatnonzero(~mask):               # the bound is not vacuous: close pairs are kept
      kept_total += kernel_depths(cloud, ref[0], cur_inv[c]).min() < 50.0
    culled_total += int(mask.sum())
  assert culled_total > 20 and kept_total > 10


def test_cull_never_on_non_finite_radius():
  far = se3(0.0, t=(1e4, 0.0, 0.0))[None]
  for r in (np.nan, np.inf):
    m = gt.cull_mask(torch.eye(4, dtype=torch.float64)[None], torch.from_numpy(far), torch.tensor([r]), 50.0)
    assert not bool(m.any())
  m = gt.cull_mask(torch.eye(4, dtype=torch.float64)[None], torch.from_numpy(far), torch.tensor([10.0]), 50.0)
  assert bool(m.all())


def test_normalize_and_split_match_reference_golden(capsys):
  z = np.load(os.path.join(GOLDEN, 'gt_files.npz'))
  for seed in z['seeds']:
    np.random.seed(int(seed))
    norm = gt.normalize_data(z['mapping'])
    train, val = gt.split_train_val(norm)
    assert np.array_equal(norm, z['normalized_seed%d' % seed])
    assert np.array_equal(train, z['train_seed%d' % seed])
    assert np.array_equal(val, z['validation_seed%d' % seed])
    assert len(val) == len(norm) // 10
  out = capsys.readouterr().out
  assert 'size of normalized data:  %d' % len(z['normalized_seed0']) in out
  assert 'finished generating training data and validation data' in out


def test_split_rejects_too_few_rows():
  with pytest.raises(ValueError):
    gt.split_train_val(np.zeros((9, 4)))


def test_written_files_load_for_training(tmp_path):
  from overlapnet_b200.evaluate import load_overlap_npz
  rng = np.random.default_rng(4)
  m = np.zeros((50, 4))
  m[:, 0], m[:, 1], m[:, 2], m[:, 3] = 3, np.arange(50), rng.uniform(0, 1, 50), rng.integers(0, 360, 50)
  d = gt.write_gt_files(str(tmp_path), m, m[:45], m[45:], '07')
  assert sorted(os.listdir(d)) == ['ground_truth_overlap_yaw.npz', 'train_set.npz', 'validation_set.npz']
  f1, f2, d1, d2, ov, yaw = load_overlap_npz([os.path.join(d, 'ground_truth_overlap_yaw.npz')], shuffle=False)
  assert f1 == ['000003'] * 50 and f2 == ['%06d' % i for i in range(50)]
  assert d1 == ['07'] * 50 and d2 == ['07'] * 50
  assert np.array_equal(ov, m[:, 2]) and np.array_equal(yaw, m[:, 3])
  f1, _, _, _, ov, _ = load_overlap_npz([os.path.join(d, 'validation_set.npz')], shuffle=False)
  assert len(f1) == 5 and np.array_equal(ov, m[45:, 2])


def test_kitti_lidar_poses_match_demo4_conversion(tmp_path):
  rng = np.random.default_rng(5)
  cam = random_poses(rng, 4, spread=0.3)
  calib = se3(0.1, 0.02, -1.5, t=(0.3, -0.1, 0.05))
  (tmp_path / 'poses.txt').write_text('\n'.join(' '.join('%.17g' % v for v in p[:3].ravel()) for p in cam))
  (tmp_path / 'calib.txt').write_text('P0: 1 0 0 0 0 1 0 0 0 0 1 0\nTr: ' + ' '.join('%.17g' % v for v in calib[:3].ravel()))
  got = gt.kitti_lidar_poses(str(tmp_path / 'poses.txt'), str(tmp_path / 'calib.txt'))
  inv_c, p0_inv = np.linalg.inv(calib), np.linalg.inv(cam[0])
  assert np.array_equal(got, np.array([inv_c.dot(p0_inv).dot(p).dot(calib) for p in cam]))
  assert np.allclose(got[0], np.eye(4), atol=1e-12)


def test_trajectory_sequence_shape():
  clouds, poses = synth.trajectory_sequence(3, 10, n_points=500)
  assert len(clouds) == 10 and poses.shape == (10, 4, 4)
  assert all(c.dtype == np.float32 and c.shape == (500, 4) for c in clouds)
  assert np.all(np.linalg.norm(clouds[4][:, :3], axis=1) < 40.5)
  again, _ = synth.trajectory_sequence(3, 10, n_points=500)
  assert all(np.array_equal(a, b) for a, b in zip(clouds, again))
