"""Seeded synthetic inputs shaped like the reference's data (SURVEY.md section 8d).

Used by bench.py and the tests; there is no network for KITTI, so every benchmark input is
generated here and labelled ``"data": "synthetic"``.
"""
import numpy as np

KITTI_POINTS = 124668   # point count of the reference fixture data/scans/000000.bin


def kitti_like_cloud(seed, n_points=KITTI_POINTS, zero_points=0, far_fraction=0.02):
  """HDL-64-shaped cloud: 64 beams with pitch in [-24.8, +2] deg (+ jitter), uniform azimuth,
  log-normal range clipped to (0.5, 80) m so that about ``far_fraction`` exceed max_range=50,
  intensity U[0,1) quantised to 0.01.  Returns (n_points, 4) float32 [x, y, z, intensity].
  ``zero_points`` rows are overwritten with [0,0,0,0] to exercise the depth>0 filter."""
  rng = np.random.default_rng(seed)
  beam = rng.integers(0, 64, size=n_points)
  pitch = np.deg2rad(-24.8 + (2.0 + 24.8) * (beam + 0.5) / 64.0 + rng.normal(0.0, 0.05, n_points))
  az = rng.uniform(-np.pi, np.pi, n_points)
  # median ~9 m; sigma chosen so P(r > 50) ~= far_fraction
  sigma = np.log(50.0 / 9.0) / 2.054 if far_fraction > 0 else 0.5
  r = np.clip(np.exp(rng.normal(np.log(9.0), sigma, n_points)), 0.5, 80.0)
  pts = np.empty((n_points, 4), dtype=np.float32)
  pts[:, 0] = r * np.cos(pitch) * np.cos(az)
  pts[:, 1] = r * np.cos(pitch) * np.sin(az)
  pts[:, 2] = r * np.sin(pitch)
  pts[:, 3] = np.floor(rng.uniform(0, 1, n_points) * 100.0) / 100.0
  if zero_points:
    pts[rng.choice(n_points, size=zero_points, replace=False)] = 0.0
  return pts


def random_probs(seed, n_points, n_classes=20):
  """Per-point class probabilities (softmax of N(0,1)), float32 (n_points, n_classes)."""
  rng = np.random.default_rng(seed)
  logits = rng.standard_normal((n_points, n_classes)).astype(np.float32)
  e = np.exp(logits - logits.max(axis=1, keepdims=True))
  return (e / e.sum(axis=1, keepdims=True)).astype(np.float32)


def range_like_images(seed, n, channels=4, H=64, W=900, empty_fraction=0.22):
  """Synthetic preprocessed network inputs (n, H, W, C) float32 in the reference's channel order
  (depth, normal x3, [probabilities], [intensity]); ``empty_fraction`` of the pixels hold -1."""
  rng = np.random.default_rng(seed)
  x = np.empty((n, H, W, channels), dtype=np.float32)
  x[..., 0] = rng.uniform(0.0, 50.0, (n, H, W))
  if channels >= 4:
    nrm = rng.standard_normal((n, H, W, 3))
    nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True)
    x[..., 1:4] = nrm
  if channels > 4:
    x[..., 4:] = rng.uniform(0.0, 1.0, (n, H, W, channels - 4))
  empty = rng.uniform(0, 1, (n, H, W)) < empty_fraction
  x[empty] = -1.0
  return x


def feature_volumes(seed, n, width=360, channels=128, sparsity=0.5, scale=1.0):
  """Synthetic leg outputs (n, 1, width, channels) float32: non-negative (post-ReLU) with about
  ``sparsity`` exact zeros."""
  rng = np.random.default_rng(seed)
  v = rng.standard_normal((n, 1, width, channels)).astype(np.float32) * np.float32(scale)
  v = np.maximum(v + np.float32(scale * (0.0 if sparsity == 0.5 else 0.3)), 0)
  return np.ascontiguousarray(v, dtype=np.float32)


def trajectory_sequence(seed, n_frames, n_points=KITTI_POINTS, step=None, radius=40.0):
  """A seeded static scene seen along a trajectory: (clouds, poses).  The sensor drives east along a
  road for half the frames, then back west 2 m to the side, heading 180 deg the other way (a revisit
  at a different heading).  The scene is a ground plane 1.73 m below the sensor, two walls 12 m either
  side of the road and vertical poles; each frame samples ``n_points`` of it within ``radius`` metres
  (plus a few zero points), so frames far apart share nothing.  ``step``: metres per frame (default:
  the outbound leg is 160 m long, but at least 1 m per frame).  ``poses``: (n, 4, 4) float64 sensor
  to world; every cloud is float32 (N, 4) in its own frame's coordinates, intensity U[0,1)."""
  rng = np.random.default_rng(seed)
  half = (n_frames + 1) // 2
  step = max(1.0, 160.0 / max(half, 1)) if step is None else float(step)
  length = step * half
  poles = np.stack([rng.uniform(-radius, length + radius, 400), rng.uniform(-30.0, 30.0, 400)], axis=1)
  poles = poles[np.abs(poles[:, 1]) > 4.0]
  poses = np.zeros((n_frames, 4, 4))
  clouds = []
  for i in range(n_frames):
    out = i < half
    x0 = step * i if out else step * (n_frames - 1 - i) + step / 2
    y0, yaw = (0.0, 0.0) if out else (2.0, np.pi + np.deg2rad(rng.normal(0.0, 2.0)))
    T = np.eye(4)
    T[:2, :2] = [[np.cos(yaw), -np.sin(yaw)], [np.sin(yaw), np.cos(yaw)]]
    T[:3, 3] = [x0, y0, 0.0]
    poses[i] = T
    n_ground, n_wall = n_points // 2, n_points * 3 // 10
    n_pole = n_points - n_ground - n_wall
    r = radius * np.sqrt(rng.uniform(0.0, 1.0, n_ground))
    a = rng.uniform(-np.pi, np.pi, n_ground)
    ground = np.stack([x0 + r * np.cos(a), y0 + r * np.sin(a), np.full(n_ground, -1.73)], axis=1)
    wx = x0 + rng.uniform(-radius * 0.9, radius * 0.9, n_wall)
    wall = np.stack([wx, np.where(rng.random(n_wall) < 0.5, -12.0, 12.0), rng.uniform(-1.73, 3.0, n_wall)], axis=1)
    near = poles[np.hypot(poles[:, 0] - x0, poles[:, 1] - y0) < radius - 1.0]
    if len(near) == 0:
      near = np.array([[x0 + 5.0, y0 + 5.0]])
    k = rng.integers(0, len(near), n_pole)
    pa = rng.uniform(-np.pi, np.pi, n_pole)
    pole = np.stack([near[k, 0] + 0.2 * np.cos(pa), near[k, 1] + 0.2 * np.sin(pa), rng.uniform(-1.73, 4.0, n_pole)], axis=1)
    world = np.concatenate([ground, wall, pole])
    local = (world - T[:3, 3]) @ T[:3, :3]                  # R^T (p - t)
    pts = np.empty((n_points, 4), dtype=np.float32)
    pts[:, :3] = local
    pts[:, 3] = rng.uniform(0.0, 1.0, n_points)
    pts[rng.choice(n_points, size=min(8, n_points), replace=False)] = 0.0
    clouds.append(pts)
  return clouds, poses
