"""GPU drop-in for the reference's ground-truth generator ``com_overlap_yaw``
(``src/utils/com_overlap_yaw.py:10-68``, used by ``demo/demo4_gen_gt_files.py:77``): same name,
arguments and return value.  The O(N) pose-transformed float64 range projections and the pixel
comparisons run in csrc/gt_overlap.cu through the C ABI (``ovn_gt_range_batch``,
``ovn_gt_overlap_count``); the yaw bin is 4x4 host arithmetic exactly as the reference writes it.
``overlap_yaw_sequence`` does the same for many current frames at once (``ovn_gt_pair_counts``), and
``python -m overlapnet_b200.gt demo.yml`` is the reference's demo4_gen_gt_files.py: ground truth,
``normalize_data``, ``split_train_val`` and the three training files.  There is no CPU fallback."""
import argparse
import math
import os
import sys

import numpy as np

from .preprocess import _engine, _read_scan


def load_poses(pose_path):
  """``load_poses`` (utils.py:10-36): KITTI ``.txt`` (12 numbers per line) or ``.npz['arr_0']`` -> (n,4,4)."""
  poses = []
  try:
    if '.txt' in pose_path:
      with open(pose_path, 'r') as f:
        for line in f.readlines():
          T = np.array(line.split(), dtype=float).reshape(3, 4)
          poses.append(np.vstack((T, [0, 0, 0, 1])))
    else:
      poses = np.load(pose_path)['arr_0']
  except FileNotFoundError:
    print('Ground truth poses are not avaialble.')
  return np.array(poses)


def load_calib(calib_path):
  """``load_calib`` (utils.py:39-56): the ``Tr:`` line of a KITTI calib file -> T_cam_velo (4,4)."""
  T_cam_velo = []
  try:
    with open(calib_path, 'r') as f:
      for line in f.readlines():
        if 'Tr:' in line:
          T = np.array(line.replace('Tr:', '').split(), dtype=float).reshape(3, 4)
          T_cam_velo = np.vstack((T, [0, 0, 0, 1]))
  except FileNotFoundError:
    print('Calibrations are not avaialble.')
  return np.array(T_cam_velo)


def euler_angles_from_rotation_matrix(R):
  """(psi, theta, phi) = roll, pitch, yaw after Slabaugh, as ``utils.py:178-216``."""
  def isclose(x, y, rtol=1.e-5, atol=1.e-8):
    return abs(x - y) <= atol + rtol * abs(y)
  phi = 0.0
  if isclose(R[2, 0], -1.0):
    theta = math.pi / 2.0
    psi = math.atan2(R[0, 1], R[0, 2])
  elif isclose(R[2, 0], 1.0):
    theta = -math.pi / 2.0
    psi = math.atan2(-R[0, 1], -R[0, 2])
  else:
    theta = -math.asin(R[2, 0])
    cos_theta = math.cos(theta)
    psi = math.atan2(R[2, 1] / cos_theta, R[2, 2] / cos_theta)
    phi = math.atan2(R[1, 0] / cos_theta, R[0, 0] / cos_theta)
  return psi, theta, phi


def overlap_yaw_from_clouds(clouds, poses, frame_idx, leg_output_width=360, scans_per_launch=16):
  """The body of ``com_overlap_yaw``: rows [frame_idx, reference_idx, overlap, yaw bin] as float64.
  ``clouds``: list of (N,4) float32 arrays, or of zero-argument callables returning one (read lazily,
  ``scans_per_launch`` at a time, so a whole KITTI sequence never sits in host memory)."""
  poses = np.asarray(poses, dtype=np.float64)
  n = len(clouds)
  eng = _engine(3.0, -25.0, 64, 900, 50)

  def get(i):
    c = clouds[i]
    return np.ascontiguousarray(c() if callable(c) else c, np.float32)

  cur = eng.gt_range(eng.upload_clouds([get(frame_idx)]))[0]
  current_pose = poses[frame_idx]
  cur_inv = np.linalg.inv(current_pose)
  counts = np.zeros(n, np.int64)
  valid_num = 0
  for s0 in range(0, n, scans_per_launch):
    s1 = min(n, s0 + scans_per_launch)
    batch = eng.upload_clouds([get(i) for i in range(s0, s1)])
    ref = eng.gt_range(batch, pose_ref=poses[s0:s1], pose_cur_inv=cur_inv)
    c = eng.gt_overlap_count(ref, cur).cpu().numpy()
    counts[s0:s1] = c[:-1]
    valid_num = int(c[-1])
  mapping = np.zeros((n, 4))
  mapping[:, 0] = np.ones(n) * frame_idx
  mapping[:, 1] = np.arange(n)
  for r in range(n):
    mapping[r, 2] = int(counts[r]) / valid_num                                   # com_overlap_yaw.py:44-46
    mapping[r, 3] = _yaw_bin_scalar(cur_inv, poses[r], leg_output_width)
  return mapping


def _yaw_bin_scalar(cur_inv, pose, yaw_resolution):
  """Yaw bin of ``pose`` seen from the frame whose inverse pose is ``cur_inv``, as com_overlap_yaw.py:49-54."""
  relative_transform = cur_inv.dot(pose)                                       # :49
  _, _, yaw = euler_angles_from_rotation_matrix(relative_transform[:3, :3])    # :50-51
  return int(- (yaw / np.pi) * yaw_resolution//2 + yaw_resolution//2)          # :54, same expression


def com_overlap_yaw(scan_paths, poses, frame_idx, leg_output_width=360):
  """Drop-in for ``com_overlap_yaw`` (com_overlap_yaw.py:10-68): ground-truth overlap and yaw bin of
  every scan in ``scan_paths`` against scan ``frame_idx``, from the ground-truth ``poses`` (n,4,4).
  Returns the (n, 4) float64 array [current_frame_idx, reference_frame_idx, overlap, yaw]."""
  print('Start to compute ground truth overlap and yaw ...')
  clouds = [(lambda p=p: _read_scan(p)) for p in scan_paths]      # streamed like the reference (one scan at a time there)
  mapping = overlap_yaw_from_clouds(clouds, poses, frame_idx, leg_output_width)
  print('Finish generating ground_truth_mapping!')
  return mapping


# ---- sequence-wide ground truth ----------------------------------------------------------------------
_ISCLOSE_ATOL, _ISCLOSE_RTOL = 1.e-8, 1.e-5     # euler_angles_from_rotation_matrix's isclose
_IMG_BYTES = 64 * 900 * 4


def yaw_bins(cur_inv, poses, leg_output_width=360):
  """int64 yaw bins of every pose in ``poses`` (n,4,4) seen from the frame whose inverse pose is
  ``cur_inv``, equal to ``_yaw_bin_scalar`` row by row.

  The relative transforms come from one stacked product ``cur_inv @ poses``, which equals the
  per-row ``cur_inv.dot(pose)``; the angles come from NumPy's arctan2 / arcsin / cos, which may differ
  from ``math``'s in the last bit.  Both sides are then within a few ulp of the same yaw (the common
  1/cos(theta) factor cancels inside atan2), so x = -(yaw/pi)*W differs by about 1e-13 at most, and
  floor(x/2) can only differ where x/2 lies that close to an integer.  Every row with x/2 within
  1e-9*(1 + |x/2|) of an integer, with R[2,0] within 1e-12 of an isclose threshold, or with a
  non-finite value is recomputed with the scalar code, so the result is the scalar result."""
  cur_inv = np.asarray(cur_inv, np.float64)
  poses = np.asarray(poses, np.float64)
  W = leg_output_width
  rel = cur_inv @ poses
  r20 = rel[:, 2, 0]
  thr = _ISCLOSE_ATOL + _ISCLOSE_RTOL * 1.0
  with np.errstate(all='ignore'):
    theta = -np.arcsin(r20)
    cos_theta = np.cos(theta)
    phi = np.arctan2(rel[:, 1, 0] / cos_theta, rel[:, 0, 0] / cos_theta)
    pole = (np.abs(r20 - (-1.0)) <= thr) | (np.abs(r20 - 1.0) <= thr)      # theta = +-pi/2 branches: yaw 0
    yaw = np.where(pole, 0.0, phi)
    x = -(yaw / np.pi) * W
    half = x / 2
    recheck = ((np.abs(half - np.round(half)) <= 1e-9 * (1.0 + np.abs(half)))
               | (np.abs(np.abs(r20 + 1.0) - thr) <= 1e-12) | (np.abs(np.abs(r20 - 1.0) - thr) <= 1e-12)
               | ~np.isfinite(x) | ~np.isfinite(rel[:, :3, :3]).all(axis=(1, 2)))
    bins = np.where(np.isfinite(x), x // 2 + W // 2, 0).astype(np.int64)
  for i in np.flatnonzero(recheck):
    bins[i] = _yaw_bin_scalar(cur_inv, poses[i], W)
  return bins


def cull_mask(cur_inv, pose_ref, radius, max_range):
  """Bool torch tensor (C, R): True where scan r, moved by ``pose_ref[r]`` and then ``cur_inv[c]``,
  provably has no point with depth < ``max_range``, so its range image is empty and its count is 0.
  ``cur_inv`` (C,4,4), ``pose_ref`` (R,4,4), ``radius`` (R,) = max |(x,y,z)| of each scan: float64
  torch tensors on any device.  A NaN or infinite radius never culls.

  With M = cur_inv[c] @ pose_ref[r], A = M[:3,:3], b = M[:3,3]: every moved point is M[:3,:]·(p,1)
  (whatever the bottom rows), so its exact depth is >= |b| - |A|_2 |p| >= |b| - |A|_F r.  The kernel
  rounds: the two 4x4 products err by at most 2·gamma_4·|C|_F|P|_F(r+1) in the coordinates
  (gamma_4 = 4u/(1-4u), u = 2^-53), and its depth is within 4u relative of the norm of those
  coordinates.  Here M, |b|, |A|_F and r carry rounding errors of the same kind, bounded by
  about 10·gamma_4·|C|_F|P|_F(r+1).  All of it is below 1e-13·(|C|_F|P|_F(r+1) + max_range), and
  the margin used is 1e-9·(|C|_F|P|_F(r+1) + max_range + 1), so a culled pair's computed depths are
  all >= max_range and the kernel's filter drops every point."""
  import torch
  M = torch.matmul(cur_inv[:, None, :3, :], pose_ref[None])                 # (C, R, 3, 4)
  b = torch.linalg.vector_norm(M[..., 3], dim=-1)
  a = torch.linalg.matrix_norm(M[..., :3])
  scale = torch.linalg.matrix_norm(cur_inv)[:, None] * torch.linalg.matrix_norm(pose_ref)[None] * (radius[None] + 1.0)
  margin = 1e-9 * (scale + max_range + 1.0)
  return (b - a * radius[None] > max_range + margin) & torch.isfinite(radius)[None] & torch.isfinite(scale)


def overlap_yaw_sequence(clouds, poses, frame_idxs=None, leg_output_width=360, resident_bytes=None):
  """Ground truth of many current frames at once: float64 rows [frame, reference, overlap, yaw bin],
  shaped (len(frame_idxs)·n, 4), equal to
  ``np.concatenate([overlap_yaw_from_clouds(clouds, poses, f) for f in frame_idxs])``.
  ``frame_idxs`` None = every frame; rows follow the list, repeats included.  ``clouds`` as in
  ``overlap_yaw_from_clouds``.

  The reference scans stay resident on the GPU and every (current, reference) pair is counted by
  ``Engine.gt_pair_counts``; pairs that ``cull_mask`` proves empty get 0 without a launch.  While the
  points fit ``resident_bytes`` (default: half the free device memory) every cloud is read and
  uploaded once; otherwise the reference scans go in resident chunks and each chunk is read again."""
  import torch
  poses = np.asarray(poses, dtype=np.float64)
  n = len(clouds)
  frames = np.arange(n) if frame_idxs is None else np.asarray(frame_idxs, dtype=np.int64).reshape(-1)
  if frames.size and (frames.min() < 0 or frames.max() >= n):
    raise IndexError('frame_idxs must lie in [0, %d)' % n)
  if frames.size == 0 or n == 0:
    return np.zeros((0, 4))
  eng = _engine(3.0, -25.0, 64, 900, 50)
  dev = eng.device
  max_range = float(eng.cfg.max_range)
  uniq, slot = np.unique(frames, return_inverse=True)
  if resident_bytes is None:
    resident_bytes = torch.cuda.mem_get_info(dev)[0] // 2
  cur_chunk = max(1, int(resident_bytes // 4) // _IMG_BYTES)
  ref_budget = max(1, int(resident_bytes) - min(cur_chunk, uniq.size) * _IMG_BYTES)

  def get(i):
    c = clouds[i]
    return np.ascontiguousarray(c() if callable(c) else c, np.float32)

  cur_on_dev = uniq.size <= cur_chunk
  cur_img = torch.empty((uniq.size, 64, 900), dtype=torch.float32, device=dev if cur_on_dev else 'cpu')
  radius = torch.zeros(n, dtype=torch.float64, device=dev)
  chunks, batch = [], None

  def flush(s0, arrays):
    # one resident chunk of reference scans: its radii and the images of the current frames in it
    b = eng.upload_clouds(arrays)
    s1 = s0 + len(arrays)
    seg = torch.repeat_interleave(torch.arange(len(arrays), device=dev), torch.diff(b.offsets))
    norm = torch.linalg.vector_norm(b.points[:, :3].double(), dim=1)
    rad = torch.zeros(len(arrays), dtype=torch.float64, device=dev).scatter_reduce_(0, seg, norm, 'amax')
    bad = torch.zeros(len(arrays), dtype=torch.float64, device=dev).scatter_reduce_(
        0, seg, (~torch.isfinite(norm)).double(), 'amax')
    radius[s0:s1] = torch.where(bad > 0, torch.full_like(rad, float('nan')), rad)
    us = np.flatnonzero((uniq >= s0) & (uniq < s1))
    for g0 in range(0, us.size, eng.max_batch_scans):
      g = us[g0:g0 + eng.max_batch_scans]
      local = [int(uniq[u]) - s0 for u in g]
      sub = _sub_batch(b, local)
      cur_img[g[0]:g[-1] + 1] = eng.gt_range(sub).to(cur_img.device)
    chunks.append((s0, s1))
    return b

  pending, pending_bytes, s0 = [], 0, 0
  for i in range(n):
    a = get(i)
    if pending and pending_bytes + a.nbytes > ref_budget:
      batch = None
      batch = flush(s0, pending)
      s0, pending, pending_bytes = i, [], 0
    pending.append(a)
    pending_bytes += a.nbytes
  batch = flush(s0, pending)
  del pending

  valid = (cur_img > 0).sum(dim=(1, 2)).cpu().numpy().astype(np.int64)
  if np.any(valid == 0):
    raise ZeroDivisionError('division by zero')               # what int(count) / valid_num raises per frame
  cur_inv = np.stack([np.linalg.inv(poses[f]) for f in uniq])
  cur_inv_dev = torch.from_numpy(cur_inv).to(dev)
  poses_dev = torch.from_numpy(poses).to(dev)
  counts = np.zeros((uniq.size, n), dtype=np.int64)
  for s0, s1 in chunks:
    if len(chunks) > 1:
      batch = None
      batch = eng.upload_clouds([get(i) for i in range(s0, s1)])
    for u0 in range(0, uniq.size, cur_chunk):
      u1 = min(uniq.size, u0 + cur_chunk)
      keep = torch.cat([~cull_mask(cur_inv_dev[c0:min(u1, c0 + 256)], poses_dev[s0:s1], radius[s0:s1], max_range)
                        for c0 in range(u0, u1, 256)])                 # (u1-u0, s1-s0)
      rc = torch.nonzero(keep.T)                                        # reference-major
      block = torch.zeros((u1 - u0, s1 - s0), dtype=torch.int32, device=dev)
      if rc.shape[0]:
        pairs = torch.stack([rc[:, 1], rc[:, 0]], dim=1).to(torch.int32)
        got = eng.gt_pair_counts(batch, poses_dev[s0:s1], cur_inv_dev[u0:u1], cur_img[u0:u1].to(dev), pairs)
        block[rc[:, 1], rc[:, 0]] = got
      counts[u0:u1, s0:s1] = block.cpu().numpy()
  eng.check()

  W = leg_output_width
  out = np.empty((frames.size * n, 4))
  ref_ids = np.arange(n, dtype=np.float64)
  bins = {}
  for k, (f, u) in enumerate(zip(frames.tolist(), slot.tolist())):
    if u not in bins:
      bins[u] = yaw_bins(cur_inv[u], poses, W).astype(np.float64)
    rows = out[k * n:(k + 1) * n]
    rows[:, 0] = f
    rows[:, 1] = ref_ids
    rows[:, 2] = counts[u].astype(np.float64) / float(valid[u])     # correctly rounded, as int / int
    rows[:, 3] = bins[u]
  return out


def _sub_batch(batch, local):
  """CloudBatch of scans ``local`` of ``batch``, copied on the device."""
  import torch
  from .engine import CloudBatch
  offs = batch.offsets_host
  parts = [batch.points[offs[i]:offs[i + 1]] for i in local]
  sizes = np.array([offs[i + 1] - offs[i] for i in local], np.int64)
  o = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
  return CloudBatch(torch.cat(parts), torch.from_numpy(o).to(batch.points.device), o)


def com_overlap_yaw_sequence(scan_paths, poses, frame_idxs=None, leg_output_width=360):
  """``com_overlap_yaw`` for many current frames (default: every frame): the rows of each frame in
  ``frame_idxs`` back to back, as ``overlap_yaw_sequence``.  Each ``.bin`` is read once while the
  sequence fits in device memory."""
  print('Start to compute ground truth overlap and yaw ...')
  clouds = [(lambda p=p: _read_scan(p)) for p in scan_paths]
  mapping = overlap_yaw_sequence(clouds, poses, frame_idxs, leg_output_width)
  print('Finish generating ground_truth_mapping!')
  return mapping


def normalize_data(ground_truth_mapping):
  """Drop-in for ``normalize_data`` (normalize_data.py:10-49): resample the overlap bins below 0.5 to
  the size of the [0.4, 0.5) bin, with the same global ``np.random`` draws in the same order."""
  gt_map = ground_truth_mapping
  ov = gt_map[:, 2]
  bins = [gt_map[np.where(ov < 0.1)]]
  for lo in range(1, 9):
    bins.append(gt_map[(ov < (lo + 1) / 10) & (ov >= lo / 10)])
  bins.append(gt_map[(ov <= 1) & (ov >= 0.9)])
  m = len(bins[4])
  for b in range(5):
    bins[b] = bins[b][np.random.choice(len(bins[b]), m)]
  dist_norm_data = np.concatenate(bins)
  print("size of normalized data: ", len(dist_norm_data))
  return dist_norm_data


def split_train_val(ground_truth_mapping):
  """Drop-in for ``split_train_val`` (split_train_val.py:10-26), which is sklearn's
  ``train_test_split(test_size=int(n/10))``: one ``np.random.permutation(n)`` from the global
  generator, validation = its first n//10 entries, training = the rest."""
  n = len(ground_truth_mapping)
  test_size = int(n / 10)
  if test_size <= 0 or test_size >= n:
    raise ValueError('test_size=%d should be either positive and smaller than the number of samples %d'
                     % (test_size, n))
  perm = np.random.permutation(n)
  test_set = ground_truth_mapping[perm[:test_size]]
  train_set = ground_truth_mapping[perm[test_size:]]
  print('finished generating training data and validation data')
  return train_set, test_set


def _load_files(folder):
  """``load_files`` (utils.py:233-239): every file under ``folder``, sorted."""
  paths = [os.path.join(dp, f) for dp, dn, fn in os.walk(os.path.expanduser(folder)) for f in fn]
  paths.sort()
  return paths


def kitti_lidar_poses(poses_file, calib_file):
  """Poses of a KITTI sequence moved into the LiDAR frame of scan 0, as demo4_gen_gt_files.py:60-74."""
  T_cam_velo = np.asarray(load_calib(calib_file)).reshape((4, 4))
  T_velo_cam = np.linalg.inv(T_cam_velo)
  poses = load_poses(poses_file)
  pose0_inv = np.linalg.inv(poses[0])
  return np.array([T_velo_cam.dot(pose0_inv).dot(pose).dot(T_cam_velo) for pose in poses])


def write_gt_files(dst_folder, ground_truth_mapping, train_data, validation_data, seq_idx):
  """``dst_folder/ground_truth/{train_set, validation_set, ground_truth_overlap_yaw}.npz`` with
  ``overlaps=`` and the object ``seq=`` column pair, as demo4_gen_gt_files.py:85-112."""
  dst_folder = os.path.join(dst_folder, 'ground_truth')
  try:
    os.stat(dst_folder)
    print('generating depth data in: ', dst_folder)
  except OSError:
    print('creating new depth folder: ', dst_folder)
    os.mkdir(dst_folder)
  for name, data in (('train_set', train_data), ('validation_set', validation_data),
                     ('ground_truth_overlap_yaw', ground_truth_mapping)):
    seq = np.empty((data.shape[0], 2), dtype=object)
    seq[:] = seq_idx
    np.savez_compressed(os.path.join(dst_folder, name), overlaps=data, seq=seq)
  print('Finish saving the ground truth data for training and testing at: ', dst_folder)
  return dst_folder


def main(argv=None):
  """demo4_gen_gt_files.py without the plot: ground truth of frame 0 (or of every frame with
  --all-pairs), normalised, split and written next to the sequence."""
  ap = argparse.ArgumentParser(prog='python -m overlapnet_b200.gt', description=main.__doc__)
  ap.add_argument('config', nargs='?', default='config/demo.yml', help='demo YAML with a Demo4 section')
  ap.add_argument('--all-pairs', action='store_true', help='every frame as the current frame, not only frame 0')
  ap.add_argument('--seq', default='07', help="sequence label stored in the files' seq column")
  args = ap.parse_args(argv)
  import yaml
  with open(args.config) as f:
    config = yaml.safe_load(f)['Demo4']
  scan_paths = _load_files(config['scan_folder'])
  poses = kitti_lidar_poses(config['poses_file'], config['calib_file'])
  if args.all_pairs:
    ground_truth_mapping = com_overlap_yaw_sequence(scan_paths, poses)
  else:
    ground_truth_mapping = com_overlap_yaw(scan_paths, poses, frame_idx=0)
  dist_norm_data = normalize_data(ground_truth_mapping)
  train_data, validation_data = split_train_val(dist_norm_data)
  write_gt_files(config['dst_folder'], ground_truth_mapping, train_data, validation_data, args.seq)
  return 0


if __name__ == '__main__':
  sys.exit(main())
