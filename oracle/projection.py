"""NumPy oracle for the preprocessing stage (TEST INFRASTRUCTURE, see oracle/__init__.py).

Restates, operation by operation and in float32, what the reference computes in
its ``src/utils/utils.py`` and the ``gen_*_data.py`` drivers.  Parity is PINNED:
``tests/test_oracle_projection.py`` checks every function here bit-for-bit against the golden
vectors generated from the reference (``tools/make_golden.py``, ``tools/make_golden_reference.py``).

Two places where the reference's result depends on the host's NumPy build are given a canonical,
host-independent definition here (and the CUDA kernels implement the same definition):

* ``np.arctan2`` / ``np.arcsin`` on float32 (utils.py:86-87) dispatch to SIMD routines that are
  not correctly rounded (about 39 % / 5 % of results differ in the last bit from the rounded exact
  value on this host).  The oracle uses the *correctly rounded* float32 value, obtained by
  evaluating in float64 and rounding once.  On both reference fixtures every projection bin is
  identical to the reference's; on arbitrary clouds a few points per scan that sit within one
  float32 ulp of a bin edge may land in the neighbouring bin (counted by
  ``tests/test_oracle_projection.py::test_live_reference_synthetic``).
* ``np.argsort`` (utils.py:107) is unstable, so the winner among points of *exactly equal depth*
  in one pixel is unspecified.  The oracle picks the lowest point index, which is what the
  reference produced for the tied pixels of both fixtures.
"""
import os

import numpy as np

F32 = np.float32
F64 = np.float64


def _norm3_rows(v):
  """``np.linalg.norm(v[:, :3], 2, axis=1)`` for a float32 (N,>=3) array (utils.py:75).

  NumPy evaluates ``sqrt(add.reduce(x*x, axis=1))``; for a C-contiguous (N,3) operand the reduce
  runs left to right: ((x*x + y*y) + z*z), every step rounded to float32 (verified bit-exact on
  the fixtures).
  """
  x, y, z = v[:, 0], v[:, 1], v[:, 2]
  return np.sqrt((x * x + y * y) + z * z)


def _norm3_vec(d):
  """``np.linalg.norm(d)`` for float32 3-vectors stacked on the last axis (utils.py:166-171).

  The 1-D path is ``sqrt(d.dot(d))``; NumPy's float32 dot rounds each product to float32,
  accumulates the products in a double and rounds the sum to float32 once (FLOAT_dot over
  cblas_sdot).  Verified bit-exact on both fixtures' normal maps.
  """
  p = d * d  # float32 products
  s = (p[..., 0].astype(F64) + p[..., 1].astype(F64)) + p[..., 2].astype(F64)
  return np.sqrt(s.astype(F32))


def point_depth(points):
  """float32 depth of every point, utils.py:75."""
  return _norm3_rows(np.ascontiguousarray(points[:, :3], dtype=F32))


def projection_bins(points, fov_up=3.0, fov_down=-25.0, proj_H=64, proj_W=900, max_range=50):
  """Per-point (valid mask, depth, proj_y, proj_x) following utils.py:69-104.

  ``valid`` is the filter of utils.py:76-77; bins are int32 and only meaningful where valid.
  """
  points = np.asarray(points)
  if points.dtype != F32:
    raise TypeError('oracle.projection handles the float32 path only (gen_*_data.py read .bin as float32)')
  fov_up_r = fov_up / 180.0 * np.pi          # Python floats (float64), utils.py:70-72
  fov_down_r = fov_down / 180.0 * np.pi
  fov = abs(fov_down_r) + abs(fov_up_r)

  depth = point_depth(points)                # utils.py:75
  with np.errstate(invalid='ignore'):
    valid = (depth > 0) & (depth < F32(max_range))          # utils.py:76-77 (weak scalar -> float32)
  x, y, z = points[:, 0], points[:, 1], points[:, 2]

  with np.errstate(all='ignore'):
    # utils.py:86-87, correctly rounded float32 (see module docstring)
    yaw = (-np.arctan2(y.astype(F64), x.astype(F64))).astype(F32)
    q = z / depth                             # float32 division
    pitch = np.arcsin(q.astype(F64)).astype(F32)

    # utils.py:90-95 -- Python scalars are weak: every operation stays float32
    proj_x = F32(0.5) * (yaw / F32(np.pi) + F32(1.0))
    proj_y = F32(1.0) - (pitch + F32(abs(fov_down_r))) / F32(fov)
    proj_x = proj_x * F32(proj_W)
    proj_y = proj_y * F32(proj_H)

    # utils.py:98-104
    proj_x = np.maximum(F32(0), np.minimum(F32(proj_W - 1), np.floor(proj_x)))
    proj_y = np.maximum(F32(0), np.minimum(F32(proj_H - 1), np.floor(proj_y)))
  px = np.where(valid, proj_x, 0).astype(np.int32)
  py = np.where(valid, proj_y, 0).astype(np.int32)
  return valid, depth, py, px


def range_projection(current_vertex, fov_up=3.0, fov_down=-25.0, proj_H=64, proj_W=900, max_range=50):
  """Oracle of ``range_projection`` (utils.py:59-134).

  Returns (proj_range (H,W) f32, proj_vertex (H,W,4) f32, proj_intensity (H,W) f32,
  proj_idx (H,W) i32).  ``proj_idx`` indexes the *filtered* cloud (utils.py:76,117-118).
  """
  pts = np.asarray(current_vertex)
  valid, depth, py, px = projection_bins(pts, fov_up, fov_down, proj_H, proj_W, max_range)
  sel = np.nonzero(valid)[0]
  d = depth[sel]
  yy = py[sel].astype(np.int64)
  xx = px[sel].astype(np.int64)
  filt_idx = np.arange(sel.shape[0], dtype=np.int64)      # index into the filtered cloud

  # nearest point wins (utils.py:107-132); exact-depth ties -> lowest index
  key = (d.view(np.uint32).astype(np.uint64) << np.uint64(32)) | filt_idx.astype(np.uint64)
  pix = yy * proj_W + xx
  win = np.full(proj_H * proj_W, np.iinfo(np.uint64).max, dtype=np.uint64)
  np.minimum.at(win, pix, key)
  has = win != np.iinfo(np.uint64).max
  widx = (win[has] & np.uint64(0xFFFFFFFF)).astype(np.int64)   # filtered index of the winner

  proj_range = np.full((proj_H, proj_W), -1, dtype=F32)       # utils.py:120-127
  proj_vertex = np.full((proj_H, proj_W, 4), -1, dtype=F32)
  proj_idx = np.full((proj_H, proj_W), -1, dtype=np.int32)
  proj_intensity = np.full((proj_H, proj_W), -1, dtype=F32)

  src = sel[widx]
  proj_range.reshape(-1)[has] = d[widx]
  v = proj_vertex.reshape(-1, 4)
  v[has, 0] = pts[src, 0]
  v[has, 1] = pts[src, 1]
  v[has, 2] = pts[src, 2]
  v[has, 3] = 1.0
  proj_idx.reshape(-1)[has] = widx.astype(np.int32)
  proj_intensity.reshape(-1)[has] = pts[src, 3]
  return proj_range, proj_vertex, proj_intensity, proj_idx


def gen_normal_map(current_range, current_vertex, proj_H=64, proj_W=900):
  """Oracle of ``gen_normal_map`` (utils.py:137-175), vectorised over the pixel loop.

  For x in [0,W), y in [0,H-1): p = vertex[y,x], u = vertex[y, (x+1) mod W], v = vertex[y+1, x];
  needs range>0 at all three; normal = normalise(normalise(v-p) x normalise(u-p)); stays -1 when
  invalid or when the cross product's norm is not > 0 (nan included).  Row H-1 is never written.
  """
  r = np.asarray(current_range, dtype=F32)
  vert = np.asarray(current_vertex, dtype=F32)
  out = np.full((proj_H, proj_W, 3), -1, dtype=F32)
  p = vert[:proj_H - 1, :, :3]
  u = np.roll(vert, -1, axis=1)[:proj_H - 1, :, :3]          # wrap(x+1, W), utils.py:155,178-186
  v = vert[1:, :, :3]
  ok = (r[:proj_H - 1] > 0) & (np.roll(r, -1, axis=1)[:proj_H - 1] > 0) & (r[1:] > 0)
  with np.errstate(all='ignore'):
    du = u - p
    dv = v - p
    un = du / _norm3_vec(du)[..., None]                      # utils.py:166
    vn = dv / _norm3_vec(dv)[..., None]                      # utils.py:167
    w = np.empty_like(un)                                    # np.cross(v_norm, u_norm), utils.py:169
    w[..., 0] = vn[..., 1] * un[..., 2] - vn[..., 2] * un[..., 1]
    w[..., 1] = vn[..., 2] * un[..., 0] - vn[..., 0] * un[..., 2]
    w[..., 2] = vn[..., 0] * un[..., 1] - vn[..., 1] * un[..., 0]
    nw = _norm3_vec(w)                                       # utils.py:170
    n = w / nw[..., None]                                    # utils.py:172
    ok = ok & (nw > 0)                                       # utils.py:171 (nan > 0 is False)
  out[:proj_H - 1][ok] = n[ok]
  return out


def gen_semantic_image(points, probs, proj_H=64, proj_W=900):
  """Oracle of the per-scan body of ``gen_semantic_data`` (gen_semantic_data.py:36-46).

  Reproduces the reference's quirk: ``proj_idx`` indexes the filtered cloud but is used to index
  the unfiltered ``probs``.
  """
  _, _, _, proj_idx = range_projection(points, proj_H=proj_H, proj_W=proj_W, max_range=np.inf)
  proj_prob = np.full((proj_H, proj_W, probs.shape[1]), -1, dtype=F32)
  proj_prob[proj_idx >= 0] = probs[proj_idx[proj_idx >= 0]]
  return proj_prob


def pack_input(depth=None, normal=None, probability=None, intensity=None):
  """Channel packing of ``prepareOneInput`` (ImagePairOverlapOrientationSequence.py:130-207):
  depth, normal(3), probabilities(20 or 3), intensity; raw values, empty = -1.  Returns (H,W,C) f32
  (the reference builds float64 and Keras casts to float32)."""
  chans = []
  if depth is not None:
    chans.append(np.asarray(depth, F32)[..., None])
  if normal is not None:
    chans.append(np.asarray(normal, F32))
  if probability is not None:
    chans.append(np.asarray(probability, F32))
  if intensity is not None:
    chans.append(np.asarray(intensity, F32)[..., None])
  return np.concatenate(chans, axis=-1)


def load_files(folder):
  """utils.py:233-239."""
  file_paths = [os.path.join(dp, f) for dp, dn, fn in os.walk(os.path.expanduser(folder)) for f in fn]
  file_paths.sort()
  return file_paths


def gen_cue_folder(scan_folder, dst_folder, cue, semantic_folder=None):
  """Oracle of the folder drivers gen_depth_data.py:10-48, gen_normal_data.py:10-46,
  gen_intensity_data.py:10-43, gen_semantic_data.py:11-57: same sub-folder names, file naming
  (enumeration index for depth/normal/intensity, scan basename for semantic) and .npy format."""
  sub = {'depth': 'depth', 'normal': 'normal', 'intensity': 'intensity', 'semantic': 'semantic'}[cue]
  dst = os.path.join(dst_folder, sub)
  os.makedirs(dst, exist_ok=True)
  scan_paths = load_files(scan_folder)
  prob_paths = load_files(semantic_folder) if cue == 'semantic' else None
  n = len(prob_paths) if cue == 'semantic' else len(scan_paths)
  out = []
  for idx in range(n):
    pts = np.fromfile(scan_paths[idx], dtype=F32).reshape((-1, 4))
    if cue == 'semantic':
      probs = np.fromfile(prob_paths[idx], dtype=F32).reshape((-1, 20))
      img = gen_semantic_image(pts, probs)
      name = os.path.basename(scan_paths[idx]).replace('.bin', '')
    else:
      rng, vert, inten, _ = range_projection(pts)
      img = {'depth': rng, 'intensity': inten}.get(cue)
      if cue == 'normal':
        img = gen_normal_map(rng, vert)
      name = str(idx).zfill(6)
    np.save(os.path.join(dst, name), img)
    out.append(img)
  return out
