"""Thin torch-facing wrapper of the C ABI (include/ovn_b200.h).

PyTorch is plumbing here: it owns device memory and streams; every compute step is a call into
libovn_b200.so.  All methods take / return CUDA tensors and are asynchronous on the current torch
stream unless stated otherwise.
"""
import ctypes as C

import numpy as np
import torch

from . import _cabi
from ._cabi import OvnConfig, OvnError, check, lib

FEAT_C = 128


def _ptr(t):
  return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class CloudBatch:
  """Clouds back to back on the device: points [sum N, 4] f32, offsets [n+1] i64 (+ a host copy)."""

  def __init__(self, points, offsets, offsets_host):
    self.points, self.offsets, self.offsets_host = points, offsets, np.asarray(offsets_host, np.int64)
    self.n = int(self.offsets_host.shape[0] - 1)


class Engine:
  """One handle per GPU.  ``use`` = dict of cue flags like the reference's config
  (config/network.yml:20-24); ``model`` = the ``model:`` section (network.yml:64-82)."""

  def __init__(self, use=None, model=None, precision='f16_tc', device=None, max_batch_scans=16,
               max_batch_pairs=1101, proj_H=64, proj_W=900, fov_up=3.0, fov_down=-25.0, max_range=50.0):
    L = lib()
    if not torch.cuda.is_available():
      raise OvnError('no CUDA device: overlapnet_b200 has no CPU fallback')
    self.device = torch.device('cuda', torch.cuda.current_device() if device is None else device)
    use = dict(use or {})
    model = dict(model or {})
    cfg = OvnConfig()
    L.ovn_default_config(C.byref(cfg))
    cfg.proj_H, cfg.proj_W = proj_H, proj_W
    cfg.fov_up_deg, cfg.fov_down_deg, cfg.max_range = fov_up, fov_down, max_range
    cfg.use_depth = int(bool(use.get('use_depth', True)))
    cfg.use_normals = int(bool(use.get('use_normals', True)))
    cfg.use_intensity = int(bool(use.get('use_intensity', False)))
    if use.get('use_class_probabilities', False):
      cfg.n_prob_channels = 3 if use.get('use_class_probabilities_pca', False) else 20
    else:
      cfg.n_prob_channels = 0
    s1 = model.get('strides_layer1', (2, 2))
    cfg.strides_layer1[0], cfg.strides_layer1[1] = int(s1[0]), int(s1[1])
    cfg.additional_unsymmetric_layer3a = int(bool(model.get('additional_unsymmetric_layer3a', False)))
    cfg.leg_output_width = int(model.get('leg_output_width', 360))
    cfg.conv1size = int(model.get('conv1NetworkHead_conv1size', 15))
    cfg.precision = {'fp32': _cabi.PREC_FP32, 'f16_tc': _cabi.PREC_F16_TC}[precision]
    cfg.max_batch_scans = int(max_batch_scans)
    cfg.max_batch_pairs = int(max_batch_pairs)
    self.cfg = cfg
    self._model = model
    self.precision = precision
    self.H, self.W = proj_H, proj_W
    self._h = C.c_void_p(0)
    with torch.cuda.device(self.device):
      st = L.ovn_create(C.byref(cfg), C.byref(self._h))
    if st != 0:
      raise OvnError('ovn_create failed: %s (%s)' % (L.ovn_status_string(st).decode(),
                                                     L.ovn_last_error(None).decode()))
    self.C = L.ovn_input_channels(self._h)
    self.Wf = L.ovn_feature_width(self._h)
    self.max_batch_scans = int(max_batch_scans)
    self.max_batch_pairs = int(max_batch_pairs)

  def close(self):
    if getattr(self, '_h', None) is not None and self._h.value:
      lib().ovn_destroy(self._h)
      self._h = C.c_void_p(0)

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass

  # ------------------------------------------------------------------------------------------
  def _stream(self):
    return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

  def launch_count(self):
    return int(lib().ovn_launch_count(self._h))

  def check(self):
    """ovn_check: synchronises the current stream and raises OvnError if a kernel flagged an error
    since the last check (index out of range, unprepared resident row, pipeline barrier time-out);
    the affected outputs hold NaN / INT32_MIN."""
    check(self._h, lib().ovn_check(self._h, self._stream()), 'ovn_check')

  def set_feature_center(self, mu=None):
    """Fix the per-channel centre of the fp16 operand copies (None = calibrate at first use)."""
    ptr = None
    if mu is not None:
      mu = np.ascontiguousarray(mu, np.float32).reshape(FEAT_C)
      ptr = mu.ctypes.data_as(C.c_void_p)
    check(self._h, lib().ovn_set_feature_center(self._h, ptr), 'ovn_set_feature_center')

  def peer_signal(self, flag_addrs, value):
    """ovn_peer_signal: one launch stores ``value`` (release.sys) to each peer-mapped flag address."""
    arr = (C.c_uint64 * len(flag_addrs))(*[int(a) for a in flag_addrs])
    check(self._h, lib().ovn_peer_signal(self._h, arr, len(flag_addrs), int(value), self._stream()), 'ovn_peer_signal')

  def peer_wait(self, flags, n, skip, value):
    """ovn_peer_wait: one launch waits until flags[i] >= value for every i < n except ``skip``."""
    check(self._h, lib().ovn_peer_wait(self._h, _ptr(flags), int(n), int(skip), int(value), self._stream()), 'ovn_peer_wait')

  def calibrate(self, volume):
    """ovn_calibrate: derive the three centres of the tensor-core heads from this [360,128] volume."""
    v = volume.to(device=self.device, dtype=torch.float32).contiguous()
    check(self._h, lib().ovn_calibrate(self._h, _ptr(v), self._stream()), 'ovn_calibrate')

  def get_feature_center(self):
    mu = np.zeros(FEAT_C, np.float32)
    is_set = C.c_int32(0)
    check(self._h, lib().ovn_get_feature_center(self._h, mu.ctypes.data_as(C.c_void_p), C.byref(is_set)),
          'ovn_get_feature_center')
    return mu, bool(is_set.value)

  def profile_enable(self, on=True):
    check(self._h, lib().ovn_profile_enable(self._h, int(bool(on))), 'ovn_profile_enable')

  def profile_read(self, kernel):
    """(total milliseconds, launches) of the named kernel since the last read; synchronises."""
    ms, n = C.c_double(0), C.c_int64(0)
    check(self._h, lib().ovn_profile_read(self._h, kernel.encode(), C.byref(ms), C.byref(n)), 'ovn_profile_read')
    return ms.value, int(n.value)

  def load_weights(self, weights):
    """weights: {layer name: (kernel, bias)} in Keras layouts (overlapnet_b200.weights)."""
    L = lib()
    for name, (k, b) in weights.items():
      k = np.ascontiguousarray(k, dtype=np.float32)
      b = np.ascontiguousarray(b, dtype=np.float32)
      dims = (C.c_int64 * k.ndim)(*k.shape)
      check(self._h, L.ovn_set_weights(self._h, name.encode(), k.ctypes.data_as(C.c_void_p), dims, k.ndim,
                                       b.ctypes.data_as(C.c_void_p), b.size), 'ovn_set_weights(%s)' % name)
    check(self._h, L.ovn_finalize_weights(self._h), 'ovn_finalize_weights')

  # ---- clouds --------------------------------------------------------------------------------
  def upload_clouds(self, clouds):
    """list of (N_i, 4) float32 arrays -> CloudBatch (points [sum N, 4] cuda, offsets [n+1] int64)."""
    offs = np.zeros(len(clouds) + 1, np.int64)
    for i, c in enumerate(clouds):
      offs[i + 1] = offs[i] + c.shape[0]
    flat = np.concatenate([np.ascontiguousarray(c, np.float32).reshape(-1, 4) for c in clouds]) if clouds \
        else np.zeros((0, 4), np.float32)
    return CloudBatch(torch.from_numpy(flat).to(self.device), torch.from_numpy(offs).to(self.device), offs)

  def _chunks(self, batch):
    n = batch.n
    for s0 in range(0, n, self.max_batch_scans):
      s1 = min(n, s0 + self.max_batch_scans)
      p0, p1 = int(batch.offsets_host[s0]), int(batch.offsets_host[s1])
      pts = batch.points[p0:p1]
      offs = batch.offsets[s0:s1 + 1] if p0 == 0 else (batch.offsets[s0:s1 + 1] - p0)
      yield s0, s1, p0, p1, pts, offs.contiguous()

  def project(self, batch, max_range=-1.0, want=('range', 'vertex', 'intensity', 'idx')):
    """ovn_project_batch: range_projection (utils.py:59-134) for a CloudBatch."""
    n = batch.n
    dev = self.device
    out = {}
    if 'range' in want: out['range'] = torch.empty((n, self.H, self.W), dtype=torch.float32, device=dev)
    if 'vertex' in want: out['vertex'] = torch.empty((n, self.H, self.W, 4), dtype=torch.float32, device=dev)
    if 'intensity' in want: out['intensity'] = torch.empty((n, self.H, self.W), dtype=torch.float32, device=dev)
    if 'idx' in want: out['idx'] = torch.empty((n, self.H, self.W), dtype=torch.int32, device=dev)
    L = lib()
    for s0, s1, p0, p1, pts, offs in self._chunks(batch):
      sl = {k: v[s0:s1] for k, v in out.items()}
      check(self._h, L.ovn_project_batch(
          self._h, _ptr(pts), _ptr(offs), s1 - s0, p1 - p0, float(max_range),
          _ptr(sl.get('range')), _ptr(sl.get('vertex')), _ptr(sl.get('intensity')), _ptr(sl.get('idx')),
          self._stream()), 'ovn_project_batch')
    return out

  def gt_range(self, batch, pose_ref=None, pose_cur_inv=None, max_range=-1.0):
    """ovn_gt_range_batch: float32 range images of the scans of a CloudBatch after the two float64
    pose products of com_overlap_yaw.py:39-40 (``pose_ref``: (n,4,4) float64 or None, ``pose_cur_inv``:
    (4,4) float64 or None), projected in float64 like the reference's GT generator."""
    n = batch.n
    dev = self.device
    out = torch.empty((n, self.H, self.W), dtype=torch.float32, device=dev)
    pr = None if pose_ref is None else torch.as_tensor(pose_ref, dtype=torch.float64).reshape(n, 16).to(dev).contiguous()
    pc = None if pose_cur_inv is None else torch.as_tensor(pose_cur_inv, dtype=torch.float64).reshape(16).to(dev).contiguous()
    L = lib()
    for s0, s1, p0, p1, pts, offs in self._chunks(batch):
      check(self._h, L.ovn_gt_range_batch(
          self._h, _ptr(pts), _ptr(offs), s1 - s0, p1 - p0, _ptr(pr[s0:s1]) if pr is not None else None, _ptr(pc),
          float(max_range), _ptr(out[s0:s1]), self._stream()), 'ovn_gt_range_batch')
    return out

  def gt_overlap_count(self, ref_ranges, cur_range):
    """ovn_gt_overlap_count: int32 [n + 1]: per reference image the number of pixels with ref > 0 and
    |ref - cur| < 1 (com_overlap_yaw.py:44-45); last entry = number of valid pixels of ``cur_range``."""
    n = ref_ranges.shape[0]
    counts = torch.empty((n + 1,), dtype=torch.int32, device=self.device)
    check(self._h, lib().ovn_gt_overlap_count(self._h, _ptr(ref_ranges), _ptr(cur_range), n, _ptr(counts),
                                             self._stream()), 'ovn_gt_overlap_count')
    return counts

  def normals(self, rng, vertex):
    n = rng.shape[0]
    out = torch.empty((n, self.H, self.W, 3), dtype=torch.float32, device=self.device)
    check(self._h, lib().ovn_normals_batch(self._h, _ptr(rng), _ptr(vertex), n, _ptr(out), self._stream()),
          'ovn_normals_batch')
    return out

  def semantic(self, idx, probs, offsets):
    n = idx.shape[0]
    ncls = probs.shape[1]
    out = torch.empty((n, self.H, self.W, ncls), dtype=torch.float32, device=self.device)
    check(self._h, lib().ovn_semantic_batch(self._h, _ptr(idx), _ptr(probs), _ptr(offsets), n, ncls, _ptr(out),
                                           self._stream()), 'ovn_semantic_batch')
    return out

  def preprocess(self, batch, probs=None):
    """Fused raw clouds (CloudBatch) -> packed NHWC network input [n, H, W, C]."""
    n = batch.n
    out = torch.empty((n, self.H, self.W, self.C), dtype=torch.float32, device=self.device)
    L = lib()
    for s0, s1, p0, p1, pts, offs in self._chunks(batch):
      pr = probs[p0:p1] if probs is not None else None
      check(self._h, L.ovn_preprocess_batch(self._h, _ptr(pts), _ptr(offs), s1 - s0, p1 - p0, _ptr(pr),
                                            _ptr(out[s0:s1]), self._stream()), 'ovn_preprocess_batch')
    return out

  def pack_input(self, depth=None, normal=None, prob=None, intensity=None):
    first = next(t for t in (depth, normal, prob, intensity) if t is not None)
    n = first.shape[0]
    out = torch.empty((n, self.H, self.W, self.C), dtype=torch.float32, device=self.device)
    check(self._h, lib().ovn_pack_input(self._h, _ptr(depth), _ptr(normal), _ptr(prob), _ptr(intensity), n,
                                       _ptr(out), self._stream()), 'ovn_pack_input')
    return out

  # ---- network -------------------------------------------------------------------------------
  def leg(self, x_nhwc):
    """[n, H, W, C] float32 cuda -> feature volumes [n, 360, 128] float32 cuda."""
    x = x_nhwc.contiguous()
    n = x.shape[0]
    out = torch.empty((n, self.Wf, FEAT_C), dtype=torch.float32, device=self.device)
    check(self._h, lib().ovn_leg_forward(self._h, _ptr(x), n, _ptr(out), self._stream()), 'ovn_leg_forward')
    return out

  def heads(self, bank, left_idx, right_idx, want_corr=False):
    """LEFT = bank[left_idx], RIGHT = bank[right_idx] -> (overlap [n] f32, yaw [n] i32, corr|None)."""
    n = left_idx.numel()
    ov = torch.empty((n,), dtype=torch.float32, device=self.device)
    yaw = torch.empty((n,), dtype=torch.int32, device=self.device)
    corr = torch.empty((n, self.Wf), dtype=torch.float32, device=self.device) if want_corr else None
    li = left_idx.to(device=self.device, dtype=torch.int32).contiguous()
    ri = right_idx.to(device=self.device, dtype=torch.int32).contiguous()
    check(self._h, lib().ovn_heads_forward(self._h, _ptr(bank), int(bank.shape[0]), _ptr(li), _ptr(ri), n, _ptr(ov),
                                          _ptr(yaw), _ptr(corr), self._stream()), 'ovn_heads_forward')
    return ov, yaw, corr

  def heads_1vsN(self, bank, query, cand_idx=None, n_cand=None, want_corr=False, out=None):
    """RIGHT = query [360,128] for every pair, LEFT = bank[cand_idx] (None = first n_cand rows).
    ``out`` = (overlap f32 [n], yaw i32 [n]) tensors to write into -- they may live in another GPU's
    peer-mapped memory (search.py transport 'symm'): the kernels that finish a pair store there directly."""
    if cand_idx is not None:
      ci = cand_idx.to(device=self.device, dtype=torch.int32).contiguous()
      n = ci.numel()
    else:
      ci = None
      n = int(bank.shape[0] if n_cand is None else n_cand)
    if out is not None:
      ov, yaw = out
      assert ov.numel() == n and yaw.numel() == n and ov.dtype == torch.float32 and yaw.dtype == torch.int32
      assert ov.is_contiguous() and yaw.is_contiguous()
    else:
      ov = torch.empty((n,), dtype=torch.float32, device=self.device)
      yaw = torch.empty((n,), dtype=torch.int32, device=self.device)
    corr = torch.empty((n, self.Wf), dtype=torch.float32, device=self.device) if want_corr else None
    check(self._h, lib().ovn_heads_1vsN(self._h, _ptr(bank), int(bank.shape[0]), _ptr(query), _ptr(ci), n, _ptr(ov),
                                       _ptr(yaw), _ptr(corr), self._stream()), 'ovn_heads_1vsN')
    return ov, yaw, corr

  def heads_rows_vs_bank(self, bank, row_lo, row_hi):
    """Rows [row_lo, row_hi) of the ordered all-pairs matrix of ``bank`` (RIGHT = bank[i], LEFT = every
    row): (overlap [rows, n] f32, yaw [rows, n] i32).  One C-ABI call; the row loop runs in the library."""
    n = int(bank.shape[0])
    rows = int(row_hi) - int(row_lo)
    ov = torch.empty((rows, n), dtype=torch.float32, device=self.device)
    yaw = torch.empty((rows, n), dtype=torch.int32, device=self.device)
    check(self._h, lib().ovn_heads_rows_vs_bank(self._h, _ptr(bank), n, int(row_lo), int(row_hi), _ptr(ov), _ptr(yaw),
                                               self._stream()), 'ovn_heads_rows_vs_bank')
    return ov, yaw

  def bank_prepare(self, bank, first=0, count=None):
    """Keep the tensor-core operand copies of bank rows [first, first+count) resident: later heads
    calls on this same tensor skip the per-call conversion (ovn_bank_prepare)."""
    count = int(bank.shape[0]) - first if count is None else int(count)
    check(self._h, lib().ovn_bank_prepare(self._h, _ptr(bank), int(bank.shape[0]), int(first), count, self._stream()),
          'ovn_bank_prepare')

  def bank_release(self, bank=None):
    check(self._h, lib().ovn_bank_release(self._h, _ptr(bank)), 'ovn_bank_release')

  # ---- overlap-head training on a frozen leg (precision fp32) ---------------------------------
  HEAD_LAYERS = ('c_conv1', 'c_conv2', 'c_conv3', 'overlap_output')

  def heads_backward(self, bank, left_idx, right_idx, overlap_gt, yaw_bin_gt, min_overlap_for_angle=0.7):
    """ovn_heads_backward: losses and head gradients of one batch (LEFT = bank[left_idx], RIGHT =
    bank[right_idx]).  Returns a float32 cuda tensor [3] = (5 L_ov + L_or, L_ov, L_or); the gradients
    stay in the handle (``gradients()``, ``adagrad_step``)."""
    n = left_idx.numel()
    dev = self.device
    li = left_idx.to(device=dev, dtype=torch.int32).contiguous()
    ri = right_idx.to(device=dev, dtype=torch.int32).contiguous()
    ov = torch.as_tensor(overlap_gt).to(device=dev, dtype=torch.float32).contiguous()
    yb = torch.as_tensor(yaw_bin_gt).to(device=dev, dtype=torch.int32).contiguous()
    losses = torch.empty((3,), dtype=torch.float32, device=dev)
    check(self._h, lib().ovn_heads_backward(self._h, _ptr(bank), int(bank.shape[0]), _ptr(li), _ptr(ri), n, _ptr(ov),
                                           _ptr(yb), float(min_overlap_for_angle), _ptr(losses), self._stream()),
          'ovn_heads_backward')
    return losses

  def _layer_arrays(self, fn, what, names=None):
    from .weights import layer_shapes
    shapes = layer_shapes(self.C, self._model, self.H, self.W)
    out = {}
    for name in (names or list(shapes)):
      ks, bs = shapes[name]
      k, b = np.empty(ks, np.float32), np.empty(bs, np.float32)
      check(self._h, fn(self._h, name.encode(), k.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p)),
            '%s(%s)' % (what, name))
      out[name] = (k, b)
    return out

  def gradients(self):
    """{layer: (kernel grad, bias grad)} of the head layers after the last ``heads_backward``, keyed
    like ``weights.glorot_init``; synchronises."""
    return self._layer_arrays(lib().ovn_get_gradient, 'ovn_get_gradient', self.HEAD_LAYERS)

  def get_weights(self):
    """{layer: (kernel, bias)} of every layer, trained head weights included; synchronises."""
    return self._layer_arrays(lib().ovn_get_weights, 'ovn_get_weights')

  def adagrad_step(self, lr):
    """ovn_adagrad_step: one Keras Adagrad update of the head weights with the last gradients."""
    check(self._h, lib().ovn_adagrad_step(self._h, float(lr), self._stream()), 'ovn_adagrad_step')

  def finalize_weights(self):
    """ovn_finalize_weights: repack the inference path from the (trained) weights."""
    check(self._h, lib().ovn_finalize_weights(self._h), 'ovn_finalize_weights')

  # ---- host-buffer entry points (synchronous) ------------------------------------------------
  def encode_clouds_host(self, clouds):
    offs = np.zeros(len(clouds) + 1, np.int64)
    for i, c in enumerate(clouds):
      offs[i + 1] = offs[i] + c.shape[0]
    flat = np.ascontiguousarray(np.concatenate([np.asarray(c, np.float32).reshape(-1, 4) for c in clouds]))
    out = np.empty((len(clouds), self.Wf, FEAT_C), np.float32)
    check(self._h, lib().ovn_encode_clouds_host(self._h, flat.ctypes.data_as(C.c_void_p),
                                               offs.ctypes.data_as(C.c_void_p), len(clouds),
                                               out.ctypes.data_as(C.c_void_p)), 'ovn_encode_clouds_host')
    return out

  def query_cloud_vs_bank_host(self, points_host, bank, cand_idx_host=None, n_cand=None, out_overlap=None,
                               out_yaw=None, out_query_fv=None):
    """points_host: (N,4) float32 numpy or pinned CPU tensor; bank: cuda [n,360,128].
    Returns (overlap float32 [n_cand], yaw int32 [n_cand]) host arrays."""
    if isinstance(points_host, torch.Tensor):
      p_ptr, npts = C.c_void_p(points_host.data_ptr()), int(points_host.shape[0])
    else:
      points_host = np.ascontiguousarray(points_host, np.float32)
      p_ptr, npts = points_host.ctypes.data_as(C.c_void_p), int(points_host.shape[0])
    if cand_idx_host is not None:
      cand_idx_host = np.ascontiguousarray(cand_idx_host, np.int32)
      n = cand_idx_host.size
      c_ptr = cand_idx_host.ctypes.data_as(C.c_void_p)
    else:
      n = int(bank.shape[0] if n_cand is None else n_cand)
      c_ptr = C.c_void_p(0)
    ov = out_overlap if out_overlap is not None else np.empty((n,), np.float32)
    yw = out_yaw if out_yaw is not None else np.empty((n,), np.int32)
    def hp(a):
      if a is None: return C.c_void_p(0)
      return C.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a.ctypes.data_as(C.c_void_p)
    check(self._h, lib().ovn_query_cloud_vs_bank_host(self._h, p_ptr, npts, _ptr(bank), int(bank.shape[0]), c_ptr,
                                                     n, hp(ov), hp(yw), hp(out_query_fv)),
          'ovn_query_cloud_vs_bank_host')
    return ov, yw
