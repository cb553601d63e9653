"""Host side of full-network training: the float64 oracle's autograd gradients through the leg and both
heads against central differences at full size (64 x 900), the RIGHT-roll shift schedule against the
reference's own sequence class (tests/golden/rotation_shifts.npz), and the legsType dispatch."""
import os

import numpy as np
import pytest
import torch

from oracle import network as onet
from oracle import projection as oproj
from oracle import train_network_ref as TN
from oracle import train_ref as T
from overlapnet_b200 import synth
from overlapnet_b200 import train as TR

MODEL = {'additional_unsymmetric_layer3a': True, 'strides_layer1': [2, 2]}
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _inputs(n_scans, seed=0):
  imgs = []
  for s in range(n_scans):
    rng, vert, _, _ = oproj.range_projection(synth.kitti_like_cloud(seed + s, n_points=20000))
    imgs.append(oproj.pack_input(rng, oproj.gen_normal_map(rng, vert)))
  return np.stack(imgs).astype(np.float64)


def _total_loss(x, w, y, bins, roll):
  params = {k: (torch.tensor(np.asarray(v[0], np.float64)), torch.tensor(np.asarray(v[1], np.float64)))
            for k, v in w.items()}
  xl = torch.tensor(x[:1])
  xr = torch.tensor(np.roll(x[1:2], roll, axis=2))
  fl, fr = TN.leg_forward_torch(xl, params, MODEL), TN.leg_forward_torch(xr, params, MODEL)
  o = T.head_overlap(fl, fr, params, MODEL)
  lor = TN.orientation_loss_torch(TN.correlation_head_torch(fl, fr), bins, y)
  return float(5.0 * T.overlap_loss(o, y) + lor)


def test_network_gradients_match_central_differences():
  """One pair at full size with a RIGHT roll; the largest-gradient entries of s_conv1 (kernel), s_conv3a
  (kernel), s_conv10 (bias) and c_conv1 (kernel) against float64 central differences."""
  # Scaled to unit range: the correlation logits (and the loss) stay O(1), so the roundoff of the loss does
  # not swamp small steps, and a step moves few pre-activations across their ReLU kink.
  x = _inputs(2) * 0.05
  w = onet.glorot_weights(4, MODEL, seed=4)
  fv = onet.leg_forward(x, w, MODEL)
  _, _, _, z = onet.heads_forward(fv[:1], onet.leg_forward(np.roll(x[1:2], 300, axis=2), w, MODEL), w, MODEL,
                                  return_logit=True)
  w = onet.spread_dense(w, np.concatenate([z, z + 1.0]), target_std=1.5)
  kd, bd = w['overlap_output']
  w['overlap_output'] = (kd, bd + np.float32(1.5))                 # overlap ~0.68: L_ov is not saturated
  y, bins, roll = np.array([0.75]), np.array([37]), 300          # a positive bin: L_or has a gradient
  losses, grads, _ = TN.network_gradients(x[:1], x[1:2], w, y, bins, MODEL, right_roll=[roll])
  assert losses[0] == pytest.approx(_total_loss(x, w, y, bins, roll), rel=1e-12)
  # A leg weight moves ~1M pre-activations, so its step is smaller than a head weight's: fewer of them cross
  # their ReLU kink within the step.
  for name, part, eps in (('s_conv1', 0, 1e-7), ('s_conv3a', 0, 1e-7), ('s_conv10', 1, 1e-7), ('c_conv1', 0, 1e-6)):
    g = grads[name][part]
    assert g.shape == w[name][part].shape
    for fi in np.argsort(-np.abs(g).ravel())[:2]:
      idx = np.unravel_index(fi, g.shape)
      vals = []
      for sgn in (1, -1):
        arr = np.asarray(w[name][part], np.float64).copy()
        arr[idx] += sgn * eps
        wp = dict(w)
        wp[name] = (arr, w[name][1]) if part == 0 else (w[name][0], arr)
        vals.append(_total_loss(x, wp, y, bins, roll))
      fd = (vals[0] - vals[1]) / (2 * eps)
      assert abs(fd - g[idx]) <= 1e-6 * abs(g[idx]), (name, part, idx, fd, g[idx])


def test_rotation_schedule_matches_reference_sequence():
  gold = np.load(os.path.join(GOLDEN, 'rotation_shifts.npz'))
  n, bs, width = int(gold['n_pairs']), int(gold['batch_size']), int(gold['width'])
  for mode in (1, 2):
    sched = TR.RightRollSchedule(mode, n, width)
    got = []
    for idx in gold['calls_mode%d' % mode]:
      size = min(n, (idx + 1) * bs) - idx * bs
      got.append(sched.batch(int(idx), size))
    got = np.concatenate(got) % width                              # a shift of width is no roll
    assert np.array_equal(got, gold['shifts_mode%d' % mode]), mode
  assert TR.RightRollSchedule(0, n, width).batch(0, bs) is None


def _config(**over):
  cfg = {'model': {'legsType': '360OutputkLegs'}, 'rotate_training_data': 0}
  cfg['model'].update(over.pop('model', {}))
  cfg.update(over)
  return cfg


def test_network_config_checks_and_dispatch(monkeypatch, tmp_path):
  for rot in (0, 1, 2):
    TR.check_network_config(_config(rotate_training_data=rot))
  TR.check_network_config({'model': {'legsType': '360OutputkLegs'}})
  for bad in (3, -1, '1'):
    with pytest.raises(Exception, match='rotate_training_data must be 0'):
      TR.check_network_config(_config(rotate_training_data=bad))
  with pytest.raises(Exception, match='360OutputkLegs'):
    TR.check_network_config(_config(model={'legsType': '360OutputkLegsFixed'}))
  with pytest.raises(Exception, match='leg gradients'):                # the frozen-leg trainer still refuses
    TR.check_training_config(_config())

  made = []

  class Stop(Exception):
    pass

  def fake(kind):
    def init(self, config, precision='f16_tc', device=None, seed=0):
      made.append(kind)
      raise Stop()
    return init

  monkeypatch.setattr(TR.NetworkTrainer, '__init__', fake('network'))
  monkeypatch.setattr(TR.Trainer, '__init__', fake('heads'))
  for legs, kind in (('360OutputkLegs', 'network'), ('360OutputkLegsFixed', 'heads')):
    cfg = {'experiments_path': str(tmp_path), 'testname': 't', 'model': {'legsType': legs}}
    with pytest.raises(Stop):
      TR.run_training(cfg)
    assert made[-1] == kind
  log = {0: 'NO rotation', 1: 'same sequence for every epoch', 2: 'different sequence for every epoch'}
  for mode, text in log.items():
    assert text in TR.RightRollSchedule(mode, 4, 900).log()
