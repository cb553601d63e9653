"""Host side of overlap-head training (training.py): the oracle's autograd gradients against finite
differences, the two losses on hand-computed cases, the LR schedule, batch truncation, the
(seq, scan) bank mapping and the rejected configurations."""
import math

import numpy as np
import pytest
import torch

from oracle import network as onet
from oracle import train_ref as T
from overlapnet_b200 import train as TR

SMALL = {'conv1NetworkHead_conv1size': 5}          # 25-wide volumes: o1 25x5, o2 5x5, o3 3x3


def _small_case(seed=0, n=2, width=25):
  rng = np.random.default_rng(seed)
  w = onet.glorot_weights(4, SMALL, seed=seed, leg_out_width=width)
  head = {k: w[k] for k in T.HEAD_LAYERS}
  l = rng.uniform(0, 1, (n, 1, width, 128))
  r = rng.uniform(0, 1, (n, 1, width, 128))
  y = rng.uniform(0, 1, n)
  return head, l, r, y


def test_differentiable_head_matches_oracle_forward():
  head, l, r, _ = _small_case()
  params = {k: (torch.tensor(head[k][0], dtype=torch.float64), torch.tensor(head[k][1], dtype=torch.float64))
            for k in T.HEAD_LAYERS}
  got = T.head_overlap(torch.tensor(l), torch.tensor(r), params, SMALL).numpy()
  _, z, _ = onet.delta_head(l, r, head, SMALL, return_all=True)
  assert np.allclose(got, 1 / (1 + np.exp(-z[:, 0])), rtol=0, atol=1e-12)


def test_autograd_gradients_match_finite_differences():
  head, l, r, y = _small_case(seed=1)
  # a larger Dense scale spreads the overlaps so that every layer has a sizeable gradient
  head['overlap_output'] = (head['overlap_output'][0] * 20, head['overlap_output'][1])
  _, grads, _ = T.head_gradients(l, r, head, y, np.zeros(len(y), np.int64), SMALL)
  lt, rt = torch.tensor(l), torch.tensor(r)

  def loss(wts):
    params = {k: (torch.tensor(np.asarray(wts[k][0], np.float64)), torch.tensor(np.asarray(wts[k][1], np.float64)))
              for k in T.HEAD_LAYERS}
    return 5.0 * float(T.overlap_loss(T.head_overlap(lt, rt, params, SMALL), y))

  rng = np.random.default_rng(7)
  eps = 1e-6
  for name in T.HEAD_LAYERS:
    for part in (0, 1):
      arr = np.asarray(head[name][part], np.float64)
      g = grads[name][part]
      assert g.shape == arr.shape
      flat_idx = rng.choice(arr.size, size=min(4, arr.size), replace=False)
      for fi in flat_idx:
        idx = np.unravel_index(fi, arr.shape)
        plus, minus = arr.copy(), arr.copy()
        plus[idx] += eps
        minus[idx] -= eps
        wp = dict(head); wm = dict(head)
        wp[name] = (plus, head[name][1]) if part == 0 else (head[name][0], plus)
        wm[name] = (minus, head[name][1]) if part == 0 else (head[name][0], minus)
        fd = (loss(wp) - loss(wm)) / (2 * eps)
        scale = max(np.abs(g).max(), 1e-12)
        assert abs(fd - g[idx]) <= 1e-6 * scale + 1e-9, (name, part, idx, fd, g[idx])


def test_overlap_loss_hand_cases():
  sig = lambda x: 1 / (1 + math.exp(-x))
  assert T.overlap_loss([0.3], [0.3]) == pytest.approx(sig(-6.0), rel=1e-15)
  assert T.overlap_loss([1.0, 0.0], [0.0, 0.5]) == pytest.approx((sig(18.0) + sig(6.0)) / 2, rel=1e-15)
  # at yhat = y the gradient of |.| is 0, as in TF
  yh = torch.tensor([0.4, 0.9], dtype=torch.float64, requires_grad=True)
  T.overlap_loss(yh, [0.4, 0.1]).backward()
  assert yh.grad[0].item() == 0.0 and yh.grad[1].item() > 0


def test_orientation_loss_hand_cases_and_threshold():
  x = np.zeros((2, 360))
  ln2 = math.log(2.0)
  # no positive bin (overlap 0.7 is not > 0.7): every bin costs log 2
  assert T.orientation_loss(x, [5, 9], [0.7, 0.2]) == pytest.approx(ln2, rel=1e-14)
  # a positive bin costs (1 + 359) log 2 at x = 0
  assert T.orientation_loss(x[:1], [5], [0.71]) == pytest.approx((359 * ln2 + 360 * ln2) / 360, rel=1e-14)
  assert T.orientation_loss(x[:1], [5], [0.71], min_overlap_for_angle=0.8) == pytest.approx(ln2, rel=1e-14)
  # the stable form equals q t (-log s(x)) + (1 - t)(-log(1 - s(x)))
  rng = np.random.default_rng(3)
  xs = rng.normal(0, 4, (3, 360))
  bins, ov = [0, 100, 359], [0.9, 0.5, 0.75]
  t = T.orientation_target(bins, ov)
  s = 1 / (1 + np.exp(-xs))
  naive = np.mean(360 * t * -np.log(s) + (1 - t) * -np.log(1 - s))
  assert T.orientation_loss(xs, bins, ov) == pytest.approx(naive, rel=1e-12)


def test_lr_schedule_and_adagrad():
  for sched in (T.lr_schedule, TR.lr_schedule):
    assert sched(0, 1e-3) == pytest.approx(1e-4)
    assert sched(1, 1e-3) == pytest.approx(1e-3)
    assert sched(3, 1e-3) == pytest.approx(1e-3 * 0.99 ** 2)
    assert sched(3, 1e-3, alpha=0.5) == pytest.approx(1e-3 * 0.25)
  w, a = T.adagrad(np.float32([1.0]), np.float32([2.0]), np.float32([0.0]), 0.1)
  assert a[0] == 4.0 and w[0] == np.float32(1.0) - np.float32(0.1) * np.float32(2.0) / (np.float32(2.0) + np.float32(1e-7))
  w2, a2 = T.adagrad(w, np.float32([2.0]), a, 0.1)          # accumulators persist
  assert a2[0] == 8.0 and w2[0] < w[0]


def test_no_batches_in_epoch_truncation():
  assert TR.truncate_train(100, 16, 3) == (48, 3)            # cut to batch_size * no_batches_in_epoch
  assert TR.truncate_train(50, 16, 10) == (50, 4)            # all pairs, last batch short
  assert TR.truncate_train(48, 16, 10 ** 11) == (48, 3)


def test_bank_rows_keep_sequences_apart():
  keys, left, right = TR.bank_rows(['00', '01', '00'], ['000003', '000003', '000001'],
                                   ['01', '00', '00'], ['000001', '000001', '000003'])
  assert keys == [('00', '000001'), ('00', '000003'), ('01', '000001'), ('01', '000003')]
  assert left.tolist() == [1, 3, 0] and right.tolist() == [2, 0, 1]


def _config(**over):
  cfg = {'model': {'legsType': '360OutputkLegsFixed'}, 'rotate_training_data': 0}
  cfg['model'].update(over.pop('model', {}))
  cfg.update(over)
  return cfg


def test_rejected_configs_raise():
  TR.check_training_config(_config())
  with pytest.raises(Exception, match='leg gradients'):
    TR.check_training_config(_config(model={'legsType': '360OutputkLegs'}))
  with pytest.raises(Exception, match='rotate_training_data'):
    TR.check_training_config(_config(rotate_training_data=1))


def test_data_files_follow_training_py(tmp_path):
  tr, va = TR.data_files({'data_root_folder': '/d', 'training_seqs': '00 07'})
  assert tr == ['/d/00/ground_truth/train_set.npz', '/d/07/ground_truth/train_set.npz']
  assert va == ['/d/00/ground_truth/validation_set.npz', '/d/07/ground_truth/validation_set.npz']
  assert TR.data_files({'traindata_npzfile': 'a.npz', 'validationdata_npzfile': 'b.npz'}) == (['a.npz'], ['b.npz'])
  cfg = {'experiments_path': str(tmp_path), 'testname': 't1', 'model': {'modelType': 'M'}}
  assert TR.weights_path(cfg) == str(tmp_path / 't1' / 'M_t1.npz')
