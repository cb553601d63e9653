"""Full-network training through the C ABI on the GPU (ovn_network_backward, csrc/train.cu) against the
float64 oracle (oracle/train_network_ref.network_gradients): losses and the gradients of all 15 layers, reuse of
the head gradients, the RIGHT roll, reproducibility, Adagrad over the leg, stale-pack refusal, errors, a
teacher/student run with a trainable leg and run_training with legsType 360OutputkLegs end to end."""
import os

import numpy as np
import pytest
import torch

from oracle import network as onet
from oracle import train_network_ref as TN
from oracle import train_ref as T
from overlapnet_b200 import weights as W
from overlapnet_b200._cabi import OvnError, lib
from overlapnet_b200.engine import Engine

pytestmark = pytest.mark.gpu

MODEL = {'additional_unsymmetric_layer3a': True, 'strides_layer1': [2, 2]}
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
SCANS = ('kitti_000000', 'kitti_000001', 'synth_3', 'synth_5')
LEFT, RIGHT = np.array([0, 1, 2]), np.array([1, 0, 3])
ROLL = np.array([0, 137, -1250], np.int32)               # -1250 = 550 modulo 900
LAYERS = [n for n, *_ in onet.leg_layers(MODEL)] + list(T.HEAD_LAYERS)


def rel_fro(a, b):
  return float(np.linalg.norm(np.asarray(a, np.float64) - b) / max(np.linalg.norm(b), 1e-30))


def bits_equal(a, b):
  return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def engine(w, precision='fp32', max_batch_pairs=8):
  e = Engine(model=MODEL, precision=precision, max_batch_scans=4, max_batch_pairs=max_batch_pairs)
  e.load_weights(w)
  return e


@pytest.fixture(scope='module')
def case():
  e = Engine(model=MODEL, precision='fp32', max_batch_scans=4, max_batch_pairs=4)
  clouds = [np.load(os.path.join(GOLDEN, s + '.npz'))['points'] for s in SCANS]
  x = e.preprocess(e.upload_clouds(clouds)).cpu().numpy()          # engine preprocessing of the fixtures
  e.close()
  w = onet.glorot_weights(4, MODEL, seed=1)
  fv = onet.leg_forward(x, w, MODEL)
  xr = np.stack([np.roll(x[RIGHT[p]], ROLL[p], axis=1) for p in range(len(LEFT))])
  fr = onet.leg_forward(xr, w, MODEL)
  _, _, _, z = onet.heads_forward(fv[LEFT], fr, w, MODEL, return_logit=True)
  w = onet.spread_dense(w, z, target_std=1.5)
  y = np.array([0.95, 0.3, 0.72], np.float32)                       # two positives for the yaw loss
  bins = np.array([10, 200, 359], np.int32)
  losses, grads, yh = TN.network_gradients(x[LEFT], x[RIGHT], w, y, bins, MODEL, right_roll=ROLL)
  return dict(x=x, w=w, y=y, bins=bins, losses=losses, grads=grads, yh=yh)


def net_backward(e, c, roll=ROLL, n=None, left=LEFT, right=RIGHT, bins=None, x=None):
  n = len(left) if n is None else n
  xs = torch.from_numpy(c['x'] if x is None else x).cuda()
  b = c['bins'] if bins is None else bins
  out = e.network_backward(xs, torch.from_numpy(left[:n]), torch.from_numpy(right[:n]),
                           torch.from_numpy(c['y'][:n]), torch.from_numpy(b[:n]),
                           None if roll is None else torch.from_numpy(roll[:n]))
  return out.cpu().numpy()


# Gates (relative error vs float64; DESIGN §10).  Measured on a B200 at fp32: losses <= 1.9e-5 (L_ov), head
# gradients 7.2e-5, s_conv10 bias 1.5e-5, leg kernels and biases 4.4-9.3e-4.  torch's own fp32 autograd on
# this case gives the same pattern (L_ov 1.3e-5, heads 5e-5, leg 1.5-3.4e-4): the leg weight gradients are
# sums with heavy cancellation of fp32 activations, so they carry ~10x the forward's relative error.
# At f16_tc only dW1 of c_conv1 changes (fp16 operands on tensor cores, 2e-3); every other gradient must
# equal the fp32 handle's bits.
@pytest.fixture(scope='module')
def fp32_grads(case):
  e = engine(case['w'], 'fp32')
  losses = net_backward(e, case)
  e.check()
  g = e.gradients()
  net_backward(e, case)
  g2 = e.gradients()
  e.close()
  return losses, g, g2


def test_network_gradients_match_float64_autograd_fp32(case, fp32_grads):
  losses, g, g2 = fp32_grads
  rel_l = np.abs(losses - np.array(case['losses'])) / np.abs(case['losses'])
  errs = {}
  for name in LAYERS:
    for part, tag in ((0, 'kernel'), (1, 'bias')):
      errs[name + '/' + tag] = rel_fro(g[name][part], case['grads'][name][part])
  print('fp32 loss rel err', rel_l.tolist(), 'losses', list(case['losses']))
  print('fp32 gradient rel Frobenius err', {k: '%.2e' % v for k, v in errs.items()})
  assert set(g) == set(LAYERS)
  assert rel_l.max() <= 5e-5, rel_l
  assert max(v for k, v in errs.items() if not k.startswith('s_')) <= 1e-4, errs
  assert max(errs.values()) <= 2e-3, errs
  for name in LAYERS:                                               # bit-identical on a second call
    for part in (0, 1):
      assert bits_equal(g[name][part], g2[name][part]), name


def test_f16_tc_changes_only_dW1(case, fp32_grads):
  losses32, g32, _ = fp32_grads
  e = engine(case['w'], 'f16_tc')
  losses = net_backward(e, case)
  e.check()
  g = e.gradients()
  net_backward(e, case)
  g2 = e.gradients()
  e.close()
  err = rel_fro(g['c_conv1'][0], case['grads']['c_conv1'][0])
  print('f16_tc c_conv1 kernel rel err %.2e' % err)
  assert err <= 2e-3
  assert bits_equal(losses, losses32)
  for name in LAYERS:
    for part in (0, 1):
      assert bits_equal(g[name][part], g2[name][part]), name
      if (name, part) != ('c_conv1', 0):
        assert bits_equal(g[name][part], g32[name][part]), name


@pytest.mark.parametrize('prec', ['fp32', 'f16_tc'])
def test_head_gradients_equal_heads_backward_and_roll_equals_prerolled(case, prec):
  n = len(LEFT)
  x = case['x']
  xr = np.stack([np.roll(x[RIGHT[p]], ROLL[p], axis=1) for p in range(n)])
  imgs = np.concatenate([x[LEFT], xr])                              # LEFT images, then rolled RIGHT images
  e = engine(case['w'], prec)
  l_net = net_backward(e, case)
  g_net = e.gradients()
  # the same call on inputs rolled beforehand
  l_pre = net_backward(e, case, roll=None, left=np.arange(n), right=np.arange(n, 2 * n), x=imgs)
  g_pre = e.gradients()
  assert bits_equal(l_net, l_pre)
  for name in LAYERS:
    for part in (0, 1):
      assert bits_equal(g_net[name][part], g_pre[name][part]), name
  # heads_backward on a bank made by the fp32 leg from the same 2n images
  e32 = engine(case['w'], 'fp32')
  bank = e32.leg(torch.from_numpy(imgs).cuda())
  e32.close()
  l_h = e.heads_backward(bank, torch.arange(n), torch.arange(n, 2 * n), torch.from_numpy(case['y']),
                         torch.from_numpy(case['bins'])).cpu().numpy()
  g_h = e.gradients()
  e.check()
  assert set(g_h) == set(T.HEAD_LAYERS)
  assert bits_equal(l_net, l_h)
  for name in T.HEAD_LAYERS:
    for part in (0, 1):
      assert bits_equal(g_net[name][part], g_h[name][part]), name
  with pytest.raises(OvnError, match='leg gradients need ovn_network_backward'):
    e._layer_arrays(lib().ovn_get_gradient, 'ovn_get_gradient', ['s_conv1'])
  e.close()


def test_adagrad_all_layers_reset_and_stale_leg(case):
  e = engine(case['w'])
  net_backward(e, case)
  g = e.gradients()
  lr = 1e-5                                                         # a small step keeps the overlaps spread
  e.adagrad_step(lr)
  w1 = e.get_weights()
  for name in LAYERS:
    for part in (0, 1):
      ref, _ = T.adagrad(case['w'][name][part], g[name][part], np.zeros_like(g[name][part]), lr)
      assert rel_fro(w1[name][part], ref) <= 1e-6, name
  # the leg changed: the leg and the heads refuse until finalize
  with pytest.raises(OvnError, match='weights changed by training'):
    e.leg(torch.from_numpy(case['x']).cuda())
  with pytest.raises(OvnError, match='weights changed by training'):
    e.heads(torch.zeros((2, 360, 128), device='cuda'), torch.tensor([0]), torch.tensor([1]))
  # a second step uses the accumulated squares of every layer
  net_backward(e, case)
  g2 = e.gradients()
  e.adagrad_step(lr)
  w2 = e.get_weights()
  for name in LAYERS:
    for part in (0, 1):
      k1, a1 = T.adagrad(case['w'][name][part], g[name][part], np.zeros_like(g[name][part]), lr)
      k2, _ = T.adagrad(k1, g2[name][part], a1, lr)
      assert rel_fro(w2[name][part], k2) <= 1e-6, name
  # ovn_set_weights resets the leg accumulators too: the first step from the original weights repeats
  e.load_weights(case['w'])
  net_backward(e, case)
  e.adagrad_step(lr)
  w3 = e.get_weights()
  for name in LAYERS:
    assert bits_equal(w3[name][0], w1[name][0]) and bits_equal(w3[name][1], w1[name][1]), name
  # finalize: Engine.leg + heads on the trained weights match the float64 oracle
  e.finalize_weights()
  fv = e.leg(torch.from_numpy(case['x']).cuda())
  ov, _, _ = e.heads(fv, torch.from_numpy(LEFT), torch.from_numpy(RIGHT))
  e.check()
  fv_ref = onet.leg_forward(case['x'], w3, MODEL)
  ov_ref, _, _ = onet.heads_forward(fv_ref[LEFT], fv_ref[RIGHT], w3, MODEL)
  d = float(np.abs(ov.cpu().numpy() - ov_ref).max())
  print('forward on trained weights, max |overlap - oracle|', d, 'overlaps', np.round(ov_ref, 3).tolist())
  assert d <= 1e-3
  e.close()


def test_capacity_and_index_checks(case):
  e = engine(case['w'], max_batch_pairs=2)
  with pytest.raises(OvnError, match='OVN_ERR_CAPACITY'):
    net_backward(e, case)
  bad = case['bins'].copy()
  bad[0] = 360
  losses = net_backward(e, case, n=2, bins=bad)
  with pytest.raises(OvnError, match='yaw-bin'):
    e.check()
  assert np.isnan(losses).all()
  losses = net_backward(e, case, n=2, right=np.array([1, 4]))
  with pytest.raises(OvnError, match='outside'):
    e.check()
  assert np.isnan(losses).all()
  e.close()


def learning_curve(case, prec, lr=1e-5, epochs=10):
  x = case['x']
  left = np.array([i for i in range(4) for j in range(4) if i != j])
  right = np.array([j for i in range(4) for j in range(4) if i != j])
  teacher = onet.glorot_weights(4, MODEL, seed=2)
  fv_t = onet.leg_forward(x, teacher, MODEL)
  _, _, _, z = onet.heads_forward(fv_t[left], fv_t[right], teacher, MODEL, return_logit=True)
  teacher = onet.spread_dense(teacher, z, target_std=1.5)
  y_t, _, _ = onet.heads_forward(fv_t[left], fv_t[right], teacher, MODEL)
  student = onet.glorot_weights(4, MODEL, seed=3)
  fv_s = onet.leg_forward(x, student, MODEL)
  _, _, _, zs = onet.heads_forward(fv_s[left], fv_s[right], student, MODEL, return_logit=True)
  student = onet.spread_dense(student, zs, target_std=1.5)
  e = engine(student, prec)
  xs = torch.from_numpy(x).cuda()
  bins = torch.zeros(len(left), dtype=torch.int32)
  means = []
  for _ in range(epochs):
    ls = []
    for b in range(3):
      sl = slice(4 * b, 4 * b + 4)
      l = e.network_backward(xs, torch.from_numpy(left[sl]), torch.from_numpy(right[sl]),
                             torch.from_numpy(y_t[sl].astype(np.float32)), bins[sl])
      e.adagrad_step(lr)
      ls.append(l)
    means.append(float(torch.stack(ls)[:, 1].mean()))
  e.check()
  e.close()
  return np.array(means)


def test_student_with_trainable_leg_learns_teacher_overlaps(case):
  """Targets from a teacher network with another seed; 30 Adagrad steps on every layer of the student lower
  its overlap loss, and the f16_tc curve tracks the fp32 one.  (The yaw loss dominates the leg's gradient
  direction, and Adagrad moves every coordinate by ~lr per step: at lr 2e-4 the student's overlaps collapse
  to 0 within a few steps.)"""
  c32, c16 = learning_curve(case, 'fp32'), learning_curve(case, 'f16_tc')
  print('overlap-loss epoch means fp32', c32.tolist(), 'f16_tc', c16.tolist())
  for c in (c32, c16):
    assert c[-1] < 0.8 * c[0], c
  assert np.abs(c16 - c32).max() <= 0.05 * c32.max(), (c32, c16)


def _write_dataset(root, seq, scans, rng):
  for cue, shape in (('depth', (64, 900)), ('normal', (64, 900, 3))):
    os.makedirs(os.path.join(root, seq, cue), exist_ok=True)
    for s in scans:
      a = rng.uniform(0, 20 if cue == 'depth' else 1, shape).astype(np.float32)
      np.save(os.path.join(root, seq, cue, '%06d.npy' % s), a)


def _write_gt(path, pairs, seq):
  os.makedirs(os.path.dirname(path), exist_ok=True)
  t = np.array(pairs, np.float64)
  sq = np.empty((len(pairs), 2), dtype=object)
  sq[:] = seq
  np.savez_compressed(path, overlaps=t, seq=sq)


def test_run_training_network_end_to_end(tmp_path):
  from overlapnet_b200.evaluate import evaluate_pairs
  from overlapnet_b200.infer import Infer
  from overlapnet_b200.train import NetworkTrainer, run_training, weights_path
  rng = np.random.default_rng(0)
  root = str(tmp_path / 'data')
  _write_dataset(root, '00', range(6), rng)
  train = [[i, j, rng.uniform(), rng.integers(0, 360)] for i in range(6) for j in range(6) if i != j][:10]
  val = [[0, 5, 0.9, 10.0], [2, 3, 0.3, 200.0], [4, 1, 0.75, 359.0]]
  _write_gt(os.path.join(root, '00', 'ground_truth', 'train_set.npz'), train, '00')
  _write_gt(os.path.join(root, '00', 'ground_truth', 'validation_set.npz'), val, '00')
  config = {'experiments_path': str(tmp_path / 'exp'), 'testname': 't', 'pretrained_weightsfilename': '',
            'use_depth': True, 'use_normals': True, 'data_root_folder': root, 'training_seqs': '00',
            'batch_size': 4, 'no_batches_in_epoch': 100, 'no_epochs': 2, 'no_test_pairs': 100,
            'learning_rate': 1e-3, 'momentum': 0.5, 'rotate_training_data': 2,
            'model': {'modelType': 'SiameseNetworkTemplate', 'legsType': '360OutputkLegs',
                      'overlap_head': 'DeltaLayerConv1NetworkHead', 'orientation_head': 'CorrelationHead',
                      'inputShape': [64, 900], 'leg_output_width': 360, 'strides_layer1': [2, 2],
                      'additional_unsymmetric_layer3a': True}}
  tr, hist = run_training(config, precision='fp32')
  assert isinstance(tr, NetworkTrainer) and tr.no_batches == 3 and [h['epoch'] for h in hist] == [0, 1]
  log = open(os.path.join(str(tmp_path / 'exp'), 't', 'training.log')).read()
  assert 'rotation of training data, different sequence for every epoch' in log
  assert 'Evaluation: mean overlap difference' in log
  wp = weights_path(config)
  saved, init = W.load_npz(wp), W.glorot_init(4, config['model'], seed=0)
  assert not np.array_equal(saved['s_conv1'][0], init['s_conv1'][0])     # the leg is trained
  assert not np.array_equal(saved['c_conv1'][0], init['c_conv1'][0])
  ov_trainer, stats = tr.validate()
  assert stats['overlap_mean'] == pytest.approx(hist[-1]['overlap_mean'])
  icfg = dict(config, infer_seqs='00', use_class_probabilities=False, use_class_probabilities_pca=False,
              use_intensity=False, pretrained_weightsfilename=wp)
  icfg['model'] = dict(config['model'], inputShape=[64, 900])
  inf = Infer(icfg, precision='fp32')
  m, _ = evaluate_pairs(inf, ['%06d' % p[0] for p in val], ['%06d' % p[1] for p in val],
                        np.array([p[2] for p in val]), np.array([p[3] for p in val]))
  print('validation overlaps: trainer', ov_trainer.tolist(), 'Infer', m[:, 2].tolist())
  assert np.allclose(m[:, 2], ov_trainer, rtol=0, atol=1e-6)
  # the default precision runs the same flow
  tr16, hist16 = run_training(dict(config, testname='t16', no_epochs=1))
  assert np.isfinite(hist16[0]['loss']) and os.path.exists(weights_path(dict(config, testname='t16')))
