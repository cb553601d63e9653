"""Overlap-head training through the C ABI on the GPU (csrc/train.cu) against the float64 oracle
(oracle/train_ref.py): losses, gradients of all four head layers, Adagrad, stale-pack refusal,
capacity, a teacher-student learning run and run_training end to end."""
import os

import numpy as np
import pytest
import torch

from oracle import network as onet
from oracle import train_ref as T
from overlapnet_b200 import weights as W
from overlapnet_b200._cabi import OvnError
from overlapnet_b200.engine import Engine

pytestmark = pytest.mark.gpu

MODEL = {'additional_unsymmetric_layer3a': True, 'strides_layer1': [2, 2]}
N_BANK, N_PAIRS = 8, 12
LR_LEARN = 1e-5


def rel_fro(a, b):
  return float(np.linalg.norm(np.asarray(a, np.float64) - b) / max(np.linalg.norm(b), 1e-30))


def make_bank(seed, n=N_BANK):
  rng = np.random.default_rng(seed)
  return rng.uniform(0, 1, (n, 360, 128)).astype(np.float32)       # leg outputs are ReLU >= 0


def spread_weights(seed, bank, left, right):
  w = onet.glorot_weights(4, MODEL, seed=seed)
  _, _, _, z = onet.heads_forward(bank[left][:, None], bank[right][:, None], w, MODEL, return_logit=True)
  return onet.spread_dense(w, z, target_std=1.5)


@pytest.fixture(scope='module')
def case():
  rng = np.random.default_rng(11)
  bank = make_bank(0)
  left = rng.integers(0, N_BANK, N_PAIRS)
  right = rng.integers(0, N_BANK, N_PAIRS)
  w = spread_weights(1, bank, left, right)
  y = np.linspace(0.02, 0.98, N_PAIRS)
  rng.shuffle(y)
  y[:3] = [0.95, 0.7, 0.71]                                         # positives and the 0.7 threshold
  bins = rng.integers(0, 360, N_PAIRS)
  losses, grads, yh = T.head_gradients(bank[left][:, None], bank[right][:, None], w, y, bins, MODEL)
  return dict(bank=bank, left=left, right=right, w=w, y=y.astype(np.float32), bins=bins, losses=losses,
              grads=grads, yh=yh)


def engine(w, precision='fp32', max_batch_pairs=16):
  e = Engine(model=MODEL, precision=precision, max_batch_scans=4, max_batch_pairs=max_batch_pairs)
  e.load_weights(w)
  return e


def backward(e, c, n=None):
  n = N_PAIRS if n is None else n
  bank = torch.from_numpy(c['bank']).cuda()
  out = e.heads_backward(bank, torch.from_numpy(c['left'][:n]), torch.from_numpy(c['right'][:n]),
                         torch.from_numpy(c['y'][:n]), torch.from_numpy(c['bins'][:n]))
  return out.cpu().numpy()


# gradient gates (relative Frobenius error per layer and part).  fp32: measured on a B200 2.0-4.4e-5, the
# same for every layer -- the fp32 forward's error in dL/dz, which every gradient is a multiple of.
# f16_tc: dW1 from fp16 operands on tensor cores (measured 3.6e-4), the rest as fp32.
@pytest.mark.parametrize('prec,grad_tol', [('fp32', 1e-4), ('f16_tc', 2e-3)])
def test_losses_and_gradients_match_float64_autograd(case, prec, grad_tol):
  e = engine(case['w'], prec)
  losses = backward(e, case)
  e.check()
  rel_l = np.abs(losses - np.array(case['losses'])) / np.abs(case['losses'])
  g = e.gradients()
  errs = {}
  for name in T.HEAD_LAYERS:
    for part, tag in ((0, 'kernel'), (1, 'bias')):
      errs[name + '/' + tag] = rel_fro(g[name][part], case['grads'][name][part])
  print(prec, 'loss rel err', rel_l.tolist(), 'gradient rel Frobenius err', errs)
  assert rel_l.max() <= 1e-5, rel_l                    # the forward is fp32 in both precisions
  assert max(errs.values()) <= grad_tol, errs
  # bit-identical on a second call
  backward(e, case)
  g2 = e.gradients()
  for name in T.HEAD_LAYERS:
    for part in (0, 1):
      assert np.array_equal(g[name][part].view(np.uint32), g2[name][part].view(np.uint32)), name
  e.close()


def test_adagrad_step_matches_keras_and_set_weights_resets(case):
  e = engine(case['w'])
  backward(e, case)
  g = e.gradients()
  lr = 1e-3
  e.adagrad_step(lr)
  w1 = e.get_weights()
  for name in T.HEAD_LAYERS:
    for part in (0, 1):
      ref, _ = T.adagrad(case['w'][name][part], g[name][part], np.zeros_like(g[name][part]), lr)
      assert rel_fro(w1[name][part], ref) <= 1e-6, name
  for name in ('s_conv1', 's_conv10'):                              # the leg is frozen
    assert np.array_equal(w1[name][0], case['w'][name][0])
  # a second step uses the accumulated squares
  backward(e, case)
  g2 = e.gradients()
  e.adagrad_step(lr)
  w2 = e.get_weights()
  k1, a1 = T.adagrad(case['w']['c_conv2'][0], g['c_conv2'][0], np.zeros_like(g['c_conv2'][0]), lr)
  k2, _ = T.adagrad(k1, g2['c_conv2'][0], a1, lr)
  assert rel_fro(w2['c_conv2'][0], k2) <= 1e-6
  # ovn_set_weights resets the accumulators: the first step from the original weights repeats exactly
  e.load_weights(case['w'])
  backward(e, case)
  e.adagrad_step(lr)
  w3 = e.get_weights()
  for name in T.HEAD_LAYERS:
    assert np.array_equal(w3[name][0], w1[name][0]) and np.array_equal(w3[name][1], w1[name][1]), name
  e.close()


def test_inference_refuses_stale_packs_until_finalized(case):
  e = engine(case['w'])
  bank = torch.from_numpy(case['bank']).cuda()
  li, ri = torch.from_numpy(case['left']), torch.from_numpy(case['right'])
  for _ in range(3):                                                # a small rate keeps the overlaps spread
    backward(e, case)
    e.adagrad_step(LR_LEARN)
  with pytest.raises(OvnError, match='weights changed by training'):
    e.heads(bank, li, ri)
  e.finalize_weights()
  trained = e.get_weights()
  ov_ref, _, _ = onet.heads_forward(case['bank'][case['left']][:, None], case['bank'][case['right']][:, None],
                                    trained, MODEL)
  ov, _, _ = e.heads(bank, li, ri)
  e.check()
  d = {'fp32': float(np.abs(ov.cpu().numpy() - ov_ref).max())}
  tc = engine(trained, 'f16_tc')
  ov16, _, _ = tc.heads(bank, li, ri)
  tc.check()
  d['f16_tc'] = float(np.abs(ov16.cpu().numpy() - ov_ref).max())
  print('forward on trained weights, max |overlap - oracle|', d, 'overlaps', np.round(ov_ref, 3).tolist())
  assert max(d.values()) <= 1e-3, d
  tc.close()
  e.close()


def test_capacity_and_index_checks(case):
  e = engine(case['w'], max_batch_pairs=8)
  with pytest.raises(OvnError, match='OVN_ERR_CAPACITY'):
    backward(e, case)
  c = dict(case)
  c['bins'] = case['bins'].copy()
  c['bins'][0] = 360
  losses = backward(e, c, n=8)
  with pytest.raises(OvnError, match='yaw-bin'):
    e.check()
  assert np.isnan(losses).all()
  e.close()


def learning_curve(case, prec):
  bank = case['bank']
  rng = np.random.default_rng(5)
  n = 16
  left, right = rng.integers(0, N_BANK, n), rng.integers(0, N_BANK, n)
  teacher = spread_weights(2, bank, left, right)
  y_t, _, _ = onet.heads_forward(bank[left][:, None], bank[right][:, None], teacher, MODEL)
  student = spread_weights(3, bank, left, right)
  e = engine(student, prec)
  tb = torch.from_numpy(bank).cuda()
  bins = torch.zeros(n, dtype=torch.int32)
  epoch_means = []
  for epoch in range(5):                                            # 5 epochs x 8 steps = 40 Adagrad steps
    ls = []
    for _ in range(4):
      for b in range(2):
        sl = slice(8 * b, 8 * b + 8)
        l = e.heads_backward(tb, torch.from_numpy(left[sl]), torch.from_numpy(right[sl]),
                             torch.from_numpy(y_t[sl]), bins[sl])
        e.adagrad_step(LR_LEARN)
        ls.append(l)
    epoch_means.append(float(torch.stack(ls)[:, 1].mean()))
  e.check()
  e.close()
  return np.array(epoch_means)


def test_student_learns_teacher_overlaps(case):
  """Targets from a teacher head with another seed; Adagrad on the student lowers the overlap loss, and
  the f16_tc curve tracks the fp32 one."""
  c32, c16 = learning_curve(case, 'fp32'), learning_curve(case, 'f16_tc')
  print('overlap-loss epoch means fp32', c32.tolist(), 'f16_tc', c16.tolist())   # B200 fp32: 0.308 0.251 0.203 0.135 0.130
  for c in (c32, c16):
    assert np.all(np.diff(c) < 0), c
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
  np.savez_compressed(path, overlaps=t, seq=sq)                      # demo4_gen_gt_files.py:111


def test_run_training_end_to_end(tmp_path):
  from overlapnet_b200.evaluate import evaluate_pairs
  from overlapnet_b200.infer import Infer
  from overlapnet_b200.train import run_training, weights_path
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
            'learning_rate': 1e-3, 'momentum': 0.5,
            'model': {'modelType': 'SiameseNetworkTemplate', 'legsType': '360OutputkLegsFixed',
                      'overlap_head': 'DeltaLayerConv1NetworkHead', 'orientation_head': 'CorrelationHead',
                      'inputShape': [64, 900], 'leg_output_width': 360, 'strides_layer1': [2, 2],
                      'additional_unsymmetric_layer3a': True}}
  tr, hist = run_training(config, precision='fp32')
  assert [h['epoch'] for h in hist] == [0, 1] and tr.no_batches == 3
  assert hist[0]['lr'] == pytest.approx(1e-4) and hist[1]['lr'] == pytest.approx(1e-3)
  log = open(os.path.join(str(tmp_path / 'exp'), 't', 'training.log')).read()
  assert 'Evaluation: mean overlap difference' in log
  wp = weights_path(config)
  assert os.path.exists(wp)
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
  # the default precision (f16_tc: tensor-core leg, heads and dW1) runs the same flow
  tr16, hist16 = run_training(dict(config, testname='t16', no_epochs=1))
  assert np.isfinite(hist16[0]['loss']) and os.path.exists(weights_path(dict(config, testname='t16')))
  saved, init = W.load_npz(wp), W.glorot_init(4, config['model'], seed=0)
  assert np.array_equal(saved['s_conv1'][0], init['s_conv1'][0])     # frozen leg
  assert not np.array_equal(saved['c_conv1'][0], init['c_conv1'][0])
