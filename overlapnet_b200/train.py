"""Training of the overlap head on a frozen leg: the script body of the reference's
``src/two_heads/training.py`` for ``legsType: 360OutputkLegsFixed`` (generateNet.py:222-324), where
every leg layer is frozen and only c_conv1..3 and overlap_output are fitted.

Because the leg is frozen, every distinct (sequence, scan) of the train and validation pairs is
encoded once into a GPU-resident feature bank; a training step then only needs pair indices into
that bank.  Losses, gradients and the Adagrad update run in CUDA behind the C ABI
(``ovn_heads_backward`` / ``ovn_adagrad_step``, csrc/train.cu).  With precision 'f16_tc' the leg and the
validation heads run on tensor cores and dW1, the dominant gradient, on the tcgen05 kernel
``k_delta_wgrad_tc``; precision 'fp32' is the all-SIMT reference.

Not reproduced: full-network training (leg gradients), ``rotate_training_data`` (a column roll of
the 900-wide input is not a roll of the 360-wide feature volume), HDF5 weights and tensorboard logs.

Usage: ``python -m overlapnet_b200.train network.yml``
"""
import logging
import os
import sys

import numpy as np
import torch

from . import weights as _weights
from .evaluate import error_statistics, load_overlap_npz

logger = logging.getLogger('overlapnet_b200.train')

FROZEN_LEG = '360OutputkLegsFixed'


def check_training_config(config):
  """Reject what this trainer cannot fit, naming what is missing."""
  legs = config['model'].get('legsType')
  if legs != FROZEN_LEG:
    raise Exception("legsType '%s' trains the leg, which needs leg gradients; this trainer fits only the "
                    "overlap head on a frozen leg (legsType: %s)" % (legs, FROZEN_LEG))
  if int(config.get('rotate_training_data', 0)) > 0:
    raise Exception('rotate_training_data > 0 rolls the 900-wide input image; that is not a roll of the '
                    '360-wide feature volume, so it cannot be applied to the frozen-leg feature bank')


def lr_schedule(epoch, initial_lr, alpha=0.99):
  """learning_rate_schedule (training.py:47-57)."""
  return initial_lr * 0.1 if epoch < 1 else initial_lr * np.power(alpha, epoch - 1.0)


def truncate_train(n, batch_size, no_batches_in_epoch):
  """training.py:275-286: (pairs used, batches per epoch).  When the set is larger than
  batch_size * no_batches_in_epoch it is cut to that; otherwise every pair is used and Keras runs
  ceil(n / batch_size) batches, the last one short (ImagePairOverlapOrientationSequence.py:82-85)."""
  if batch_size * no_batches_in_epoch < n:
    n = batch_size * no_batches_in_epoch
  return n, int(np.ceil(n / float(batch_size)))


def bank_rows(dir1, imgf1, dir2, imgf2):
  """One bank row per distinct (sequence, scan) -- several sequences can share scan ids.
  Returns (sorted list of (seq, scan) keys, left rows (n,), right rows (n,))."""
  keys = sorted(set(zip(dir1, imgf1)) | set(zip(dir2, imgf2)))
  pos = {k: i for i, k in enumerate(keys)}
  left = np.array([pos[k] for k in zip(dir1, imgf1)], np.int64)
  right = np.array([pos[k] for k in zip(dir2, imgf2)], np.int64)
  return keys, left, right


def data_files(config):
  """training.py:119-134: per-sequence ground truth, else the two single npz files."""
  root = config.get('data_root_folder', '')
  if 'training_seqs' in config:
    seqs = config['training_seqs'].split()
    return ([os.path.join(root, s, 'ground_truth/train_set.npz') for s in seqs],
            [os.path.join(root, s, 'ground_truth/validation_set.npz') for s in seqs])
  return [config['traindata_npzfile']], [config['validationdata_npzfile']]


class Trainer:
  """Fits the overlap head for the YAML dict of training.py.  ``seed`` drives the Glorot init (when
  no pretrained weights are given), the shuffle of the training pairs and the batch order."""

  def __init__(self, config, precision='f16_tc', device=None, seed=0):
    from .infer import Infer
    check_training_config(config)
    self.config = config
    self.rng = np.random.default_rng(seed)
    self.batch_size = int(config['batch_size'])
    self.initial_lr = float(config['learning_rate'])
    self.lr_alpha = float(config.get('lr_alpha', 0.99))
    self.min_overlap_for_angle = float(config.get('min_overlap_for_angle', 0.7))

    train_files, val_files = data_files(config)
    t1, t2, td1, td2, tov, tor = load_overlap_npz(train_files, shuffle=False)
    perm = self.rng.permutation(len(t1))                 # the training pairs are shuffled, validation not
    t1, t2, td1, td2 = [np.asarray(a)[perm] for a in (t1, t2, td1, td2)]
    tov, tor = tov[perm], tor[perm]
    n, self.no_batches = truncate_train(len(t1), self.batch_size, int(config['no_batches_in_epoch']))
    t1, t2, td1, td2, tov, tor = t1[:n], t2[:n], td1[:n], td2[:n], tov[:n], tor[:n]
    v1, v2, vd1, vd2, vov, vor = load_overlap_npz(val_files, shuffle=False)
    nt = min(int(config.get('no_test_pairs', len(v1))), len(v1))
    v1, v2, vd1, vd2, vov, vor = [np.asarray(a)[:nt] for a in (v1, v2, vd1, vd2, vov, vor)]
    self.n_train, self.n_val = n, nt

    keys, left, right = bank_rows(list(td1) + list(vd1), list(t1) + list(v1), list(td2) + list(vd2),
                                  list(t2) + list(v2))
    self.train_left, self.val_left = left[:n], left[n:]
    self.train_right, self.val_right = right[:n], right[n:]
    self.train_overlap, self.train_bin = tov.astype(np.float32), tor.astype(np.int32)
    self.val_overlap, self.val_orientation = vov, vor

    cfg = dict(config)
    for key, default in (('use_depth', True), ('use_normals', True), ('use_class_probabilities', False),
                         ('use_class_probabilities_pca', False), ('use_intensity', False)):
      cfg.setdefault(key, default)                       # training.py:137-160 defaults
    cfg['data_root_folder'] = config.get('imgpath', config.get('data_root_folder', ''))
    cfg['infer_seqs'] = ''
    cfg['model'] = dict(config['model'])
    cfg['model']['inputShape'] = list(config['model']['inputShape'])
    self.infer = Infer(cfg, precision=precision, device=device, max_batch_pairs=max(self.batch_size, 1))
    self.engine = self.infer._engine
    if len(config.get('pretrained_weightsfilename', '')) == 0:
      self.engine.load_weights(_weights.glorot_init(self.infer.no_input_channels, cfg['model'], seed=seed,
                                                    H=self.infer.inputShape[0], W=self.infer.inputShape[1]))
    self.bank = self._encode(keys)

  def _encode(self, keys):
    """Feature volumes of the (seq, scan) keys, in key order, through the frozen leg."""
    out = torch.empty((len(keys), self.engine.Wf, 128), dtype=torch.float32, device=self.engine.device)
    by_seq = {}
    for i, (seq, scan) in enumerate(keys):
      by_seq.setdefault(seq, []).append((i, scan))
    for seq, items in by_seq.items():
      self.infer.seq = seq
      rows = torch.tensor([i for i, _ in items], dtype=torch.int64, device=self.engine.device)
      out[rows] = self.infer._create_feature_volumes_device([s for _, s in items])
    logger.info('  Number of feature volumes: %d', len(keys))
    return out

  def step(self, idx, lr):
    """One batch (positions ``idx`` of the training set): backward + Adagrad.  Returns the losses
    (total, overlap, orientation) as float32 numpy."""
    e = self.engine
    losses = e.heads_backward(self.bank, torch.from_numpy(self.train_left[idx]),
                              torch.from_numpy(self.train_right[idx]), torch.from_numpy(self.train_overlap[idx]),
                              torch.from_numpy(self.train_bin[idx]), self.min_overlap_for_angle)
    e.adagrad_step(lr)
    out = losses.cpu().numpy()
    e.check()
    return out

  def train_epoch(self, epoch):
    """One Keras epoch: batches in a seeded random order; returns the batch-size-weighted mean loss
    and the per-batch (total, overlap, orientation) losses."""
    lr = lr_schedule(epoch, self.initial_lr, self.lr_alpha)
    total, hist = 0.0, []
    for b in self.rng.permutation(self.no_batches):
      idx = np.arange(b * self.batch_size, min(self.n_train, (b + 1) * self.batch_size))
      l = self.step(idx, lr)
      hist.append(l)
      total += float(l[0]) * len(idx)
    return total / self.n_train, np.array(hist), lr

  def validate(self):
    """Overlaps of the validation pairs with the current weights and their error statistics
    (training.py:365-374)."""
    e = self.engine
    e.finalize_weights()
    ov, yaw, _ = e.heads(self.bank, torch.from_numpy(self.val_left), torch.from_numpy(self.val_right))
    e.check()
    ov = ov.cpu().numpy()
    argmax = e.Wf // 2 - yaw.cpu().numpy().astype(np.int64)
    return ov, error_statistics(ov, argmax, self.val_overlap, self.val_orientation, e.Wf)

  def weights(self):
    return self.engine.get_weights()


def weights_path(config):
  """<experiments_path>/<testname>/<modelType>_<testname>.npz (training.py:207-209 with .npz)."""
  return os.path.join(config['experiments_path'], config['testname'],
                      config['model']['modelType'] + '_' + config['testname'] + '.npz')


def run_training(config, precision='f16_tc', device=None, seed=0):
  """The body of training.py for a loaded YAML dict.  Returns (trainer, history) with one dict per
  epoch: loss, learning rate and the validation statistics."""
  out_dir = os.path.join(config['experiments_path'], config['testname'])
  os.makedirs(out_dir, exist_ok=True)
  fh = logging.FileHandler(os.path.join(out_dir, 'training.log'), mode='w')
  fh.setFormatter(logging.Formatter(fmt='%(asctime)s %(message)s', datefmt='%H:%M:%S'))
  logger.addHandler(fh)
  logger.setLevel(logging.INFO)                           # training.py:103-105 logs at DEBUG level
  try:
    tr = Trainer(config, precision=precision, device=device, seed=seed)
    wpath = weights_path(config)
    logger.info('compiled model with learning_rate=%f, lr_alpha=%f, momentum=%f', tr.initial_lr, tr.lr_alpha,
                float(config.get('momentum', 0.0)))        # momentum is logged, unused (Adagrad)
    logger.info('Training loop, saving weights to %s', wpath)
    logger.info('  batch size is           : %d', tr.batch_size)
    logger.info('  number of training pairs: %d', tr.n_train)
    logger.info('  number of test pairs    : %d', tr.n_val)
    logger.info('  NO rotation of training data')
    history = []
    for epoch in range(int(config['no_epochs'])):
      loss, _, lr = tr.train_epoch(epoch)
      logger.info('Epoch %d: loss %f, learning rate %f', epoch, loss, lr)
      logger.info('                  saving model weights ...')
      _weights.save_npz(wpath, tr.weights())
      logger.info('  Evaluation on test data ...')
      _, stats = tr.validate()
      logger.info('  Evaluation on test data results: ')
      logger.info('           Evaluation: mean overlap difference:   %f', stats['overlap_mean'])
      logger.info('           Evaluation: max  overlap difference:   %f', stats['overlap_max'])
      logger.info('           Evaluation: RMS  overlap error        : %f', stats['overlap_rms'])
      history.append(dict(epoch=epoch, loss=loss, lr=lr, **stats))
    return tr, history
  finally:
    logger.removeHandler(fh)
    fh.close()


def main(argv):
  from .config import load_config
  logging.basicConfig(format='%(message)s', level=logging.INFO)
  path = argv[1] if len(argv) > 1 else 'network.yml'
  config = load_config(path)
  logger.info('Using configuration file %s.', path)
  run_training(config)


if __name__ == '__main__':
  main(sys.argv)
