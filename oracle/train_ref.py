"""CPU oracle of overlap-head training on a frozen leg (TEST INFRASTRUCTURE, see oracle/__init__.py).

Restates, from the reference's ``src/two_heads/training.py``:
  ``overlap_loss``       my_sigmoid_loss (:71-83)
  ``orientation_loss``   my_entropy (:86-92) = tf.nn.weighted_cross_entropy_with_logits, pos_weight 360
  ``lr_schedule``        learning_rate_schedule (:47-57)
  ``adagrad``            keras.optimizers.Adagrad of Keras 2.1.5 (:253)
and gets the head gradients by torch.autograd through the overlap head of ``oracle.network``
(same ``delta_layer``, same layer table) with the weights as float64 leaf tensors.
"""
import numpy as np
import torch
import torch.nn.functional as F

from . import network as onet

HEAD_LAYERS = ('c_conv1', 'c_conv2', 'c_conv3', 'overlap_output')


def overlap_loss(yhat, y):
  """my_sigmoid_loss (training.py:71-83): mean sigmoid((|yhat - y| + 0.25) * 24 - 12)."""
  if isinstance(yhat, torch.Tensor):
    y = torch.as_tensor(np.asarray(y), dtype=yhat.dtype)
    return torch.mean(1.0 / (1.0 + torch.exp(-((torch.abs(yhat - y) + 0.25) * 24 - 12))))
  d = np.abs(np.asarray(yhat, np.float64) - np.asarray(y, np.float64))
  return float(np.mean(1.0 / (1.0 + np.exp(-((d + 0.25) * 24 - 12)))))


def orientation_target(yaw_bin, overlap, n_bins=360, min_overlap_for_angle=0.7):
  """ImagePairOverlapOrientationSequence.py:118-121 (t[b] = overlap) thresholded like my_entropy."""
  t = np.zeros((len(yaw_bin), n_bins))
  t[np.arange(len(yaw_bin)), np.asarray(yaw_bin, np.int64)] = overlap
  return (t > min_overlap_for_angle).astype(np.float64)


def orientation_loss(corr, yaw_bin, overlap, min_overlap_for_angle=0.7):
  """my_entropy (training.py:86-92): TF's stable weighted sigmoid cross entropy with pos_weight =
  the number of bins, (1 - t) x + (1 + (q - 1) t) (log1p(exp(-|x|)) + max(-x, 0)), averaged over the
  bins and then over the batch (Keras' _weighted_masked_objective)."""
  x = np.asarray(corr, np.float64)
  q = x.shape[1]
  t = orientation_target(yaw_bin, overlap, q, min_overlap_for_angle)
  l = (1 - t) * x + (1 + (q - 1) * t) * (np.log1p(np.exp(-np.abs(x))) + np.maximum(-x, 0))
  return float(np.mean(np.mean(l, axis=1)))


def lr_schedule(epoch, initial_lr, alpha=0.99):
  """learning_rate_schedule (training.py:47-57)."""
  return initial_lr * 0.1 if epoch < 1 else initial_lr * np.power(alpha, epoch - 1.0)


def adagrad(w, g, a, lr, eps=1e-7):
  """Keras 2.1.5 Adagrad in float32: a += g^2; w -= lr * g / (sqrt(a) + eps).  Returns (w, a)."""
  w = np.asarray(w, np.float32)
  g = np.asarray(g, np.float32)
  a = np.asarray(a, np.float32) + g * g
  return (w - np.float32(lr) * g / (np.sqrt(a) + np.float32(eps))).astype(np.float32), a.astype(np.float32)


def head_overlap(l_fv, r_fv, params, model_cfg=None):
  """The overlap head of oracle.network.delta_head with torch weights (differentiable):
  l_fv, r_fv (B, 1, W, 128) float64 tensors, params {layer: (kernel HWIO, bias)} -> overlap (B,)."""
  x = onet.delta_layer(l_fv, r_fv).permute(0, 3, 1, 2)
  for name, _, stride, _, act in onet.head_layers(model_cfg):
    k, b = params[name]
    x = F.conv2d(x, k.permute(3, 2, 0, 1), b, stride=stride)
    if act == 'relu':
      x = torch.relu(x)
  flat = x.permute(0, 2, 3, 1).reshape(x.shape[0], -1)
  kd, bd = params['overlap_output']
  return torch.sigmoid(flat @ kd + bd)[:, 0]


def head_gradients(l_fv, r_fv, weights, overlap, yaw_bin, model_cfg=None, min_overlap_for_angle=0.7, chunk=2):
  """float64 losses and gradients of 5 L_ov + L_or for pairs (LEFT l_fv[p], RIGHT r_fv[p]).
  Returns ((total, L_ov, L_or), {layer: (dkernel, dbias)} float64, overlaps (n,))."""
  n = l_fv.shape[0]
  params = {k: (torch.tensor(np.asarray(weights[k][0], np.float64), requires_grad=True),
                torch.tensor(np.asarray(weights[k][1], np.float64), requires_grad=True)) for k in HEAD_LAYERS}
  y = np.asarray(overlap, np.float64)
  yh = []
  for s in range(0, n, chunk):
    l = torch.as_tensor(np.asarray(l_fv[s:s + chunk]), dtype=torch.float64)
    r = torch.as_tensor(np.asarray(r_fv[s:s + chunk]), dtype=torch.float64)
    o = head_overlap(l, r, params, model_cfg)
    # L_ov is a mean over the whole batch: each chunk contributes its share of 5 * L_ov
    part = overlap_loss(o, y[s:s + chunk]) * (5.0 * o.shape[0] / n)
    part.backward()
    yh.append(o.detach().numpy())
  yh = np.concatenate(yh)
  corr = onet.correlation_head(l_fv, r_fv)
  lov = overlap_loss(yh, y)
  lor = orientation_loss(corr, yaw_bin, y, min_overlap_for_angle)
  grads = {k: (params[k][0].grad.numpy(), params[k][1].grad.numpy()) for k in HEAD_LAYERS}
  return (5.0 * lov + lor, lov, lor), grads, yh
