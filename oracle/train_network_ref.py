"""CPU oracle of full-network training (legsType 360OutputkLegs; TEST INFRASTRUCTURE, see oracle/__init__.py).

Differentiable torch forms of the leg (``oracle.network.leg_forward``) and the correlation head
(``oracle.network.correlation_head``), the yaw loss (``oracle.train_ref.orientation_loss``) on torch tensors,
and ``network_gradients``: float64 autograd through the leg, both heads and both losses with all 15 layers
as leaf tensors.  The overlap head is ``oracle.train_ref.head_overlap``; the layer tables are those of
``oracle.network``.
"""
import numpy as np
import torch
import torch.nn.functional as F

from . import network as onet
from . import train_ref as T


def leg_forward_torch(x_nhwc, params, model_cfg=None):
  """``oracle.network.leg_forward`` on torch tensors, differentiable: x (B, H, W, C), params {layer: (kernel
  HWIO, bias)} -> feature volumes (B, 1, W_out, 128) in the dtype of the inputs."""
  x = x_nhwc.permute(0, 3, 1, 2).contiguous()
  for name, _, stride, _ in onet.leg_layers(model_cfg):
    k, b = params[name]
    x = torch.relu(F.conv2d(x, k.permute(3, 2, 0, 1).contiguous(), b, stride=stride))
  return x.permute(0, 2, 3, 1)


def correlation_head_torch(l, r):
  """``oracle.network.correlation_head`` on torch tensors, differentiable: l, r (B, 1, W, 128) -> corr (B, W)
  with corr[b, k] = sum_{j,c} L[b, 0, (k + j + W//2) mod W, c] R[b, 0, j, c]."""
  W = l.shape[2]
  pad = onet.range_padding(l, W // 2)
  return torch.stack([F.conv2d(pad[b:b + 1].permute(0, 3, 1, 2), r[b].permute(2, 0, 1).unsqueeze(0)).reshape(-1)
                      for b in range(l.shape[0])])


def orientation_loss_torch(corr, yaw_bin, overlap, min_overlap_for_angle=0.7):
  """``oracle.train_ref.orientation_loss`` on a torch (B, q) tensor, differentiable; returns the SUM over the
  batch of the per-pair mean over bins (divide by the batch size for my_entropy)."""
  q = corr.shape[1]
  t = torch.as_tensor(T.orientation_target(yaw_bin, overlap, q, min_overlap_for_angle), dtype=corr.dtype)
  l = (1 - t) * corr + (1 + (q - 1) * t) * (torch.log1p(torch.exp(-corr.abs())) + torch.clamp(-corr, min=0))
  return l.mean(dim=1).sum()


def network_gradients(x_left, x_right, weights, overlap, yaw_bin, model_cfg=None, min_overlap_for_angle=0.7,
                      right_roll=None, chunk=1):
  """float64 losses and gradients of 5 L_ov + L_or for full-network training (legsType 360OutputkLegs):
  pair p runs LEFT image x_left[p] and RIGHT image x_right[p] (B, H, W, C), the latter rolled by
  right_roll[p] columns (np.roll along the width; None = no roll), through the same leg
  (generateNet.py:119-219), then both heads.  Every layer is a float64 leaf tensor, so each leg weight
  gets the sum of its gradients from both images of every pair, and L_or has a gradient.
  Returns ((total, L_ov, L_or), {layer: (dkernel, dbias)} float64, overlaps (n,))."""
  n = len(x_left)
  params = {k: (torch.tensor(np.asarray(weights[k][0], np.float64), requires_grad=True),
                torch.tensor(np.asarray(weights[k][1], np.float64), requires_grad=True)) for k in weights}
  y = np.asarray(overlap, np.float64)
  bins = np.asarray(yaw_bin, np.int64)
  yh, lov_sum, lor_sum = [], 0.0, 0.0
  for s in range(0, n, chunk):
    xl = np.asarray(x_left[s:s + chunk], np.float64)
    xr = np.asarray(x_right[s:s + chunk], np.float64)
    if right_roll is not None:
      xr = np.stack([np.roll(xr[i], int(right_roll[s + i]), axis=1) for i in range(len(xr))])
    fl = leg_forward_torch(torch.tensor(xl), params, model_cfg)
    fr = leg_forward_torch(torch.tensor(xr), params, model_cfg)
    o = T.head_overlap(fl, fr, params, model_cfg)
    lov = T.overlap_loss(o, y[s:s + chunk]) * o.shape[0]           # sum over the chunk
    lor = orientation_loss_torch(correlation_head_torch(fl, fr), bins[s:s + chunk], y[s:s + chunk],
                                 min_overlap_for_angle)
    ((5.0 * lov + lor) / n).backward()
    yh.append(o.detach().numpy())
    lov_sum += float(lov.detach())
    lor_sum += float(lor.detach())
  grads = {k: (params[k][0].grad.numpy(), params[k][1].grad.numpy()) for k in params}
  lov, lor = lov_sum / n, lor_sum / n
  return (5.0 * lov + lor, lov, lor), grads, np.concatenate(yh)
