"""Time one training step for precisions fp32 and f16_tc at the batch sizes of network.yml (16) and 64:
the overlap head on a frozen leg (ovn_heads_backward + ovn_adagrad_step, dW1's achieved rate), or with
--network the full network (ovn_network_backward + ovn_adagrad_step on packed 64 x 900 inputs).

Method: the step time comes from CUDA events around the timed steps of an unprofiled run.  The
per-kernel split comes from torch.profiler (CUPTI kernel records) over the same number of steps in a
SEPARATE run right after it, so its shares are not from the timed window and may include profiler
overhead; they size the kernels, the events give the step time.

  python tools/time_train.py [--network] [--steps 20] [--warmup 3] [--out DIR]

Work per pair (MAC), from the shapes of generateNet.py:64-116 with 360-wide volumes:
  forward  c_conv1 1 061 683 200, c_conv2 70 778 880, c_conv3 142 737 408, Dense 123 904,
           correlation 16 588 800  -> 2.55 GFLOP
  backward dW1 1 061 683 200, dO1 70 778 880, dW2 70 778 880, dX2 142 737 408, dW3 142 737 408,
           Dense 2 x 123 904       -> 2.98 GFLOP
Full network, per pair (two scans): leg forward, dW and useful dX 2 x (866 611 072 + 866 611 072 +
802 819 072), the head as above, the new dD 1 061 683 200 and the correlation backward 33 177 600 MAC.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MAC_FWD = 1061683200 + 70778880 + 142737408 + 123904 + 16588800
MAC_BWD = 1061683200 + 70778880 + 70778880 + 142737408 + 142737408 + 2 * 123904
MAC_DW1 = 1061683200
MAC_NET = 2 * (866611072 + 866611072 + 802819072) + MAC_FWD + MAC_BWD + 1061683200 + 33177600
DATASHEET_F16_DENSE_TFLOPS = 2250.0       # HGX B200 data sheet, one GPU, dense FP16/BF16 (not a reached rate)
MODEL = {'additional_unsymmetric_layer3a': True, 'strides_layer1': [2, 2]}


def card():
  q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                     capture_output=True, text=True)
  return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def setup(batch, precision, n_bank=64):
  from overlapnet_b200 import weights as W
  from overlapnet_b200.engine import Engine
  rng = np.random.default_rng(0)
  e = Engine(model=MODEL, precision=precision, max_batch_scans=4, max_batch_pairs=batch)
  e.load_weights(W.glorot_init(4, MODEL, seed=0))
  bank = torch.from_numpy(rng.uniform(0, 1, (n_bank, 360, 128)).astype(np.float32)).cuda()
  args = (bank, torch.from_numpy(rng.integers(0, n_bank, batch)), torch.from_numpy(rng.integers(0, n_bank, batch)),
          torch.from_numpy(rng.uniform(0, 1, batch).astype(np.float32)),
          torch.from_numpy(rng.integers(0, 360, batch)))
  return e, args


def setup_network(batch, precision, n_inputs=32):
  from overlapnet_b200 import weights as W
  from overlapnet_b200.engine import Engine
  rng = np.random.default_rng(0)
  e = Engine(model=MODEL, precision=precision, max_batch_scans=4, max_batch_pairs=batch)
  e.load_weights(W.glorot_init(4, MODEL, seed=0))
  x = rng.uniform(0, 1, (n_inputs, 64, 900, 4)).astype(np.float32)
  x[..., 0] *= 50.0                                                  # depth channel in metres
  args = (torch.from_numpy(x).cuda(), torch.from_numpy(rng.integers(0, n_inputs, batch)),
          torch.from_numpy(rng.integers(0, n_inputs, batch)), torch.from_numpy(rng.uniform(0, 1, batch).astype(np.float32)),
          torch.from_numpy(rng.integers(0, 360, batch)), torch.from_numpy(rng.integers(0, 901, batch)))
  return e, args


def step(e, args):
  if len(args) == 6:
    e.network_backward(*args)
  else:
    e.heads_backward(*args)
  e.adagrad_step(1e-3)


def time_batch(batch, precision, steps, warmup, network=False):
  e, args = (setup_network if network else setup)(batch, precision)
  for _ in range(warmup):
    step(e, args)
  e.check()
  t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  t0.record()
  for _ in range(steps):
    step(e, args)
  t1.record()
  torch.cuda.synchronize()
  e.check()
  ms = t0.elapsed_time(t1) / steps
  # per-kernel split in a separate profiled run
  from torch.profiler import ProfilerActivity, profile
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(steps):
      step(e, args)
    torch.cuda.synchronize()
  kern = {}
  for ev in prof.key_averages():
    if ev.device_type is not None and 'CUDA' in str(ev.device_type) and ev.self_device_time_total > 0:
      kern[ev.key] = kern.get(ev.key, 0.0) + ev.self_device_time_total / 1e3 / steps     # ms per step
  total = sum(kern.values())
  split = sorted(({'kernel': k, 'ms_per_step': v, 'share': v / total} for k, v in kern.items()),
                 key=lambda d: -d['ms_per_step'])
  dw1 = sum(v for k, v in kern.items() if ('k_wgrad' in k and 'DeltaOperand' in k) or 'k_delta_wgrad_tc' in k or 'k_dO1_' in k)
  e.close()
  if network:
    names = (('conv forward: leg, c_conv2, c_conv3 (k_simt_gemm<ConvOperand>)', 'k_simt_gemm<ovn::ConvOperand'),
             ('data gradients: leg, c_conv3 (k_simt_gemm<ConvTOperand>)', 'k_simt_gemm<ovn::ConvTOperand'),
             ('weight gradients: every layer (k_wgrad, k_delta_wgrad_tc)', 'wgrad'),
             ('dFV from the overlap head (k_dfv_overlap)', 'k_dfv_overlap'))
    groups = {g: 0.0 for g, _ in names}
    for k, v in kern.items():
      for g, key in names:
        if key in k:
          groups[g] += v
    return {'precision': precision, 'batch': batch, 'ms_per_step': ms, 'pairs_per_s': batch / ms * 1e3,
            'gflop_per_pair': 2 * MAC_NET / 1e9, 'step_tflops': batch * 2 * MAC_NET / (ms * 1e-3) / 1e12,
            'groups_ms': groups, 'kernels': split}
  return {'precision': precision, 'batch': batch, 'ms_per_step': ms, 'pairs_per_s': batch / ms * 1e3,
          'gflop_per_pair': 2 * (MAC_FWD + MAC_BWD) / 1e9,
          'step_tflops': batch * 2 * (MAC_FWD + MAC_BWD) / (ms * 1e-3) / 1e12,
          'dW1_ms': dw1, 'dW1_tflops': batch * 2 * MAC_DW1 / (dw1 * 1e-3) / 1e12 if dw1 else None,
          'kernels': split}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--steps', type=int, default=20)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--out', default=None)
  ap.add_argument('--network', action='store_true', help='time full-network steps (ovn_network_backward)')
  a = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('time_train.py needs a CUDA device')
  res = {'card': card(), 'method': 'step time: CUDA events, unprofiled run; kernel split: torch.profiler, separate run',
         'datasheet_dense_f16_tflops': DATASHEET_F16_DENSE_TFLOPS, 'network': a.network,
         'runs': [time_batch(b, p, a.steps, a.warmup, a.network) for p in ('fp32', 'f16_tc') for b in (16, 64)]}
  print('# %s; %s; data-sheet dense fp16 rate %.0f TFLOP/s (not a reached rate)' % (
      res['card'], res['method'], DATASHEET_F16_DENSE_TFLOPS))
  if a.network:
    for r in res['runs']:
      print('%-6s batch %3d: %.2f ms/step, %.0f pairs/s, %.1f GFLOP/pair, %.1f TFLOP/s per step' % (
          r['precision'], r['batch'], r['ms_per_step'], r['pairs_per_s'], r['gflop_per_pair'], r['step_tflops']))
      for g, v in r['groups_ms'].items():
        print('   %7.2f ms  %s' % (v, g))
      for k in r['kernels'][:10]:
        print('   %7.2f ms %5.1f%%  %s' % (k['ms_per_step'], 100 * k['share'], k['kernel'][:100]))
    print(json.dumps(res))
    return
  for r in res['runs']:
    print('%-6s batch %3d: %.2f ms/step, %.0f pairs/s, %.1f TFLOP/s per step; dW1 %.2f ms = %.1f TFLOP/s' % (
        r['precision'], r['batch'], r['ms_per_step'], r['pairs_per_s'], r['step_tflops'], r['dW1_ms'], r['dW1_tflops'] or 0))
    for k in r['kernels'][:8]:
      print('   %6.2f ms %5.1f%%  %s' % (k['ms_per_step'], 100 * k['share'], k['kernel'][:100]))
  print(json.dumps(res))
  if a.out:
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, 'time_train.json'), 'w') as f:
      json.dump(res, f, indent=1)


if __name__ == '__main__':
  main()
