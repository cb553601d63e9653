#!/usr/bin/env python3
"""Time sequence-wide ground truth (overlapnet_b200.gt.overlap_yaw_sequence) on a synthetic
KITTI-sized sequence, against the per-frame loop it replaces.

  python tools/time_gt.py [--frames 1000] [--points 124668] [--loop-frames 3]

The sequence is ``synth.trajectory_sequence`` (2 MB of points per scan, 2 GB in all: larger than L2).
Reported, all in one run with the card's name and power limit:
  - all-pairs wall time (host clock around the call, which ends in a device synchronise), pairs/s and
    point projections/s (points of every scan of every pair that was not culled);
  - the culled fraction;
  - pair-kernel time from CUDA events around every ovn_gt_pair_counts call;
  - FP64 instructions per point, counted in the SASS of k_gt_pair_counts (the per-point loop between
    the two barriers: both sides of its in-loop branches, none of the out-of-line slow paths), and the
    kernel's share of the data-sheet FP64 rate at that count;
  - the per-frame loop (overlap_yaw_from_clouds per frame, same in-memory clouds) timed on
    ``--loop-frames`` frames and extrapolated to all frames (labelled as extrapolated).
"""
import argparse
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# NVIDIA HGX B200 data sheet: FP64 / FP64 Tensor Core 296 TFLOP/s for eight GPUs, so 37 TFLOP/s for one
# (at up to 1000 W).  One FP64 pipe instruction (DFMA counted as 2 FLOP) per lane: 18.5e12 per second.
DATASHEET_FP64_FLOPS = 37e12
FP64_OPS = re.compile(r'^(DFMA|DMUL|DADD|DSETP|DMNMX|DRND|F2F\.F64|F2F\.F32\.F64|I2F\.F64|F2I\.F64|FRND\.F64|'
                      r'MUFU\.(RCP64H|RSQ64H))')


def card():
  import torch
  name = torch.cuda.get_device_name(0)
  try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True, timeout=60).stdout.strip()
  except (OSError, subprocess.SubprocessError):
    q = 'nvidia-smi not available'
  return name, q


def fp64_per_point():
  """(FP64 instructions in the per-point loop of k_gt_pair_counts, its SASS text length)."""
  from overlapnet_b200 import _cabi
  lib = _cabi.LIB_PATH
  sass = subprocess.run(['cuobjdump', '-sass', lib], capture_output=True, text=True).stdout
  fn = re.search(r'Function : (\S*k_gt_pair_counts\S*)\n(.*?)(?=\n\s*Function : |\Z)', sass, re.S)
  if not fn:
    return None, 0
  ops = [m.group(1) for m in re.finditer(r'/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9_.]+)', fn.group(2))]
  bars = [i for i, o in enumerate(ops) if o.startswith('BAR')]
  loop = ops[bars[0] + 1:bars[1]]
  return sum(1 for o in loop if FP64_OPS.match(o)), len(ops)


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument('--frames', type=int, default=1000)
  ap.add_argument('--points', type=int, default=124668)
  ap.add_argument('--loop-frames', type=int, default=3)
  ap.add_argument('--seed', type=int, default=0)
  args = ap.parse_args()
  import torch
  from overlapnet_b200 import engine, gt, synth

  name, smi = card()
  print('card: %s | nvidia-smi name, power.limit, clocks.max.sm: %s' % (name, smi))
  t0 = time.perf_counter()
  clouds, poses = synth.trajectory_sequence(args.seed, args.frames, n_points=args.points)
  n = len(clouds)
  print('sequence: synth.trajectory_sequence(seed=%d): %d frames x %d points (%.2f GB of points), generated in %.1f s'
        % (args.seed, n, args.points, n * args.points * 16 / 1e9, time.perf_counter() - t0))

  stats = {'ms': 0.0, 'pairs': 0, 'points': 0, 'launches': 0}
  orig = engine.Engine.gt_pair_counts

  def timed(self, batch, pose_ref, pose_cur_inv, cur_ranges, pairs, **kw):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    out = orig(self, batch, pose_ref, pose_cur_inv, cur_ranges, pairs, **kw)
    stop.record()
    stop.synchronize()
    stats['ms'] += start.elapsed_time(stop)
    sizes = torch.diff(batch.offsets)
    stats['points'] += int(sizes[pairs[:, 1].long()].sum())
    stats['pairs'] += int(pairs.shape[0])
    stats['launches'] += 1
    return out

  gt.overlap_yaw_sequence(clouds[:3], poses[:3])              # warm-up: modules, handle, every code path
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  rows = gt.overlap_yaw_sequence(clouds, poses)
  torch.cuda.synchronize()
  wall = time.perf_counter() - t0
  total = n * n
  print('all-pairs wall time: %.2f s for %d pairs = %.3g pairs/s (rows %s, ends in a device synchronise)'
        % (wall, total, total / wall, rows.shape))

  engine.Engine.gt_pair_counts = timed                       # second run: per-launch events (synchronises each launch)
  rows2 = gt.overlap_yaw_sequence(clouds, poses)
  engine.Engine.gt_pair_counts = orig
  assert np.array_equal(rows, rows2)
  culled = 1.0 - stats['pairs'] / total
  kern_s = stats['ms'] / 1e3
  print('culled: %d of %d pairs (%.1f %%); %d pairs launched in %d launches' % (total - stats['pairs'], total,
                                                                                100 * culled, stats['pairs'],
                                                                                stats['launches']))
  print('point projections: %.4g (points of the reference scan of every launched pair); %.3g /s over the all-pairs '
        'wall time, %.3g /s over pair-kernel time' % (stats['points'], stats['points'] / wall, stats['points'] / kern_s))
  print('pair-kernel time (CUDA events): %.3f s, %.2f us per launched pair, %.1f %% of the all-pairs wall time'
        % (kern_s, 1e6 * kern_s / max(stats['pairs'], 1), 100 * kern_s / wall))
  per_point, n_sass = fp64_per_point()
  if per_point:
    rate = DATASHEET_FP64_FLOPS / 2
    share = per_point * stats['points'] / kern_s / rate
    print('FP64 instructions per point: %d (SASS of k_gt_pair_counts, per-point loop, static count of both sides of '
          'its branches; %d SASS instructions in the kernel)' % (per_point, n_sass))
    print('FP64 pipe: %.3g instructions/s = %.1f %% of the data-sheet FP64 rate (HGX B200 data sheet, 37 TFLOP/s '
          'per GPU = 18.5e12 FP64 instructions/s; a data-sheet figure, not a measured peak)'
          % (per_point * stats['points'] / kern_s, 100 * share))
  else:
    print('FP64 instructions per point: not measured (cuobjdump not available)')

  k = min(args.loop_frames, n)
  frames = np.linspace(0, n - 1, k).astype(int)
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  loop_rows = [gt.overlap_yaw_from_clouds(clouds, poses, int(f)) for f in frames]
  torch.cuda.synchronize()
  per = (time.perf_counter() - t0) / k
  for f, r in zip(frames, loop_rows):
    assert np.array_equal(r, rows[f * n:(f + 1) * n]), f
  print('per-frame loop: %.2f s per frame measured on frames %s (rows equal the all-pairs rows); '
        '%.0f s for all %d frames (EXTRAPOLATED, not measured) = %.1fx the all-pairs wall time'
        % (per, frames.tolist(), per * n, n, per * n / wall))


if __name__ == '__main__':
  main()
