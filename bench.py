#!/usr/bin/env python3
"""bench.py -- BASELINE.json's metric: scan-pairs/s (overlap + yaw) of the 1-query-vs-N-candidate
loop-closure search at 64x900, on synthetic KITTI-shaped data.

  python bench.py --gpus N --steps K --warmup W            # this repo's B200 path
  python bench.py --impl reference --steps K --warmup W    # the CPU port of the reference, host cores
  (N > 1: python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...)
  --dump-outputs DIR   also write what the last timed headline step returned (every candidate's
                       overlap and yaw, float32 .npy) so that two builds can be compared output for
                       output; the inputs depend only on the arguments.

Headline (`value`, `e2e`): BASELINE config 2 -- one query scan through the whole hot path,
  raw cloud (124 668 pts) -> projection + normals (64x900x4) -> leg -> 1 x 1101 delta + correlation
  heads over the rank's candidate bank -> (overlap, yaw) per candidate.
N > 1 is weak scaling (every rank holds its own 1101-candidate shard): rank 0 encodes the query; the
other ranks read the 184 KB query volume straight out of rank 0's symmetric (peer-mapped) buffer and
their finalize kernels store (overlap, yaw) straight into rank 0's result table over NVLink -- no
collective on the data path (fallback when symmetric memory is unavailable: ONE NCCL broadcast + ONE
gather of packed 8-byte records).

The same JSON line carries the other BASELINE configs as extra objects (each measured in this run):
  "latency_1pair"  config 1  one scan pair through Infer-equivalent calls (ms per pair)
  "leg_batch256"   config 3  4-cue C=25 input, batch-256 leg encode (scans/s, TFLOP/s)
  "bank4541"       config 4  4541-volume bank SHARDED over the N ranks (strong scaling)
  "all_pairs"      config 5  rows of the 4541 x 4541 ordered pair matrix + streamed raw-cloud encode
  "range_proj"               batched projection + normals (Mpts/s, GB/s against the measured HBM peak)
`roofline` = k_delta_conv1_tc (the dominant kernel) against the measured bf16 tensor peaks (burst and
sustained); `cpu_baseline` = the oracle port of the reference graph on a bounded sample, whose float64
twin also spot-checks the timed GPU output in-run (`parity_check`).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

MODEL = {'additional_unsymmetric_layer3a': True, 'strides_layer1': [2, 2]}
N_CAND = 1101                     # KITTI-07 length (BASELINE config 2)
N_BANK4 = 4541                    # KITTI-00 length (BASELINE configs 4, 5)
N_SRC_SCANS = 32                  # distinct synthetic scans behind a bank (yaw-rolled to the bank size)
FLOP_DELTA_CONV1 = 2 * 1061683200 # per pair, c_conv1 (SURVEY 8a row 9)
FLOP_PAIR = 2 * (1275323392 + 16588800)
FLOP_LEG_C4 = 2 * 866611072
FLOP_LEG_C25 = 2 * 1201519072
METRIC = 'scan-pairs/sec (overlap+yaw) at 64x900'
WORKLOAD = '1 query x 1101 candidates per GPU, geo-only 64x900 (BASELINE config 2)'
LOGIT_SPREAD = 1.5                # the Dense layer is rescaled so that the bank's logits have this std (parity_check)


def parse():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=20)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--precision', default='f16_tc', choices=['f16_tc', 'fp32'])
  ap.add_argument('--cpu-pairs', type=int, default=8, help='pairs per step in the CPU sample')
  ap.add_argument('--transport', default='auto', choices=['auto', 'symm', 'collective'])
  ap.add_argument('--no-extras', action='store_true', help='only the headline config (fast)')
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='write the overlaps and yaws of the last timed headline step to DIR/{overlap,yaw}.npy')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  return args


def peaks():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    with open(p) as f:
      d = json.load(f)
    return {'burst': d.get('bf16_tflops'), 'sustained': d.get('bf16_tflops_sustained'), 'hbm': d.get('hbm_gbs'),
            'source': 'measured (MEASURED_PEAKS.json)'}
  return {'burst': 1590.0, 'sustained': 1400.0, 'hbm': 6650.0, 'source': 'fallback (B200_PROFILING.md)'}


class ClockSampler(threading.Thread):
  """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

  def __init__(self, index=0):
    super().__init__(daemon=True)
    self.index, self.rows, self.proc = index, [], None

  def wait_first_sample(self, timeout=5.0):
    t0 = time.time()
    while not self.rows and time.time() - t0 < timeout:
      time.sleep(0.02)

  def run(self):
    q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    try:
      self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                    '--format=csv,noheader,nounits', '-lms', '20'],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      for line in self.proc.stdout:
        self.rows.append([x.strip() for x in line.split(',')])
    except Exception:
      pass

  def stop(self):
    if self.proc:
      self.proc.terminate()
    sm, mx, reasons = [], 0, set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for r in self.rows:
      try:
        sm.append(float(r[0]))
        mx = max(mx, float(r[1]))
        for i, n in enumerate(names):
          if r[2 + i].lower().startswith('active'):
            reasons.add(n)
      except Exception:
        continue
    busy = sorted(s for s in sm if s > 0.5 * mx) or sorted(sm)
    return {'sm_mhz': busy[len(busy) // 2] if busy else None, 'sm_max_mhz': mx or None,
            'reasons': sorted(reasons), 'samples': len(sm)}


def make_weights(channels=4):
  """Seeded Glorot-uniform kernels keyed by the Keras layer names (what the reference runs with when no
  pretrained file is given, infer.py:117-122) + small random biases so that the bias path is exercised."""
  from overlapnet_b200 import weights as W
  w = W.glorot_init(channels, MODEL, seed=0)
  rng = np.random.default_rng(1)
  return {k: (kern, rng.uniform(-0.05, 0.05, b.shape).astype(np.float32)) for k, (kern, b) in w.items()}


def spread_dense(w, overlaps, target_std=LOGIT_SPREAD):
  """Rescale / recentre Dense(1) from the overlaps the product path produced with the raw weights:
  Glorot heads put every overlap at 0.5 +- 0.003, where an absolute 1e-3 gate says nothing."""
  ov = np.clip(np.asarray(overlaps, np.float64), 1e-7, 1 - 1e-7)
  z = np.log(ov / (1 - ov))
  k, b = w['overlap_output']
  raw = z - float(b[0])
  g = target_std / max(float(raw.std()), 1e-12)
  w2 = dict(w)
  w2['overlap_output'] = ((k.astype(np.float64) * g).astype(np.float32), np.array([-g * float(np.median(raw))], np.float32))
  return w2


# ---- the CPU port of the reference graph (oracle/) -----------------------------------------------------
def cpu_sample(w, bank_np, query_cloud, n_pairs, dtype=torch.float32):
  """One bounded sample of the config-2 step on the host cores: projection + normals + leg of the
  query scan, then the two heads on ``n_pairs`` candidates (delta tensor materialised like Keras,
  batch 16 like config/network.yml:41).  Returns the three stage times and the outputs."""
  from oracle import network as onet
  from oracle import projection as oproj
  t0 = time.perf_counter()
  rng, vert, _, _ = oproj.range_projection(query_cloud)
  x = oproj.pack_input(rng, oproj.gen_normal_map(rng, vert))[None]
  t1 = time.perf_counter()
  q = onet.leg_forward(x, w, MODEL, dtype=dtype)
  t2 = time.perf_counter()
  ov, yaw, _ = onet.heads_forward(bank_np[:n_pairs, None], np.repeat(q, n_pairs, 0), w, MODEL, dtype=dtype, batch=16)
  t3 = time.perf_counter()
  return {'t_proj': t1 - t0, 't_leg': t2 - t1, 't_heads': t3 - t2, 'ov': ov, 'yaw': yaw, 'qfv': q}


def cpu_extrapolate(samples, n_pairs):
  """pairs/s of the full 1 x 1101 step from the measured stages: projection and leg happen once per
  query, the heads scale with the candidates."""
  t_proj = float(np.mean([s['t_proj'] for s in samples]))
  t_leg = float(np.mean([s['t_leg'] for s in samples]))
  t_pair = float(np.mean([s['t_heads'] for s in samples])) / n_pairs
  t_step = t_proj + t_leg + N_CAND * t_pair
  return N_CAND / t_step, {'t_projection_normals_s': t_proj, 't_leg_s': t_leg, 't_heads_per_pair_s': t_pair,
                           't_step_1101_s': t_step}


def synth_bank_np(n, seed=7):
  from overlapnet_b200 import synth
  return synth.feature_volumes(seed, n)[:, 0]


def run_reference(args):
  """--impl reference: the reference's own implementation is Python/TF and cannot be installed
  offline, so this arm times the oracle port on all host cores (kind = "port").  Every step is a bounded
  sample of the config-2 step (1 projection + normals, 1 leg, --cpu-pairs head pairs); the full-step
  figure is the explicit extrapolation  t_proj + t_leg + 1101 * t_pair."""
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  from overlapnet_b200 import synth
  w = make_weights()
  cores = os.cpu_count()
  torch.set_num_threads(cores)
  n = args.cpu_pairs
  bank = synth_bank_np(n)
  clouds = [synth.kitti_like_cloud(50000 + s) for s in range(4)]
  for i in range(args.warmup):
    cpu_sample(w, bank, clouds[i % 4], n)
  samples = [cpu_sample(w, bank, clouds[(args.warmup + i) % 4], n) for i in range(args.steps)]
  val, parts = cpu_extrapolate(samples, n)
  sample = ('%d of the 1101 pairs per step + 1 projection/normals + 1 leg, torch-CPU fp32, delta tensor '
            'materialised; value = 1101 / (t_proj + t_leg + 1101 * t_pair)' % n)
  print(json.dumps({
      'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'pairs/s', 'n_gpus': args.gpus, 'steps': args.steps,
      'warmup': args.warmup, 'ms_per_step': parts['t_step_1101_s'] * 1e3, 'higher_is_better': True,
      'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': {'workload': WORKLOAD + ', bounded sample', 'stages': parts},
      'cpu_baseline': {'value': val, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port', 'sample': sample},
      'e2e': {'value': val, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
  }))


# ---- the B200 path ---------------------------------------------------------------------------------------
def rolled_bank(eng, fv_src, n, dev):
  src = torch.arange(n, device=dev) % fv_src.shape[0]
  roll = (torch.arange(n, device=dev) // fv_src.shape[0]) * 7
  rows = (torch.arange(eng.Wf, device=dev)[None, :] - roll[:, None]) % eng.Wf
  out = torch.empty((n, eng.Wf, 128), dtype=torch.float32, device=dev)
  for s0 in range(0, n, 512):                                     # bounded temporaries
    out[s0:s0 + 512] = fv_src[src[s0:s0 + 512, None], rows[s0:s0 + 512]]
  return out


def main():
  args = parse()
  if args.impl == 'reference':
    run_reference(args)
    return
  import torch.distributed as dist
  from overlapnet_b200 import synth
  from overlapnet_b200.engine import CloudBatch, Engine
  from overlapnet_b200.search import ShardedSearch, engine_heads_fn, shard_range

  world = int(os.environ.get('WORLD_SIZE', '1'))
  rank = int(os.environ.get('RANK', '0'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  if args.gpus != world and world == 1 and args.gpus > 1:
    raise SystemExit('launch with torch.distributed.run --nproc-per-node %d for --gpus %d' % (args.gpus, args.gpus))
  torch.cuda.set_device(local)
  dev = torch.device('cuda', local)
  if world > 1:
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    dist.init_process_group('nccl', device_id=dev)

  def timed(fn, steps, warmup):
    for i in range(warmup):
      fn(i)
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
      fn(warmup + i)
    b.record()
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b)], device=dev)
    if world > 1:
      dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())

  w = make_weights()
  eng = Engine(model=MODEL, precision=args.precision, device=local, max_batch_scans=N_SRC_SCANS,
               max_batch_pairs=N_CAND)
  eng.load_weights(w)

  # ---- candidate bank of this rank: 32 synthetic scans encoded by the product path, yaw-rolled to 1101
  clouds = [synth.kitti_like_cloud(1000 * rank + s) for s in range(N_SRC_SCANS)]
  cloud_batch = eng.upload_clouds(clouds)
  fv_src = eng.leg(eng.preprocess(cloud_batch))
  bank = rolled_bank(eng, fv_src, N_CAND, dev)
  # query clouds: a fresh scan per step (pinned host copies for the e2e leg); the same on every rank
  n_q = 4
  q_np = [synth.kitti_like_cloud(50000 + s) for s in range(n_q)]
  q_host = [torch.from_numpy(q).pin_memory() for q in q_np]
  q_dev = [eng.upload_clouds([q]) for q in q_np]
  # Dense layer rescaled from a first pass of the product path (logit spread 1.5 over this bank)
  ov0, _, _ = eng.heads_1vsN(bank, eng.leg(eng.preprocess(q_dev[0]))[0], n_cand=N_CAND)
  eng.check()
  ov0 = ov0.cpu().numpy()
  if world > 1:                                             # every rank must run the same weights
    t0 = torch.from_numpy(ov0).to(dev)
    dist.broadcast(t0, 0)
    ov0 = t0.cpu().numpy()
  w = spread_dense(w, ov0)
  eng.load_weights(w)
  eng.bank_prepare(bank)          # the candidate bank is static: keep its tensor-core operand copies resident

  ss = ShardedSearch(engine_heads_fn(eng), bank, N_CAND * world, transport=args.transport) if world > 1 else None
  transport = ss.transport if ss else 'single GPU'
  qfv = torch.empty((eng.Wf, 128), dtype=torch.float32, device=dev)
  last = {}

  def step(i):
    """Device-resident step: query cloud already in HBM (on rank 0)."""
    if rank == 0:
      qfv.copy_(eng.leg(eng.preprocess(q_dev[i % n_q]))[0])
    if world == 1:
      last['res'] = eng.heads_1vsN(bank, qfv, n_cand=N_CAND)[:2]
    else:
      last['res'] = ss.query(qfv)

  ov_h = np.empty((N_CAND,), np.float32)
  yaw_h = np.empty((N_CAND,), np.int32)

  def step_e2e(i):
    """Public host-buffer entry point: H2D of the query cloud + D2H of the results every step."""
    if world == 1:
      eng.query_cloud_vs_bank_host(q_host[i % n_q], bank, n_cand=N_CAND, out_overlap=ov_h, out_yaw=yaw_h)
      return
    if rank == 0:
      qd = q_host[i % n_q].to(dev, non_blocking=True)
      off = torch.tensor([0, qd.shape[0]], dtype=torch.int64, device=dev)
      qfv.copy_(eng.leg(eng.preprocess(CloudBatch(qd, off, [0, qd.shape[0]])))[0])
    res = ss.query(qfv)
    if rank == 0:
      last['host'] = (res[0].cpu(), res[1].cpu())               # D2H of every rank's records; synchronises

  # ---- timed region 1: device-resident, per-kernel events on
  sampler = ClockSampler(local) if rank == 0 else None
  if sampler:
    sampler.start()
    sampler.wait_first_sample()
  kernels = ('delta_conv1', 'conv2', 'conv3', 'corr', 'leg', 'project_scatter', 'project_gather')
  eng.profile_enable(True)
  timed(step, 0, args.warmup)
  for k in kernels:
    eng.profile_read(k)
  l0 = eng.launch_count()
  ms = timed(step, args.steps, 0)
  launches = eng.launch_count() - l0
  prof = {k: eng.profile_read(k) for k in kernels}
  eng.profile_enable(False)
  eng.check()
  gpu_ov = last['res'][0][:N_CAND].cpu().numpy() if rank == 0 else None     # rank 0's own shard of the last timed step
  gpu_yaw = last['res'][1][:N_CAND].cpu().numpy() if rank == 0 else None
  if rank == 0 and args.dump_outputs:                        # every rank's candidates, in bank order
    dump = {'overlap': last['res'][0].cpu().numpy().astype(np.float32),
            'yaw': last['res'][1].cpu().numpy().astype(np.float32)}
  last_q = (args.steps - 1) % n_q if args.steps else 0
  # ---- timed region 2: end to end through the host-buffer entry point
  ms_e2e = timed(step_e2e, args.steps, args.warmup)
  clocks = sampler.stop() if sampler else None

  extras = {}
  if not args.no_extras:
    leg_ms = prof['leg'][0] / max(args.steps, 1)
    per_pair_ms = max(ms / max(args.steps, 1) - leg_ms, 1e-6) / N_CAND
    disc = torch.tensor([int(round(leg_ms / per_pair_ms))], dtype=torch.int32, device=dev)
    if world > 1:
      dist.broadcast(disc, 0)
    try:
      extras = measure_extras(args, eng, w, dev, rank, world, local, timed, q_dev, q_host, cloud_batch, fv_src, bank,
                              int(disc.item()))
    except Exception as e:                                   # the headline line must survive a failing extra
      extras = {'extras_error': repr(e)[:300]}

  if rank == 0:
    pk = peaks()
    pairs = world * N_CAND * args.steps
    value = pairs / (ms * 1e-3)
    e2e = pairs / (ms_e2e * 1e-3)
    k_ms, k_n = prof['delta_conv1']
    ach = (N_CAND * FLOP_DELTA_CONV1 / 1e12) / (k_ms / max(k_n, 1) * 1e-3) if k_n else None
    shares = {k: round(v[0] / ms, 4) for k, v in prof.items()}
    # ---- CPU port on a bounded sample of this workload + in-run parity spot check of the timed output
    torch.set_num_threads(os.cpu_count())
    bank_np = bank[:args.cpu_pairs].cpu().numpy()
    t_cpu0 = time.perf_counter()
    samples = [cpu_sample(w, bank_np, q_np[last_q], args.cpu_pairs) for _ in range(3)]
    cpu_val, cpu_parts = cpu_extrapolate(samples[1:], args.cpu_pairs)
    t_cpu = time.perf_counter() - t_cpu0
    chk = cpu_sample(w, bank_np, q_np[last_q], args.cpu_pairs, dtype=torch.float64)     # float64 twin = the checker
    d_ov = np.abs(gpu_ov[:args.cpu_pairs] - chk['ov'])
    parity = {'pairs_checked': int(args.cpu_pairs), 'max_abs_overlap_err': float(d_ov.max()),
              'yaw_equal': int((gpu_yaw[:args.cpu_pairs] == chk['yaw']).sum()), 'gate': 1e-3,
              'logit_spread': LOGIT_SPREAD,
              'overlap_range_checked': [float(chk['ov'].min()), float(chk['ov'].max())],
              'checker': 'oracle float64 on the first %d candidates of the last timed step (query scan %d)'
                         % (args.cpu_pairs, last_q)}
    traffic = None
    tp = os.path.join(ROOT, 'profiles', 'r2_delta_traffic.json')
    if os.path.exists(tp) and args.precision == 'f16_tc':
      with open(tp) as f:
        tj = json.load(f)
      traffic = (tj['dram_bytes_read'] + tj['dram_bytes_write']) * N_CAND / tj['pairs_per_launch']
    line = {
        'metric': METRIC, 'value': value, 'unit': 'pairs/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f16' if args.precision == 'f16_tc' else 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'candidates_per_gpu': N_CAND, 'query_points': int(q_host[0].shape[0]),
                   'l2': 'inputs larger than L2: the fp32 candidate bank is 203 MB per step',
                   'parallelism': 'bank sharded x%d; transport: %s' % (world, transport),
                   'precision': args.precision,
                   'weights': 'seeded Glorot (no pretrained weights offline), Dense rescaled to logit spread %.1f' % LOGIT_SPREAD},
        'gpu_launches': int(launches),
        'e2e': {'value': e2e, 'unit': 'pairs/s', 'ms_per_step': ms_e2e / args.steps,
                'h2d_bytes_per_step': int(q_host[0].numel() * 4),
                'd2h_bytes_per_step': int(N_CAND * 8 * world)},
        'roofline': {'kernel': 'k_delta_conv1_tc' if args.precision == 'f16_tc' else 'k_simt_gemm<DeltaOperand>',
                     'bound': 'tensor', 'achieved': ach, 'peak': pk['burst'], 'unit': 'TFLOP/s',
                     'frac': (ach / pk['burst']) if ach else None,
                     'frac_burst': (ach / pk['burst']) if ach else None,
                     'frac_sustained': (ach / pk['sustained']) if ach else None,
                     'peak_burst': pk['burst'], 'peak_sustained': pk['sustained'],
                     'peak_note': 'the kernel is timed inside a ~60 ms region at full clock: the burst peak applies',
                     'traffic': traffic, 'peak_source': pk['source'],
                     'flop_per_launch': N_CAND * FLOP_DELTA_CONV1, 'avg_launch_ms': k_ms / max(k_n, 1),
                     'share_of_step': shares},
        'whole_path_tflops': pairs * FLOP_PAIR / 1e12 / (ms * 1e-3),
        'parity_check': parity,
        'cpu_baseline': {'value': cpu_val, 'unit': 'pairs/s', 'cores': os.cpu_count(), 'kind': 'port',
                         'sample': '2 x (%d of the 1101 pairs + 1 projection/normals + 1 leg) in %.1f s, torch-CPU fp32; '
                                   'value = 1101 / (t_proj + t_leg + 1101 * t_pair)' % (args.cpu_pairs, t_cpu),
                         'stages': cpu_parts},
        'clocks': clocks,
    }
    line.update(extras)
    if args.dump_outputs:
      os.makedirs(args.dump_outputs, exist_ok=True)
      for name, a in dump.items():
        np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
    print(json.dumps(line))
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


def measure_extras(args, eng, w, dev, rank, world, local, timed, q_dev, q_host, cloud_batch, fv_src, bank, src_discount):
  """The other BASELINE configs, each a short measurement in the same run (see the module docstring)."""
  import torch.distributed as dist
  from overlapnet_b200 import synth
  from overlapnet_b200.engine import CloudBatch, Engine
  from overlapnet_b200.search import ShardedSearch, balanced_sizes, engine_heads_fn, shard_range
  out = {}
  pk = peaks()
  n_q = len(q_dev)

  # ---- config 1: one scan pair (demo2_infer: encode both scans, one pair through both heads) -----------
  if rank == 0:
    pair_batch = eng.upload_clouds([synth.kitti_like_cloud(77), synth.kitti_like_cloud(78)])
    li, ri = torch.tensor([0], dtype=torch.int32, device=dev), torch.tensor([1], dtype=torch.int32, device=dev)

    def one_pair(i):
      fv = eng.leg(eng.preprocess(pair_batch))
      eng.heads(fv, li, ri)
    eng.bank_release(None)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(5):
      one_pair(i)
    torch.cuda.synchronize()
    a.record()
    for i in range(50):
      one_pair(i)
    b.record()
    torch.cuda.synchronize()
    ms1 = a.elapsed_time(b) / 50
    # same work replayed from a CUDA graph (launch-bound chain of ~40 small kernels)
    ms1_graph = None
    try:
      g = torch.cuda.CUDAGraph()
      s = torch.cuda.Stream()
      s.wait_stream(torch.cuda.current_stream())
      with torch.cuda.stream(s):
        one_pair(0)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
          one_pair(0)
      torch.cuda.synchronize()
      a.record()
      for i in range(50):
        g.replay()
      b.record()
      torch.cuda.synchronize()
      ms1_graph = a.elapsed_time(b) / 50
    except Exception as e:                                   # capture is an optimisation, never a requirement
      ms1_graph = None
      out['latency_1pair_graph_error'] = repr(e)[:200]
      torch.cuda.synchronize()
    out['latency_1pair'] = {'workload': 'BASELINE config 1: two raw clouds -> projection -> leg x2 -> one pair through both heads',
                            'ms_per_pair': ms1, 'ms_per_pair_cuda_graph': ms1_graph,
                            'pairs_per_s': 1e3 / min(ms1, ms1_graph or ms1)}
    eng.bank_prepare(bank)

  # ---- batched projection (BASELINE metric "range-proj Mpts/s") ---------------------------------------
  if rank == 0:
    def proj(i):
      eng.preprocess(cloud_batch)
    eng.profile_enable(True)
    for k in ('project_scatter', 'project_gather'):
      eng.profile_read(k)
    for i in range(3):
      proj(i)
    for k in ('project_scatter', 'project_gather'):
      eng.profile_read(k)
    for i in range(10):
      proj(i)
    ps, pg = eng.profile_read('project_scatter'), eng.profile_read('project_gather')
    eng.profile_enable(False)
    n_scans = cloud_batch.n
    npts = int(cloud_batch.offsets_host[-1])
    ms_p = (ps[0] + pg[0]) / 10
    byts = npts * 16 + n_scans * 64 * 900 * 16
    out['range_proj'] = {'scans_per_launch': n_scans, 'points': npts, 'ms_per_launch': ms_p,
                         'mpts_per_s': npts / (ms_p * 1e-3) / 1e6, 'algorithmic_bytes': byts,
                         'gb_per_s': byts / (ms_p * 1e-3) / 1e9, 'hbm_peak_gb_per_s': pk['hbm'],
                         'frac_of_hbm_peak': byts / (ms_p * 1e-3) / 1e9 / pk['hbm'],
                         'kernels_ms': {'scatter': ps[0] / 10, 'gather_normals_pack': pg[0] / 10},
                         'note': 'fused projection + normals + channel packing of %d clouds in one launch pair; '
                                 'bytes = 16 B/point read once + 16 B/pixel written once (SURVEY 8d)' % n_scans}

  # ---- config 3: 4-cue input (C = 25), batch-256 leg encode -------------------------------------------
  if rank == 0:
    try:
      use = {'use_intensity': True, 'use_class_probabilities': True}
      eng25 = Engine(use=use, model=MODEL, precision=args.precision, device=local, max_batch_scans=256, max_batch_pairs=1)
      eng25.load_weights(make_weights(25))
      x_small = torch.from_numpy(synth.range_like_images(5, 8, 25)).to(dev)
      x25 = x_small.repeat(32, 1, 1, 1)                      # 256 scans, 1.47 GB of NHWC input (> L2)
      for i in range(2):
        eng25.leg(x25)
      torch.cuda.synchronize()
      a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a.record()
      for i in range(5):
        eng25.leg(x25)
      b.record()
      torch.cuda.synchronize()
      ms3 = a.elapsed_time(b) / 5
      tf = 256 * FLOP_LEG_C25 / 1e12 / (ms3 * 1e-3)
      out['leg_batch256'] = {'workload': 'BASELINE config 3: 4-cue C=25 64x900 input, batch-256 leg encode',
                             'ms_per_batch': ms3, 'scans_per_s': 256 / (ms3 * 1e-3), 'tflops': tf,
                             'frac_burst': tf / pk['burst'], 'frac_sustained': tf / pk['sustained'],
                             'note': 'algorithmic FLOPs (2 x 1 201 519 072 per scan); the kernels issue 3x that '
                                     '(hi/lo split fp16 operands, fp32-grade accuracy)'}
      del x25
      eng25.close()
      torch.cuda.empty_cache()
    except Exception as e:
      out['leg_batch256'] = {'error': repr(e)[:300]}

  # ---- config 4: 4541-volume bank SHARDED over the ranks (strong scaling) -----------------------------
  # rank 0 also encodes the query: its shard is shorter by (encode time / time per candidate) candidates
  sizes4 = balanced_sizes(N_BANK4, world, 0, src_discount)
  lo = int(sum(sizes4[:rank]))
  hi = lo + sizes4[rank]
  eng.bank_release(None)
  big = rolled_bank(eng, fv_src, N_BANK4, dev)[lo:hi].contiguous()
  eng.bank_prepare(big)
  qfv = torch.empty((eng.Wf, 128), dtype=torch.float32, device=dev)
  ss4 = ShardedSearch(engine_heads_fn(eng), big, N_BANK4, transport=args.transport, sizes=sizes4) if world > 1 else None

  def step4(i):
    if rank == 0:
      qfv.copy_(eng.leg(eng.preprocess(q_dev[i % n_q]))[0])
    if world == 1:
      eng.heads_1vsN(big, qfv, n_cand=N_BANK4)
    else:
      ss4.query(qfv)
  k4 = max(3, min(10, args.steps))
  ms4 = timed(step4, k4, 2)
  eng.check()
  if rank == 0:
    out['bank4541'] = {'workload': 'BASELINE config 4: 1 query x 4541-volume bank sharded over %d GPU(s), shard sizes %s '
                                   '(rank 0 also encodes the query)' % (world, sizes4),
                       'scaling': 'strong', 'pairs_per_s': N_BANK4 * k4 / (ms4 * 1e-3), 'ms_per_query': ms4 / k4,
                       'steps': k4, 'transport': ss4.transport if ss4 else 'single GPU'}

  # ---- config 5: all-pairs 4541 x 4541 with streamed raw-cloud projection -----------------------------
  # (a) streamed encode: raw clouds from pinned host memory -> H2D -> projection/normals -> leg, 32 per launch
  host_clouds = torch.from_numpy(cloud_batch.points.cpu().numpy()).pin_memory()
  offs_dev = cloud_batch.offsets
  offs_host = cloud_batch.offsets_host
  stage = torch.empty_like(cloud_batch.points)

  def encode32(i):
    stage.copy_(host_clouds, non_blocking=True)
    eng.leg(eng.preprocess(CloudBatch(stage, offs_dev, offs_host)))
  ms_enc = timed(encode32, 5, 2) / 5
  # (b) rows of the ordered pair matrix: every rank holds the whole bank (one all_gather in a real run;
  #     here the shards are re-generated locally) and scores ROWS rows against all 4541 volumes
  eng.bank_release(None)
  del big
  torch.cuda.empty_cache()
  full = rolled_bank(eng, fv_src, N_BANK4, dev)
  eng.bank_prepare(full)
  rows = 2
  r_lo = shard_range(N_BANK4, rank, world)[0]

  def rows_step(i):
    eng.heads_rows_vs_bank(full, r_lo, r_lo + rows)
  ms_rows = timed(rows_step, 3, 1) / 3
  eng.check()
  t_ag = None
  lo, hi = shard_range(N_BANK4, rank, world)
  if world > 1:
    shard = full[lo:hi].contiguous()
    pad = torch.zeros((shard_range(N_BANK4, 0, world)[1],) + tuple(shard.shape[1:]), dtype=shard.dtype, device=dev)
    pad[:shard.shape[0]] = shard
    parts = [torch.empty_like(pad) for _ in range(world)]

    def ag(i):
      dist.all_gather(parts, pad)
    t_ag = timed(ag, 3, 1) / 3
    del parts, pad, shard
  if rank == 0:
    per_rank_rows = (N_BANK4 + world - 1) // world
    t_rows_full = per_rank_rows * (ms_rows / rows) * 1e-3
    t_enc_full = (per_rank_rows / cloud_batch.n) * ms_enc * 1e-3
    t_full = t_enc_full + (t_ag or 0) * 1e-3 + t_rows_full
    out['all_pairs'] = {
        'workload': 'BASELINE config 5: ordered all-pairs 4541 x 4541 on %d GPU(s), raw clouds streamed from pinned host memory' % world,
        'measured': {'rows_per_rank': rows, 'ms_per_row_of_4541_pairs': ms_rows / rows,
                     'pairs_per_s': world * rows * N_BANK4 / (ms_rows * 1e-3),
                     'streamed_encode_ms_per_32_scans': ms_enc,
                     'streamed_encode_scans_per_s': world * cloud_batch.n / (ms_enc * 1e-3),
                     'streamed_encode_h2d_bytes_per_scan': int(cloud_batch.points.numel() * 4 // cloud_batch.n),
                     'bank_all_gather_ms': t_ag},
        'projected_full_matrix_s': t_full,
        'projection_note': 'full run = %d rows per rank x measured row time + %d streamed encodes per rank + one all_gather; '
                           'only %d rows per rank are executed here to keep the default bench run short'
                           % (per_rank_rows, per_rank_rows, rows)}
  eng.bank_release(None)
  return out


if __name__ == '__main__':
  main()
