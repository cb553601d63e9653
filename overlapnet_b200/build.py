"""In-tree build of libovn_b200.so (nvcc, sm_100a only).  The built .so is git-ignored but ships
with the repo snapshot to the GPU box; nothing is JIT-compiled at import time."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libovn_b200.so')
PROBE = os.path.join(HERE, 'umma_probe')
SOURCES = ['api.cu', 'projection.cu', 'gt_overlap.cu', 'network_fp32.cu', 'network_tc.cu', 'train.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC'] + os.environ.get('OVN_NVCC_EXTRA', '').split()      # e.g. -DOVN_K4_ROT=0 for A/B timing


def _newer(target, deps):
  if not os.path.exists(target):
    return True
  t = os.path.getmtime(target)
  return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
  """Compile every CUDA source for sm_100a into overlapnet_b200/libovn_b200.so."""
  nvcc = os.environ.get('NVCC', 'nvcc')
  srcs = [os.path.join(CSRC, s) for s in SOURCES]
  deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h'))]
  deps.append(os.path.join(HERE, '..', 'include', 'ovn_b200.h'))
  if force or _newer(LIB, deps):
    # one object per translation unit, compiled in parallel, then linked
    objdir = os.path.join(HERE, 'build')
    os.makedirs(objdir, exist_ok=True)
    hdrs = [d for d in deps if d not in srcs]

    def compile_one(src):
      obj = os.path.join(objdir, os.path.basename(src)[:-3] + '.o')
      if force or _newer(obj, [src] + hdrs):
        cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas=-v'] if verbose else []) + ['-c', '-o', obj, src]
        if verbose:
          print(' '.join(cmd), file=sys.stderr)
        subprocess.check_call(cmd)
      return obj

    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:
      objs = list(ex.map(compile_one, srcs))
    subprocess.check_call([nvcc] + NVCC_FLAGS + ['-shared', '-o', LIB] + objs)
  # standalone known-answer / rate probes of the tcgen05 building blocks (tools, not linked into the library)
  for name in ('umma_probe', 'cta2_probe', 'ss_rate_probe'):
    probe_src, probe_bin = os.path.join(CSRC, name + '.cu'), os.path.join(HERE, name)
    if os.path.exists(probe_src) and (force or _newer(probe_bin, [probe_src] + deps)):
      subprocess.check_call([nvcc] + NVCC_FLAGS + ['-o', probe_bin, probe_src])
  return LIB


if __name__ == '__main__':
  print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
