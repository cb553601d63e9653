import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
  config.addinivalue_line('markers', 'gpu: needs a real B200 (run with -m gpu on the GPU box)')


def pytest_collection_modifyitems(config, items):
  # GPU tests must never silently pass on a box without CUDA
  try:
    import torch
    has_cuda = torch.cuda.is_available()
  except Exception:
    has_cuda = False
  if not has_cuda:
    skip = pytest.mark.skip(reason='no CUDA device in this container (run under gpurun)')
    for item in items:
      if 'gpu' in item.keywords:
        item.add_marker(skip)


@pytest.fixture(scope='session')
def manifest():
  with open(os.path.join(GOLDEN, 'MANIFEST.json')) as f:
    return json.load(f)


@pytest.fixture(scope='session')
def reference_outputs():
  """What the reference computed on the parity inputs (tools/make_golden_reference.py)."""
  with open(os.path.join(GOLDEN, 'reference_outputs.json')) as f:
    return json.load(f)


def load_golden(name):
  z = np.load(os.path.join(GOLDEN, name + '.npz'))
  return {k: z[k] for k in z.files}


GOLDEN_CASES = ['kitti_000000', 'kitti_000001', 'synth_3', 'synth_5', 'synth_11']


@pytest.fixture(scope='session')
def engine_fp32():
  from overlapnet_b200.engine import Engine
  return Engine(precision='fp32', model={'additional_unsymmetric_layer3a': True, 'strides_layer1': [2, 2]},
                max_batch_scans=8, max_batch_pairs=64)
