"""overlapnet_b200 -- Blackwell-native (sm_100a) OverlapNet inference hot path.

Public surface mirrors the reference (PRBonn/OverlapNet):
  Infer                         src/two_heads/infer.py:22
  range_projection, gen_normal_map, gen_*_data   src/utils/utils.py, src/utils/gen_*_data.py
  com_overlap_yaw               src/utils/com_overlap_yaw.py:10
  normalize_data, split_train_val   src/utils/normalize_data.py:10, split_train_val.py:10
Everything computes through hand-written CUDA kernels behind the C ABI in include/ovn_b200.h;
there is no CPU fallback.
"""
from .config import load_config  # noqa: F401


def __getattr__(name):
  # lazy: importing the package must not require torch+CUDA (the C-ABI symbol test runs on CPU)
  if name == 'Infer':
    from .infer import Infer
    return Infer
  if name == 'Trainer':
    from .train import Trainer
    return Trainer
  if name == 'Engine':
    from .engine import Engine
    return Engine
  if name in ('range_projection', 'gen_normal_map', 'gen_depth_data', 'gen_normal_data',
              'gen_intensity_data', 'gen_semantic_data'):
    from . import preprocess
    return getattr(preprocess, name)
  if name in ('com_overlap_yaw', 'com_overlap_yaw_sequence', 'overlap_yaw_sequence', 'normalize_data',
              'split_train_val', 'load_poses', 'load_calib', 'euler_angles_from_rotation_matrix'):
    from . import gt
    return getattr(gt, name)
  raise AttributeError(name)
