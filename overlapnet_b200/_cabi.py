"""ctypes binding of include/ovn_b200.h.  The product path has NO CPU fallback: if the shared
library is missing or a call fails, an exception is raised."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libovn_b200.so')

OVN_ABI_VERSION = 1
PREC_FP32 = 0
PREC_F16_TC = 1

# every symbol include/ovn_b200.h declares (tests/test_cabi.py checks the .so exports them all)
SYMBOLS = [
    'ovn_default_config', 'ovn_create', 'ovn_destroy', 'ovn_last_error', 'ovn_status_string',
    'ovn_abi_version', 'ovn_input_channels', 'ovn_feature_width', 'ovn_feature_channels',
    'ovn_launch_count', 'ovn_profile_enable', 'ovn_profile_read', 'ovn_set_weights', 'ovn_finalize_weights', 'ovn_project_batch',
    'ovn_normals_batch', 'ovn_semantic_batch', 'ovn_gt_range_batch', 'ovn_gt_overlap_count', 'ovn_preprocess_batch',
    'ovn_pack_input',
    'ovn_leg_forward', 'ovn_heads_forward', 'ovn_heads_1vsN', 'ovn_bank_prepare', 'ovn_bank_release', 'ovn_encode_clouds_host',
    'ovn_query_cloud_vs_bank_host', 'ovn_check', 'ovn_set_feature_center', 'ovn_get_feature_center',
    'ovn_heads_rows_vs_bank', 'ovn_calibrate', 'ovn_peer_signal', 'ovn_peer_wait',
    'ovn_heads_backward', 'ovn_get_gradient', 'ovn_adagrad_step', 'ovn_get_weights',
    'ovn_network_backward', 'ovn_gt_pair_counts',
]


class OvnConfig(C.Structure):
  _fields_ = [
      ('abi_version', C.c_int32),
      ('proj_H', C.c_int32), ('proj_W', C.c_int32),
      ('fov_up_deg', C.c_float), ('fov_down_deg', C.c_float), ('max_range', C.c_float),
      ('use_depth', C.c_int32), ('use_normals', C.c_int32), ('n_prob_channels', C.c_int32),
      ('use_intensity', C.c_int32),
      ('strides_layer1', C.c_int32 * 2),
      ('additional_unsymmetric_layer3a', C.c_int32),
      ('leg_output_width', C.c_int32),
      ('conv1size', C.c_int32),
      ('precision', C.c_int32),
      ('max_batch_scans', C.c_int32), ('max_batch_pairs', C.c_int32),
  ]


class OvnError(Exception):
  """Raised for any non-zero ovn_status (plain Exception subclass, like the reference's errors)."""


_lib = None


def lib():
  """Load libovn_b200.so (built in-tree by overlapnet_b200.build).  Fails loudly when absent."""
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.exists(LIB_PATH):
    raise OvnError('libovn_b200.so is not built: run `python -m overlapnet_b200.build` '
                   '(there is no CPU fallback for the CUDA path)')
  L = C.CDLL(LIB_PATH)
  vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
  L.ovn_default_config.argtypes = [C.POINTER(OvnConfig)]
  L.ovn_default_config.restype = None
  L.ovn_create.argtypes = [C.POINTER(OvnConfig), C.POINTER(vp)]
  L.ovn_destroy.argtypes = [vp]
  L.ovn_last_error.argtypes = [vp]
  L.ovn_last_error.restype = C.c_char_p
  L.ovn_status_string.argtypes = [C.c_int]
  L.ovn_status_string.restype = C.c_char_p
  L.ovn_abi_version.restype = C.c_int
  for f in ('ovn_input_channels', 'ovn_feature_width', 'ovn_feature_channels'):
    getattr(L, f).argtypes = [vp]
  L.ovn_launch_count.argtypes = [vp]
  L.ovn_launch_count.restype = i64
  L.ovn_profile_enable.argtypes = [vp, C.c_int]
  L.ovn_profile_read.argtypes = [vp, C.c_char_p, C.POINTER(C.c_double), C.POINTER(i64)]
  L.ovn_set_weights.argtypes = [vp, C.c_char_p, vp, C.POINTER(i64), i32, vp, i64]
  L.ovn_finalize_weights.argtypes = [vp]
  L.ovn_project_batch.argtypes = [vp, vp, vp, i32, i64, f32, vp, vp, vp, vp, vp]
  L.ovn_normals_batch.argtypes = [vp, vp, vp, i32, vp, vp]
  L.ovn_gt_range_batch.argtypes = [vp, vp, vp, i32, i64, vp, vp, f32, vp, vp]
  L.ovn_gt_overlap_count.argtypes = [vp, vp, vp, i32, vp, vp]
  L.ovn_gt_pair_counts.argtypes = [vp, vp, vp, i32, i64, vp, vp, vp, i32, vp, i64, f32, vp, vp]
  L.ovn_semantic_batch.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp]
  L.ovn_preprocess_batch.argtypes = [vp, vp, vp, i32, i64, vp, vp, vp]
  L.ovn_pack_input.argtypes = [vp, vp, vp, vp, vp, i32, vp, vp]
  L.ovn_leg_forward.argtypes = [vp, vp, i32, vp, vp]
  L.ovn_heads_forward.argtypes = [vp, vp, i64, vp, vp, i32, vp, vp, vp, vp]
  L.ovn_heads_1vsN.argtypes = [vp, vp, i64, vp, vp, i32, vp, vp, vp, vp]
  L.ovn_bank_prepare.argtypes = [vp, vp, i64, i64, i64, vp]
  L.ovn_heads_rows_vs_bank.argtypes = [vp, vp, i64, i64, i64, vp, vp, vp]
  L.ovn_bank_release.argtypes = [vp, vp]
  L.ovn_check.argtypes = [vp, vp]
  L.ovn_set_feature_center.argtypes = [vp, vp]
  L.ovn_get_feature_center.argtypes = [vp, vp, C.POINTER(i32)]
  L.ovn_calibrate.argtypes = [vp, vp, vp]
  L.ovn_peer_signal.argtypes = [vp, vp, i32, i32, vp]
  L.ovn_peer_wait.argtypes = [vp, vp, i32, i32, i32, vp]
  L.ovn_heads_backward.argtypes = [vp, vp, i64, vp, vp, i32, vp, vp, f32, vp, vp]
  L.ovn_get_gradient.argtypes = [vp, C.c_char_p, vp, vp]
  L.ovn_adagrad_step.argtypes = [vp, f32, vp]
  L.ovn_get_weights.argtypes = [vp, C.c_char_p, vp, vp]
  L.ovn_network_backward.argtypes = [vp, vp, i64, vp, vp, vp, i32, vp, vp, f32, vp, vp]
  L.ovn_encode_clouds_host.argtypes = [vp, vp, vp, i32, vp]
  L.ovn_query_cloud_vs_bank_host.argtypes = [vp, vp, i64, vp, i64, vp, i32, vp, vp, vp]
  _lib = L
  return L


def check(handle, status, what=''):
  if status != 0:
    L = lib()
    msg = L.ovn_last_error(handle).decode(errors='replace') if L.ovn_last_error(handle) else ''
    raise OvnError('%s failed: %s (%s)' % (what or 'ovn call', L.ovn_status_string(status).decode(), msg))
