"""ctypes binding of libwavenet_b200.so (include/wavenet_b200.h).

There is NO CPU fallback: if the shared library is missing this module raises, and every
compute entry point fails with RuntimeError when no sm_100 GPU is present.
"""
from __future__ import annotations

import ctypes as C
import os

WN_MAX_LIST = 8
WN_MAX_DILATIONS = 512

WN_OK, WN_ERR_VALUE, WN_ERR_UNSUPPORTED, WN_ERR_CUDA, WN_ERR_STATE = 0, -1, -2, -3, -4
ACTIVATIONS = {None: 0, 'linear': 0, 'relu': 1, 'leaky_relu': 2, 'tanh': 3, 'sigmoid': 4}
SAMPLING = {'categorical': 0, 'logistic': 1, 'gaussian': 2}
PRECISION = {'fp32': 0, 'float32': 0, 'bf16': 1, 'bfloat16': 1}

EXPORTS = [
  'wn_create', 'wn_destroy', 'wn_last_error', 'wn_receptive_field', 'wn_dilation', 'wn_num_params',
  'wn_param_count', 'wn_param_info', 'wn_params_dev', 'wn_grads_dev', 'wn_set_param', 'wn_get_param',
  'wn_get_grad', 'wn_params_changed', 'wn_quantize', 'wn_forward', 'wn_train_step', 'wn_test_step',
  'wn_train_step_host', 'wn_layer_forward', 'wn_layer_backward', 'wn_last_launch_count',
  'wn_fused_forward_blocks', 'wn_grouped_wgrad_tiles', 'wn_stack_forward_layers', 'wn_profile_begin', 'wn_profile_end', 'wn_profile_get', 'wn_build_info', 'wn_set_dropout_masks', 'wn_set_dropout_seed', 'wn_layer_forward_ex', 'wn_num_frames', 'wn_preprocess_frames', 'wn_inverse_mu_law', 'wn_one_hot', 'wn_sample_waveform', 'wn_sample_last_step', 'wn_generate', 'wn_adam_init', 'wn_clip_grads', 'wn_adam_step', 'wn_adam_state', 'wn_debug_conv_gemm', 'wn_debug_wgrad', 'wn_debug_bench',
  'wn_forward_ex', 'wn_loss_fn', 'wn_adam_restore', 'wn_nccl_unique_id', 'wn_comm_init', 'wn_comm_attach', 'wn_comm_fuse_allreduce',
  'wn_allreduce_grads', 'wn_nccl_info', 'wn_grouped_wgrad_info', 'wn_debug_tensor', 'wn_stack_backward_layers',
  'wn_allreduce_buckets', 'wn_layer_forward_seq',
]


class WnConfig(C.Structure):
  _fields_ = [
    ('kernel_size', C.c_int32), ('channels', C.c_int32), ('blocks', C.c_int32), ('layers_per_block', C.c_int32),
    ('activation', C.c_int32), ('conditioning', C.c_int32), ('n_mapping', C.c_int32),
    ('mapping_layers', C.c_int32 * WN_MAX_LIST), ('mapping_activation', C.c_int32), ('cond_in', C.c_int32),
    ('dilation_bound', C.c_int32), ('num_mixtures', C.c_int32), ('sampling_function', C.c_int32), ('bits', C.c_int32),
    ('skip_channels', C.c_int32), ('dilation_channels', C.c_int32), ('use_residual', C.c_int32), ('use_skip', C.c_int32),
    ('n_final', C.c_int32), ('final_layers_channels', C.c_int32 * WN_MAX_LIST),
    ('l2_reg_factor', C.c_float), ('dropout', C.c_float),
    ('n_dilations', C.c_int32), ('dilations', C.c_int32 * WN_MAX_DILATIONS),
    ('has_input_conv', C.c_int32), ('has_head', C.c_int32), ('precision', C.c_int32),
    ('max_batch', C.c_int32), ('max_time', C.c_int32), ('device', C.c_int32),
  ]


def lib_path() -> str:
  # WN_LIB selects an alternative build of the same library (another revision from scripts/build_rev.sh, the precise / tl flavours)
  return os.environ.get('WN_LIB') or os.path.join(os.path.dirname(os.path.abspath(__file__)), 'libwavenet_b200.so')


_LIB = None


def load():
  """Load the shared library (build it with `python -m wavenets_b200.build`)."""
  global _LIB
  if _LIB is not None:
    return _LIB
  path = lib_path()
  if not os.path.exists(path):
    raise ImportError(
      f'{path} is missing: build the CUDA extension with `python -m wavenets_b200.build` '
      '(wavenets_b200 has no CPU fallback)')
  lib = C.CDLL(path)
  vp, i32, i64, fp = C.c_void_p, C.c_int, C.c_int64, C.POINTER(C.c_float)
  lib.wn_create.argtypes = [C.POINTER(WnConfig), C.POINTER(vp)]
  lib.wn_destroy.argtypes = [vp]
  lib.wn_destroy.restype = None
  lib.wn_last_error.restype = C.c_char_p
  lib.wn_build_info.restype = C.c_char_p
  lib.wn_receptive_field.argtypes = [vp]
  lib.wn_dilation.argtypes = [vp, i32, i32]
  lib.wn_num_params.argtypes = [vp]
  lib.wn_param_count.argtypes = [vp]
  lib.wn_param_count.restype = i64
  lib.wn_param_info.argtypes = [vp, i32, C.c_char_p, i32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(i64)]
  lib.wn_params_dev.argtypes = [vp]
  lib.wn_params_dev.restype = vp
  lib.wn_grads_dev.argtypes = [vp]
  lib.wn_grads_dev.restype = vp
  lib.wn_set_param.argtypes = [vp, i32, vp]
  lib.wn_get_param.argtypes = [vp, i32, vp]
  lib.wn_get_grad.argtypes = [vp, i32, vp]
  lib.wn_params_changed.argtypes = [vp, vp]
  lib.wn_quantize.argtypes = [vp, vp, i64, i32, vp]
  lib.wn_forward.argtypes = [vp, vp, vp, i32, i32, vp, vp]
  lib.wn_forward_ex.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
  lib.wn_loss_fn.argtypes = [vp, vp, i32, vp, i32, i32, vp, vp]
  lib.wn_adam_restore.argtypes = [vp, vp, vp, i64]
  lib.wn_nccl_unique_id.argtypes = [vp]
  lib.wn_comm_init.argtypes = [vp, vp, i32, i32]
  lib.wn_comm_attach.argtypes = [vp, vp, i32, i32]
  lib.wn_comm_fuse_allreduce.argtypes = [vp, i32]
  lib.wn_allreduce_grads.argtypes = [vp, vp]
  lib.wn_nccl_info.restype = C.c_char_p
  lib.wn_train_step.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
  lib.wn_test_step.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
  lib.wn_train_step_host.argtypes = [vp, vp, vp, i32, i32, i32, vp]
  lib.wn_layer_forward.argtypes = [vp, i32, vp, vp, i32, i32, vp, vp, vp]
  lib.wn_layer_forward_ex.argtypes = [vp, i32, vp, vp, i32, i32, i32, vp, vp, vp]
  lib.wn_layer_forward_seq.argtypes = [vp, i32, vp, vp, i32, i32, i32, vp, vp, vp]
  lib.wn_layer_backward.argtypes = [vp, i32, vp, vp, vp, vp, vp]
  lib.wn_last_launch_count.argtypes = [vp]
  lib.wn_last_launch_count.restype = i64
  lib.wn_fused_forward_blocks.argtypes = [vp]
  lib.wn_grouped_wgrad_tiles.argtypes = [vp, C.POINTER(C.c_int)]
  lib.wn_stack_forward_layers.argtypes = [vp]
  lib.wn_stack_backward_layers.argtypes = [vp]
  lib.wn_allreduce_buckets.argtypes = [vp]
  lib.wn_debug_tensor.argtypes = [vp, C.c_char_p, i32, vp, i64]
  lib.wn_grouped_wgrad_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
  lib.wn_profile_begin.argtypes = [vp, i32]
  lib.wn_profile_end.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(i64)]
  lib.wn_profile_get.argtypes = [vp, i32, C.POINTER(C.c_double), C.c_char_p, i32]
  lib.wn_set_dropout_masks.argtypes = [vp, vp, i32, i32]
  lib.wn_set_dropout_seed.argtypes = [vp, C.c_uint64]
  f32 = C.c_float
  lib.wn_generate.argtypes = [vp, vp, i32, vp, i32, i32, i32, C.c_uint64, vp, vp, vp, vp]
  lib.wn_num_frames.argtypes = [i64, i32]
  lib.wn_num_frames.restype = i64
  lib.wn_preprocess_frames.argtypes = [vp, i32, i64, i32, i32, vp, vp, vp]
  lib.wn_inverse_mu_law.argtypes = [vp, vp, i64, vp]
  lib.wn_one_hot.argtypes = [vp, i32, i32, vp, vp]
  lib.wn_sample_waveform.argtypes = [vp, vp, i32, i32, i32, C.c_uint64, vp, vp]
  lib.wn_sample_last_step.argtypes = [vp, vp, i32, C.c_uint64, vp, vp, vp]
  lib.wn_adam_init.argtypes = [vp, f32, f32, f32, f32, f32]
  lib.wn_clip_grads.argtypes = [vp, vp]
  lib.wn_adam_step.argtypes = [vp, f32, vp]
  lib.wn_adam_state.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(i64)]
  ip = C.POINTER(C.c_int)
  lib.wn_debug_conv_gemm.argtypes = [vp, i32, i32, i32, i32, ip, i32, vp, i32, i32, i32, vp, vp]
  lib.wn_debug_wgrad.argtypes = [vp, i32, vp, i32, i32, i32, i32, ip, i32, i32, vp, vp]
  lib.wn_debug_bench.argtypes = [i32, i32, vp, i32, vp, i32, i32, i32, i32, ip, i32, i32, vp, i32, C.POINTER(C.c_float)]
  _LIB = lib
  return lib


def check(rc: int):
  """Translate C status codes into the reference's Python exceptions."""
  if rc >= 0:
    return rc
  msg = load().wn_last_error().decode('utf-8', 'replace')
  if rc == WN_ERR_VALUE:
    raise ValueError(msg)
  if rc == WN_ERR_UNSUPPORTED:
    raise NotImplementedError(msg)
  raise RuntimeError(f'libwavenet_b200: {msg} (status {rc})')


def activation_code(name):
  if callable(name) and not isinstance(name, str):
    name = getattr(name, '__name__', str(name))
  if name not in ACTIVATIONS:
    raise NotImplementedError(f'activation {name!r} is not built (supported: {sorted(k for k in ACTIVATIONS if k)})')
  return ACTIVATIONS[name]
