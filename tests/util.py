"""Shared helpers for the parity tests: one set of kwargs drives both the oracle and the product."""
import contextlib
import os

import numpy as np

from oracle import wavenet_oracle as wo


def oracle_config(kw: dict, cond_in: int = 0) -> wo.Config:
  return wo.config_from_kwargs(kw, cond_in)


@contextlib.contextmanager
def env_vars(env):
  """sets the environment variables in env (the library reads its switches at wn_create), restores them on exit"""
  old = {k: os.environ.get(k) for k in env}
  os.environ.update(env)
  try:
    yield
  finally:
    for k, v in old.items():
      if v is None:
        os.environ.pop(k, None)
      else:
        os.environ[k] = v


def make_inputs(B, T, cond_in=0, seed=0):
  rng = np.random.default_rng(seed)
  x = np.clip(rng.standard_normal((B, T + 1, 1)) * 0.4, -1, 1).astype(np.float32)
  cond = None
  if cond_in:
    ids = rng.integers(0, cond_in, B)
    cond = np.eye(cond_in, dtype=np.float32)[ids]
  return x, cond


def rel_err(a, b):
  a = np.asarray(a, dtype=np.float64)
  b = np.asarray(b, dtype=np.float64)
  return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


def rel_l2(a, b):
  a = np.asarray(a, dtype=np.float64).ravel()
  b = np.asarray(b, dtype=np.float64).ravel()
  return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))


# small model configurations shared by the CPU oracle tests and the GPU parity tests
SMALL_MODELS = {
  'categorical_multidil': dict(channels=8, blocks=3, layers_per_block=2, activation='leaky_relu', dilation_bound=8,
                               final_layers_channels=[12, 16], bits=8),
  'cond_skip': dict(channels=8, blocks=4, layers_per_block=1, dilation_bound=8, final_layers_channels=[12],
                    skip_channels=6, dilation_channels=10, conditioning='global', mapping_layers=[4, 6],
                    mapping_activation='leaky_relu', activation='relu'),
  'logistic_cond': dict(channels=8, blocks=3, layers_per_block=3, activation='tanh', dilation_bound=4,
                        final_layers_channels=[12], num_mixtures=3, sampling_function='logistic', bits=16,
                        conditioning='global', mapping_layers=[4], mapping_activation='relu'),
  'gaussian_noskip': dict(channels=8, blocks=3, layers_per_block=1, dilation_bound=4, final_layers_channels=[12],
                          num_mixtures=4, sampling_function='gaussian', use_skip=False, skip_channels=5),
  'k3_nores': dict(channels=8, blocks=3, layers_per_block=1, dilation_bound=9, final_layers_channels=[],
                   use_residual=False, kernel_size=3),
  # more mixture components than a half warp: the mixture-loss kernel runs with 32 lanes per row (17, 20 components)
  'logistic_m20': dict(channels=8, blocks=2, layers_per_block=1, dilation_bound=4, final_layers_channels=[16], num_mixtures=20,
                       sampling_function='logistic', bits=16),
  'gaussian_m17': dict(channels=8, blocks=2, layers_per_block=1, dilation_bound=4, final_layers_channels=[16], num_mixtures=17,
                       sampling_function='gaussian'),
  'wide_ragged': dict(channels=40, blocks=2, layers_per_block=2, activation='sigmoid', dilation_bound=4,
                      final_layers_channels=[70], skip_channels=72, dilation_channels=36, bits=8),
  # L2 on convs whose output nothing reads: conv1 of the last block under use_skip, conv_skip without use_skip —
  # their data gradient is zero, the regulariser's is not (model.py:331-334)
  'l2_skip': dict(channels=8, blocks=2, layers_per_block=1, dilation_bound=4, final_layers_channels=[8], l2_reg_factor=0.01, skip_channels=6),
  'l2_unused_skip': dict(channels=8, blocks=2, layers_per_block=1, dilation_bound=4, final_layers_channels=[8], l2_reg_factor=0.01,
                         skip_channels=6, use_skip=False),
  'l2': dict(channels=8, blocks=2, layers_per_block=1, dilation_bound=4, final_layers_channels=[8],
             l2_reg_factor=0.01, conditioning='global', mapping_layers=[4], mapping_activation='tanh'),
}
COND_IN = 5


def device_tensor(model, name, index, B, T, width):
  """An intermediate tensor of the model's last step from the device (wn_debug_tensor), (B,T,width) fp32, or None."""
  import ctypes as C
  h = model.handle
  buf = np.empty(B * T * width, dtype=np.float32)
  w = h.lib.wn_debug_tensor(h.h, name.encode(), index, buf.ctypes.data_as(C.c_void_p), buf.size)
  if w < 0:
    return None
  return buf[:B * T * w].reshape(B, T, w)


def device_slope_masks(model, kw, B, T):
  """Which elements of every relu / leaky_relu output of the model's LAST step sit on the positive branch, read back from the
  device: {('hact', i) | ('act', block, j): bool (B,T,C)} for oracle.faithful.train_step(slope_masks=...).  The derivative of
  a piecewise-linear activation is discontinuous: a pre-activation within one bf16 rounding flip of zero falls on different
  sides in two correct implementations and changes that gradient element five-fold (leaky_relu).  With the masks of the
  implementation under test, its backward arithmetic is compared like for like; its forward values are checked separately."""
  act = kw.get('activation')
  if act not in ('relu', 'leaky_relu'):
    return None
  pos = (lambda y: y > 0) if act == 'relu' else (lambda y: y >= 0)
  masks = {}
  for i, w in enumerate(kw.get('final_layers_channels') or []):
    y = device_tensor(model, 'hact', i, B, T, w)
    if y is not None:
      masks[('hact', i)] = pos(y)
  lpb = kw.get('layers_per_block', 1)
  D = kw.get('dilation_channels') or kw.get('channels', 32)
  for b in range(kw.get('blocks', 10)):
    for j in range(lpb - 1):
      y = device_tensor(model, 'act', 16 * b + j, B, T, D)
      if y is not None:
        masks[('act', b, j)] = pos(y)
  return masks
