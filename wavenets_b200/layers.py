"""WaveNetLayer — B200-native stand-in for the reference Keras layer.

Mirrors /root/reference/src/layers.py: same constructor kwargs (:10-20), `build` (:122-164),
`compute_output_shape` (:166-176) and `call(inputs, training=False) -> (x_out, skip)`
(:178-224), same ValueErrors.  The arithmetic runs in libwavenet_b200.so (`wn_layer_forward` /
`wn_layer_backward`); torch only holds the device buffers.  `generate` (:226-290) is
inference-only and out of scope.

Conditioning (`condition=True`) takes either form the reference accepts: a (B,Cc) vector, or a (B,T,Cc)
sequence that is constant in time, runs as a per-batch bias of the gated conv; a (B,T,Cc) sequence that
varies in time (local conditioning, one feature vector per sample) runs through `wn_layer_forward_seq`,
where conv_cond is one more segment of the gated conv's contraction.  `backward` returns `dcond` in the
shape of the conditioning that ran: (B,Cc) for the time-constant forms, (B,T,Cc) for a sequence.
"""
from __future__ import annotations

from types import SimpleNamespace

import torch

from . import _lib
from ._engine import Handle, as_dev


class WaveNetLayer:
  """WaveNet layer (gated dilated causal conv block with residual and skip outputs)."""

  def __init__(self, kernel=2, dilation_rate=1, activation=None, channels=32, residual=True,
               dilation_channels=None, skip_channels=None, l2_reg_factor=None, condition=False,
               dropout=0, precision='fp32', device=0, **kwargs):
    # layers.py:46-59
    self.l2_reg_factor = 0 if l2_reg_factor is None else l2_reg_factor
    if dilation_channels is None:
      dilation_channels = channels
    if not isinstance(dilation_rate, list):
      dilation_rate = [dilation_rate]
    self.input_dilation = dilation_rate[0]
    self.depth = len(dilation_rate)
    self.kernel_size = kernel
    self.channels = channels
    self.residual = residual
    self.activation = activation
    self.condition = condition
    self.dilation_rates = list(dilation_rate)
    self.dilation_channels = dilation_channels
    self.skip_channels = skip_channels
    self.dropout_rate = dropout
    self.name = kwargs.get('name', 'wave_net_layer')
    # descriptors standing in for the Keras sub-layers (layers.py:64-120)
    self.dilated_stack = [
      SimpleNamespace(filters=dilation_channels, kernel_size=kernel, dilation_rate=d, padding='causal', activation=activation)
      for d in dilation_rate[:-1]]
    self.dilated_stack.append(
      SimpleNamespace(filters=2 * dilation_channels, kernel_size=kernel, dilation_rate=dilation_rate[-1], padding='causal', activation=None))
    self.conv1 = SimpleNamespace(filters=channels, kernel_size=1)
    self.conv_skip = SimpleNamespace(filters=skip_channels, kernel_size=1) if skip_channels is not None else None
    self.dropout = SimpleNamespace(rate=dropout) if dropout > 0 else None
    if condition:
      self.conv_cond = SimpleNamespace(filters=2 * dilation_channels, kernel_size=1)
    self.precision = precision
    self.device_index = device
    self.built = False
    self._handle = None
    self._act_code = _lib.activation_code(activation)
    if precision not in _lib.PRECISION:
      raise ValueError(f'precision must be one of {sorted(_lib.PRECISION)}')

  # ------------------------------------------------------------------ build (layers.py:122-164)
  def build(self, input_shape):
    if self.condition:
      x_shape, cond_shape = input_shape
      if len(cond_shape) == 3 and x_shape[1] != cond_shape[1]:
        raise ValueError('Condition tensor must have the same length as input')
    else:
      x_shape = input_shape
      cond_shape = None
    x_shape = tuple(x_shape)
    if self.residual and x_shape[2] != self.channels:
      # conv1 maps to `channels`; a different input width breaks the residual add (layers.py:161-162)
      raise ValueError('Residual connection must have the same shape as input')
    if x_shape[2] != self.channels:
      raise NotImplementedError('input width != channels is only reachable with residual=False and is not built')
    cfg = _lib.WnConfig()
    cfg.kernel_size = self.kernel_size
    cfg.channels = self.channels
    cfg.blocks = 1
    cfg.layers_per_block = self.depth
    cfg.activation = self._act_code if self.depth > 1 else 0
    cfg.conditioning = 1 if self.condition else 0
    cfg.n_mapping = 0
    cfg.cond_in = int(cond_shape[-1]) if self.condition else 0
    self._cond_in = cfg.cond_in
    cfg.dilation_bound = 1
    cfg.num_mixtures = 0
    cfg.sampling_function = 0
    cfg.bits = 8
    cfg.skip_channels = 0 if self.skip_channels is None else self.skip_channels
    cfg.dilation_channels = self.dilation_channels
    cfg.use_residual = 1 if self.residual else 0
    cfg.use_skip = 1
    cfg.n_final = 0
    cfg.l2_reg_factor = float(self.l2_reg_factor)
    cfg.dropout = float(self.dropout_rate)
    cfg.n_dilations = self.depth
    for i, d in enumerate(self.dilation_rates):
      cfg.dilations[i] = d
    cfg.has_input_conv = 0
    cfg.has_head = 0
    cfg.precision = _lib.PRECISION[self.precision]
    cfg.max_batch = int(x_shape[0])
    cfg.max_time = int(x_shape[1])
    cfg.device = self.device_index
    if self._handle is not None:
      old = self._handle.get_weights()
      self._handle.close()
      self._handle = Handle(cfg)
      self._handle.set_weights(old)
    else:
      self._handle = Handle(cfg)
      self._handle.glorot_init(seed=1, bias_std=0.0)
    skip_ch = self.channels if self.skip_channels is None else self.skip_channels
    x_out_shape = (x_shape[0], x_shape[1], self.channels)
    self.built = True
    self._output_shape = (x_out_shape, (x_shape[0], x_shape[1], skip_ch))
    self._built_for = (int(x_shape[0]), int(x_shape[1]))

  def compute_output_shape(self, input_shape):
    if not self.built:
      raise ValueError('Layer is not built')
    return self._output_shape

  # ------------------------------------------------------------------ weights (Keras layouts)
  _ALIASES = {'dil': 'block0/dil', 'conv1': 'block0/conv1', 'conv_skip': 'block0/conv_skip', 'conv_cond': 'block0/conv_cond'}

  @property
  def weight_names(self):
    return [n[len('block0/'):] for n in self._handle.names]

  def get_weights(self):
    return {n[len('block0/'):]: w for n, w in self._handle.get_weights().items()}

  def set_weights(self, weights):
    self._handle.set_weights({'block0/' + n: w for n, w in weights.items()})

  def get_grads(self):
    return {n[len('block0/'):]: w for n, w in self._handle.get_grads().items()}

  # ------------------------------------------------------------------ dropout (layers.py:109-112,195-196)
  def set_dropout_mask(self, keep):
    """Inject the keep-mask (B,T,channels) bool used by `call(training=True)` and its `backward` (parity runs); None returns
    to fresh Philox masks per call."""
    import ctypes as C
    import numpy as np
    if self.dropout is None:
      raise ValueError('layer was built with dropout == 0')
    if not self.built:
      raise ValueError('Layer is not built')
    h = self._handle
    if keep is None:
      _lib.check(h.lib.wn_set_dropout_masks(h.h, None, 1, 1))
      return
    a = np.ascontiguousarray(np.asarray(keep).astype(np.uint8))
    if a.ndim != 3 or a.shape[2] != self.channels:
      raise ValueError('keep-mask must be (batch, samples, channels)')
    _lib.check(h.lib.wn_set_dropout_masks(h.h, a.ctypes.data_as(C.c_void_p), a.shape[0], a.shape[1]))

  def set_dropout_seed(self, seed: int):
    import ctypes as C
    if self._handle is not None:
      _lib.check(self._handle.lib.wn_set_dropout_seed(self._handle.h, C.c_uint64(int(seed) & (2 ** 64 - 1))))

  # ------------------------------------------------------------------ call (layers.py:178-224)
  def _split_inputs(self, inputs):
    if self.condition:
      x, cond = inputs
    else:
      x, cond = inputs, None
    return x, cond

  def call(self, inputs, training=False):
    x, cond = self._split_inputs(inputs)
    dev = torch.device('cuda', self.device_index)
    x = as_dev(x, dev)
    if x.dim() != 3:
      raise ValueError('input must be (batch, samples, channels)')
    B, T, _ = x.shape
    cond2 = None
    seq = None
    if self.condition:
      cond = as_dev(cond, dev)
      if cond.dim() == 3:
        if cond.shape[1] != T:
          raise ValueError('Condition tensor must have the same length as input')
        if T > 1 and not bool((cond == cond[:, :1, :]).all()):
          # local conditioning: conv_cond(cond) joins the gated conv's pre-activation at every step (layers.py:203-204)
          if self.built and cond.shape[2] != self._cond_in:
            raise ValueError(f'Condition tensor has {cond.shape[2]} channels; the layer was built for {self._cond_in}')
          seq = cond
        else:
          cond2 = cond[:, 0, :].contiguous()
      else:
        cond2 = cond
    if not self.built or (B, T) != self._built_for and (B > self._built_for[0] or T > self._built_for[1]):
      self.build((x.shape, cond.shape) if self.condition else x.shape)
    h = self._handle
    skip_ch = self.channels if self.skip_channels is None else self.skip_channels
    x_out = torch.empty((B, T, self.channels), dtype=torch.float32, device=dev)
    skip = torch.empty((B, T, skip_ch), dtype=torch.float32, device=dev)
    # training=True: inverted dropout on the conv branch, residual from the un-masked input (layers.py:192-196); the keep-mask
    # is a fresh Philox draw unless one was injected with set_dropout_mask (TF's RNG stream is not reproducible)
    drop = 1 if (training and self.dropout is not None) else 0
    if seq is not None:
      _lib.check(h.lib.wn_layer_forward_seq(h.h, 0, h.ptr(x), h.ptr(seq), B, T, drop, h.ptr(x_out), h.ptr(skip), h.stream_ptr()))
      self._last = (x, seq)   # the library reads the sequence again in backward
    else:
      _lib.check(h.lib.wn_layer_forward_ex(h.h, 0, h.ptr(x), h.ptr(cond2), B, T, drop, h.ptr(x_out), h.ptr(skip), h.stream_ptr()))
      self._last = (x, cond2)
    return x_out, skip

  __call__ = call

  def backward(self, dx_out=None, dskip=None):
    """Adjoint of the last `call` (what tf.GradientTape would compute): returns (dx, dcond);
    parameter gradients are available from `get_grads()`."""
    h = self._handle
    dev = h.device
    x, cond2 = self._last
    dxo = None if dx_out is None else as_dev(dx_out, dev)
    dsk = None if dskip is None else as_dev(dskip, dev)
    dx = torch.empty_like(x)
    dcond = torch.empty_like(cond2) if cond2 is not None else None
    _lib.check(h.lib.wn_layer_backward(h.h, 0, h.ptr(dxo), h.ptr(dsk), h.ptr(dx), h.ptr(dcond), h.stream_ptr()))
    return dx, dcond

  def generate(self, inputs):
    raise NotImplementedError('fast-wavenet single-step generation (layers.py:226-290) is inference-only and out of scope')
