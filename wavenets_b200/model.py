"""WaveNet — B200-native stand-in for the reference Keras model (training pass).

Mirrors /root/reference/src/model.py: constructor kwargs and validation (:14-70), dilation
schedule and receptive field (:79-81,122), `build` (:171-211), `call` (:213-239),
`train_step` / `test_step` (:309-391, up to and including the gradients), `prepare_target`
(:151-155), `compute_receptive_field` (:553-556).  The arithmetic runs in libwavenet_b200.so;
torch holds device buffers, streams and (multi-GPU) the NCCL process group.

`generate` uses per-conv input histories (the fast single-step form of layers.py:226-290); observability
(callbacks, TensorBoard) stays out of scope (SURVEY.md section 8).
"""
from __future__ import annotations

import ctypes as C
import math
import warnings
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._engine import Handle, as_dev
from .layers import WaveNetLayer  # noqa: F401  (re-export, like `from src.layers import WaveNetLayer`)
from .metrics import Mean


class _PendingLogs:
  """Metrics of one deferred training step (see WaveNet.train_step_deferred)."""

  def __init__(self, model, slot, event):
    self._model, self._slot, self._event, self._out = model, slot, event, None

  def result(self):
    if self._out is None:
      self._event.synchronize()
      m = self._model
      self._out = m._logs_from_values(m._pin_logs[self._slot].tolist(), train=True)
    return self._out


class _RawView:
  """Zero-copy view of `n` fp32 values at a device address owned by the C library."""

  def __init__(self, ptr: int, n: int):
    self.__cuda_array_interface__ = {'shape': (n,), 'typestr': '<f4', 'data': (ptr, False), 'version': 2, 'strides': None}


class WaveNet:
  """WaveNet model class (same kwargs as the reference)."""

  def __init__(self, kernel_size: int = 2, channels: int = 32, blocks: int = 10, layers_per_block: int = 1,
               activation=None, conditioning=None, mapping_layers=None, mapping_activation=None,
               dropout: float = 0, dilation_bound: int = 512, num_mixtures=None,
               sampling_function: str = 'categorical', bits=8, skip_channels=None, dilation_channels=None,
               use_residual=True, use_skip=True, final_layers_channels=None, l2_reg_factor: int = 0,
               precision: str = 'fp32', device: Optional[int] = None, max_batch: Optional[int] = None,
               max_time: Optional[int] = None, **kwargs):
    # model.py:52-70 (same messages)
    if conditioning not in ['global', 'local', None]:
      raise ValueError("Conditioning must be 'global', 'local' or None.")
    if kernel_size < 2:
      raise ValueError('Kernel size must be at least 2.')
    if math.log(dilation_bound, kernel_size) % 1 != 0:
      raise ValueError('dilation bound must be power of kernel_size.')
    if layers_per_block < 1:
      raise ValueError('Layers per block must be at least 1.')
    if blocks < 1:
      raise ValueError('Blocks must be at least 1.')
    if num_mixtures is not None and num_mixtures < 1:
      raise ValueError('Number of mixtures must be at least 1 or None.')
    if dropout < 0 or dropout > 1:
      raise ValueError('Dropout must be between 0 and 1.')
    if sampling_function not in ['categorical', 'logistic', 'gaussian']:
      raise ValueError('Sampling function must be categorical, logistic or gaussian.')
    if sampling_function == 'categorical' and num_mixtures is not None:
      raise ValueError('Categorical sampling cannot be used with mixtures.')
    if conditioning == 'local':
      # the reference raises at construction too (model.py:137 passes `kernel=` to Conv1D)
      raise NotImplementedError('local conditioning is untested/broken upstream (README.md:13) and not built')
    if final_layers_channels is None:
      raise TypeError("'NoneType' object is not iterable: final_layers_channels must be a list (model.py:111)")
    if mapping_layers is None:
      mapping_layers = []
    elif isinstance(mapping_layers, int):
      mapping_layers = [mapping_layers]
    elif not isinstance(mapping_layers, list):
      raise ValueError('Mapping layers must be a list of integers.')
    if precision not in _lib.PRECISION:
      raise ValueError(f'precision must be one of {sorted(_lib.PRECISION)}')

    self.regularization = l2_reg_factor > 0
    self.l2_reg_factor = l2_reg_factor
    self.num_mixtures = num_mixtures
    self.use_skip = use_skip
    self.use_residual = use_residual
    self.sampling_function = sampling_function
    self.bits = bits
    self.kernel_size = kernel_size
    self.channels = channels
    self.blocks = blocks
    self.layers_per_block = layers_per_block
    self.activation = activation
    self.mapping_layers = list(mapping_layers)
    self.mapping_activation = mapping_activation
    self.dropout = dropout
    self.dilation_bound = dilation_bound
    self.skip_channels = skip_channels
    self.dilation_channels = dilation_channels
    self.final_layers_channels = list(final_layers_channels)
    self.conditioning = conditioning
    self.precision = precision
    self.device_index = torch.cuda.current_device() if (device is None and torch.cuda.is_available()) else (device or 0)
    self._max_batch, self._max_time = max_batch, max_time

    # model.py:79-81: dilations never reach dilation_bound
    max_power = int(math.log(dilation_bound, kernel_size))
    self.dilations = [kernel_size ** (i % max_power) for i in range(layers_per_block * blocks)]
    # model.py:122
    self.receptive_field = 1 + sum(self.dilations) * (kernel_size - 1) + 1

    self._act = _lib.activation_code(activation)
    self._map_act = _lib.activation_code(mapping_activation)
    self.optimizer = None
    self.built = False
    self._handle: Optional[Handle] = None
    self._pending_weights = None
    self._staging = {}
    self._metrics_from_compilation = []
    self.loss_tracker = None          # created by compile(), like model.py:166-168
    self.reg_loss = None
    self.last_step_logs = {}
    self._sample_seed, self._sample_calls = 0x42, 0
    self._pin_logs, self._pin_events, self._pending_slot = None, None, 0
    self._last_frames, self._last_rows = None, 0
    self._last_call = None       # (x, cond, output shape) of the last call: backward() reads them again
    self.n_replicas = 1          # MirroredStrategy replica count (train.py:203); set by parallel.attach()
    self.replica_rank = 0        # this process's replica index: folded into the dropout key (independent masks per replica)
    self._process_group = None   # torch.distributed group (gloo tests / fallback when NCCL cannot be loaded)
    self._comm = None            # (id bytes, nranks, rank) of the NCCL communicator living inside the C library
    self._dropout_seed = 0x243F6A8885A308D3
    self._ar_fused = False

  # ------------------------------------------------------------------ compile (model.py:157-169)
  def compile(self, **kwargs):
    if 'loss' in kwargs:
      raise ValueError('Loss must be set in the model init function.')
    self.optimizer = kwargs.get('optimizer', None)
    self._metrics_from_compilation = list(kwargs.get('metrics') or [])
    # model.py:166-168: running means over the steps since the last reset_metrics() (Keras `fit` resets them every epoch);
    # what train_step / test_step of a COMPILED model report as 'loss' / 'reg_loss'
    self.loss_tracker = Mean(name='loss')
    self.reg_loss = Mean(name='reg_loss') if self.regularization else None
    if self.optimizer is not None and self.built and hasattr(self.optimizer, 'build'):
      self.optimizer.build(self)

  # ------------------------------------------------------------------ build (model.py:171-211)
  def build(self, input_shape):
    if self.conditioning == 'global':
      x_shape, cond_shape = input_shape
      cond_in = int(cond_shape[-1])
    else:
      x_shape, cond_in = input_shape, 0
    x_shape = tuple(x_shape)
    B = int(self._max_batch or x_shape[0])
    T = int(self._max_time or x_shape[1])
    cfg = _lib.WnConfig()
    cfg.kernel_size = self.kernel_size
    cfg.channels = self.channels
    cfg.blocks = self.blocks
    cfg.layers_per_block = self.layers_per_block
    cfg.activation = self._act
    cfg.conditioning = 1 if self.conditioning == 'global' else 0
    cfg.n_mapping = len(self.mapping_layers)
    for i, m in enumerate(self.mapping_layers):
      cfg.mapping_layers[i] = m
    cfg.mapping_activation = self._map_act
    cfg.cond_in = cond_in
    cfg.dilation_bound = self.dilation_bound
    cfg.num_mixtures = 0 if self.num_mixtures is None else self.num_mixtures
    cfg.sampling_function = _lib.SAMPLING[self.sampling_function]
    cfg.bits = self.bits
    cfg.skip_channels = 0 if self.skip_channels is None else self.skip_channels
    cfg.dilation_channels = 0 if self.dilation_channels is None else self.dilation_channels
    cfg.use_residual = 1 if self.use_residual else 0
    cfg.use_skip = 1 if self.use_skip else 0
    cfg.n_final = len(self.final_layers_channels)
    for i, m in enumerate(self.final_layers_channels):
      cfg.final_layers_channels[i] = m
    cfg.l2_reg_factor = float(self.l2_reg_factor)
    cfg.dropout = float(self.dropout)
    cfg.n_dilations = 0
    cfg.has_input_conv = 1
    cfg.has_head = 1
    cfg.precision = _lib.PRECISION[self.precision]
    cfg.max_batch = B
    cfg.max_time = T
    cfg.device = self.device_index
    old, old_opt = None, None
    if self._handle is not None:
      # a rebuild (larger batch / longer segments than the workspace was sized for) moves every device buffer: views handed
      # out earlier (trainable_variables, handle.flat_grads, ...) die with the old handle; weights and Adam's state move over
      warnings.warn(f'wavenets_b200: workspace rebuilt for (batch, time) = ({B}, {T}); device views of the previous handle '
                    '(trainable_variables, flat_grads, flat_params) are invalid now — pass max_batch / max_time to size it once')
      old = self._handle.get_weights()
      opt = self.optimizer
      if opt is not None and getattr(opt, '_handle', None) is self._handle:
        m, v, step = C.c_void_p(), C.c_void_p(), C.c_int64()
        _lib.check(self._handle.lib.wn_adam_state(self._handle.h, C.byref(m), C.byref(v), None, C.byref(step)))
        n = self._handle.n_scalars
        torch.cuda.synchronize(self._handle.device)
        old_opt = (torch.as_tensor(_RawView(m.value, n), device=self._handle.device).clone(),
                   torch.as_tensor(_RawView(v.value, n), device=self._handle.device).clone(), int(step.value))
      self._handle.close()
      self._staging = {}
    self._handle = Handle(cfg)
    self._ar_fused = False
    assert self._handle.lib.wn_receptive_field(self._handle.h) == self.receptive_field
    if self.dropout > 0:
      # tf.distribute draws independent dropout masks on every replica: the replica index is part of the Philox key
      _lib.check(self._handle.lib.wn_set_dropout_seed(self._handle.h, C.c_uint64((self._dropout_seed + self.replica_rank) & (2 ** 64 - 1))))
    if self._comm is not None:
      self._init_comm(*self._comm)
    if old is not None:
      self._handle.set_weights(old)
    elif self._pending_weights is not None:
      self._handle.set_weights(self._pending_weights)
      self._pending_weights = None
    else:
      self._handle.glorot_init(seed=1, bias_std=0.0)   # Keras defaults: glorot-uniform, zero bias
    self.built = True
    self._built_for = (B, T)
    if self._pin_logs is None:
      self._pin_logs = [torch.zeros(4, dtype=torch.float32).pin_memory() for _ in range(4)]
      self._pin_events = [torch.cuda.Event() for _ in range(4)]
    if self.optimizer is not None and hasattr(self.optimizer, 'build'):
      self.optimizer.build(self)      # model.py:211
      if old_opt is not None:
        h = self._handle
        _lib.check(h.lib.wn_adam_restore(h.h, h.ptr(old_opt[0]), h.ptr(old_opt[1]), old_opt[2]))

  def _init_comm(self, id_bytes: bytes, nranks: int, rank: int):
    """NCCL communicator of the replicas inside the C library (wn_comm_init): the gradient all-reduce of MirroredStrategy
    (train.py:203, model.py:336) then runs behind the C ABI (wn_allreduce_grads)."""
    h = self._handle
    buf = (C.c_uint8 * 128).from_buffer_copy(id_bytes)
    _lib.check(h.lib.wn_comm_init(h.h, buf, int(nranks), int(rank)))

  def _ensure_built(self, x, cond):
    B, T = int(x.shape[0]), int(x.shape[1])
    if not self.built or B > self._built_for[0] or T > self._built_for[1]:
      if self.built:
        self._max_batch = max(B, self._built_for[0])
        self._max_time = max(T, self._built_for[1])
      self.build((x.shape, cond.shape) if self.conditioning == 'global' else x.shape)

  # ------------------------------------------------------------------ weights
  @property
  def handle(self) -> Handle:
    if self._handle is None:
      raise ValueError('Model is not built')
    return self._handle

  @property
  def trainable_variables(self):
    """Zero-copy device views in Keras tracking order and layouts."""
    h = self.handle
    return [h.param(i) for i in range(h.n_params)]

  @property
  def variable_names(self):
    return list(self.handle.names)

  def get_weights(self):
    return self.handle.get_weights()

  def set_weights(self, weights):
    if self._handle is None:
      self._pending_weights = dict(weights)
    else:
      self._handle.set_weights(weights)

  def get_grads(self):
    return self.handle.get_grads()

  # ------------------------------------------------------------------ dropout (layers.py:109-112,195-196)
  def set_dropout_masks(self, keep_masks):
    """Inject per-block keep-masks, each (B,T,channels) bool, for the next training steps (parity runs:
    TF's dropout RNG stream cannot be reproduced).  None returns to the built-in Philox masks."""
    h = self.handle
    if keep_masks is None:
      _lib.check(h.lib.wn_set_dropout_masks(h.h, None, 1, 1))
      return
    if len(keep_masks) != self.blocks:
      raise ValueError('one keep-mask per block expected')
    B, T = keep_masks[0].shape[0], keep_masks[0].shape[1]
    a = np.ascontiguousarray(np.stack([np.asarray(k).reshape(B, T, self.channels) for k in keep_masks]).astype(np.uint8))
    _lib.check(h.lib.wn_set_dropout_masks(h.h, a.ctypes.data_as(C.c_void_p), B, T))

  def set_dropout_seed(self, seed: int):
    """Base seed of the dropout masks; every replica adds its rank (independent masks per replica, like tf.distribute)."""
    self._dropout_seed = int(seed)
    if self._handle is not None:
      h = self.handle
      _lib.check(h.lib.wn_set_dropout_seed(h.h, C.c_uint64((self._dropout_seed + self.replica_rank) & (2 ** 64 - 1))))

  # ------------------------------------------------------------------ call (model.py:213-239)
  def _unpack(self, inputs):
    if self.conditioning == 'global':
      x, cond = inputs
    else:
      x, cond = inputs, None
    return x, cond

  def call(self, inputs, training=False):
    x, cond = self._unpack(inputs)
    dev = torch.device('cuda', self.device_index)
    x = as_dev(x, dev)
    if x.dim() == 3:
      if x.shape[2] != 1:
        raise ValueError('input must be (batch, samples, 1)')
      x2 = x[:, :, 0].contiguous()
    else:
      x2 = x
    cond = as_dev(cond, dev) if cond is not None else None
    self._ensure_built(x2, cond)
    h = self.handle
    B, T = x2.shape
    cout = 3 * self.num_mixtures if self.num_mixtures is not None else 2 ** self.bits
    out = torch.empty((B, T, cout), dtype=torch.float32, device=dev)
    self._last_call = None
    # training=True: Keras runs the blocks' Dropout layers (layers.py:195-196) — fresh masks per call
    _lib.check(h.lib.wn_forward_ex(h.h, h.ptr(x2), h.ptr(cond), B, T, 1 if training else 0, h.ptr(out), h.stream_ptr()))
    self._last_call = (x2, cond, (B, T, cout), tuple(x.shape))
    return out

  __call__ = call

  def backward(self, dpred, input_grad=False, param_grads=True):
    """Gradients of the last `call` for a loss the caller computes on its output (tf.GradientTape over model(inputs),
    then tape.gradient(loss, model.trainable_variables)).  `dpred` (B, T, C) = d loss / d pred, pred being what `call`
    returned (probabilities or mixture parameters).  The gradients land in `get_grads()` / `handle.flat_grads` as after
    `train_step`: clipped per replica when the optimizer has clipnorm, then summed over the replicas, ready for
    `optimizer.apply_gradients(model)`; no L2 term (model.py:331-334 belongs to train_step, not to call).  Returns
    d loss / d cond ((B, cond_in) tensor), or None without conditioning.  Anything that changes the weights, the
    activations or the dropout masks (train_step, generate, set_weights, optimizer.apply_gradients, ...) between the
    call and this one makes it raise.

    input_grad=True also gives d loss / d x (tape.gradient(loss, x)) and returns (dx, dcond): dx has the shape of the
    waveform passed to `call`, (B, T, 1) or (B, T), and is this replica's own (never reduced).  param_grads=False computes
    no parameter gradient at all (a frozen model used as a differentiable function of its input): `get_grads()` keeps what
    it held, and no clipnorm or all-reduce runs.  It needs something to compute: input_grad=True or conditioning."""
    last = self._last_call
    if last is None:
      raise RuntimeError('backward needs a preceding call on this model')
    x2, cond, shape, x_shape = last
    if not param_grads and not input_grad and cond is None:
      raise ValueError('backward(param_grads=False) needs input_grad=True or a conditioned model: nothing to compute')
    h = self.handle
    dpred = as_dev(dpred, h.device)
    if tuple(dpred.shape) != shape:
      raise ValueError(f'dpred must have the shape {shape} of the last call output, got {tuple(dpred.shape)}')
    if dpred.data_ptr() % 16:
      dpred = dpred.clone()
    dcond = torch.empty((shape[0], int(cond.shape[-1])), dtype=torch.float32, device=h.device) if cond is not None else None
    dx = torch.empty(shape[:2], dtype=torch.float32, device=h.device) if input_grad else None
    _lib.check(h.lib.wn_backward_ex(h.h, h.ptr(dpred), h.ptr(dcond), h.ptr(dx), 1 if param_grads else 0, h.stream_ptr()))
    if param_grads:
      # the library reduces inside wn_train_step only (wn_comm_fuse_allreduce): here the all-reduce always follows
      self._reduce_grads(allreduce_done=False)
    if input_grad:
      return dx.reshape(x_shape), dcond
    return dcond

  # ------------------------------------------------------------------ targets (model.py:151-155)
  def prepare_target(self, x):
    if self.num_mixtures is not None:
      return x
    dev = torch.device('cuda', self.device_index)
    xt = as_dev(x, dev)
    idx = torch.empty(xt.shape, dtype=torch.int64, device=dev)
    lib = _lib.load()
    _lib.check(lib.wn_quantize(C.c_void_p(xt.data_ptr()), C.c_void_p(idx.data_ptr()), xt.numel(), self.bits,
                               C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return idx

  # ------------------------------------------------------------------ steps (model.py:309-391)
  def _stage(self, name, src, shape, dev):
    """Host input -> persistent device staging buffer (fixed address, so the captured step graph is
    replayed instead of being re-captured for every fresh allocation); device input -> used in place."""
    if isinstance(src, torch.Tensor) and src.is_cuda:
      t = src.detach()
      if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.to(dtype=torch.float32).contiguous()
      return t.reshape(shape)
    t = src.detach() if isinstance(src, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(src, dtype=np.float32)))
    buf = self._staging.get(name)
    if buf is None or tuple(buf.shape) != tuple(shape) or buf.device != dev:
      buf = torch.empty(shape, dtype=torch.float32, device=dev)
      self._staging[name] = buf
    buf.copy_(t.reshape(shape), non_blocking=True)
    return buf

  def _step(self, data, train: bool):
    x, cond = self._unpack(data) if self.conditioning == 'global' else (data, None)
    if not torch.cuda.is_available():
      raise RuntimeError('wavenets_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
    dev = torch.device('cuda', self.device_index)
    if len(x.shape) == 3 and x.shape[2] != 1:
      raise ValueError('input must be (batch, samples, 1)')
    B, T = int(x.shape[0]), int(x.shape[1]) - 1
    frames = self._stage('frames', x, (B, T + 1), dev)
    cond = self._stage('cond', cond, (B, int(cond.shape[-1])), dev) if cond is not None else None
    self._ensure_built(frames[:, :-1], cond)
    h = self.handle
    self._last_frames, self._last_rows = frames, B * T
    fn = h.lib.wn_train_step if train else h.lib.wn_test_step
    if train and self._comm is not None:
      # nothing runs between backward and all-reduce unless the optimizer clips per replica first
      fuse = not (self.optimizer is not None and getattr(self.optimizer, 'clipnorm', None))
      if fuse != self._ar_fused:
        _lib.check(h.lib.wn_comm_fuse_allreduce(h.h, 1 if fuse else 0))
        self._ar_fused = fuse
    _lib.check(fn(h.h, h.ptr(frames), h.ptr(cond), B, T, self.n_replicas, h.ptr(h._loss), h.stream_ptr()))
    if train:
      # (fused: wn_train_step enqueued the all-reduce behind the backward pass, inside the step graph)
      self._reduce_grads(allreduce_done=self._ar_fused)
    return h._loss[:2]

  def _reduce_grads(self, allreduce_done: bool):
    """What follows the gradients of one replica: per-replica clipnorm (Keras clips on every replica before the sum), then
    MirroredStrategy's gradient all-reduce (SUM: the loss is already divided by the global batch, model.py:328)."""
    h = self.handle
    if self.optimizer is not None and getattr(self.optimizer, 'clipnorm', None):
      self.optimizer.clip(self)
    if self.n_replicas > 1:
      if self._comm is not None:
        if not allreduce_done:
          _lib.check(h.lib.wn_allreduce_grads(h.h, h.stream_ptr()))
      elif self._process_group is not None:
        torch.distributed.all_reduce(h.flat_grads, op=torch.distributed.ReduceOp.SUM, group=self._process_group)

  def train_step(self, data):
    """Forward + loss + backward; gradients land in `get_grads()` / `handle.flat_grads`.
    Returns {'loss': float} like the Keras metrics dict (optimizer/MSE metric: out of scope)."""
    loss = self._step(data, True)
    if self.optimizer is not None:
      self.optimizer.apply_gradients(self)
    return self._metrics_dict(loss)

  def _metrics_dict(self, loss_dev, train=True):
    # model.py:338-348: 'loss' excludes the regulariser, which is reported as 'reg_loss'; every compiled metric is
    # fed (y_true, waveform sampled from this step's predictions)
    mse = None
    if self._metrics_from_compilation:
      h = self.handle
      self._sample_calls += 1
      out_buf = self._stage_like('sample', (self._last_rows,))
      _lib.check(h.lib.wn_sample_last_step(h.h, h.ptr(self._last_frames), 0, C.c_uint64(self._sample_seed + self._sample_calls),
                                           h.ptr(out_buf), h.ptr(h._loss[2:]), h.stream_ptr()))
    vals = loss_dev.tolist() if not self._metrics_from_compilation else self.handle._loss.tolist()
    return self._logs_from_values(vals, train=train)

  def _logs_from_values(self, vals, train):
    """The logs dict of one step from [loss, reg_loss, per-step metric value].  A compiled model reports what Keras does
    (model.py:340-348): the running means of `loss_tracker` / `reg_loss` and of every compiled metric since the last
    `reset_metrics()`; this step's own values stay readable as `last_step_logs`.  Without `compile()` (which the reference
    cannot run at all: its trackers are created there) the dict holds the step's own values."""
    step = {'loss': vals[0]}
    if self.regularization:
      step['reg_loss'] = vals[1]
    out = dict(step)
    if self.loss_tracker is not None:
      self.loss_tracker.update_state(vals[0])
      out['loss'] = self.loss_tracker.result()
      if self.reg_loss is not None:
        if train:                      # (test_step has no regulariser value to feed, model.py:376-389)
          self.reg_loss.update_state(vals[1])
        out['reg_loss'] = self.reg_loss.result()
    for metric in self._metrics_from_compilation:
      metric.update_state(vals[2])
      step[metric.name] = vals[2]
      out[metric.name] = metric.result()
    self.last_step_logs = step
    return out

  @property
  def metrics(self):
    """model.py:350-360: compiled metrics, then the loss trackers."""
    extra = [t for t in (self.loss_tracker, self.reg_loss) if t is not None]
    return list(self._metrics_from_compilation) + extra

  def _stage_like(self, name, shape):
    buf = self._staging.get(name)
    dev = torch.device('cuda', self.device_index)
    if buf is None or tuple(buf.shape) != tuple(shape):
      buf = torch.empty(shape, dtype=torch.float32, device=dev)
      self._staging[name] = buf
    return buf

  def reset_metrics(self):
    for metric in self.metrics:
      metric.reset_state()

  def train_step_async(self, data):
    """Same as train_step without the host read-back: returns a device tensor [loss, reg_loss]."""
    return self._step(data, True)

  def train_step_deferred(self, data):
    """train_step whose metrics are read one call later, the way Keras `fit` fetches its logs asynchronously:
    enqueues the H2D copy of the inputs, the step, the optimizer (if compiled), the metrics and a D2H copy of the
    loss floats into pinned memory, and returns a handle; `handle.result()` waits for THAT step only and returns
    the same dict as `train_step`.  The host never idles the GPU between steps."""
    loss = self._step(data, True)
    if self.optimizer is not None:
      self.optimizer.apply_gradients(self)
    h = self.handle
    if self._metrics_from_compilation:
      self._sample_calls += 1
      out_buf = self._stage_like('sample', (self._last_rows,))
      _lib.check(h.lib.wn_sample_last_step(h.h, h.ptr(self._last_frames), 0, C.c_uint64(self._sample_seed + self._sample_calls),
                                           h.ptr(out_buf), h.ptr(h._loss[2:]), h.stream_ptr()))
    slot = self._pending_slot
    self._pending_slot = (slot + 1) % len(self._pin_logs)
    self._pin_logs[slot].copy_(h._loss, non_blocking=True)
    ev = self._pin_events[slot]
    ev.record(torch.cuda.current_stream(h.device))
    return _PendingLogs(self, slot, ev)

  def test_step(self, data):
    out = self._metrics_dict(self._step(data, False), train=False)
    out.pop('reg_loss', None)     # model.py:384-389: test_step reports the loss and the compiled metrics only
    return out

  def loss_fn(self, target, pred):
    """model.py:505-551 on materialised predictions: `pred` (B,T,C) as `call` returns it (softmax probabilities or mixture
    parameters), `target` as `prepare_target` returns it ((B,T,1) int64 bins, or the waveform for mixtures).  Returns the
    un-reduced (B,T) loss tensor like the reference (train_step applies compute_average_loss to it, model.py:328)."""
    dev = torch.device('cuda', self.device_index)
    pred = as_dev(pred, dev)
    if pred.dim() != 3:
      raise ValueError('pred must be (batch, samples, channels)')
    B, T, Cp = (int(v) for v in pred.shape)
    cout = 3 * self.num_mixtures if self.num_mixtures is not None else 2 ** self.bits
    if Cp != cout:
      raise ValueError(f'pred has {Cp} channels, the model predicts {cout}')
    is_idx = False
    if isinstance(target, torch.Tensor):
      is_idx = not target.dtype.is_floating_point
    else:
      target = np.asarray(target)
      is_idx = target.dtype.kind in 'iu'
    if is_idx and self.num_mixtures is not None:
      raise ValueError('mixture losses take the waveform itself as target (model.py:155)')
    tgt = as_dev(target, dev, dtype=torch.int64 if is_idx else torch.float32).reshape(-1)
    if tgt.numel() != B * T:
      raise ValueError('target must hold one value per (batch, sample)')
    if not self.built:
      raise ValueError('Model is not built')
    h = self.handle
    out = torch.empty((B, T), dtype=torch.float32, device=dev)
    _lib.check(h.lib.wn_loss_fn(h.h, h.ptr(tgt), 1 if is_idx else 0, h.ptr(pred), B, T, h.ptr(out), h.stream_ptr()))
    return out

  def compute_receptive_field(self, sampling_frequency):
    return self.receptive_field / sampling_frequency

  def sample_waveform(self, inputs, deterministic=False, seed=None):
    """model.py:393-503 on a `call` output (probabilities or mixture parameters), (B,T,C) -> (B,T,1)
    ((B,T) for deterministic categorical, like the reference).  Stochastic draws use a Philox stream keyed by
    `seed` (TF's stateless seed-(4,2) stream cannot be reproduced: statistical parity)."""
    dev = torch.device('cuda', self.device_index)
    pred = as_dev(inputs, dev)
    if pred.dim() != 3:
      raise ValueError('pred must be (batch, samples, channels)')
    B, T = int(pred.shape[0]), int(pred.shape[1])
    h = self.handle
    out = torch.empty((B, T), dtype=torch.float32, device=dev)
    if seed is None:
      self._sample_calls += 1
      seed = self._sample_seed + self._sample_calls
    _lib.check(h.lib.wn_sample_waveform(h.h, h.ptr(pred), B, T, 1 if deterministic else 0, C.c_uint64(int(seed)), h.ptr(out), h.stream_ptr()))
    if deterministic and self.num_mixtures is None:
      return out
    return out.unsqueeze(-1)

  def generate(self, length, batch_size: int = 1, condition=None, sample=None, use_queues=True, deterministic=False, seed=None):
    """model.py:258-307 with the per-layer single-step form (layers.py:226-290): returns (B, length, 1).
    `sample` (B, n, 1) primes the model (the reference uses n = receptive_field; zeros when deterministic, N(0,1)
    noise otherwise).  Histories of every dilated conv's input replace the sliding window, so a new sample costs one
    matrix-vector product per conv instead of a forward pass over the receptive field (`use_queues` is accepted for
    signature compatibility; the windowed loop is not built).  Draws as in `sample_waveform`; upstream's
    `_generation` always samples deterministically (model.py:255) — pass deterministic=True for that."""
    if self.conditioning is not None and condition is None:
      raise ValueError('Conditioning must be provided.')
    dev = torch.device('cuda', self.device_index)
    cond = as_dev(condition, dev) if condition is not None else None
    if cond is not None:
      batch_size = int(cond.shape[0])
    if sample is not None:
      prime = as_dev(sample, dev)
      if cond is not None and int(prime.shape[0]) != batch_size:
        raise ValueError('Condition and sample must have same batch size.')
      batch_size = int(prime.shape[0])
    elif deterministic:
      prime = torch.zeros((batch_size, self.receptive_field, 1), dtype=torch.float32, device=dev)
    else:
      gen = torch.Generator(device=dev)
      gen.manual_seed(42 if seed is None else int(seed))
      prime = torch.randn((batch_size, self.receptive_field, 1), dtype=torch.float32, device=dev, generator=gen)
    prime2 = prime.reshape(batch_size, -1).contiguous()
    if not self.built:
      self.build(((batch_size, prime2.shape[1], 1), cond.shape) if cond is not None else (batch_size, prime2.shape[1], 1))
    h = self.handle
    out = torch.empty((batch_size, int(length)), dtype=torch.float32, device=dev)
    if seed is None:
      self._sample_calls += 1
      seed = self._sample_seed + self._sample_calls
    _lib.check(h.lib.wn_generate(h.h, h.ptr(prime2), int(prime2.shape[1]), h.ptr(cond), batch_size, int(length), 1 if deterministic else 0,
                                 C.c_uint64(int(seed)), h.ptr(out), None, None, h.stream_ptr()))
    return out.unsqueeze(-1)

  def _teacher_forced_step_predictions(self, prime, teacher, condition=None):
    """Test hook: run the generation step teacher-forced on prime ++ teacher and return the predictive distribution of
    every teacher position, (B, len(teacher), C) — must equal `call` on the same waveform."""
    dev = torch.device('cuda', self.device_index)
    p2 = as_dev(prime, dev).reshape(prime.shape[0], -1).contiguous()
    t2 = as_dev(teacher, dev).reshape(teacher.shape[0], -1).contiguous()
    cond = as_dev(condition, dev) if condition is not None else None
    h = self.handle
    cout = 3 * self.num_mixtures if self.num_mixtures is not None else 2 ** self.bits
    pred = torch.empty((p2.shape[0], t2.shape[1], cout), dtype=torch.float32, device=dev)
    _lib.check(h.lib.wn_generate(h.h, h.ptr(p2), int(p2.shape[1]), h.ptr(cond), int(p2.shape[0]), int(t2.shape[1]), 1, C.c_uint64(0),
                                 None, h.ptr(pred), h.ptr(t2), h.stream_ptr()))
    return pred
