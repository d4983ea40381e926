"""Calls smaller than the workspace a handle was built for, on both precision tiers.

A handle sized for (maxB, maxT) addresses every per-layer slab with capacity rows, maxB * maxT (gate outputs, the kept d z /
d x_out slabs, dropout masks; the conditioning biases per maxB), while tensor maps, tile counts, splits and plans follow the
call's (B, T).  The last partial batch of an epoch, a validation set with shorter segments or `call` on a short input all run
in that regime; a call that fills its workspace cannot tell the two row counts apart.  So every case here takes one model
and two handles with the same weights: `big`, built for the workspace, and `exact`, built for the call's (B, T).  Before
the checked calls `big` runs one training step and one `call` at full capacity on other inputs (amplitude near +-1, another
speaker in every row), which leaves stale data in every slab row the smaller call must not read.  At each smaller shape:
  (a) loss, reg_loss, every gradient, `call`'s output and test_step's loss against the float64 oracle (fp32 tier, 1e-4 as in
      test_gpu_parity_fp32.py), or against the bf16-faithful and the float64 oracle (bf16 tier, tolerances of
      test_gpu_parity_bf16.py / test_gpu_configs.py);
  (b) loss, gradients, `call`'s output and the schedule counters bit-equal to `exact`: every split and plan derives from
      the call's (B, T);
  (c) eager, eager and CUDA-graph replay bit-equal, and the first shape replayed again after the others ran;
  (d) call(training=True) + backward (against `exact` and the reference of test_gpu_model_backward.py), train_step_deferred
      on host inputs, wn_train_step_host and loss_fn.
Injected dropout masks belong to the (B, T) they were packed for: a training pass at another shape is rejected.

`test_case_table` (no GPU) pins the table for a B200's 74 CTA pairs, so that an edit cannot quietly drop a regime.  Run
with -s for the largest errors per case."""
import ctypes as C
import json
import time

import numpy as np
import pytest

from oracle import faithful
from oracle import wavenet_oracle as wo
from tests.util import SMALL_MODELS, device_slope_masks, oracle_config, rel_err, rel_l2

TILE = 256
B200_PAIRS = 74

# fp32 tier (tolerance of tests/test_gpu_parity_fp32.py)
TOL_FP32 = 1e-4
# bf16 tier: tests/test_gpu_parity_bf16.py ...
TOL_OUT, TOL_LOSS, TOL_GRAD, TOL_GRAD_PWL, MIN_COS_PWL = 1e-2, 1e-2, 1.5e-2, 1e-1, 0.995
TOL_GRAD_FAITHFUL, TOL_LOSS_FAITHFUL, TOL_OUT_FAITHFUL = 8e-3, 3e-4, 3e-3
# ... and tests/test_gpu_configs.py for the 256-wide models on the persistent stack launches
TOL_LOSS_FAITHFUL_STACK, TOL_GLOBAL_FAITHFUL = 5e-5, 4e-3
TOL_GRAD_FAITHFUL_DROPOUT, TOL_GLOBAL_FAITHFUL_DROPOUT = 1.2e-2, 5e-3
TOL_LOSS_BF16, TOL_GRAD_BF16 = 1e-2, 6e-2

FP32_COND_IN, BF16_COND_IN = 5, 9      # >= the workspace batch: every row gets a speaker of its own

# (what is smaller than the workspace, B, T); T % 128 and T % 256 are non-zero everywhere (ragged last tiles)
FP32_WS = (4, 160)
FP32_SHAPES = [('B', 3, 160), ('T', 4, 151), ('BT', 2, 97)]
BF16_WS = (4, 400)
BF16_SHAPES = [('B', 3, 400), ('T', 4, 333), ('BT', 2, 269)]


def _bf16_models():
  from tests.test_gpu_parity_bf16 import BF16_MODELS
  return BF16_MODELS


FP32_CASES = ['cond_skip', 'categorical_multidil', 'logistic_cond', 'gaussian_noskip', 'k3_nores', 'wide_ragged', 'l2']
BF16_CASES = ['single_dil_skip_cond', 'fused128_multidil_cond', 'group256_cond_l2', 'group256_alias_multidil', 'narrow32_cond_skip96',
              'logistic', 'gaussian_k3']

# one handle through the schedule regimes (side_launches of tests/test_gpu_group_wgrad.py: 256 channels, 6 blocks, conditioning)
STACK_KW = dict(channels=256, blocks=6, layers_per_block=1, dilation_bound=16, skip_channels=256, final_layers_channels=[256],
                activation='tanh', conditioning='global', mapping_layers=[8], mapping_activation='tanh')
STACK_WS = (4, 8000)


def stack_shapes(pairs):
  """(kind, B, T, persistent launches expected): stack forward / backward and grouped weight gradients, a second shape of that
  regime, fewer 256-row tiles than CTA pairs (per-block launches), then the first shape again"""
  fallback_tiles = pairs // 4                        # 2 sequences: half as many tiles as pairs
  return [('B', 3, 8000, True), ('T', 4, 6500, True), ('BT', 2, TILE * (fallback_tiles - 1) + 100, False), ('B', 3, 8000, True)]


# 256 wide, dropout 0.1, on the persistent stack launches (masks applied inside them)
DROPOUT_KW = dict(channels=256, blocks=4, layers_per_block=1, dilation_bound=16, skip_channels=256, final_layers_channels=[256],
                  activation='tanh', dropout=0.1)
DROPOUT_WS, DROPOUT_SHAPE = (4, 8000), ('BT', 3, 6500)
DROPOUT_FP32_KW = dict(SMALL_MODELS['cond_skip'], dropout=0.25)
DROPOUT_FP32_SHAPE = ('BT', 3, 151)

LAYER_WS = (4, 64)
LAYER_SHAPES = [('BT', 2, 37), ('T', 4, 50)]
LAYER_CASES = {
  # (precision, WaveNetLayer kwargs, conditioning: None | 'vector' (B, Cc) | 'sequence' (B, T, Cc) varying in time)
  'fp32_cond': ('fp32', dict(dilation_rate=2, channels=8, skip_channels=4), 'vector'),
  'fp32_multi_leaky': ('fp32', dict(dilation_rate=[1, 2, 4], activation='leaky_relu', channels=8, dilation_channels=12, skip_channels=6), None),
  'bf16_sequence': ('bf16', dict(dilation_rate=[1, 2], activation='tanh', channels=64, skip_channels=32), 'sequence'),
}


def _tiles(B, T):
  return B * -(-T // TILE)


# ----------------------------------------------------------------------------------------------------------- no GPU
def _table():
  """(case, workspace, [(kind, B, T)]) of every model case"""
  rows = [(f'fp32/{n}', FP32_WS, FP32_SHAPES) for n in FP32_CASES] + [(f'bf16/{n}', BF16_WS, BF16_SHAPES) for n in BF16_CASES]
  rows.append(('stack', STACK_WS, [s[:3] for s in stack_shapes(B200_PAIRS)]))
  rows.append(('dropout/bf16', DROPOUT_WS, [DROPOUT_SHAPE]))
  rows.append(('dropout/fp32', FP32_WS, [DROPOUT_FP32_SHAPE]))
  rows.append(('layer', LAYER_WS, LAYER_SHAPES))
  return rows


@pytest.mark.parametrize('case,ws,shapes', _table(), ids=[r[0] for r in _table()])
def test_case_table(case, ws, shapes):
  maxB, maxT = ws
  kinds = {k for k, _, _ in shapes}
  for kind, B, T in shapes:
    assert B <= maxB and T <= maxT, (case, B, T)
    assert (B < maxB) == ('B' in kind) and (T < maxT) == ('T' in kind), (case, kind, B, T)
    if case != 'layer':
      assert T % 128 != 0 and T % 256 != 0, (case, T)      # ragged last tile of both tile heights
  if case.startswith(('fp32/', 'bf16/')):
    assert kinds == {'B', 'T', 'BT'}, case
    assert ws[0] <= (FP32_COND_IN if case.startswith('fp32/') else BF16_COND_IN)
  if case == 'stack':
    s = stack_shapes(B200_PAIRS)
    assert [x[1:3] for x in s[:2]] == [(3, 8000), (4, 6500)] and s[3] == s[0]
    for _, B, T, persistent in s:
      assert (_tiles(B, T) > B200_PAIRS) == persistent, (B, T, _tiles(B, T))
    assert kinds == {'B', 'T', 'BT'}
  if case == 'dropout/bf16':
    _, B, T = DROPOUT_SHAPE
    assert _tiles(B, T) > B200_PAIRS                       # the keep-masks are applied inside the persistent launches
  if case == 'layer':
    assert {(B, T) for _, B, T in shapes} == {(2, 37), (4, 50)}


def test_cases_are_known_models():
  from tests.test_gpu_parity_bf16 import BF16_MODELS
  assert set(FP32_CASES) <= set(SMALL_MODELS) and set(BF16_CASES) <= set(BF16_MODELS)
  assert any(SMALL_MODELS[n].get('conditioning') for n in FP32_CASES)
  assert any(BF16_MODELS[n].get('conditioning') for n in BF16_CASES)
  assert SMALL_MODELS['l2']['l2_reg_factor'] > 0


# ----------------------------------------------------------------------------------------------------------- GPU helpers
def _pairs():
  import torch
  return torch.cuda.get_device_properties(0).multi_processor_count // 2


class _Memory:
  """device memory in use at the end of a case beyond what was in use when the first case started (cudaMemGetInfo: the
  library allocates with cudaMalloc, outside torch's allocator), handles of earlier cases not yet collected included"""
  base = None

  @classmethod
  def used_gib(cls):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if cls.base is None:
      cls.base = free
    return (cls.base - free) / 2 ** 30


def _report(case, res, t0):
  res.update(case=case, seconds=round(time.time() - t0, 1), device_memory_gib=round(_Memory.used_gib(), 3))
  print(json.dumps(res, default=float))


def _speakers(B, cond_in, offset):
  return np.eye(cond_in, dtype=np.float32)[(np.arange(B) + offset) % cond_in]


def _inputs(B, T, cond_in, seed):
  rng = np.random.default_rng(seed)
  x = np.clip(rng.standard_normal((B, T + 1, 1)) * 0.4, -1, 1).astype(np.float32)
  return x, (_speakers(B, cond_in, 0) if cond_in else None)


def _poison_inputs(B, T, cond_in):
  rng = np.random.default_rng(12345)
  x = (np.where(rng.random((B, T + 1, 1)) < 0.5, -1.0, 1.0) * rng.uniform(0.8, 1.0, (B, T + 1, 1))).astype(np.float32)
  return x, (_speakers(B, cond_in, 2) if cond_in else None)


def _pack(x, cond):
  return (x, cond) if cond is not None else x


def _dev(a):
  import torch
  return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _model(kw, precision, B, T, cond_in, p):
  from wavenets_b200 import WaveNet
  m = WaveNet(**kw, precision=precision, max_batch=B, max_time=T)
  m.build(((B, T, 1), (B, cond_in)) if cond_in else (B, T, 1))
  m.set_weights({k: v.astype(np.float32) for k, v in p.items()})
  return m


def _poison(m, ws, cond_in):
  """a training step and a call at full capacity: non-zero data in every slab row beyond the smaller calls"""
  x, cond = _poison_inputs(*ws, cond_in)
  m.train_step(_pack(x, cond))
  m(_pack(x[:, :-1], cond))


def _counters(m):
  lib, h = m.handle.lib, m.handle.h
  t, pt, side = C.c_int(), C.c_int(), C.c_int()
  assert lib.wn_grouped_wgrad_info(h, C.byref(t), C.byref(pt), C.byref(side)) == 0
  return dict(launches=int(lib.wn_last_launch_count(h)), fused_fwd=int(lib.wn_fused_forward_blocks(h)),
              stack_fwd=int(lib.wn_stack_forward_layers(h)), stack_bwd=int(lib.wn_stack_backward_layers(h)),
              grouped=(t.value, pt.value, side.value))


def _steps(m, data, n=3):
  """n training steps on device inputs (eager, eager + capture, graph replay): [(loss, reg_loss, flat gradients)]"""
  out = []
  for _ in range(n):
    r = m.train_step(data)
    out.append((r['loss'], r.get('reg_loss'), m.handle.flat_grads.clone()))
  return out


def _same_step(a, b):
  import torch
  return a[0] == b[0] and a[1] == b[1] and torch.equal(a[2], b[2])


def _loss_grad(m, pred, x):
  from tests.test_gpu_model_backward import _loss_grad
  return _loss_grad(m, pred, x)


def _errors(g, ref):
  """worst per-tensor relative L2 over the tensors with a non-zero reference gradient (zero ones must be zero), and the
  relative L2 of all gradients together"""
  from tests.config_parity import errors
  e = errors(g, ref)
  glob = float(np.sqrt(sum(np.sum((g[k].astype(np.float64) - ref[k]) ** 2) for k in ref) / sum(np.sum(ref[k] ** 2) for k in ref)))
  return e[0], glob


def _cos(a, b):
  a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
  return float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-300))


class _Reference:
  """the oracle side of one case: bounds per tier, the largest error seen per quantity"""

  def __init__(self, kw, cfg, p, precision, stack=False, keep=None):
    self.kw, self.cfg, self.p, self.precision, self.stack, self.keep = kw, cfg, p, precision, stack, keep
    self.p32 = {k: v.astype(np.float32).astype(np.float64) for k, v in p.items()}
    self.worst = {}

  def note(self, name, err, bound):
    self.worst[name] = max(self.worst.get(name, (0.0, bound))[0], float(err)), bound
    assert err <= bound, (name, err, bound)

  def pwl(self):
    return self.kw.get('activation') in ('relu', 'leaky_relu') or self.kw.get('mapping_activation') in ('relu', 'leaky_relu')

  def train(self, m, x, cond, step, B, T):
    loss, reg, _ = step
    g = m.get_grads()
    c64 = None if cond is None else cond.astype(np.float64)
    if self.precision == 'fp32':
      loss_o, g_o, aux = wo.train_step(self.p, self.cfg, x.astype(np.float64), c64, keep_masks=self.keep)
      self.note('loss_fp64', abs(loss - aux['loss_no_reg']) / abs(loss_o), TOL_FP32)
      self.note('reg_loss_fp64', abs((reg or 0.0) - aux['reg_loss']) / abs(loss_o), TOL_FP32)
      assert (reg is not None) == (self.cfg.l2_reg_factor > 0)
      self.note('grad_fp64', max(rel_err(g[k], g_o[k]) for k in g_o), TOL_FP32)
      return aux['loss_no_reg']
    masks = device_slope_masks(m, self.kw, B, T)
    l_f, g_f = faithful.train_step(self.p32, self.cfg, x, cond, faithful=True, slope_masks=masks, keep_masks=self.keep)
    (e_f, k_f), glob = _errors(g, g_f)
    if self.stack:
      dropout = self.keep is not None
      self.note('loss_faithful', abs(loss - l_f) / abs(l_f), TOL_LOSS_FAITHFUL_STACK)
      self.note('grad_faithful', e_f, TOL_GRAD_FAITHFUL_DROPOUT if dropout else TOL_GRAD_FAITHFUL)
      self.note('grad_faithful_global', glob, TOL_GLOBAL_FAITHFUL_DROPOUT if dropout else TOL_GLOBAL_FAITHFUL)
      l_64, g_64 = faithful.train_step(self.p32, self.cfg, x, cond, faithful=False, keep_masks=self.keep)
      self.note('loss_fp64', abs(loss - l_64) / abs(l_64), TOL_LOSS_BF16)
      self.note('grad_fp64', _errors(g, g_64)[0][0], TOL_GRAD_BF16)
      return l_64
    self.note('loss_faithful', abs(loss - l_f) / abs(l_f), TOL_LOSS_FAITHFUL)
    self.note('grad_faithful', e_f, TOL_GRAD_FAITHFUL)
    loss_o, g_o, aux = wo.train_step(self.p, self.cfg, x.astype(np.float64), c64)
    self.note('loss_fp64', abs(loss - aux['loss_no_reg']) / abs(loss_o), TOL_LOSS)
    self.note('reg_loss_fp64', abs((reg or 0.0) - aux['reg_loss']) / abs(loss_o), TOL_LOSS)
    nz = [k for k in g_o if np.linalg.norm(g_o[k]) > 0]
    self.note('grad_fp64', max(rel_l2(g[k], g_o[k]) for k in nz), TOL_GRAD_PWL if self.pwl() else TOL_GRAD)
    if self.pwl():
      self.note('grad_fp64_1-cos', 1 - min(_cos(g[k], g_o[k]) for k in nz), 1 - MIN_COS_PWL)
    return aux['loss_no_reg']

  def forward(self, pred, x, cond):
    xin = x[:, :-1]
    c64 = None if cond is None else cond.astype(np.float64)
    if self.precision == 'fp32':
      pred_o, _ = wo.model_forward(self.p, self.cfg, xin.astype(np.float64), c64)
      self.note('call_fp64', rel_err(pred, pred_o), TOL_FP32)
      return
    pred_o, _ = wo.model_forward(self.p, self.cfg, xin.astype(np.float64), c64)
    self.note('call_fp64', rel_l2(pred, pred_o), TOL_OUT)
    self.note('call_faithful', rel_l2(pred, faithful.forward(self.p32, self.cfg, xin, cond, faithful=True)), TOL_OUT_FAITHFUL)

  def loss(self, name, got, ref):
    self.note(name, abs(got - ref) / abs(ref), TOL_FP32 if self.precision == 'fp32' else TOL_LOSS)

  def backward(self, m, g, dcond, x, cond, dp, masks):
    from tests.test_gpu_model_backward import vjp_reference
    if self.precision == 'fp32':
      g_o, dc_o = vjp_reference(self.p, self.cfg, x[:, :-1], cond, dp)
      scale = max(np.abs(v).max() for v in g_o.values())
      for k in g_o:
        if np.abs(g_o[k]).max() == 0:
          assert np.abs(g[k]).max() <= 1e-6 * scale, k
      self.note('backward_fp64', max(rel_err(g[k], g_o[k]) for k in g_o if np.abs(g_o[k]).max() > 0), TOL_FP32)
      if cond is not None:
        self.note('dcond_fp64', rel_err(dcond, dc_o), TOL_FP32)
      return
    g_f, dc_f = vjp_reference(self.p32, self.cfg, x[:, :-1], cond, dp, True, masks)
    scale = max(np.linalg.norm(v) for v in g_f.values())
    self.note('backward_faithful', max(rel_l2(g[k], g_f[k]) for k in g_f if np.linalg.norm(g_f[k]) > 1e-9 * scale), TOL_GRAD_FAITHFUL)
    if cond is not None:
      self.note('dcond_faithful', rel_l2(dcond, dc_f), TOL_GRAD_FAITHFUL)

  def summary(self):
    return {k: f'{v[0]:.2e} <= {v[1]:.0e}' for k, v in sorted(self.worst.items())}


def _host_step(m, x, cond):
  """wn_train_step_host: pinned host staging buffers sized for the workspace"""
  h = m.handle
  B, T = x.shape[0], x.shape[1] - 1
  frames = np.ascontiguousarray(x.reshape(B, T + 1))
  loss = np.zeros(2, np.float32)
  c = None if cond is None else np.ascontiguousarray(cond)
  rc = h.lib.wn_train_step_host(h.h, frames.ctypes.data, None if c is None else c.ctypes.data, B, T, 1, loss.ctypes.data)
  return rc, loss


def _check_shape(big, exact, ref, kw, x, cond, data, first, with_backward_ref=True):
  """(a), (b) and (d) at one smaller shape, after the steps of every shape ran on both handles (`first`: big's first step here)"""
  import torch
  B, T = x.shape[0], x.shape[1] - 1
  assert _same_step(_steps(big, data, 1)[0], first), (B, T)      # (big's activations of this shape again, for the slope masks)
  masks = device_slope_masks(big, kw, B, T) if ref.precision == 'bf16' else None
  ref_loss = ref.train(big, x, cond, first, B, T)
  # call, test_step, loss_fn
  inputs = _pack(_dev(x[:, :-1]), _dev(cond))
  pred, pred_x = big(inputs), exact(inputs)
  assert torch.equal(pred, pred_x), (B, T)
  ref.forward(pred.cpu().numpy(), x, cond)
  t_loss = big.test_step(data)['loss']
  assert t_loss == exact.test_step(data)['loss']
  ref.loss('test_step_fp64', t_loss, ref_loss)
  target = big.prepare_target(_dev(x[:, 1:])) if big.num_mixtures is None else _dev(x[:, 1:, 0])
  lf = big.loss_fn(target, pred)
  assert torch.equal(lf, exact.loss_fn(target, pred_x))
  ref.loss('loss_fn_fp64', float(lf.double().sum()) / B, ref_loss)
  # (d) call(training=True) + backward
  if ref.precision == 'fp32':
    dp = np.random.default_rng(7).standard_normal(tuple(pred.shape)).astype(np.float32)
  else:
    dp = _loss_grad(big, pred, x)
  dps = []
  for m in (big, exact):
    m(inputs, training=True)
    dc = m.backward(dp)
    dps.append((m.handle.flat_grads.clone(), None if dc is None else dc.clone()))
  assert torch.equal(dps[0][0], dps[1][0]), (B, T)
  assert (dps[0][1] is None) == (cond is None) and (cond is None or torch.equal(dps[0][1], dps[1][1]))
  if with_backward_ref:
    ref.backward(big, big.get_grads(), None if cond is None else dps[0][1].cpu().numpy(), x, cond, dp, masks)
  # train_step_deferred on host arrays (staged through the model's own buffers) and wn_train_step_host: train_step's result
  pending = big.train_step_deferred(_pack(x, cond))
  assert pending.result()['loss'] == first[0] and torch.equal(big.handle.flat_grads, first[2]), (B, T)
  rc, loss = _host_step(big, x, cond)
  assert rc == 0, big.handle.lib.wn_last_error()
  assert float(loss[0]) == first[0] and torch.equal(big.handle.flat_grads, first[2]), (B, T)


def _run_model_case(kw, precision, ws, shapes, cond_in, case, stack=False, check=None):
  t0 = time.time()
  _Memory.used_gib()
  cfg = oracle_config(kw, cond_in)
  p = wo.init_params(cfg, seed=1)
  ref = _Reference(kw, cfg, p, precision, stack=stack)
  big = _model(kw, precision, *ws, cond_in, p)
  _poison(big, ws, cond_in)
  res = {'counters': {}}
  seen = {}
  # (c) every shape in turn: eager, eager + capture, graph replay; a shape met again replays its graph over the rows the
  # others left behind.  (b) `exact` gives the same steps and counters.
  for i, (kind, B, T) in enumerate(shapes):
    if (B, T) in seen:
      assert _same_step(_steps(big, seen[(B, T)][2], 1)[0], seen[(B, T)][3]), (B, T, 'replayed after the other shapes')
      continue
    x, cond = _inputs(B, T, cond_in, seed=1000 * B + T)
    data = _pack(_dev(x), _dev(cond))
    steps = _steps(big, data)
    n = _counters(big)
    exact = _model(kw, precision, B, T, cond_in, p)
    for s in steps[1:] + _steps(exact, data):
      assert _same_step(s, steps[0]), (B, T)
    assert n == _counters(exact), (B, T, n, _counters(exact))
    res['counters'][f'{B}x{T}'] = n
    if check is not None:
      check(i, n)
    seen[(B, T)] = (x, cond, data, steps[0], exact)
  A = shapes[0][1:]
  assert _same_step(_steps(big, seen[A][2], 1)[0], seen[A][3]), 'the first shape replayed after the others'
  # (a), (d)
  for x, cond, data, first, exact in seen.values():
    _check_shape(big, exact, ref, kw, x, cond, data, first, with_backward_ref=not stack)
  res['worst'] = ref.summary()
  res['big_equals_exact'] = 'bit-equal'
  _report(case, res, t0)


# ----------------------------------------------------------------------------------------------------------- GPU: models
@pytest.mark.gpu
@pytest.mark.parametrize('name', FP32_CASES)
def test_fp32_smaller_than_workspace(name):
  kw = SMALL_MODELS[name]
  _run_model_case(kw, 'fp32', FP32_WS, FP32_SHAPES, FP32_COND_IN if kw.get('conditioning') else 0, f'fp32/{name}')


@pytest.mark.gpu
@pytest.mark.parametrize('name', BF16_CASES)
def test_bf16_smaller_than_workspace(name):
  kw = _bf16_models()[name]
  _run_model_case(kw, 'bf16', BF16_WS, BF16_SHAPES, BF16_COND_IN if kw.get('conditioning') else 0, f'bf16/{name}')


@pytest.mark.gpu
def test_schedule_switches_in_one_handle():
  """One 4 x 8000 handle through the persistent stack launches with grouped weight gradients (3 x 8000, 4 x 6500), the per-block
  launches (fewer 256-row tiles than CTA pairs) and back to 3 x 8000 (a graph replay over the leftovers of all the others)."""
  shapes = stack_shapes(_pairs())
  L = STACK_KW['blocks']

  def check(i, n):
    _, B, T, persistent = shapes[i]
    assert (_tiles(B, T) > _pairs()) == persistent
    if persistent:
      assert n['stack_fwd'] == L and n['stack_bwd'] == L and n['grouped'][0] > 0, n
    else:
      assert n['stack_fwd'] == 0 and n['stack_bwd'] == 0, n

  _run_model_case(STACK_KW, 'bf16', STACK_WS, [s[:3] for s in shapes], BF16_COND_IN, 'stack', stack=True, check=check)


# ----------------------------------------------------------------------------------------------------------- GPU: dropout
def _keep(kw, B, T, seed=17):
  rng = np.random.default_rng(seed)
  return [(rng.random((B, T, kw['channels'])) >= kw['dropout']).astype(np.uint8) for _ in range(kw['blocks'])]


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_dropout_smaller_than_workspace(precision):
  """Injected masks at the smaller shape against the oracle with the same masks (bf16: 256 wide, masks applied inside the
  persistent stack launches) and bit-equal to `exact`; then Philox masks, bit-equal to `exact` with the same seed and steps."""
  import torch
  t0 = time.time()
  _Memory.used_gib()
  kw, ws, (_, B, T) = (DROPOUT_FP32_KW, FP32_WS, DROPOUT_FP32_SHAPE) if precision == 'fp32' else (DROPOUT_KW, DROPOUT_WS, DROPOUT_SHAPE)
  cond_in = FP32_COND_IN if kw.get('conditioning') else 0
  cfg = oracle_config(kw, cond_in)
  p = wo.init_params(cfg, seed=1)
  keep = _keep(kw, B, T)
  ref = _Reference(kw, cfg, p, precision, stack=precision == 'bf16', keep=keep)
  big = _model(kw, precision, *ws, cond_in, p)
  _poison(big, ws, cond_in)                                   # (Philox masks at full capacity)
  exact = _model(kw, precision, B, T, cond_in, p)
  x, cond = _inputs(B, T, cond_in, seed=5)
  data = _pack(_dev(x), _dev(cond))
  res = {}
  for m in (big, exact):
    m.set_dropout_masks(keep)
  steps = _steps(big, data)
  ref.train(big, x, cond, steps[0], B, T)
  c_big = _counters(big)
  if precision == 'bf16':
    assert c_big['stack_fwd'] == kw['blocks'] and c_big['stack_bwd'] == kw['blocks'], c_big
  for s in steps[1:] + _steps(exact, data):
    assert _same_step(s, steps[0])
  assert c_big == _counters(exact)
  res['counters'] = c_big
  # Philox masks drawn for the smaller shape: same seed, same step count
  philox = []
  for m in (big, exact):
    m.set_dropout_masks(None)
    m.set_dropout_seed(2024)
    philox.append(_steps(m, data, 2))
  for a, b in zip(*philox):
    assert _same_step(a, b)
  # fresh masks every step, not the injected ones (the gradients tell: a loss summed over 19,500 rows of a 3 x 6500 batch can land
  # on the same float32 for two mask sets)
  assert not torch.equal(philox[0][0][2], philox[0][1][2]) and not torch.equal(philox[0][0][2], steps[0][2])
  assert torch.equal(big(_pack(_dev(x[:, :-1]), _dev(cond))), exact(_pack(_dev(x[:, :-1]), _dev(cond))))
  res['worst'] = ref.summary()
  res['big_equals_exact'] = 'bit-equal'
  _report(f'dropout/{precision}', res, t0)


@pytest.mark.gpu
def test_injected_masks_reject_another_shape():
  """Masks injected for (2, 100) are packed as b * 100 + t: a training pass at (2, 90) would read them with its own packing."""
  from wavenets_b200 import WaveNetLayer, _lib
  kw = DROPOUT_FP32_KW
  cond_in = FP32_COND_IN
  p = wo.init_params(oracle_config(kw, cond_in), seed=1)
  m = _model(kw, 'fp32', 2, 100, cond_in, p)
  m.set_dropout_masks(_keep(kw, 2, 100))
  x100, c100 = _inputs(2, 100, cond_in, seed=1)
  x90, c90 = _inputs(2, 90, cond_in, seed=2)
  msg = r'\(2, 100\).*\(2, 90\)'
  with pytest.raises(RuntimeError, match=msg):
    m.train_step((x90, c90))
  with pytest.raises(RuntimeError, match=msg):
    m((x90[:, :-1], c90), training=True)
  rc, _ = _host_step(m, x90, c90)
  assert rc == _lib.WN_ERR_STATE
  # the passes without dropout run at any shape; the injected shape still trains
  assert np.isfinite(m.test_step((x100, c100))['loss'])
  assert bool(m((x90[:, :-1], c90)).isfinite().all())
  assert np.isfinite(m.train_step((x100, c100))['loss'])
  m.set_dropout_masks(None)
  assert np.isfinite(m.train_step((x90, c90))['loss'])
  # the layer API: the same rule
  rng = np.random.default_rng(0)
  lay = WaveNetLayer(dilation_rate=2, channels=8, dropout=0.25)
  lay.build((2, 100, 8))
  lay.set_dropout_mask(rng.random((2, 100, 8)) >= 0.25)
  xl90 = rng.standard_normal((2, 90, 8)).astype(np.float32)
  with pytest.raises(RuntimeError, match=msg):
    lay.call(xl90, training=True)
  lay.call(xl90)
  lay.call(rng.standard_normal((2, 100, 8)).astype(np.float32), training=True)
  lay.set_dropout_mask(None)
  lay.call(xl90, training=True)


# ----------------------------------------------------------------------------------------------------------- GPU: WaveNetLayer
def _layer(precision, kw, cond, B, T, w=None):
  from wavenets_b200 import WaveNetLayer
  R, Cc = kw['channels'], 6
  lay = WaveNetLayer(**kw, condition=cond is not None, precision=precision)
  cshape = None if cond is None else ((B, Cc) if cond == 'vector' else (B, T, Cc))
  lay.build(((B, T, R), cshape) if cond is not None else (B, T, R))
  if w is None:
    rng = np.random.default_rng(3)
    w = {n: ((rng.standard_normal(s) / np.sqrt(np.prod(s[:-1]))) if n.endswith('kernel') else rng.standard_normal(s) * 0.1).astype(np.float32)
         for n, s in zip(lay.weight_names, lay._handle.shapes)}
  lay.set_weights(w)
  return lay, w


def _layer_inputs(kw, cond, B, T, seed, amp=1.0):
  rng = np.random.default_rng(seed)
  R, Cc = kw['channels'], 6
  S = kw.get('skip_channels') or R
  x = (rng.standard_normal((B, T, R)) * amp).astype(np.float32)
  c = None
  if cond == 'vector':
    c = rng.standard_normal((B, Cc)).astype(np.float32)
  elif cond == 'sequence':
    c = rng.standard_normal((B, T, Cc)).astype(np.float32)
  return x, c, rng.standard_normal((B, T, R)).astype(np.float32), rng.standard_normal((B, T, S)).astype(np.float32)


def _layer_run(lay, x, c, dxo, dsk):
  xo, sk = lay.call((x, c) if c is not None else x)
  dx, dc = lay.backward(dxo, dsk)
  return [xo.cpu().numpy(), sk.cpu().numpy(), dx.cpu().numpy(), None if dc is None else dc.cpu().numpy()], lay.get_grads()


@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(LAYER_CASES))
def test_layer_smaller_than_workspace(name):
  t0 = time.time()
  _Memory.used_gib()
  precision, kw, cond = LAYER_CASES[name]
  lay, w = _layer(precision, kw, cond, *LAYER_WS)
  x, c, dxo, dsk = _layer_inputs(kw, cond, *LAYER_WS, seed=99, amp=3.0)    # stale rows at full capacity
  _layer_run(lay, x, c, dxo, dsk)
  ref = _Reference(kw, None, {}, precision)
  dils = kw['dilation_rate'] if isinstance(kw['dilation_rate'], list) else [kw['dilation_rate']]
  lc = dict(dilations=dils, activation=kw.get('activation'), residual=kw.get('residual', True), has_skip=kw.get('skip_channels') is not None,
            condition=cond is not None)
  p = {'block0/' + k: v.astype(np.float64) for k, v in w.items()}
  smooth = len(dils) == 1 or kw.get('activation') in (None, 'tanh', 'sigmoid')
  for _, B, T in LAYER_SHAPES:
    x, c, dxo, dsk = _layer_inputs(kw, cond, B, T, seed=B * 1000 + T)
    out, g = _layer_run(lay, x, c, dxo, dsk)
    exact, _ = _layer(precision, kw, cond, B, T, w)
    out_x, g_x = _layer_run(exact, x, c, dxo, dsk)
    for a, b in zip(out, out_x):
      assert (a is None and b is None) or np.array_equal(a, b), (B, T)
    for k in g_x:
      assert np.array_equal(g[k], g_x[k]), (B, T, k)
    xo_o, sk_o, cache = wo.layer_forward(p, 'block0', lc, x.astype(np.float64), None if c is None else c.astype(np.float64))
    dx_o, dc_o, g_o = wo.layer_backward(p, 'block0', lc, cache, dxo.astype(np.float64), dsk.astype(np.float64))
    pairs = [('x_out', out[0], xo_o), ('skip', out[1], sk_o), ('dx', out[2], dx_o)] + ([('dcond', out[3], dc_o)] if c is not None else [])
    pairs += [(k, g[k[len('block0/'):]], v) for k, v in g_o.items()]
    for n, a, b in pairs:
      assert a.shape == b.shape, n
      if precision == 'fp32':
        ref.note(n, rel_err(a, b), TOL_FP32)
      elif n in ('x_out', 'skip'):
        ref.note(n, rel_l2(a, b), TOL_OUT)
      else:
        ref.note(n, rel_l2(a, b), TOL_GRAD if smooth else TOL_GRAD_PWL)
  _report(f'layer/{name}', {'worst': ref.summary(), 'big_equals_exact': 'bit-equal'}, t0)
