"""WaveNet.backward(input_grad=True, param_grads=...) (wn_backward_ex): d loss / d x of the waveform passed to `call`, what
tape.gradient(loss, x) gives in the reference, with or without the parameter gradients.

Checker: `input_grad_reference` (tests/test_oracle_input_grad_cpu.py, pinned there against central differences of
oracle/wavenet_oracle.model_forward): float64 on the fp32 tier (<= 1e-4), the bf16-faithful forward on the bf16 tier with the
tolerances of the backward tests (tests/test_gpu_model_backward.py)."""
import gc

import numpy as np
import pytest
import torch

from tests import config_parity
from tests.test_gpu_model_backward import (BF16_COND_IN, TOL_FP32, TOL_GRAD_FAITHFUL, TOL_GRAD_FAITHFUL_DROPOUT, _bf16_models, _dpred,
                                           _inputs, _loss_grad, _model)
from tests.test_oracle_input_grad_cpu import input_grad_reference
from tests.util import COND_IN, SMALL_MODELS, device_slope_masks, rel_err, rel_l2

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _free_handles():
  """A model's handle and its zero-copy flat parameter / gradient tensors refer to each other through torch's storage, a cycle
  the garbage collector cannot see: the handles made here would keep their device workspaces (C2: several GB) for the rest of
  the session.  Each test's handles are closed when it ends."""
  from wavenets_b200._engine import Handle
  before = {id(o) for o in gc.get_objects() if type(o) is Handle}
  yield
  for o in gc.get_objects():
    if type(o) is Handle and id(o) not in before:
      o.close()


def _kw(precision, name):
  return SMALL_MODELS[name] if precision == 'fp32' else _bf16_models()[name]


def _cond_in(precision, kw):
  return 0 if not kw.get('conditioning') else (COND_IN if precision == 'fp32' else BF16_COND_IN)


def _check(precision, m, kw, cfg, p, x, cond, dp, dx, B, T, keep=None, tol=None):
  """dx against the reference of its tier"""
  dx = dx.cpu().numpy().reshape(B, T)
  if precision == 'fp32':
    ref = input_grad_reference(p, cfg, x[:, :-1], cond, dp, keep_masks=keep)
    assert rel_err(dx, ref) < TOL_FP32, rel_err(dx, ref)
  else:
    ref = input_grad_reference(p, cfg, x[:, :-1], cond, dp, True, device_slope_masks(m, kw, B, T), keep)
    assert rel_l2(dx, ref) < (tol or TOL_GRAD_FAITHFUL), rel_l2(dx, ref)


# ------------------------------------------------------------------ fp32 tier
@pytest.mark.parametrize('name', sorted(SMALL_MODELS))
@pytest.mark.parametrize('BT', [(2, 100), (3, 257)])
def test_input_grad_fp32_vs_fp64(name, BT):
  kw = SMALL_MODELS[name]
  B, T = BT
  m, cfg, p, x, cond = _model(kw, B, T, 'fp32', _cond_in('fp32', kw))
  dp = _dpred(m, B, T)
  m(_inputs(x, cond))
  d_full = m.backward(dp)
  g_full = m.handle.flat_grads.clone()
  dx, dcond = m.backward(dp, input_grad=True)
  assert dx.shape == (B, T, 1)
  _check('fp32', m, kw, cfg, p, x, cond, dp, dx, B, T)
  # the parameter gradients and d cond do not depend on whether dx is asked for
  assert torch.equal(g_full, m.handle.flat_grads)
  assert (dcond is None) == (d_full is None)
  if dcond is not None:
    assert torch.equal(dcond, d_full)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_input_grad_training_pass_with_injected_masks(precision):
  name = 'cond_skip' if precision == 'fp32' else 'single_dil_skip_cond'
  kw = dict(_kw(precision, name), dropout=0.2)
  B, T = 2, 300
  m, cfg, p, x, cond = _model(kw, B, T, precision, _cond_in(precision, kw))
  rng = np.random.default_rng(3)
  keep = [(rng.random((B, T, kw['channels'])) >= kw['dropout']).astype(np.uint8) for _ in range(kw['blocks'])]
  m.set_dropout_masks(keep)
  pred = m(_inputs(x, cond), training=True)
  dp = _dpred(m, B, T) if precision == 'fp32' else _loss_grad(m, pred, x)
  dx, _ = m.backward(dp, input_grad=True)
  _check(precision, m, kw, cfg, p, x, cond, dp, dx, B, T, keep, TOL_GRAD_FAITHFUL_DROPOUT)


# ------------------------------------------------------------------ bf16 tier
@pytest.mark.parametrize('name', sorted(_bf16_models()))
def test_input_grad_bf16_vs_faithful(name):
  kw = _bf16_models()[name]
  B, T = 2, 100
  m, cfg, p, x, cond = _model(kw, B, T, 'bf16', _cond_in('bf16', kw))
  dp = _loss_grad(m, m(_inputs(x, cond)), x)
  dx, _ = m.backward(dp, input_grad=True)
  _check('bf16', m, kw, cfg, p, x, cond, dp, dx, B, T)


# C2's d h0 (softmax head, 30 blocks) carries the bf16 storage noise of the whole gradient chain, which the faithful oracle does
# not round, and dx is a sum over only R * K terms of it (the weight gradients average it over B * T rows): on a B200, 1.47e-2
# (dropout 0) and 1.54e-2 (dropout 0.1) against the faithful oracle.  C4 runs the same chain and the same dgrad launch with a
# mixture head and meets TOL_GRAD_FAITHFUL; the fp32 tier checks the kernel itself to 1e-4.
TOL_C2 = 2e-2


@pytest.mark.parametrize('name,dropout', [('c2', 0.0), ('c2', 0.1), ('c3', 0.0), ('c3', 0.1), ('c4', 0.0)])
def test_input_grad_persistent_stack_vs_faithful(name, dropout):
  m, ocfg, p, x, cond, _, _, _, kw = config_parity.setup(name, dropout)
  B, T = config_parity.SHAPES[name][:2]
  h = m.handle
  keep = None
  if dropout > 0:
    rng = np.random.default_rng(17)
    keep = [(rng.random((B, T, kw['channels'])) >= dropout).astype(np.uint8) for _ in range(kw['blocks'])]
    m.set_dropout_masks(keep)
  dp = _loss_grad(m, m(_inputs(x, cond), training=dropout > 0), x)
  dx, _ = m.backward(dp, input_grad=True)
  assert int(h.lib.wn_stack_backward_layers(h.h)) == m.blocks
  tol = TOL_C2 if name == 'c2' else TOL_GRAD_FAITHFUL_DROPOUT if dropout > 0 else TOL_GRAD_FAITHFUL
  _check('bf16', m, kw, ocfg, p, x, cond, dp, dx, B, T, keep, tol)


# ------------------------------------------------------------------ input-only mode
def _setup_mode(case):
  if case == 'c2':
    m, _, _, x, cond, _, _, _, _ = config_parity.setup('c2', 0.1)
    B, T = config_parity.SHAPES['c2'][:2]
    return m, x, cond, B, T, True
  precision, name = case
  kw = _kw(precision, name)
  B, T = 3, 700
  m, _, _, x, cond = _model(kw, B, T, precision, _cond_in(precision, kw))
  return m, x, cond, B, T, False


@pytest.mark.parametrize('case', [('fp32', 'cond_skip'), ('bf16', 'group256_cond_l2'), 'c2'], ids=['fp32', 'group256', 'c2'])
def test_input_only_mode(case):
  m, x, cond, B, T, training = _setup_mode(case)
  h = m.handle
  dp = _dpred(m, B, T)
  m(_inputs(x, cond), training=training)
  h.flat_grads.fill_(-1.25)
  sentinel = h.flat_grads.clone()
  dx_in, dc_in = m.backward(dp, input_grad=True, param_grads=False)
  torch.cuda.synchronize()
  assert torch.equal(h.flat_grads, sentinel)
  launches_in = int(h.lib.wn_last_launch_count(h.h))
  assert int(h.lib.wn_grouped_wgrad_tiles(h.h, None)) == 0
  if case == 'c2':
    assert int(h.lib.wn_stack_backward_layers(h.h)) == m.blocks
  dx_full, dc_full = m.backward(dp, input_grad=True)
  launches_full = int(h.lib.wn_last_launch_count(h.h))
  assert launches_in < launches_full, (launches_in, launches_full)
  assert torch.equal(dx_in, dx_full)
  if cond is not None:
    # (the per-batch sums of d z and the mapping MLP's dgrads run in their own fp32 summation order without the weight gradients)
    assert rel_err(dc_in.cpu().numpy(), dc_full.cpu().numpy()) < 1e-5
  # and d cond alone, without dx
  if cond is not None:
    dc_only = m.backward(dp, param_grads=False)
    assert torch.equal(dc_only, dc_in)


# ------------------------------------------------------------------ edges
EDGE_MODELS = {'fp32': ('k3_nores', 'cond_skip'), 'bf16': ('gaussian_k3', 'single_dil_skip_cond')}


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_input_grad_sequence_shorter_than_kernel(precision):
  name = EDGE_MODELS[precision][0]           # kernel_size 3
  kw = _kw(precision, name)
  B, T = 2, 2
  m, cfg, p, x, cond = _model(kw, B, T, precision, _cond_in(precision, kw))
  pred = m(_inputs(x, cond))
  dp = _dpred(m, B, T) if precision == 'fp32' else _loss_grad(m, pred, x)
  dx, _ = m.backward(dp, input_grad=True, param_grads=False)
  _check(precision, m, kw, cfg, p, x, cond, dp, dx, B, T)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('BT', [(2, 130), (3, 65)])
def test_input_grad_smaller_than_workspace(precision, BT):
  """B < max_batch, T < max_time and not a multiple of the kernel's 64-row tile: the rows of a batch row stay T apart"""
  from wavenets_b200 import WaveNet
  name = EDGE_MODELS[precision][1]
  kw = _kw(precision, name)
  cond_in = _cond_in(precision, kw)
  B, T = BT
  m0, cfg, p, x, cond = _model(kw, B, T, precision, cond_in)
  m = WaveNet(**kw, precision=precision, max_batch=4, max_time=300)
  m.build(((4, 300, 1), (4, cond_in)) if cond_in else (4, 300, 1))
  m.set_weights(m0.get_weights())
  pred = m(_inputs(x, cond))
  dp = _dpred(m, B, T) if precision == 'fp32' else _loss_grad(m, pred, x)
  dx, _ = m.backward(dp, input_grad=True)
  _check(precision, m, kw, cfg, p, x, cond, dp, dx, B, T)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('param_grads', [True, False])
def test_input_grad_causal_and_rows_apart(precision, param_grads):
  name = EDGE_MODELS[precision][1]
  kw = _kw(precision, name)
  B, T, last = 3, 257, 190
  m, _, _, x, cond = _model(kw, B, T, precision, _cond_in(precision, kw))
  dp = _dpred(m, B, T)
  dp[:, last + 1:] = 0
  dp[1] = 0
  m(_inputs(x, cond))
  dx, _ = m.backward(dp, input_grad=True, param_grads=param_grads)
  dx = dx.cpu().numpy()[:, :, 0]
  assert np.all(dx[:, last + 1:] == 0)
  assert np.all(dx[1] == 0)
  assert np.abs(dx[0, :last + 1]).max() > 0 and np.abs(dx[2, :last + 1]).max() > 0


def test_input_grad_of_a_2d_input_is_2d():
  kw = SMALL_MODELS['categorical_multidil']
  B, T = 2, 64
  m, _, _, x, _ = _model(kw, B, T, 'fp32', 0)
  m(np.ascontiguousarray(x[:, :-1, 0]))
  dx, dcond = m.backward(_dpred(m, B, T), input_grad=True, param_grads=False)
  assert dx.shape == (B, T) and dcond is None


# ------------------------------------------------------------------ repeatability
@pytest.mark.parametrize('precision,name', [('fp32', 'cond_skip'), ('bf16', 'r256'), ('bf16', 'c2')])
def test_input_grad_repeatable_and_independent_of_mode_order(precision, name):
  case = 'c2' if name == 'c2' else (precision, name)
  m, x, cond, B, T, training = _setup_mode(case)
  h = m.handle
  dp = _dpred(m, B, T)
  m(_inputs(x, cond), training=training)
  dx1, dc1 = m.backward(dp, input_grad=True)
  g1 = h.flat_grads.clone()
  dx2, dc2 = m.backward(dp, input_grad=True)
  assert torch.equal(dx1, dx2) and torch.equal(g1, h.flat_grads)
  if dc1 is not None:
    assert torch.equal(dc1, dc2)
  # input-only, then full: the same as full alone
  m.backward(dp, input_grad=True, param_grads=False)
  dx3, dc3 = m.backward(dp, input_grad=True)
  assert torch.equal(dx1, dx3) and torch.equal(g1, h.flat_grads)
  if dc1 is not None:
    assert torch.equal(dc1, dc3)


@pytest.mark.parametrize('precision,name', [('fp32', 'cond_skip'), ('bf16', 'r256')])
@pytest.mark.parametrize('param_grads', [True, False])
def test_input_grad_leaves_train_step_unchanged(precision, name, param_grads):
  kw = _kw(precision, name)
  B, T = 3, 700
  cond_in = _cond_in(precision, kw)
  runs = []
  for with_backward in (False, True):
    m, _, _, x, cond = _model(kw, B, T, precision, cond_in)
    data = (x, cond) if cond is not None else x
    m.train_step(data)
    if with_backward:
      m(_inputs(x, cond))
      m.backward(_dpred(m, B, T), input_grad=True, param_grads=param_grads)
    out = m.train_step(data)
    runs.append((out['loss'], m.handle.flat_grads.clone()))
  assert runs[0][0] == runs[1][0]
  assert torch.equal(runs[0][1], runs[1][1])


# ------------------------------------------------------------------ errors
def test_input_grad_errors():
  kw = SMALL_MODELS['categorical_multidil']
  B, T = 2, 120
  m, _, _, x, _ = _model(kw, B, T, 'fp32', 0)
  h = m.handle
  dp = torch.as_tensor(_dpred(m, B, T), device=h.device)
  dx = torch.empty((B, T), dtype=torch.float32, device=h.device)
  assert h.lib.wn_backward_ex(h.h, h.ptr(dp), None, h.ptr(dx), 0, h.stream_ptr()) == -4      # WN_ERR_STATE: no call yet
  with pytest.raises(RuntimeError):
    m.backward(dp, input_grad=True, param_grads=False)
  m(x[:, :-1])
  with pytest.raises(ValueError):
    m.backward(dp, param_grads=False)       # no conditioning, no dx: nothing to compute
  assert h.lib.wn_backward_ex(h.h, h.ptr(dp), None, None, 0, h.stream_ptr()) == -1         # WN_ERR_VALUE
  m.backward(dp, input_grad=True, param_grads=False)      # the handle's state is intact
