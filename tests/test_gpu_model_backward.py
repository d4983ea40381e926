"""WaveNet.backward (wn_backward): the adjoint of WaveNet.call for a loss the caller computes on its output — what a
tf.GradientTape over `model(inputs, training=True)` followed by `tape.gradient(loss, model.trainable_variables)` gives in the
reference (model.py:213-239).

Checker: `vjp_reference` below — oracle/faithful.py's forward on torch float64 with autograd, the softmax on top for categorical
heads, and (pred * dpred).sum() differentiated with respect to every parameter and to the conditioning input.  faithful=False is
the reference path in float64 (fp32 tier: <= 1e-4 relative, the tier's stated tolerance); faithful=True rounds to bf16 exactly
where the kernels do (bf16 tier: every tensor within TOL_GRAD_FAITHFUL, as train_step at the same shapes).  It is pinned against
oracle/wavenet_oracle.model_backward in tests/test_oracle_vjp_cpu.py.
"""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import faithful
from oracle import wavenet_oracle as wo
from tests import config_parity
from tests.util import COND_IN, SMALL_MODELS, device_slope_masks, device_tensor, make_inputs, oracle_config, rel_err, rel_l2

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL_FP32 = 1e-4
TOL_GRAD_FAITHFUL, TOL_GLOBAL_FAITHFUL = 8e-3, 4e-3                     # = tests/test_gpu_configs.py (train_step at these shapes)
TOL_GRAD_FAITHFUL_DROPOUT, TOL_GLOBAL_FAITHFUL_DROPOUT = 1.2e-2, 5e-3
BF16_COND_IN = 9


def vjp_reference(p_np, cfg: wo.Config, x, cond_in, dpred, faithful_mode=False, slope_masks=None, keep_masks=None):
  """Gradients of sum(pred * dpred), pred = WaveNet.call(x, cond_in) (softmax probabilities or mixture parameters).
  x (B,T,1), cond_in (B,cond_in) or None, dpred (B,T,C).  Returns ({name: gradient}, d cond_in or None), float64 numpy."""
  R = faithful.Rounding(faithful_mode)
  dt = torch.float64
  p = {k: torch.tensor(np.asarray(v), dtype=dt, requires_grad=True) for k, v in p_np.items()}
  xx = torch.tensor(np.asarray(x), dtype=dt)
  c = None if cond_in is None else torch.tensor(np.asarray(cond_in), dtype=dt, requires_grad=True)
  logits = faithful.forward_logits(p, cfg, xx, c, R, None, slope_masks, keep_masks)
  if faithful_mode:
    logits = logits.to(torch.float32).to(dt)      # the logits live in fp32
  pred = torch.softmax(logits, dim=-1) if cfg.sampling_function == 'categorical' else logits
  (pred * torch.tensor(np.asarray(dpred), dtype=dt)).sum().backward()
  grads = {k: (v.grad.numpy() if v.grad is not None else np.zeros(v.shape)) for k, v in p.items()}
  return grads, None if c is None else c.grad.numpy()


def _model(kw, B, T, precision, cond_in, seed=1):
  from wavenets_b200 import WaveNet
  cfg = oracle_config(kw, cond_in)
  p = wo.init_params(cfg, seed=seed)
  m = WaveNet(**kw, precision=precision)
  x, cond = make_inputs(B, T, cond_in)
  m.build((x[:, :-1].shape, cond.shape) if cond is not None else x[:, :-1].shape)
  m.set_weights({k: v.astype(np.float32) for k, v in p.items()})
  p32 = {k: v.astype(np.float32).astype(np.float64) for k, v in p.items()}
  return m, cfg, p32, x, cond


def _inputs(x, cond):
  return (x[:, :-1], cond) if cond is not None else x[:, :-1]


def _dpred(m, B, T, seed=7):
  cout = 3 * m.num_mixtures if m.num_mixtures is not None else 2 ** m.bits
  return np.random.default_rng(seed).standard_normal((B, T, cout)).astype(np.float32)


def _loss_grad(m, pred, x, seed=5):
  """d loss / d pred of a loss of the caller's making: cross entropy with per-position weights in [0, 2) and the first quarter of
  every sequence masked out (categorical), or a weighted quadratic on the mixture parameters.  The bf16 tier is checked with it:
  like any real loss its gradient is coherent over the batch, so the weight gradients (sums over B*T rows) grow with B*T while the
  bf16 storage noise grows with sqrt(B*T) — the regime TOL_GRAD_FAITHFUL was set in.  An N(0,1) dpred cancels in those sums and
  leaves the noise alone (on a B200, C2: 2.3e-2 worst tensor, 1.5e-2 over all gradients against the faithful oracle; the fp32 tier
  meets 1e-4 with it, see test_backward_fp32_vs_fp64)."""
  B, T, _ = pred.shape
  w = torch.as_tensor(np.random.default_rng(seed).random((B, T, 1)) * 2, dtype=torch.float32, device=pred.device)
  w[:, :T // 4] = 0
  if m.num_mixtures is not None:
    return (w * pred / (B * T)).cpu().numpy()
  y = m.prepare_target(x[:, 1:]).reshape(B, T, 1)
  return torch.zeros_like(pred).scatter_(2, y, -w / (B * torch.gather(pred, 2, y))).cpu().numpy()


# ------------------------------------------------------------------ fp32 tier
@pytest.mark.parametrize('name', sorted(SMALL_MODELS))
@pytest.mark.parametrize('BT', [(2, 100), (3, 257)])
def test_backward_fp32_vs_fp64(name, BT):
  kw = SMALL_MODELS[name]
  B, T = BT
  cond_in = COND_IN if kw.get('conditioning') else 0
  m, cfg, p, x, cond = _model(kw, B, T, 'fp32', cond_in)
  dp = _dpred(m, B, T)
  m(_inputs(x, cond))
  dcond = m.backward(dp)
  g = m.get_grads()
  g_o, dc_o = vjp_reference(p, cfg, x[:, :-1], cond, dp)
  # (the L2 models: the regulariser belongs to train_step, not to call — a gradient with it would miss by far more than 1e-4)
  scale = max(np.abs(v).max() for v in g_o.values())
  for k in g_o:
    if np.abs(g_o[k]).max() == 0:       # a conv whose output nothing reads (conv1 of the last block under use_skip, ...)
      assert np.abs(g[k]).max() <= 1e-6 * scale, k
      continue
    assert rel_err(g[k], g_o[k]) < TOL_FP32, (k, rel_err(g[k], g_o[k]))
  if cond is None:
    assert dcond is None
  else:
    assert dcond.shape == (B, cond_in)
    assert rel_err(dcond.cpu().numpy(), dc_o) < TOL_FP32


def test_backward_fp32_training_pass_with_injected_masks():
  kw = dict(SMALL_MODELS['cond_skip'], dropout=0.25)
  B, T = 2, 150
  m, cfg, p, x, cond = _model(kw, B, T, 'fp32', COND_IN)
  rng = np.random.default_rng(3)
  keep = [(rng.random((B, T, kw['channels'])) >= kw['dropout']).astype(np.uint8) for _ in range(kw['blocks'])]
  m.set_dropout_masks(keep)
  dp = _dpred(m, B, T)
  m(_inputs(x, cond), training=True)
  dcond = m.backward(dp)
  g = m.get_grads()
  g_o, dc_o = vjp_reference(p, cfg, x[:, :-1], cond, dp, keep_masks=keep)
  for k in g_o:
    assert rel_err(g[k], g_o[k]) < TOL_FP32, (k, rel_err(g[k], g_o[k]))
  assert rel_err(dcond.cpu().numpy(), dc_o) < TOL_FP32


# ------------------------------------------------------------------ bf16 tier
def _check_faithful(g, ref, tol):
  scale = max(np.linalg.norm(v) for v in ref.values())
  worst = max((rel_l2(g[k], ref[k]), k) for k in ref if np.linalg.norm(ref[k]) > 1e-9 * scale)
  assert worst[0] < tol, worst


def _bf16_models():
  from tests.test_gpu_parity_bf16 import BF16_MODELS
  return BF16_MODELS


@pytest.mark.parametrize('name', sorted(_bf16_models()))
def test_backward_bf16_vs_faithful(name):
  kw = _bf16_models()[name]
  B, T = 2, 100
  cond_in = BF16_COND_IN if kw.get('conditioning') else 0
  m, cfg, p, x, cond = _model(kw, B, T, 'bf16', cond_in)
  dp = _loss_grad(m, m(_inputs(x, cond)), x)
  dcond = m.backward(dp)
  g = m.get_grads()
  g_f, dc_f = vjp_reference(p, cfg, x[:, :-1], cond, dp, True, device_slope_masks(m, kw, B, T))
  _check_faithful(g, g_f, TOL_GRAD_FAITHFUL)
  if cond is not None:
    assert rel_l2(dcond.cpu().numpy(), dc_f) < TOL_GRAD_FAITHFUL


def test_backward_bf16_training_pass_with_injected_masks():
  kw = dict(_bf16_models()['single_dil_skip_cond'], dropout=0.2)
  B, T = 2, 300
  m, cfg, p, x, cond = _model(kw, B, T, 'bf16', BF16_COND_IN)
  rng = np.random.default_rng(3)
  keep = [(rng.random((B, T, kw['channels'])) >= kw['dropout']).astype(np.uint8) for _ in range(kw['blocks'])]
  m.set_dropout_masks(keep)
  dp = _loss_grad(m, m(_inputs(x, cond), training=True), x)
  dcond = m.backward(dp)
  g = m.get_grads()
  g_f, dc_f = vjp_reference(p, cfg, x[:, :-1], cond, dp, True, device_slope_masks(m, kw, B, T), keep)
  _check_faithful(g, g_f, TOL_GRAD_FAITHFUL_DROPOUT)
  assert rel_l2(dcond.cpu().numpy(), dc_f) < TOL_GRAD_FAITHFUL_DROPOUT


@pytest.mark.parametrize('name,dropout', [('c2', 0.0), ('c2', 0.1), ('c3', 0.0), ('c3', 0.1)])
def test_backward_persistent_stack_vs_faithful(name, dropout):
  """C2 / C3 at 3 x 6400: the persistent stack-forward and stack-backward launches and the grouped weight gradients are on the
  checked path (asserted), with the training-pass dropout masks applied inside them."""
  m, ocfg, p, x, cond, _, _, _, kw = config_parity.setup(name, dropout)
  B, T = config_parity.SHAPES[name][:2]
  h = m.handle
  keep = None
  if dropout > 0:
    rng = np.random.default_rng(17)
    keep = [(rng.random((B, T, kw['channels'])) >= dropout).astype(np.uint8) for _ in range(kw['blocks'])]
    m.set_dropout_masks(keep)
  dp = _loss_grad(m, m(_inputs(x, cond), training=dropout > 0), x)
  dcond = m.backward(dp)
  assert int(h.lib.wn_stack_backward_layers(h.h)) == m.blocks
  assert int(h.lib.wn_grouped_wgrad_tiles(h.h, None)) > 0
  g = m.get_grads()
  g_f, dc_f = vjp_reference(p, ocfg, x[:, :-1], cond, dp, True, device_slope_masks(m, kw, B, T), keep)
  ef = config_parity.errors(g, g_f)
  glob = float(np.sqrt(sum(np.sum((g[k].astype(np.float64) - g_f[k]) ** 2) for k in g_f) / sum(np.sum(g_f[k] ** 2) for k in g_f)))
  print(json.dumps({'config': name, 'dropout': dropout, 'worst': ef[0], 'global': glob}))
  tol, tol_glob = (TOL_GRAD_FAITHFUL_DROPOUT, TOL_GLOBAL_FAITHFUL_DROPOUT) if dropout > 0 else (TOL_GRAD_FAITHFUL, TOL_GLOBAL_FAITHFUL)
  assert ef[0][0] <= tol, ef[:4]
  assert glob <= tol_glob
  if cond is not None:
    assert rel_l2(dcond.cpu().numpy(), dc_f) <= tol


# ------------------------------------------------------------------ the same gradients as train_step
def _train_step_then_backward_of_its_dlogits(m, x, cond, B, T):
  data = (x, cond) if cond is not None else x
  for _ in range(3):            # eager, plans built, CUDA-graph replay
    m.train_step(data)
  g_ts = m.handle.flat_grads.clone()
  cout = 3 * m.num_mixtures
  dl = device_tensor(m, 'dlogits', 0, B, T, cout)      # the step's d logits (bf16 values on the bf16 tier: exact in fp32)
  m(_inputs(x, cond))           # x[:, :-1] holds what the step reads through its T + 1 frame stride
  m.backward(dl)
  return g_ts, m.handle.flat_grads


def test_backward_mixture_c4_bit_equal_to_train_step():
  m, _, _, x, cond, _, _, _, _ = config_parity.setup('c4')
  B, T = config_parity.SHAPES['c4'][:2]
  g_ts, g = _train_step_then_backward_of_its_dlogits(m, x, cond, B, T)
  assert int(m.handle.lib.wn_stack_backward_layers(m.handle.h)) == m.blocks
  assert torch.equal(g_ts, g)


def test_backward_mixture_fp32_bit_equal_to_train_step():
  B, T = 2, 200
  m, _, _, x, cond = _model(SMALL_MODELS['logistic_cond'], B, T, 'fp32', COND_IN)
  g_ts, g = _train_step_then_backward_of_its_dlogits(m, x, cond, B, T)
  assert torch.equal(g_ts, g)


def test_backward_categorical_loss_gradient_reproduces_train_step():
  """dpred = d(mean cross entropy)/d p = -onehot(target) / (B p_target) through backward gives train_step's gradients."""
  B, T = 2, 200
  m, _, _, x, cond = _model(SMALL_MODELS['categorical_multidil'], B, T, 'fp32', 0)
  m.train_step(x)
  g_ts = m.get_grads()
  pred = m(x[:, :-1])
  y = m.prepare_target(x[:, 1:]).reshape(B, T, 1)
  p_y = torch.gather(pred, 2, y)
  dp = torch.zeros_like(pred).scatter_(2, y, -1.0 / (B * p_y))
  m.backward(dp)
  g = m.get_grads()
  for k in g_ts:
    assert rel_err(g[k], g_ts[k]) < TOL_FP32, (k, rel_err(g[k], g_ts[k]))


# ------------------------------------------------------------------ state and errors
def test_backward_state_errors():
  from wavenets_b200.optimizers import Adam
  kw = SMALL_MODELS['categorical_multidil']
  B, T = 2, 120
  m, _, _, x, _ = _model(kw, B, T, 'fp32', 0)
  h = m.handle
  dp = torch.as_tensor(_dpred(m, B, T), device=h.device)
  with pytest.raises(RuntimeError):
    m.backward(dp)              # no call yet
  assert h.lib.wn_backward(h.h, h.ptr(dp), None, h.stream_ptr()) == -4      # WN_ERR_STATE at the C ABI
  m(x[:, :-1])
  with pytest.raises(ValueError):
    m.backward(dp[:, :-1])
  m.train_step(x)
  with pytest.raises(RuntimeError):
    m.backward(dp)
  m(x[:, :-1])
  m.set_weights(m.get_weights())
  with pytest.raises(RuntimeError):
    m.backward(dp)
  m.compile(optimizer=Adam(learning_rate=1e-3))
  m(x[:, :-1])
  m.optimizer.apply_gradients(m)
  with pytest.raises(RuntimeError):
    m.backward(dp)
  m(x[:, :-1])
  m.generate(4, batch_size=1, deterministic=True)
  with pytest.raises(RuntimeError):
    m.backward(dp)
  m(x[:, :-1])
  m.backward(dp)                # and valid again after a call


@pytest.mark.parametrize('precision,name', [('fp32', 'cond_skip'), ('bf16', 'r256'), ('bf16', 'c2')])
def test_backward_twice_is_bit_identical(precision, name):
  if name == 'c2':
    m, _, _, x, cond, _, _, _, _ = config_parity.setup('c2', 0.1)
    B, T = config_parity.SHAPES['c2'][:2]
    training = True             # (Philox masks drawn by the call, reused by both backward passes)
  else:
    kw = SMALL_MODELS[name] if precision == 'fp32' else _bf16_models()[name]
    B, T = 3, 700
    m, _, _, x, cond = _model(kw, B, T, precision, COND_IN if kw.get('conditioning') else 0)
    training = False
  dp = _dpred(m, B, T)
  m(_inputs(x, cond), training=training)
  d1 = m.backward(dp)
  g1 = m.handle.flat_grads.clone()
  d2 = m.backward(dp)
  assert torch.equal(g1, m.handle.flat_grads)
  if d1 is not None:
    assert torch.equal(d1, d2)


@pytest.mark.parametrize('precision,name', [('fp32', 'cond_skip'), ('bf16', 'r256')])
def test_call_and_backward_leave_train_step_unchanged(precision, name):
  kw = SMALL_MODELS[name] if precision == 'fp32' else _bf16_models()[name]
  B, T = 3, 700
  cond_in = COND_IN if kw.get('conditioning') else 0
  runs = []
  for with_backward in (False, True):
    m, _, _, x, cond = _model(kw, B, T, precision, cond_in)
    data = (x, cond) if cond is not None else x
    m.train_step(data)
    if with_backward:
      m(_inputs(x, cond))
      m.backward(_dpred(m, B, T))
    out = m.train_step(data)
    runs.append((out['loss'], m.handle.flat_grads.clone()))
  assert runs[0][0] == runs[1][0]
  assert torch.equal(runs[0][1], runs[1][1])


# ------------------------------------------------------------------ data parallel
def _free_port():
  s = socket.socket()
  s.bind(('127.0.0.1', 0))
  port = s.getsockname()[1]
  s.close()
  return port


@pytest.mark.parametrize('native', [1, 0])
def test_two_gpu_backward_allreduced_grads_equal_single_gpu(native):
  if torch.cuda.device_count() < 2:
    pytest.skip('needs 2 GPUs on one box')
  cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
         '--master-port', str(_free_port()), os.path.join(ROOT, 'scripts', 'dp_backward_check.py'), '--native', str(native)]
  r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
  lines = [json.loads(l) for l in r.stdout.splitlines() if l.startswith('{')]
  assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
  assert len(lines) == 2 and all(l['ok'] for l in lines), lines
