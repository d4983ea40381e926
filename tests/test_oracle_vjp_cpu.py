"""Pins tests/test_gpu_model_backward.py's reference for WaveNet.backward: torch autograd of sum(call(x) * dpred) over
oracle/faithful.py's float64 forward must equal oracle/wavenet_oracle.model_backward (the hand-written adjoint every train_step
parity test rests on), fed the float64 softmax VJP of dpred (categorical) or dpred itself (mixture parameters)."""
import numpy as np
import pytest

from oracle import wavenet_oracle as wo
from tests.test_gpu_model_backward import vjp_reference
from tests.util import COND_IN, SMALL_MODELS, make_inputs, oracle_config, rel_err


@pytest.mark.parametrize('name', sorted(SMALL_MODELS))
def test_vjp_reference_matches_oracle_model_backward(name):
  kw = SMALL_MODELS[name]
  B, T = 2, 40
  cond_in = COND_IN if kw.get('conditioning') else 0
  cfg = oracle_config(kw, cond_in)
  p = wo.init_params(cfg, seed=1)
  x, cond = make_inputs(B, T, cond_in)
  x = x[:, :-1].astype(np.float64)
  cond = None if cond is None else cond.astype(np.float64)
  logits, cache = wo.model_forward(p, cfg, x, cond, return_logits=True)
  cout = logits.shape[-1]
  dpred = np.random.default_rng(7).standard_normal((B, T, cout))
  if cfg.sampling_function == 'categorical':
    e = np.exp(logits - logits.max(axis=-1, keepdims=True))
    prob = e / e.sum(axis=-1, keepdims=True)
    dlogits = prob * (dpred - (prob * dpred).sum(axis=-1, keepdims=True))
  else:
    dlogits = dpred
  g_o = wo.model_backward(p, cfg, cache, dlogits)
  g, dcond = vjp_reference(p, cfg, x, cond, dpred, faithful_mode=False)
  assert set(g) == set(p)
  for k in p:
    ref = g_o.get(k, np.zeros(p[k].shape))
    if np.abs(ref).max() == 0:
      assert np.abs(g[k]).max() == 0, k
      continue
    assert rel_err(g[k], ref) < 1e-10, (k, rel_err(g[k], ref))
  assert (dcond is None) == (cond is None)
  if cond is not None:
    # d cond (through the mapping MLP; wavenet_oracle.model_backward stops at the mapping weights): central differences
    def f(c):
      out, _ = wo.model_forward(p, cfg, x, c)
      return float((out * dpred).sum())
    fd = np.zeros_like(cond)
    for i in np.ndindex(cond.shape):
      cp, cm = cond.copy(), cond.copy()
      cp[i] += 1e-6
      cm[i] -= 1e-6
      fd[i] = (f(cp) - f(cm)) / 2e-6
    assert rel_err(dcond, fd) < 1e-5, rel_err(dcond, fd)
