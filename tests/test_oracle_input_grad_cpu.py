"""Pins tests/test_gpu_input_grad.py's reference for WaveNet.backward(input_grad=True): d loss / d x from torch autograd of
sum(call(x) * dpred) over oracle/faithful.py's float64 forward (x.requires_grad) must match central differences of
oracle/wavenet_oracle.model_forward, be exactly zero past the last position with a nonzero dpred (the model is causal), and
exactly zero in a batch row whose dpred is zero (rows never mix)."""
import numpy as np
import pytest
import torch

from oracle import faithful
from oracle import wavenet_oracle as wo
from tests.util import COND_IN, SMALL_MODELS, make_inputs, oracle_config, rel_err


def input_grad_reference(p_np, cfg: wo.Config, x, cond_in, dpred, faithful_mode=False, slope_masks=None, keep_masks=None):
  """d sum(pred * dpred) / d x, pred = WaveNet.call(x, cond_in) (softmax probabilities or mixture parameters).
  x (B,T,1), cond_in (B,cond_in) or None, dpred (B,T,C).  Returns dx (B,T) float64 numpy."""
  R = faithful.Rounding(faithful_mode)
  dt = torch.float64
  p = {k: torch.tensor(np.asarray(v), dtype=dt) for k, v in p_np.items()}
  xx = torch.tensor(np.asarray(x), dtype=dt, requires_grad=True)
  c = None if cond_in is None else torch.tensor(np.asarray(cond_in), dtype=dt)
  logits = faithful.forward_logits(p, cfg, xx, c, R, None, slope_masks, keep_masks)
  if faithful_mode:
    logits = logits.to(torch.float32).to(dt)      # the logits live in fp32
  pred = torch.softmax(logits, dim=-1) if cfg.sampling_function == 'categorical' else logits
  (pred * torch.tensor(np.asarray(dpred), dtype=dt)).sum().backward()
  return xx.grad.numpy()[:, :, 0]


def _case(name, B=2, T=40):
  kw = SMALL_MODELS[name]
  cond_in = COND_IN if kw.get('conditioning') else 0
  cfg = oracle_config(kw, cond_in)
  p = wo.init_params(cfg, seed=1)
  x, cond = make_inputs(B, T, cond_in)
  x = x[:, :-1].astype(np.float64)
  cond = None if cond is None else cond.astype(np.float64)
  out, _ = wo.model_forward(p, cfg, x, cond)
  dpred = np.random.default_rng(7).standard_normal(out.shape)
  return p, cfg, x, cond, dpred


@pytest.mark.parametrize('name', sorted(SMALL_MODELS))
def test_input_grad_reference_matches_central_differences(name):
  p, cfg, x, cond, dpred = _case(name)
  dx = input_grad_reference(p, cfg, x, cond, dpred)

  def f(xv):
    out, _ = wo.model_forward(p, cfg, xv, cond)
    return float((out * dpred).sum())
  fd = np.zeros(x.shape[:2])
  for i in np.ndindex(fd.shape):
    xp, xm = x.copy(), x.copy()
    xp[i + (0,)] += 1e-6
    xm[i + (0,)] -= 1e-6
    fd[i] = (f(xp) - f(xm)) / 2e-6
  assert rel_err(dx, fd) < 1e-5, rel_err(dx, fd)


@pytest.mark.parametrize('name', sorted(SMALL_MODELS))
def test_input_grad_reference_is_causal_and_keeps_rows_apart(name):
  p, cfg, x, cond, dpred = _case(name)
  last = 25
  dp = dpred.copy()
  dp[:, last + 1:] = 0
  dp[1] = 0
  dx = input_grad_reference(p, cfg, x, cond, dp)
  assert np.all(dx[:, last + 1:] == 0)
  assert np.all(dx[1] == 0)
  assert np.abs(dx[0, :last + 1]).max() > 0
