"""CPU tests of the oracle (no GPU): known-answer tests derived by hand from the reference
source, and three-way gradient agreement (manual backward / torch autograd / finite differences).
The reference ships no tests or golden vectors (SURVEY.md section 4): parity is UNPINNED and these
are the pins we create ourselves."""
import math

import numpy as np
import pytest

from oracle import torch_ref as tr
from oracle import wavenet_oracle as wo
from tests.util import COND_IN, SMALL_MODELS, make_inputs, oracle_config, rel_err


def test_dilation_schedule_defaults_yaml():
  # defaults.yaml:9-18: K=2, 5 blocks x 5 layers, bound 256 -> powers 1..128 (never 256), RF 768
  cfg = wo.Config(channels=32, blocks=5, layers_per_block=5, dilation_bound=256, final_layers_channels=[128, 256])
  per_block, rf = wo.dilation_schedule(cfg)
  assert per_block == [[1, 2, 4, 8, 16], [32, 64, 128, 1, 2], [4, 8, 16, 32, 64], [128, 1, 2, 4, 8], [16, 32, 64, 128, 1]]
  assert rf == 768
  assert wo.num_params(cfg) == 170816
  f = wo.flops_fwd_per_sample(cfg)
  assert f == {'dilated': 122880, 'pointwise': 10240, 'head': 204800, 'input': 128, 'total': 338048}


def test_dilation_schedule_deep():
  cfg = wo.Config(channels=8, blocks=40, layers_per_block=1, dilation_bound=1024, final_layers_channels=[])
  per_block, rf = wo.dilation_schedule(cfg)
  assert [d[0] for d in per_block[:11]] == [1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1]
  assert rf == 1 + 4 * 1023 + 1 == 4094


def test_validation_errors():
  with pytest.raises(ValueError):
    wo.Config(kernel_size=1).validate()
  with pytest.raises(ValueError):
    wo.Config(dilation_bound=100).validate()
  with pytest.raises(ValueError):
    wo.Config(sampling_function='categorical', num_mixtures=3).validate()
  with pytest.raises(ValueError):
    wo.Config(conditioning='speaker').validate()


def test_discretize_edges():
  # model.py:152-153: boundaries linspace(-1,1,257)[1:-1]; idx = #boundaries <= x
  x = np.array([-1.0, -1e-30, 0.0, 1.0, 0.999, -0.9921875, np.nextafter(np.float32(-0.9921875), np.float32(-2))], dtype=np.float32)
  assert wo.discretize(x, 8).tolist() == [0, 127, 128, 255, 255, 1, 0]
  # naive floor((x+1)*128) is wrong for tiny negatives: this is why the quantiser is comparison based
  assert int(math.floor((np.float32(-1e-30) + np.float32(1.0)) * 128)) == 128
  # 16 bit: every boundary exactly representable in fp32
  b = np.linspace(-1, 1, 2 ** 16 + 1)[1:-1]
  assert np.array_equal(b.astype(np.float32).astype(np.float64), b)
  assert wo.discretize(np.array([0.0, 1.0, -1.0], np.float32), 16).tolist() == [32768, 65535, 0]


def test_causal_conv_indices():
  # Keras causal Conv1D: tap k multiplies x[t-(K-1-k)d]; zero left padding per batch row
  x = np.arange(1, 13, dtype=np.float64).reshape(2, 6, 1)
  W = np.array([10.0, 1.0]).reshape(2, 1, 1)
  y = wo.causal_conv_fwd(x, W, np.zeros(1), dilation=2)
  assert y[0, :, 0].tolist() == [1, 2, 13, 24, 35, 46]
  assert y[1, :, 0].tolist() == [7, 8, 79, 90, 101, 112]   # no leakage across the batch boundary


def test_mu_law_matches_formula():
  x = np.array([-1.0, -0.5, 0.0, 0.25, 1.0], dtype=np.float32)
  y = wo.mu_law(x)
  assert y[0] == -1.0 and y[-1] == 1.0 and y[2] == 0.0
  np.testing.assert_allclose(y[3], math.log(1 + 255 * 0.25) / math.log(256), rtol=1e-6)


def test_skip_alias_is_pre_residual():
  # layers.py:216-223: with skip_channels=None, skip = conv1(g) BEFORE the residual add
  cfg = wo.Config(channels=4, blocks=1, layers_per_block=1, dilation_bound=2, final_layers_channels=[])
  p = wo.init_params(cfg, seed=3)
  x = np.random.default_rng(0).standard_normal((1, 9, 4))
  lc = wo._layer_cfgs(cfg)[0]
  xo, skip, _ = wo.layer_forward(p, 'block0', lc, x)
  np.testing.assert_allclose(xo - x, skip, atol=1e-12)


def test_causality_and_receptive_field():
  cfg = wo.Config(channels=4, blocks=3, layers_per_block=1, dilation_bound=4, final_layers_channels=[4], bits=8)
  _, rf = wo.dilation_schedule(cfg)   # dilations 1,2,1 -> rf 6
  assert rf == 6
  p = wo.init_params(cfg, seed=2)
  rng = np.random.default_rng(1)
  x = rng.standard_normal((1, 20, 1)) * 0.3
  y0, _ = wo.model_forward(p, cfg, x, return_logits=True)
  t = 15
  for dt, changed in [(1, False), (0, True), (-(rf - 1), True), (-rf, False)]:  # output[t] sees exactly x[t-rf+1..t]
    x2 = x.copy()
    x2[0, t + dt, 0] += 0.5
    y2, _ = wo.model_forward(p, cfg, x2, return_logits=True)
    assert (np.abs(y2[0, t] - y0[0, t]).max() > 1e-9) == changed, (dt, changed)


@pytest.mark.parametrize('name', sorted(SMALL_MODELS))
def test_manual_backward_matches_autograd_and_fd(name):
  kw = SMALL_MODELS[name]
  cond_in = COND_IN if kw.get('conditioning') else 0
  cfg = oracle_config(kw, cond_in)
  p = wo.init_params(cfg, seed=1)
  x, cond = make_inputs(2, 24, cond_in)
  x = x.astype(np.float64)
  cond = None if cond is None else cond.astype(np.float64)
  loss, g, _ = wo.train_step(p, cfg, x, cond)
  if cfg.l2_reg_factor == 0:
    loss_t, g_t = tr.train_step(p, cfg, x, cond)
    assert abs(loss - loss_t) <= 1e-9 * abs(loss_t)
    for k in g:
      assert rel_err(g[k], g_t[k]) < 1e-8, k
  rng = np.random.default_rng(5)
  for pname in list(p)[::3]:
    idx = tuple(int(rng.integers(0, s)) for s in p[pname].shape)
    eps = 1e-6
    pp = {k: v.copy() for k, v in p.items()}
    pp[pname][idx] += eps
    lp, _, _ = wo.train_step(pp, cfg, x, cond)
    pp[pname][idx] -= 2 * eps
    lm, _, _ = wo.train_step(pp, cfg, x, cond)
    num = (lp - lm) / (2 * eps)
    assert abs(num - g[pname][idx]) <= 1e-4 * max(1.0, abs(num)) + 5e-3 * abs(num), (pname, num, g[pname][idx])


def test_saturated_categorical_loss_three_way():
  """Keras 3's clip inside sparse_categorical_crossentropy with the clip ACTIVE (logits conv scaled x150: clipped class and target
  probabilities): the hand-derived gradient of the NumPy oracle against torch autograd of the independently written torch
  restatement and against central finite differences.  (The golden case `cat_saturated` pins both to the reference source.)"""
  kw = dict(channels=8, blocks=2, layers_per_block=1, dilation_bound=4, final_layers_channels=[16, 16], activation='tanh', bits=6)
  cfg = oracle_config(kw, 0)
  p = wo.init_params(cfg, seed=1)
  p['final2/kernel'] = p['final2/kernel'] * 150.0
  x, _ = make_inputs(2, 60, 0)
  x = x.astype(np.float64)
  loss, g, aux = wo.train_step(p, cfg, x, None)
  pred, _ = wo.model_forward(p, cfg, x[:, :-1], None)
  p_y = np.take_along_axis(pred, wo.discretize(x[:, 1:, 0], 6)[..., None], -1)[..., 0]
  assert 0.1 < (p_y < 1e-7).mean() < 0.9 and (pred < 1e-7).mean() > 0.1
  # a clipped target contributes -log(1e-7) + log(sum of clipped probabilities) and no gradient through its own probability
  assert abs(aux['loss_per_sample'].max() + np.log(1e-7)) < 1e-3
  loss_t, g_t = tr.train_step(p, cfg, x, None)
  assert abs(loss - loss_t) <= 1e-9 * abs(loss_t)
  for k in g:
    assert rel_err(g[k], g_t[k]) < 1e-7, k
  rng = np.random.default_rng(6)
  for pname in ('final2/kernel', 'final2/bias', 'final1/kernel', 'block1/dil0/kernel', 'causal/kernel'):
    idx = tuple(int(rng.integers(0, s)) for s in p[pname].shape)
    eps = 1e-7
    pp = {k: v.copy() for k, v in p.items()}
    pp[pname][idx] += eps
    lp, _, _ = wo.train_step(pp, cfg, x, None)
    pp[pname][idx] -= 2 * eps
    lm, _, _ = wo.train_step(pp, cfg, x, None)
    num = (lp - lm) / (2 * eps)
    assert abs(num - g[pname][idx]) <= 1e-4 * max(1.0, abs(num)) + 5e-3 * abs(num), (pname, num, g[pname][idx])


@pytest.mark.parametrize('bits', [1, 16])
@pytest.mark.parametrize('clipped', [False, True])
def test_categorical_loss_and_dlogits_at_extreme_class_counts(bits, clipped):
  """loss_and_dlogits at 2 and 65,536 classes (the GPU class-count tests rest on it there) against torch autograd of the torch
  restatement, with the Keras 3 clip inactive, or active on part of the targets and on many entries per row."""
  import torch
  C = 2 ** bits
  cfg = oracle_config(dict(channels=8, blocks=1, final_layers_channels=[], dilation_bound=2, bits=bits), 0)
  rng = np.random.default_rng(bits)
  B, T = 2, 12
  y = rng.uniform(-1, 1, (B, T, 1))
  idx = wo.discretize(y[..., 0], bits)
  logits = rng.standard_normal((B, T, C)) * (30.0 if clipped else 0.3)
  if clipped:       # every other row: the target at the row's maximum, so that some targets stay un-clipped
    rows = np.arange(T) % 2 == 0
    top = logits.max(-1)
    np.put_along_axis(logits, idx[..., None], np.where(rows, top, np.take_along_axis(logits, idx[..., None], -1)[..., 0])[..., None], -1)
  loss, d = wo.loss_and_dlogits(cfg, logits, y, 0.5)
  lt = torch.tensor(logits, requires_grad=True)
  loss_t = tr.loss_per_sample(cfg, lt, torch.tensor(y))
  (loss_t.sum() * 0.5).backward()
  pr = np.exp(logits - logits.max(-1, keepdims=True))
  pr /= pr.sum(-1, keepdims=True)
  p_y = np.take_along_axis(pr, idx[..., None], -1)[..., 0]
  out = (pr < 1e-7) | (pr > 1 - 1e-7)
  if clipped:
    in_y = (p_y >= 1e-7) & (p_y <= 1 - 1e-7)
    assert out.sum(-1).max() >= C // 2 and in_y.any() and not in_y.all()    # clipped and un-clipped targets both present
  else:
    assert not out.any()
  assert rel_err(loss, loss_t.detach().numpy()) < 1e-12
  assert rel_err(d, lt.grad.numpy()) < 1e-10


def test_replica_scaling():
  # compute_average_loss divides by B*replicas: two replicas' grads SUM to the 1-replica grads
  kw = SMALL_MODELS['categorical_multidil']
  cfg = oracle_config(kw)
  p = wo.init_params(cfg, seed=1)
  x, _ = make_inputs(4, 16)
  x = x.astype(np.float64)
  l_all, g_all, _ = wo.train_step(p, cfg, x)
  l0, g0, _ = wo.train_step(p, cfg, x[:2], n_replicas=2)
  l1, g1, _ = wo.train_step(p, cfg, x[2:], n_replicas=2)
  assert abs((l0 + l1) - l_all) < 1e-9
  for k in g_all:
    assert rel_err(g0[k] + g1[k], g_all[k]) < 1e-10


def test_adam_known_answer():
  """Keras 3 Adam, one scalar weight, by hand: t=1: m=0.1g, v=0.001g^2, alpha=lr*sqrt(0.001)/0.1 -> w -= lr*g/(|g|+eps*...)."""
  p = {'w': np.array([1.0])}
  g = {'w': np.array([0.5])}
  st = {}
  p1, st = wo.adam_step(p, g, st, lr=0.1)
  alpha = 0.1 * np.sqrt(1 - 0.999) / (1 - 0.9)
  expect = 1.0 - alpha * (0.1 * 0.5) / (np.sqrt(0.001 * 0.25) + 1e-7)
  assert abs(p1['w'][0] - expect) < 1e-15
  # clipnorm: a gradient of norm 5 is scaled to norm 1 per variable before the moments are updated
  p2, st2 = wo.adam_step({'w': np.array([3.0, 4.0])}, {'w': np.array([3.0, 4.0])}, {}, lr=0.1, clipnorm=1.0)
  assert np.allclose(st2['m']['w'], 0.1 * np.array([0.6, 0.8]))
  assert np.allclose(wo.clip_by_norm(np.array([0.3, 0.4]), 1.0), [0.3, 0.4])


@pytest.mark.parametrize('name', sorted(SMALL_MODELS))
def test_faithful_oracle_exact_mode_equals_oracle(name):
  """oracle/faithful.py with every rounding switched off is the same function as the NumPy oracle (hand-derived backward)
  — the bf16-faithful mode then differs from it ONLY by the roundings listed in its header."""
  from oracle import faithful
  kw = SMALL_MODELS[name]
  cond_in = COND_IN if kw.get('conditioning') else 0
  cfg = oracle_config(kw, cond_in)
  p = wo.init_params(cfg, seed=1)
  x, cond = make_inputs(2, 40, cond_in)
  _, g0, aux = wo.train_step(p, cfg, x.astype(np.float64), None if cond is None else cond.astype(np.float64))
  l1, g1 = faithful.train_step(p, cfg, x, cond, faithful=False)
  assert abs(l1 - aux['loss_no_reg']) <= 1e-9 * abs(l1)
  for k in g0:
    assert rel_err(g1[k], g0[k]) < 1e-9, k
  # faithful mode: bf16 storage moves every gradient a little, never a lot (and never not at all)
  l2, g2 = faithful.train_step(p, cfg, x, cond, faithful=True)
  assert 0 < abs(l2 - l1) <= 1e-2 * abs(l1)
  y1 = faithful.forward(p, cfg, x[:, :-1], cond, faithful=False)
  y2 = faithful.forward(p, cfg, x[:, :-1], cond, faithful=True)
  assert y1.shape == y2.shape and 0 < np.abs(y1 - y2).max() < 5e-2 * np.abs(y1).max() + 1e-3


def test_faithful_rounding_ops():
  """the rounding operators round where they say: value only / gradient only / both"""
  import torch
  from oracle import faithful
  R = faithful.Rounding(True)
  x = torch.tensor([1.0 + 2.0 ** -10, -3.0 - 2.0 ** -9], dtype=torch.float64, requires_grad=True)
  w = torch.tensor([1.0 + 2.0 ** -12, 0.3], dtype=torch.float64)
  (R.fwd(x) * w).sum().backward()
  assert torch.equal(x.grad, w)                                  # value rounded, gradient untouched
  y = R.fwd(x).detach()
  assert float(y[0]) == 1.0 and float(y[1]) == -3.0              # bf16 keeps 8 significant bits (round to nearest even)
  x.grad = None
  (R.bwd(x) * w).sum().backward()
  assert torch.equal(x.grad, w.to(torch.bfloat16).to(torch.float64))
  assert torch.equal(R.bwd(x).detach(), x.detach())


def test_faithful_gate_caches_derivative_coefficients():
  """The bf16 tier caches P = dg/dz_f and Q = dg/dz_s (evaluated on the un-rounded accumulator) instead of z; the faithful oracle's
  gate adjoint is dz = bf16([dg * bf16(P) | dg * bf16(Q)]) — within bf16 rounding of the exact derivative, and exactly that formula."""
  import torch
  from oracle import faithful
  rng = np.random.default_rng(3)
  z = torch.tensor(rng.standard_normal((2, 5, 8)) * 2.0, dtype=torch.float64, requires_grad=True)
  dg = torch.tensor(rng.standard_normal((2, 5, 4)), dtype=torch.float64)
  g = faithful.Rounding(True).gate(z)
  g.backward(dg)
  D = 4
  th, sg = torch.tanh(z[..., :D]).detach(), torch.sigmoid(z[..., D:]).detach()
  P, Q = sg * (1 - th * th), th * sg * (1 - sg)
  b = lambda t: t.to(torch.bfloat16).to(torch.float64)
  want = b(torch.cat([dg * b(P), dg * b(Q)], -1))
  assert torch.equal(z.grad, want)
  exact = torch.cat([dg * P, dg * Q], -1)
  assert float((z.grad - exact).abs().max()) <= 2.0 ** -7 * float(exact.abs().max())
  assert torch.equal(g.detach(), th * sg)                      # the gate itself is evaluated on the un-rounded accumulator


def test_faithful_oracle_dropout_equals_oracle():
  """keep-masks: oracle/faithful.py in exact mode equals the NumPy oracle with the same injected masks (layers.py:192-196:
  the conv branch sees keep * x / (1 - rate), the residual is taken before it)."""
  from oracle import faithful
  cfg = wo.Config(channels=16, blocks=3, layers_per_block=2, dilation_bound=4, skip_channels=16, final_layers_channels=[16], dropout=0.25,
                  activation='leaky_relu')
  p = wo.init_params(cfg, seed=1)
  rng = np.random.default_rng(0)
  x = np.clip(rng.standard_normal((2, 41, 1)) * 0.4, -1, 1)
  keep = [(rng.random((2, 40, 16)) >= 0.25).astype(np.uint8) for _ in range(3)]
  l0, g0, _ = wo.train_step(p, cfg, x, None, keep_masks=keep)
  l1, g1 = faithful.train_step(p, cfg, x, None, faithful=False, keep_masks=keep)
  assert abs(l0 - l1) <= 1e-12 * abs(l0)
  for k in g0:
    assert rel_err(g1[k], g0[k]) < 1e-9, k
  l2, _ = faithful.train_step(p, cfg, x, None, faithful=False)
  assert abs(l2 - l0) > 1e-6 * abs(l0)                         # the masks do something
