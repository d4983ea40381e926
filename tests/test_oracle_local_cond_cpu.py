"""CPU tests of the fp64 oracle's WaveNetLayer with a conditioning SEQUENCE (B,T,Cc) (layers.py:115-120,203-204): its adjoint
against central finite differences, and its agreement with the time-constant (B,Cc) form.  The GPU layer tests compare
`wn_layer_forward_seq` against this oracle."""
import numpy as np
import pytest

from oracle import wavenet_oracle as wo

LAYERS = {
  'multi_leaky': dict(K=2, dilations=[1, 2, 4], activation='leaky_relu', R=6, D=5, S=4),
  'k3': dict(K=3, dilations=[1, 3], activation='tanh', R=6, D=6, S=None),
}


def _setup(spec, B=2, T=13, Cc=3, seed=0):
  rng = np.random.default_rng(seed)
  K, R, D, S = spec['K'], spec['R'], spec['D'], spec['S']
  p = {}
  cin = R
  for j in range(len(spec['dilations'])):
    cout = 2 * D if j == len(spec['dilations']) - 1 else D
    p[f'b/dil{j}/kernel'] = rng.standard_normal((K, cin, cout)) * 0.4
    p[f'b/dil{j}/bias'] = rng.standard_normal(cout) * 0.1
    cin = D
  p['b/conv1/kernel'] = rng.standard_normal((1, D, R)) * 0.4
  p['b/conv1/bias'] = rng.standard_normal(R) * 0.1
  if S is not None:
    p['b/conv_skip/kernel'] = rng.standard_normal((1, D, S)) * 0.4
    p['b/conv_skip/bias'] = rng.standard_normal(S) * 0.1
  p['b/conv_cond/kernel'] = rng.standard_normal((1, Cc, 2 * D)) * 0.4
  p['b/conv_cond/bias'] = rng.standard_normal(2 * D) * 0.1
  lc = dict(dilations=spec['dilations'], activation=spec['activation'], residual=True, has_skip=S is not None, condition=True)
  x = rng.standard_normal((B, T, R))
  cond = rng.standard_normal((B, T, Cc))
  wx = rng.standard_normal((B, T, R))
  ws = rng.standard_normal((B, T, S if S is not None else R))
  return p, lc, x, cond, wx, ws


def _loss(p, lc, x, cond, wx, ws):
  xo, sk, _ = wo.layer_forward(p, 'b', lc, x, cond)
  return float((xo * wx).sum() + (sk * ws).sum())


def _fd(f, a, idx, eps=1e-6):
  a0 = a[idx]
  a[idx] = a0 + eps
  fp = f()
  a[idx] = a0 - eps
  fm = f()
  a[idx] = a0
  return (fp - fm) / (2 * eps)


@pytest.mark.parametrize('name', sorted(LAYERS))
def test_sequence_adjoint_matches_finite_differences(name):
  p, lc, x, cond, wx, ws = _setup(LAYERS[name])
  _, _, cache = wo.layer_forward(p, 'b', lc, x, cond)
  dx, dcond, g = wo.layer_backward(p, 'b', lc, cache, wx, ws)
  assert dcond.shape == cond.shape
  f = lambda: _loss(p, lc, x, cond, wx, ws)   # noqa: E731
  rng = np.random.default_rng(1)
  checks = [(x, dx), (cond, dcond), (p['b/conv_cond/kernel'], g['b/conv_cond/kernel']), (p['b/conv_cond/bias'], g['b/conv_cond/bias'])]
  for arr, grad in checks:
    for _ in range(12):
      idx = tuple(int(rng.integers(0, n)) for n in arr.shape)
      num = _fd(f, arr, idx)
      assert abs(num - grad[idx]) <= 1e-6 * max(1.0, abs(num)), (idx, num, grad[idx])


@pytest.mark.parametrize('name', sorted(LAYERS))
def test_time_constant_sequence_matches_vector_form(name):
  p, lc, x, cond, wx, ws = _setup(LAYERS[name])
  c2 = cond[:, 0, :]
  c3 = np.repeat(c2[:, None, :], x.shape[1], axis=1)
  xo2, sk2, cache2 = wo.layer_forward(p, 'b', lc, x, c2)
  xo3, sk3, cache3 = wo.layer_forward(p, 'b', lc, x, c3)
  assert np.abs(xo3 - xo2).max() <= 1e-12 and np.abs(sk3 - sk2).max() <= 1e-12
  dx2, dc2, g2 = wo.layer_backward(p, 'b', lc, cache2, wx, ws)
  dx3, dc3, g3 = wo.layer_backward(p, 'b', lc, cache3, wx, ws)
  assert dc2.shape == c2.shape and dc3.shape == c3.shape
  assert np.abs(dc3.sum(axis=1) - dc2).max() <= 1e-12 * max(1.0, np.abs(dc2).max())
  assert np.abs(dx3 - dx2).max() <= 1e-12
  for k in g2:
    assert np.abs(g3[k] - g2[k]).max() <= 1e-12 * max(1.0, np.abs(g2[k]).max()), k
