"""WaveNetLayer with a conditioning SEQUENCE (B,T,Cc) that varies in time (layers.py:115-120,203-204): `call` runs
`wn_layer_forward_seq`, `backward` returns dcond (B,T,Cc).  Both tiers against the fp64 oracle, dropout, causality and
batch isolation of the new contraction segment, agreement with the time-constant bias path, determinism, errors."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import wavenet_oracle as wo
from tests.util import rel_err, rel_l2

pytestmark = pytest.mark.gpu
TOL = 1e-4                                                         # fp32 tier (as test_gpu_parity_fp32.py)
TOL_OUT, TOL_GRAD, TOL_GRAD_PWL, MIN_COS_PWL = 1e-2, 1.5e-2, 1e-1, 0.995   # bf16 tier (as test_gpu_parity_bf16.py)

FP32_LAYERS = {
  'single': dict(dilation_rate=4, channels=8),
  'multi_leaky': dict(dilation_rate=[1, 2, 4], activation='leaky_relu', channels=8, dilation_channels=12, skip_channels=6),
  'nores': dict(dilation_rate=[3, 1], activation='tanh', channels=8, residual=False),
  'k3': dict(kernel=3, dilation_rate=[1, 3], activation='relu', channels=8, skip_channels=5),
  'k4': dict(kernel=4, dilation_rate=[2], channels=8),
}

BF16_LAYERS = {
  'r32_tanh': dict(dilation_rate=[1, 2], activation='tanh', channels=32, skip_channels=32),
  'r64_k3': dict(kernel=3, dilation_rate=4, channels=64),
  # R = D = 128 / 256 with residual: the shapes the time-constant path runs through the fused block kernel
  'r128': dict(dilation_rate=2, channels=128, skip_channels=128),
  # R = D = S = 256: a handle eligible for the grouped weight-gradient launch
  'r256_leaky': dict(dilation_rate=[1, 2], activation='leaky_relu', channels=256, skip_channels=256),
  'r256_k3': dict(kernel=3, dilation_rate=3, channels=256),
  # K = 4: four taps + the sequence = five segments of the tcgen05 contraction
  'r64_k4_tanh': dict(kernel=4, dilation_rate=[1, 4], activation='tanh', channels=64, skip_channels=32),
  'r256_k4': dict(kernel=4, dilation_rate=2, channels=256, skip_channels=256),
}


def _oracle_cfg(kw):
  dils = kw['dilation_rate'] if isinstance(kw['dilation_rate'], list) else [kw['dilation_rate']]
  return dict(dilations=dils, activation=kw.get('activation'), residual=kw.get('residual', True),
              has_skip=kw.get('skip_channels') is not None, condition=True)


def _smooth(kw):
  dils = kw['dilation_rate'] if isinstance(kw['dilation_rate'], list) else [kw['dilation_rate']]
  return len(dils) == 1 or kw.get('activation') in (None, 'tanh', 'sigmoid')


def _cos(a, b):
  a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
  return float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-300))


def _make(kw, B, T, Cc, precision, seed=3, **extra):
  """Built layer with random weights (kernels scaled by 1/sqrt(fan_in)), inputs, a time-varying sequence, fp64 weights."""
  from wavenets_b200 import WaveNetLayer
  rng = np.random.default_rng(seed)
  R = kw['channels']
  lay = WaveNetLayer(**kw, condition=True, precision=precision, **extra)
  lay.build(((B, T, R), (B, T, Cc)))
  w = {}
  for n, shape in zip(lay.weight_names, lay._handle.shapes):
    if n.endswith('kernel'):
      w[n] = (rng.standard_normal(shape) / np.sqrt(np.prod(shape[:-1]))).astype(np.float32)
    else:
      w[n] = (rng.standard_normal(shape) * 0.1).astype(np.float32)
  lay.set_weights(w)
  x = rng.standard_normal((B, T, R)).astype(np.float32)
  cond = rng.standard_normal((B, T, Cc)).astype(np.float32)
  p = {'block0/' + k: v.astype(np.float64) for k, v in w.items()}
  return lay, x, cond, p, rng


def _run(lay, x, cond, dxo, dsk, training=False):
  xo, sk = lay.call((x, cond), training=training)
  dx, dcond = lay.backward(dxo, dsk)
  return (xo.cpu().numpy(), sk.cpu().numpy(), dx.cpu().numpy(), dcond.cpu().numpy(), lay.get_grads())


def _oracle(kw, p, x, cond, dxo, dsk, keep=None, rate=0.0):
  lc = _oracle_cfg(kw)
  xo, sk, cache = wo.layer_forward(p, 'block0', lc, x.astype(np.float64), cond.astype(np.float64), keep=keep, rate=rate)
  dx, dcond, g = wo.layer_backward(p, 'block0', lc, cache, dxo.astype(np.float64), dsk.astype(np.float64))
  return xo, sk, dx, dcond, {k[len('block0/'):]: v for k, v in g.items()}


def _check_fp32(got, ref):
  names = ('x_out', 'skip', 'dx', 'dcond')
  for n, a, b in zip(names, got[:4], ref[:4]):
    assert a.shape == b.shape, n
    assert rel_err(a, b) < TOL, (n, rel_err(a, b))
  for k, v in ref[4].items():
    assert rel_err(got[4][k], v) < TOL, (k, rel_err(got[4][k], v))


def _check_bf16(kw, got, ref):
  for n, a, b in zip(('x_out', 'skip'), got[:2], ref[:2]):
    assert rel_l2(a, b) < TOL_OUT, (n, rel_l2(a, b))
  grads = [('dx', got[2], ref[2]), ('dcond', got[3], ref[3])] + [(k, got[4][k], v) for k, v in ref[4].items()]
  for n, a, b in grads:
    assert a.shape == b.shape, n
    e = rel_l2(a, b)
    if _smooth(kw):
      assert e < TOL_GRAD, (n, e)
    else:
      assert e < TOL_GRAD_PWL and _cos(a, b) >= MIN_COS_PWL, (n, e, _cos(a, b))


def _upstream(rng, x_out_shape, skip_shape):
  return rng.standard_normal(x_out_shape).astype(np.float32), rng.standard_normal(skip_shape).astype(np.float32)


# ---------------------------------------------------------------- 1. fp32 tier against the oracle
@pytest.mark.parametrize('Cc', [5, 80])
@pytest.mark.parametrize('name', sorted(FP32_LAYERS))
def test_fp32_sequence_matches_oracle(name, Cc):
  kw = FP32_LAYERS[name]
  B, T = 2, 37
  lay, x, cond, p, rng = _make(kw, B, T, Cc, 'fp32')
  S = kw.get('skip_channels') or kw['channels']
  dxo, dsk = _upstream(rng, x.shape, (B, T, S))
  got = _run(lay, x, cond, dxo, dsk)
  _check_fp32(got, _oracle(kw, p, x, cond, dxo, dsk))


# ---------------------------------------------------------------- 2. bf16 tier against the fp64 oracle
@pytest.mark.parametrize('Cc', [32, 80])
@pytest.mark.parametrize('name', sorted(BF16_LAYERS))
def test_bf16_sequence_matches_oracle(name, Cc):
  kw = BF16_LAYERS[name]
  B, T = 3, 333
  lay, x, cond, p, rng = _make(kw, B, T, Cc, 'bf16')
  S = kw.get('skip_channels') or kw['channels']
  dxo, dsk = _upstream(rng, x.shape, (B, T, S))
  got = _run(lay, x, cond, dxo, dsk)
  _check_bf16(kw, got, _oracle(kw, p, x, cond, dxo, dsk))


# ---------------------------------------------------------------- 3. dropout masks x only
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_dropout_with_injected_mask(precision):
  kw = dict(dilation_rate=[1, 2], activation='tanh', channels=8 if precision == 'fp32' else 64, skip_channels=None)
  kw = {k: v for k, v in kw.items() if v is not None}
  B, T, Cc, rate = 2, 150, 7, 0.3
  lay, x, cond, p, rng = _make(kw, B, T, Cc, precision, dropout=rate)
  keep = rng.random((B, T, kw['channels'])) >= rate
  lay.set_dropout_mask(keep)
  dxo, dsk = _upstream(rng, x.shape, x.shape)
  got = _run(lay, x, cond, dxo, dsk, training=True)
  ref = _oracle(kw, p, x, cond, dxo, dsk, keep=keep, rate=rate)
  if precision == 'fp32':
    _check_fp32(got, ref)
  else:
    _check_bf16(kw, got, ref)


# ---------------------------------------------------------------- 4. causality and batch isolation of the sequence segment
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_sequence_row_is_exact(precision):
  kw = dict(dilation_rate=[1, 4], activation='tanh', channels=8 if precision == 'fp32' else 64, skip_channels=16 if precision == 'fp32' else 32)
  B, T, Cc = 3, 200, 9
  lay, x, cond, p, rng = _make(kw, B, T, Cc, precision)
  xo0, sk0 = [a.cpu().numpy() for a in lay((x, cond))]
  b0, t0 = 1, 130
  c2 = cond.copy()
  c2[b0, t0, :] += 1.0
  xo1, sk1 = [a.cpu().numpy() for a in lay((x, c2))]
  for a0, a1 in ((xo0, xo1), (sk0, sk1)):
    diff = np.any(a0 != a1, axis=-1)
    assert diff[b0, t0]
    diff[b0, t0] = False
    assert not diff.any(), np.argwhere(diff)[:5]


# ---------------------------------------------------------------- 5. a time-constant sequence through both paths
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_constant_sequence_matches_bias_path(precision):
  kw = dict(dilation_rate=[1, 2], activation='tanh', channels=8 if precision == 'fp32' else 128, skip_channels=6 if precision == 'fp32' else 64)
  B, T, Cc = 2, 140, 11
  lay, x, _, p, rng = _make(kw, B, T, Cc, precision)
  c2 = rng.standard_normal((B, Cc)).astype(np.float32)
  c3 = np.repeat(c2[:, None, :], T, axis=1)
  dxo, dsk = _upstream(rng, x.shape, (B, T, kw['skip_channels']))
  # existing bias path: a time-constant (B,T,Cc) sequence goes through wn_layer_forward_ex with (B,Cc)
  xo_b, sk_b, dx_b, dc_b, g_b = _run(lay, x, c3, dxo, dsk)
  assert dc_b.shape == (B, Cc)
  # the same sequence through wn_layer_forward_seq
  h = lay._handle
  dev = h.device
  xt, ct = torch.from_numpy(x).to(dev), torch.from_numpy(c3).to(dev)
  xo = torch.empty((B, T, kw['channels']), device=dev)
  sk = torch.empty((B, T, kw['skip_channels']), device=dev)
  rc = h.lib.wn_layer_forward_seq(h.h, 0, h.ptr(xt), h.ptr(ct), B, T, 0, h.ptr(xo), h.ptr(sk), h.stream_ptr())
  assert rc == 0, h.lib.wn_last_error()
  dxo_t, dsk_t = torch.from_numpy(dxo).to(dev), torch.from_numpy(dsk).to(dev)
  dx, dc = torch.empty_like(xt), torch.empty_like(ct)
  rc = h.lib.wn_layer_backward(h.h, 0, h.ptr(dxo_t), h.ptr(dsk_t), h.ptr(dx), h.ptr(dc), h.stream_ptr())
  assert rc == 0, h.lib.wn_last_error()
  g_s = lay.get_grads()
  xo, sk, dx, dc = (a.cpu().numpy() for a in (xo, sk, dx, dc))
  if precision == 'fp32':
    assert rel_err(xo, xo_b) <= 1e-5 and rel_err(sk, sk_b) <= 1e-5
    err, tol = rel_err, TOL
  else:
    assert rel_l2(xo, xo_b) < TOL_OUT and rel_l2(sk, sk_b) < TOL_OUT
    err, tol = rel_l2, TOL_GRAD
  assert err(dx, dx_b) < tol
  assert err(dc.astype(np.float64).sum(axis=1), dc_b) < tol
  for k in ('conv_cond/kernel', 'conv_cond/bias'):
    assert err(g_s[k], g_b[k]) < tol, (k, err(g_s[k], g_b[k]))


# ---------------------------------------------------------------- 6. determinism
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_sequence_run_to_run_bit_identical(precision):
  kw = dict(dilation_rate=[1, 2], activation='tanh', channels=8 if precision == 'fp32' else 64, skip_channels=16 if precision == 'fp32' else 64)
  B, T, Cc = 3, 333, 80
  lay, x, cond, p, rng = _make(kw, B, T, Cc, precision)
  dxo, dsk = _upstream(rng, x.shape, (B, T, kw['skip_channels']))
  a = _run(lay, x, cond, dxo, dsk)
  b = _run(lay, x, cond, dxo, dsk)
  for u, v in zip(a[:4], b[:4]):
    assert np.array_equal(u, v)
  for k in a[4]:
    assert np.array_equal(a[4][k], b[4][k]), k


# ---------------------------------------------------------------- 7. errors and state
def test_wrong_cond_width_raises():
  kw = FP32_LAYERS['single']
  lay, x, cond, p, rng = _make(kw, 2, 20, 5, 'fp32')
  with pytest.raises(ValueError, match='channels'):
    lay((x, rng.standard_normal((2, 20, 6)).astype(np.float32)))


def test_forward_seq_rejects_null_and_unconditioned():
  from wavenets_b200 import WaveNetLayer, _lib
  B, T = 2, 16
  lay = WaveNetLayer(dilation_rate=1, channels=8)
  lay.build((B, T, 8))
  h = lay._handle
  x = torch.zeros((B, T, 8), device=h.device)
  c = torch.zeros((B, T, 3), device=h.device)
  xo, sk = torch.empty_like(x), torch.empty_like(x)
  rc = h.lib.wn_layer_forward_seq(h.h, 0, h.ptr(x), h.ptr(c), B, T, 0, h.ptr(xo), h.ptr(sk), h.stream_ptr())
  assert rc == _lib.WN_ERR_VALUE
  lay2, x2, c2, _, _ = _make(FP32_LAYERS['single'], B, T, 3, 'fp32')
  h2 = lay2._handle
  x2 = torch.from_numpy(x2).to(h2.device)
  rc = h2.lib.wn_layer_forward_seq(h2.h, 0, h2.ptr(x2), C.c_void_p(0), B, T, 0, h2.ptr(torch.empty_like(x2)), h2.ptr(torch.empty_like(x2)),
                                   h2.stream_ptr())
  assert rc == _lib.WN_ERR_VALUE


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_alternating_constant_and_sequence_calls(precision):
  kw = dict(dilation_rate=[1, 2], activation='tanh', channels=8 if precision == 'fp32' else 64)
  B, T, Cc = 2, 90, 6
  lay, x, cond, p, rng = _make(kw, B, T, Cc, precision)
  dxo, dsk = _upstream(rng, x.shape, x.shape)
  c2 = rng.standard_normal((B, Cc)).astype(np.float32)
  check = _check_fp32 if precision == 'fp32' else (lambda g, r: _check_bf16(kw, g, r))
  for step in range(2):
    got = _run(lay, x, cond, dxo, dsk)
    assert got[3].shape == (B, T, Cc)
    check(got, _oracle(kw, p, x, cond, dxo, dsk))
    got = _run(lay, x, c2, dxo, dsk)
    assert got[3].shape == (B, Cc)
    check(got, _oracle(kw, p, x, c2, dxo, dsk))
  # backward follows the last forward: a sequence forward, then the constant one, then backward
  lay((x, cond))
  xo, sk = lay((x, c2))
  dx, dcond = lay.backward(dxo, dsk)
  assert tuple(dcond.shape) == (B, Cc)
  ref = _oracle(kw, p, x, c2, dxo, dsk)
  check((xo.cpu().numpy(), sk.cpu().numpy(), dx.cpu().numpy(), dcond.cpu().numpy(), lay.get_grads()), ref)
