"""The categorical head at every class count wn_create accepts: bits in 1..16, C = 2^bits from 2 to 65,536, on both precision tiers.

The rest of the suite runs 256 classes almost everywhere, where the register-resident softmax kernels take the loss and the softmax
VJP.  Every other class count goes through the generic kernels (softmax_ce_kernel, softmax_vjp_kernel), the bf16 head with
ldd = rup(C, 64) padded d logits, the head GEMMs at N = C up to 65,536, and the sampling / generation / loss_fn kernels at N = C.
The class counts below each reach a different case of the one-warp-per-row loops (c = 4 lane, step 128):
  C = 2       fewer classes than one float4: the element-wise path (a float4 would span two rows)
  C = 4, 16   one partial float4 step, most lanes idle
  C = 128     exactly one float4 step for all 32 lanes
  C >= 512    many steps per lane; at the largest bf16 sizes the head GEMM runs hundreds of column tiles
and B*T = 3 * 37 leaves idle warps in the last CTA of those kernels (8 rows per CTA).

Checkers (no new reference code): oracle/wavenet_oracle in float64 (fp32 tier: <= 1e-4 relative), oracle/faithful with the device's
relu / leaky_relu slope masks (bf16 tier: every gradient tensor within TOL_GRAD_FAITHFUL), and vjp_reference / _loss_grad of
tests/test_gpu_model_backward.py for WaveNet.backward.  Every case prints one JSON line with its largest error (pytest -s)."""
import json

import numpy as np
import pytest
import torch

from oracle import faithful
from oracle import wavenet_oracle as wo
from tests.test_gpu_model_backward import (BF16_COND_IN, TOL_FP32, TOL_GRAD_FAITHFUL, _dpred, _inputs, _loss_grad,
                                           _model, vjp_reference)
from tests.test_gpu_parity_bf16 import BF16_MODELS, TOL_LOSS, TOL_LOSS_FAITHFUL
from tests.util import COND_IN, SMALL_MODELS, device_slope_masks, make_inputs, oracle_config, rel_err, rel_l2

pytestmark = pytest.mark.gpu

BITS = [1, 2, 4, 7, 9, 12, 16]            # C = 2, 4, 16, 128, 512, 4096, 65536
SHAPES = [(3, 37), (2, 64)]               # 111 rows: the last CTA of the one-warp-per-row kernels has 1 of 8 warps busy


def _fp32_kw(bits):
  return dict(SMALL_MODELS['categorical_multidil'], bits=bits)


def _bf16_kw(bits):
  return dict(BF16_MODELS['single_dil_skip_cond'], bits=bits)


def _report(case, **kw):
  print(json.dumps(dict(case=case, **kw)))


def _worst_rel(g, ref):
  """max over tensors of rel_err; a tensor the reference leaves at zero must stay (near) zero on the device"""
  scale = max(np.abs(v).max() for v in ref.values())
  worst = (0.0, None)
  for k in ref:
    if np.abs(ref[k]).max() == 0:
      assert np.abs(g[k]).max() <= 1e-6 * scale, k
      continue
    worst = max(worst, (rel_err(g[k], ref[k]), k))
  return worst


def _worst_faithful(g, ref):
  scale = max(np.linalg.norm(v) for v in ref.values())
  return max((rel_l2(g[k], ref[k]), k) for k in ref if np.linalg.norm(ref[k]) > 1e-9 * scale)


# ------------------------------------------------------------------ 1. fp32 tier: train_step, test_step, call
@pytest.mark.parametrize('bits', BITS)
@pytest.mark.parametrize('BT', SHAPES)
def test_fp32_train_test_call_vs_fp64(bits, BT):
  B, T = BT
  m, cfg, p, x, _ = _model(_fp32_kw(bits), B, T, 'fp32', 0)
  loss_o, g_o, _ = wo.train_step(p, cfg, x.astype(np.float64), None)
  out = m.train_step(x)
  e_loss = abs(out['loss'] - loss_o) / abs(loss_o)
  worst = _worst_rel(m.get_grads(), g_o)
  pred_o, _ = wo.model_forward(p, cfg, x[:, :-1].astype(np.float64), None)
  pred = m(x[:, :-1]).cpu().numpy()
  assert pred.shape == (B, T, 2 ** bits)
  e_pred = rel_err(pred, pred_o)
  e_test = abs(m.test_step(x)['loss'] - loss_o) / abs(loss_o)
  _report('fp32_train_step', bits=bits, BT=BT, loss=e_loss, grad=worst[0], grad_tensor=worst[1], pred=e_pred, test_loss=e_test)
  assert e_loss <= TOL_FP32, (out['loss'], loss_o)
  assert worst[0] < TOL_FP32, worst
  assert e_pred < TOL_FP32
  assert e_test <= TOL_FP32


# ------------------------------------------------------------------ 2. Keras-3 clip at many classes
@pytest.mark.parametrize('bits,scale', [(12, 1000.0), (16, 2500.0)])
def test_fp32_saturated_softmax_keras3_clip_many_classes(bits, scale):
  """test_gpu_parity_fp32.test_saturated_softmax_keras3_clip at 4,096 and 65,536 classes: the last head kernel scaled until part
  of the targets and, at 65,536 classes, tens of thousands of entries per row leave [1e-7, 1 - 1e-7].  delta = sum_j clip(p_j) - p_j
  is then the longest fp32 accumulation of the loss kernel."""
  from wavenets_b200 import WaveNet
  kw = dict(channels=8, blocks=2, layers_per_block=1, dilation_bound=4, final_layers_channels=[16, 16], activation='tanh', bits=bits)
  B, T = 2, 120
  cfg = oracle_config(kw, 0)
  p = {k: v.astype(np.float32).astype(np.float64) for k, v in wo.init_params(cfg, seed=1).items()}
  p['final2/kernel'] = (p['final2/kernel'] * scale).astype(np.float32).astype(np.float64)
  x, _ = make_inputs(B, T, 0)
  m = WaveNet(**kw)
  m.build(x[:, :-1].shape)
  m.set_weights({k: v.astype(np.float32) for k, v in p.items()})
  loss_o, g_o, _ = wo.train_step(p, cfg, x.astype(np.float64), None)
  pred_o, _ = wo.model_forward(p, cfg, x[:, :-1].astype(np.float64), None)
  p_y = np.take_along_axis(pred_o, wo.discretize(x[:, 1:, 0], bits)[..., None], -1)[..., 0]
  n_clipped = (pred_o < 1e-7).sum(-1)
  assert 0.1 < (p_y < 1e-7).mean() < 0.9                     # clipped and un-clipped targets both present
  assert n_clipped.max() > 2 ** bits // 4 and n_clipped.min() < n_clipped.max()
  out = m.train_step(x)
  e_loss = abs(out['loss'] - loss_o) / abs(loss_o)
  worst = _worst_rel(m.get_grads(), g_o)
  e_test = abs(m.test_step(x)['loss'] - loss_o) / abs(loss_o)
  _report('fp32_keras3_clip', bits=bits, max_clipped_per_row=int(n_clipped.max()), loss=e_loss, grad=worst[0], grad_tensor=worst[1],
          test_loss=e_test)
  assert e_loss <= TOL_FP32, (out['loss'], loss_o)
  assert worst[0] < TOL_FP32, worst
  assert e_test <= TOL_FP32


# ------------------------------------------------------------------ 3. bf16 tier: train_step
@pytest.mark.parametrize('bits', BITS)
@pytest.mark.parametrize('BT', SHAPES)
def test_bf16_train_step_vs_faithful(bits, BT):
  """At C = 2 and 16 the d logits are padded to ldd = 64 columns and the head dgrad contracts over all 64."""
  B, T = BT
  kw = _bf16_kw(bits)
  m, cfg, p, x, cond = _model(kw, B, T, 'bf16', BF16_COND_IN)
  out = m.train_step((x, cond))
  loss_o, _, _ = wo.train_step(p, cfg, x.astype(np.float64), cond.astype(np.float64))
  l_f, g_f = faithful.train_step(p, cfg, x, cond, faithful=True, slope_masks=device_slope_masks(m, kw, B, T))
  e_loss = abs(out['loss'] - loss_o) / abs(loss_o)
  e_loss_f = abs(out['loss'] - l_f) / abs(l_f)
  worst = _worst_faithful(m.get_grads(), g_f)
  _report('bf16_train_step', bits=bits, BT=BT, loss_fp64=e_loss, loss_faithful=e_loss_f, grad_faithful=worst[0], grad_tensor=worst[1])
  assert e_loss <= TOL_LOSS, (out['loss'], loss_o)
  assert e_loss_f <= TOL_LOSS_FAITHFUL, (out['loss'], l_f)
  assert worst[0] < TOL_GRAD_FAITHFUL, worst


# ------------------------------------------------------------------ 4. WaveNet.backward
@pytest.mark.parametrize('bits', BITS)
@pytest.mark.parametrize('BT', SHAPES)
def test_backward_fp32_vs_fp64(bits, BT):
  """An N(0,1) d pred through the generic softmax VJP (softmax_vjp_kernel: the register kernel takes 256 classes only)."""
  assert 2 ** bits != 256
  B, T = BT
  kw = dict(SMALL_MODELS['cond_skip'], bits=bits)          # (cond_skip: the fp32 model with a conditioning input, for dcond)
  m, cfg, p, x, cond = _model(kw, B, T, 'fp32', COND_IN)
  dp = _dpred(m, B, T)
  m(_inputs(x, cond))
  dcond = m.backward(dp)
  g_o, dc_o = vjp_reference(p, cfg, x[:, :-1], cond, dp)
  worst = _worst_rel(m.get_grads(), g_o)
  e_dc = rel_err(dcond.cpu().numpy(), dc_o)
  _report('fp32_backward', bits=bits, BT=BT, grad=worst[0], grad_tensor=worst[1], dcond=e_dc)
  assert worst[0] < TOL_FP32, worst
  assert e_dc < TOL_FP32


@pytest.mark.parametrize('bits', BITS)
def test_backward_bf16_vs_faithful(bits):
  assert 2 ** bits != 256
  B, T = 3, 37
  kw = _bf16_kw(bits)
  m, cfg, p, x, cond = _model(kw, B, T, 'bf16', BF16_COND_IN)
  dp = _loss_grad(m, m(_inputs(x, cond)), x)
  dcond = m.backward(dp)
  g_f, dc_f = vjp_reference(p, cfg, x[:, :-1], cond, dp, True, device_slope_masks(m, kw, B, T))
  worst = _worst_faithful(m.get_grads(), g_f)
  e_dc = rel_l2(dcond.cpu().numpy(), dc_f)
  _report('bf16_backward', bits=bits, grad_faithful=worst[0], grad_tensor=worst[1], dcond=e_dc)
  assert worst[0] < TOL_GRAD_FAITHFUL, worst
  assert e_dc < TOL_GRAD_FAITHFUL


@pytest.mark.parametrize('bits', [1, 16])
def test_backward_cross_entropy_gradient_reproduces_train_step(bits):
  """dpred = d(mean cross entropy)/d p = -onehot(target) / (B p_target) through backward gives train_step's gradients
  (nothing is clipped at these weights, so the Keras-3 clip leaves the loss the plain cross entropy)."""
  B, T = 3, 37
  m, _, _, x, _ = _model(_fp32_kw(bits), B, T, 'fp32', 0)
  m.train_step(x)
  g_ts = m.get_grads()
  pred = m(x[:, :-1])
  assert float(pred.min()) >= 1e-7 and float(pred.max()) <= 1 - 1e-7
  y = m.prepare_target(x[:, 1:]).reshape(B, T, 1)
  dp = torch.zeros_like(pred).scatter_(2, y, -1.0 / (B * torch.gather(pred, 2, y)))
  m.backward(dp)
  worst = _worst_rel(m.get_grads(), g_ts)
  _report('backward_ce_vs_train_step', bits=bits, grad=worst[0], grad_tensor=worst[1])
  assert worst[0] < TOL_FP32, worst


# ------------------------------------------------------------------ 5. loss_fn on call's output
@pytest.mark.parametrize('bits', BITS)
def test_loss_fn_on_call_output(bits):
  B, T = 3, 37
  m, cfg, p, x, _ = _model(_fp32_kw(bits), B, T, 'fp32', 0)
  _, _, aux = wo.train_step(p, cfg, x.astype(np.float64), None)
  pred = m(x[:, :-1])
  per_idx = m.loss_fn(m.prepare_target(x[:, 1:]), pred).cpu().numpy()
  per_wave = m.loss_fn(x[:, 1:], pred).cpu().numpy()
  e_idx, e_wave = rel_err(per_idx, aux['loss_per_sample']), rel_err(per_wave, aux['loss_per_sample'])
  _report('loss_fn', bits=bits, int64_target=e_idx, waveform_target=e_wave)
  assert per_idx.shape == per_wave.shape == (B, T)
  assert e_idx < TOL_FP32 and e_wave < TOL_FP32


# ------------------------------------------------------------------ 6. sampling
@pytest.mark.parametrize('bits', BITS)
def test_deterministic_sampling_equals_argmax(bits):
  """sample_waveform(deterministic=True) is the first maximum of the device's own probabilities, mapped to idx / 2^(bits-1) - 1
  (the same float32 arithmetic on both sides: exact)."""
  B, T = 3, 37
  m, cfg, _, x, _ = _model(_fp32_kw(bits), B, T, 'fp32', 0)
  pred = m(x[:, :-1])
  got = m.sample_waveform(pred, deterministic=True).cpu().numpy()
  assert np.array_equal(got, wo.sample_deterministic(cfg, pred.cpu().numpy()))


def test_deterministic_sampling_tie_takes_the_first_index():
  """Equal maxima at classes 70 and 40,000 of 65,536 (lanes 6 and 0 of the warp's stride-32 scan): the first wins, as tf.argmax."""
  from wavenets_b200 import WaveNet
  B, T, C = 2, 9, 2 ** 16
  m = WaveNet(channels=8, blocks=1, final_layers_channels=[], dilation_bound=2, bits=16)
  m.build((B, T, 1))
  rng = np.random.default_rng(4)
  pred = rng.random((B, T, C)).astype(np.float32) * 1e-3
  pred[:, :, 70] = pred[:, :, 40000] = 0.5
  pred[1, 4, 40000] = 0.75                  # (and a row whose single maximum sits in the later lane)
  got = m.sample_waveform(torch.from_numpy(pred).cuda(), deterministic=True).cpu().numpy()
  want = np.full((B, T), 70 / 2 ** 15 - 1, np.float32)
  want[1, 4] = 40000 / 2 ** 15 - 1
  assert np.array_equal(got, want)


def test_categorical_draws_two_classes():
  from wavenets_b200 import WaveNet
  m = WaveNet(channels=8, blocks=1, final_layers_channels=[], dilation_bound=2, bits=1)
  B, T = 64, 4096
  m.build((B, T, 1))
  p = np.array([0.3, 0.7], np.float32)
  pred = torch.from_numpy(np.broadcast_to(p, (B, T, 2)).copy()).cuda()
  s = m.sample_waveform(pred, seed=7)
  assert s.shape == (B, T, 1)
  idx = torch.round(s[..., 0] + 1.0).long().flatten().cpu().numpy()       # idx / 2^0 - 1
  assert idx.min() >= 0 and idx.max() <= 1
  n = idx.size
  freq1 = idx.mean()
  sigma = np.sqrt(p[1] * p[0] / n)
  _report('draws_c2', freq1=float(freq1), p1=float(p[1]), z=float((freq1 - p[1]) / sigma))
  assert abs(freq1 - p[1]) < 5 * sigma
  assert not torch.equal(s, m.sample_waveform(pred, seed=8))
  assert torch.equal(s, m.sample_waveform(pred, seed=7))


def test_categorical_draws_65536_classes_chi_square():
  """Draws over 65,536 classes from a Dirichlet p: chi-square over 64 groups of 1,024 consecutive classes."""
  from scipy import stats
  from wavenets_b200 import WaveNet
  C = 2 ** 16
  m = WaveNet(channels=8, blocks=1, final_layers_channels=[], dilation_bound=2, bits=16)
  B, T = 4, 2048
  m.build((B, T, 1))
  rng = np.random.default_rng(1)
  p = rng.dirichlet(np.full(C, 0.3)).astype(np.float32)
  pred = torch.from_numpy(p).cuda().expand(B, T, C).contiguous()
  s = m.sample_waveform(pred, seed=11)
  idx = torch.round((s[..., 0] + 1.0) * 2 ** 15).long().flatten().cpu().numpy()
  assert idx.min() >= 0 and idx.max() < C
  counts = np.bincount(idx // 1024, minlength=64)
  expect = p.astype(np.float64).reshape(64, 1024).sum(1) / p.astype(np.float64).sum() * idx.size
  chi2 = float(((counts - expect) ** 2 / expect).sum())
  pval = float(stats.chi2.sf(chi2, 63))
  _report('draws_c65536', chi2=chi2, p_value=pval)
  assert pval > 1e-4, (chi2, pval)
  assert not torch.equal(s, m.sample_waveform(pred, seed=12))
  assert torch.equal(s, m.sample_waveform(pred, seed=11))


# ------------------------------------------------------------------ 7. generation at 2 and 65,536 classes
def _gen_model(bits, precision):
  kw = _fp32_kw(bits) if precision == 'fp32' else _bf16_kw(bits)
  cond_in = BF16_COND_IN if kw.get('conditioning') else 0
  m, cfg, p, x, cond = _model(kw, 3, 90, precision, cond_in)
  return m, cfg, p, x, cond


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('bits', [1, 16])
def test_step_form_equals_call(bits, precision):
  """gen_dense_kernel with N = C and gen_pred_kernel's softmax over C.  The bf16 tier generates from the fp32 master weights, so
  its step form is held to the fp32 tolerance against float64 (and against call only on the fp32 tier)."""
  m, cfg, p, x, cond = _gen_model(bits, precision)
  n_prime = 17
  pred = m._teacher_forced_step_predictions(x[:, :n_prime], x[:, n_prime:-1], cond).cpu().numpy()
  xin = x[:, :-1]
  ref, _ = wo.model_forward(p, cfg, xin.astype(np.float64), None if cond is None else cond.astype(np.float64))
  e_ref = rel_err(pred, ref[:, n_prime - 1:-1])
  e_call = None
  if precision == 'fp32':
    full = m(_inputs(x, cond)).cpu().numpy()
    e_call = rel_err(pred, full[:, n_prime - 1:-1])
  _report('step_form', bits=bits, precision=precision, vs_fp64=e_ref, vs_call=e_call)
  assert e_ref < TOL_FP32
  if e_call is not None:
    assert e_call < TOL_FP32


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('bits', [1, 16])
def test_generate_matches_windowed_reference_loop(bits, precision):
  m, cfg, p, x, cond = _gen_model(bits, precision)
  rf = m.receptive_field
  B, L = 2, 12
  prime = x[:B, :rf]
  c = None if cond is None else cond[:B]
  got = m.generate(L, condition=c, sample=prime, deterministic=True).cpu().numpy()
  assert got.shape == (B, L, 1)
  win = prime.astype(np.float64)
  outs = []
  for _ in range(L):
    pred, _ = wo.model_forward(p, cfg, win, None if c is None else c.astype(np.float64))
    s = wo.sample_deterministic(cfg, pred[:, -1:, :]).reshape(B, 1, 1)
    outs.append(s)
    win = np.concatenate([win[:, 1:], s], axis=1)
  ref = np.concatenate(outs, axis=1)
  agree = float((np.abs(got - ref) < 1e-6).mean())
  _report('generate', bits=bits, precision=precision, agree=agree)
  assert agree >= 0.9                  # an argmax near-tie may send one trajectory elsewhere


# ------------------------------------------------------------------ 8. 64-bit element offsets at 65,536 classes
def test_bf16_65536_classes_beyond_2_pow_31_elements():
  """B * T * C > 2^31 at B = 4, T = 8,200, C = 65,536: the logits, call's output and the d logits (ldd = C) hold more elements than
  a 32-bit offset reaches, and positions t >= 8,000 of batch row 3 lie beyond element 2^31.  Row 3 is a copy of row 0, so its
  probabilities must equal row 0's bit for bit; train_step's loss must equal the cross entropy of call's output, evaluated in float64
  on the device in row chunks."""
  from wavenets_b200 import WaveNet
  B, T, bits = 4, 8200, 16
  C = 2 ** bits
  assert B * T * C > 2 ** 31 > (B - 1) * T * C
  need = 3 * B * T * C * 4 + (4 << 30)     # logits, call output, bf16 d logits + head GEMM and chunk scratch
  free = torch.cuda.mem_get_info()[0]
  if free < need:
    pytest.skip(f'needs {need / 2 ** 30:.1f} GiB of free device memory, {free / 2 ** 30:.1f} GiB free')
  kw = _bf16_kw(bits)
  cfg = oracle_config(kw, BF16_COND_IN)
  p = wo.init_params(cfg, seed=1)
  x, cond = make_inputs(B, T, BF16_COND_IN)
  x[3], cond[3] = x[0], cond[0]
  m = WaveNet(**kw, precision='bf16')
  m.build((x[:, :-1].shape, cond.shape))
  m.set_weights({k: v.astype(np.float32) for k, v in p.items()})
  out = m.train_step((x, cond))
  pred = m((x[:, :-1], cond))
  assert torch.equal(pred[3], pred[0])
  y = m.prepare_target(x[:, 1:]).reshape(B, T)
  total = torch.zeros((), dtype=torch.float64, device=pred.device)
  for b in range(B):
    for t0 in range(0, T, 1024):
      pc = pred[b, t0:t0 + 1024].double().clamp(1e-7, 1 - 1e-7)
      yc = y[b, t0:t0 + 1024]
      total += (torch.log(pc.sum(-1)) - torch.log(torch.gather(pc, 1, yc[:, None])[:, 0])).sum()
  loss_ref = float(total) / B
  e = abs(out['loss'] - loss_ref) / abs(loss_ref)
  _report('bf16_65536_64bit', loss=out['loss'], loss_ref=loss_ref, rel=e)
  assert e <= TOL_FP32, (out['loss'], loss_ref)
