"""The persistent stack launches (csrc/gemm_tc_stack.cuh forward, csrc/gemm_tc_stack_bwd.cuh backward) at shapes the BASELINE
topologies never produce.  Those all use kernel_size=2 and 256 channels, and their tile counts give one stack-backward band or two
equal ones.  Here:
  * kernel sizes 3 and 4: more tile flags per operand box, odd row shifts (dilations 3, 9, 27, ...), taps reaching 12 tiles back
    (K=4, dilation 1024: 3072 rows), plain layers with nseg * kb_tap k-steps, an odd number of taps per grouped weight-gradient unit;
  * 128 channels: `tc_stack_fwd_kernel<128,128>` has one gate sub-tile per tile (TcStackSeq<NT1=1>), so a tile's flag is published
    right behind its own stores up to 2 x pairs tiles per layer, and behind the next sub-tile beyond (`delay_publish`);
  * a stack backward whose last band of m tiles is shorter than the others, with a band boundary inside a sequence.

B x T comes from the device's CTA-pair count, so that every case lands in its regime on the GPU it runs on, and the last tile of
a sequence is ragged.  `test_case_table` (no GPU) pins the regimes for a B200's 74 pairs, so that an edit of the table cannot
quietly drop an edge.

Per case (`test_stack_launches`): the launches are on the path (counters); eager, eager and CUDA-graph replay agree bit for bit;
the stack forward equals one fused launch per block bit for bit; the stack backward agrees with the per-block chain to the bf16
storage error; the grouped weight gradients agree with the per-block ones to fp32 summation order; every gradient is checked against
the bf16-faithful oracle (tolerances of tests/test_gpu_configs.py).  `test_causality_at_tile_edges`: exact causality, receptive
field and batch isolation around tile boundaries for the longest taps and for the delayed publishing.  Run with -s for the
measured errors.

The 128-wide models run the stack forward, but their backward is the per-block chain: the stack backward needs the grouped
weight-gradient mode, which needs R, D and S to be multiples of 256 (`wn_api.cu`, use_group_wgrad and BwdSchedule::sb)."""
import json
import math

import numpy as np
import pytest

from oracle import wavenet_oracle as wo
from tests.util import env_vars, oracle_config, rel_err, rel_l2

TILE = 256
COND_IN = 109
B200_PAIRS = 74                 # 148 SMs
SB_BAND = 128                   # band target of the stack backward (m tiles per band)

W256 = dict(channels=256, final_layers_channels=[256])
W128 = dict(channels=128, final_layers_channels=[128])
COND = dict(conditioning='global', mapping_layers=[8], mapping_activation='tanh')

# name -> (model kwargs, B, tiles per sequence as a function of the CTA-pair count, rows in the last (ragged) tile)
CASES = {
  # 3 taps in both launches and in the grouped units; dilations 1..243: odd row shifts
  'k3_cond': (dict(W256, kernel_size=3, skip_channels=256, blocks=6, dilation_bound=729, activation='tanh', **COND),
              3, lambda pairs: (pairs + 6) // 3, 100),
  # dilations 1..1024 with 4 taps: the last one reaches 3072 rows (12 tiles) back; the skip is conv1's output; logistic mixture
  'k4_long_alias': (dict(W256, kernel_size=4, skip_channels=None, blocks=6, dilation_bound=4096, activation='leaky_relu',
                         num_mixtures=10, sampling_function='logistic', bits=16),
                    4, lambda pairs: (pairs + 5) // 4, 92),
  # plain layers (the conv in front of the gated conv) with 3 taps in both launches
  'k3_multidil': (dict(W256, kernel_size=3, skip_channels=256, blocks=3, layers_per_block=2, dilation_bound=27, activation='leaky_relu'),
                  3, lambda pairs: (pairs + 6) // 3, 100),
  # keep-masks applied inside both launches, 4 taps
  'k4_dropout': (dict(W256, kernel_size=4, skip_channels=256, blocks=4, dilation_bound=64, activation='tanh', dropout=0.1),
                 3, lambda pairs: (pairs + 6) // 3, 100),
  # 9 x 29 = 261 m tiles: stack-backward bands of 131 + 130, the boundary inside sequence 4, crossed by the taps
  'bands_unequal': (dict(W256, kernel_size=4, skip_channels=256, blocks=3, dilation_bound=256),
                    9, lambda pairs: 29, 100),
  # the <128,128> stack forward, NT1 = 1, fewer than 2 x pairs tiles: flags published right away
  'r128_cond': (dict(W128, kernel_size=2, skip_channels=128, blocks=6, dilation_bound=32, activation='tanh', **COND),
                3, lambda pairs: (pairs + 6) // 3, 100),
  # exactly 2 x pairs tiles: the last tile count that publishes right away
  'r128_k3_at_2pairs': (dict(W128, kernel_size=3, skip_channels=128, blocks=4, dilation_bound=27),
                        4, lambda pairs: 2 * pairs // 4, 100),
  # 2 x pairs + 1 tiles in one sequence: delayed publishing with NT1 = 1
  'r128_k4_delayed': (dict(W128, kernel_size=4, skip_channels=None, blocks=5, dilation_bound=256, activation='leaky_relu'),
                      1, lambda pairs: 2 * pairs + 1, TILE - 17),
}
CAUSALITY_CASES = ['k4_long_alias', 'r128_k4_delayed']

# tolerances of tests/test_gpu_configs.py (bf16-faithful oracle) and tests/test_gpu_group_wgrad.py / test_gpu_fullsize.py
TOL_LOSS_FAITHFUL = 5e-5
TOL_GRAD_FAITHFUL, TOL_GLOBAL_FAITHFUL = 8e-3, 4e-3
TOL_GRAD_FAITHFUL_DROPOUT, TOL_GLOBAL_FAITHFUL_DROPOUT = 1.2e-2, 5e-3
TOL_LOSS_BF16, TOL_GRAD_BF16, TOL_GRAD_BF16_PWL = 1e-2, 6e-2, 1e-1     # float64 reference; relu / leaky_relu models: 1e-1
TOL_DZ_STACK_BWD, TOL_GRAD_STACK_BWD = 2e-4, 5e-3
TOL_GROUPED = 3e-4


def shape(name, pairs):
  """(B, T, tiles per sequence) of a case on a device with `pairs` CTA pairs"""
  _, B, tiles_of, tail = CASES[name]
  tiles_t = tiles_of(pairs)
  return B, TILE * (tiles_t - 1) + tail, tiles_t


def wide(name):
  return CASES[name][0]['channels'] == 256


def sb_bands(num_mtiles, pairs, band_target=SB_BAND):
  """The stack backward's band split (tc_stack_bwd_launch_t): as many bands of ~band_target m tiles as fit, one fewer until the
  first and the last band both have more tiles than the launch has CTA pairs; every band but the last has ceil(n / nb) tiles."""
  nb = max(num_mtiles // band_target, 1)
  while nb > 1:
    bw = -(-num_mtiles // nb)
    if bw > pairs and num_mtiles - (nb - 1) * bw > pairs:
      break
    nb -= 1
  bw = -(-num_mtiles // nb)
  return [bw] * (nb - 1) + [num_mtiles - (nb - 1) * bw]


# ----------------------------------------------------------------------------------------------------------- no GPU
@pytest.mark.parametrize('name', sorted(CASES))
def test_case_table(name):
  from wavenets_b200 import WaveNet
  kw = CASES[name][0]
  B, T, tiles_t = shape(name, B200_PAIRS)
  tiles = B * tiles_t
  m = WaveNet(**kw, precision='bf16')
  cfg = oracle_config(kw, COND_IN if kw.get('conditioning') else 0)
  cfg.validate()                                          # the reference's checks, dilation bound a power of K in float
  dils, rf = wo.dilation_schedule(cfg)
  assert m.receptive_field == rf
  assert tiles_t == -(-T // TILE) and T % TILE != 0       # ragged last tile
  assert tiles > B200_PAIRS                               # the persistent launches need more tiles per layer than CTA pairs
  K = kw['kernel_size']
  shift = (K - 1) * max(max(d) for d in dils)
  expect = {                                              # (tiles vs 2 x pairs, largest tap shift in rows)
    'k3_cond': ('<=', 2 * 243), 'k4_long_alias': ('<=', 3 * 1024), 'k3_multidil': ('<=', 2 * 9), 'k4_dropout': ('<=', 3 * 16),
    'bands_unequal': ('>', 3 * 16), 'r128_cond': ('<=', 16), 'r128_k3_at_2pairs': ('<=', 2 * 9), 'r128_k4_delayed': ('>', 3 * 64),
  }[name]
  assert (tiles <= 2 * B200_PAIRS) == (expect[0] == '<='), (name, tiles)
  assert shift == expect[1], (name, shift)
  # the reference's receptive field counts one row for the input conv, which has K taps: the exact reach is K - 2 rows longer
  assert reach(kw) == rf + K - 2
  if name == 'k4_long_alias':
    assert shift // TILE == 12 and T > reach(kw)
  if name == 'r128_k3_at_2pairs':
    assert tiles == 2 * B200_PAIRS
  if name == 'r128_k4_delayed':
    assert tiles == 2 * B200_PAIRS + 1 and B == 1 and T > reach(kw)
  if name in CAUSALITY_CASES:
    t0 = edge(name, T)
    assert t0 % TILE == TILE - 1 and t0 + 1 + reach(kw) <= T - 1
  bands = sb_bands(tiles, B200_PAIRS)
  if name == 'bands_unequal':
    assert tiles == 261 and bands == [131, 130]
    # m tiles are numbered sequence by sequence; the boundary after the first band falls inside sequence 131 // 29 = 4, whose
    # later tiles run in the first band and earlier ones in the second (descending time order): the taps of the second band's
    # first tile of that sequence read d z written in the first band
    assert bands[0] % tiles_t != 0 and shift > 0
  else:
    assert len(set(bands)) == 1, (name, bands)


def reach(kw):
  """rows of input an output row depends on: its own, K - 1 taps of the input conv and (K - 1) * d of every dilated conv"""
  dils, _ = wo.dilation_schedule(oracle_config(kw))
  return 1 + (kw['kernel_size'] - 1) * (1 + sum(map(sum, dils)))


def edge(name, T):
  """an input row on the last row of a tile (the next row starts a tile)"""
  k = 2 if name == 'k4_long_alias' else (T // TILE) // 2
  return TILE * k - 1


# ----------------------------------------------------------------------------------------------------------- GPU
def _pairs():
  import torch
  return torch.cuda.get_device_properties(0).multi_processor_count // 2


def _setup(name):
  """weights, inputs and keep-masks as tests/config_parity.py makes them"""
  from wavenets_b200 import synth
  kw = CASES[name][0]
  B, T, _ = shape(name, _pairs())
  cond_in = COND_IN if kw.get('conditioning') else 0
  cfg = oracle_config(kw, cond_in)
  p = wo.init_params(cfg, seed=1)                          # glorot-uniform kernels, N(0, 0.02) biases
  x = synth.frames(B, T, seed=3)
  cond = synth.speakers_onehot(B, cond_in, seed=3) if cond_in else None
  keep = None
  if kw.get('dropout'):
    rng = np.random.default_rng(17)
    keep = [(rng.random((B, T, kw['channels'])) >= kw['dropout']).astype(np.uint8) for _ in range(kw['blocks'])]
  return kw, cfg, p, x, cond, keep, B, T


def _model(kw, p, B, T, cond, env=None):
  from wavenets_b200 import WaveNet
  with env_vars(env or {}):                                    # the switches are read at wn_create
    m = WaveNet(**kw, precision='bf16', max_batch=B, max_time=T)
    m.build(((B, T, 1), (B, cond.shape[1])) if cond is not None else (B, T, 1))
  m.set_weights({k: v.astype(np.float32) for k, v in p.items()})
  return m


def _train(name, env=None):
  """three steps (eager; eager with the plans built; CUDA-graph replay): the model, [(loss, grads)] per step, counters"""
  kw, cfg, p, x, cond, keep, B, T = _setup(name)
  m = _model(kw, p, B, T, cond, env)
  if keep is not None:
    m.set_dropout_masks(keep)
  data = (x, cond) if cond is not None else x
  steps = []
  for _ in range(3):
    loss = m.train_step(data)['loss']
    steps.append((loss, m.get_grads()))
  lib, h = m.handle.lib, m.handle.h
  n = dict(stack_fwd=int(lib.wn_stack_forward_layers(h)), stack_bwd=int(lib.wn_stack_backward_layers(h)),
           fused_fwd=int(lib.wn_fused_forward_blocks(h)), grouped=int(lib.wn_grouped_wgrad_tiles(h, None)))
  return m, steps, n


def _dz_last(m, kw, B, T):
  from tests.util import device_tensor
  dz = device_tensor(m, 'dz', kw['blocks'] - 1, B, T, 2 * kw['channels'])
  assert dz is not None, m.handle.lib.wn_last_error()
  return dz


@pytest.mark.gpu
@pytest.mark.parametrize('name', list(CASES))
def test_stack_launches(name):
  from oracle import faithful
  from tests.config_parity import errors
  from tests.util import device_slope_masks
  kw, cfg, p, x, cond, keep, B, T = _setup(name)
  L, pairs = kw['blocks'], _pairs()
  tiles = B * -(-T // TILE)
  res = {'case': name, 'B': B, 'T': T, 'tiles': tiles, 'pairs': pairs}

  # 1. the persistent launches are on the path (a silent fall-back to per-block launches would make the rest vacuous)
  m, steps, n = _train(name)
  res['counters'] = n
  assert n['stack_fwd'] == L, n
  if wide(name):
    assert n['stack_bwd'] == L and n['grouped'] > 0, n
  else:
    assert n['stack_bwd'] == 0 and n['grouped'] == 0, n      # 128 wide: stack forward, per-block backward chain
  if name == 'bands_unequal':
    bands = sb_bands(tiles, pairs)
    assert len(bands) > 1 and bands[-1] != bands[0], bands
  if name == 'r128_k4_delayed':
    assert tiles > 2 * pairs                                  # delay_publish
  if name == 'r128_k3_at_2pairs':
    assert tiles == 2 * pairs

  # 2. bit-reproducible: eager, eager, CUDA-graph replay
  loss, g = steps[0]
  assert np.isfinite(loss) and all(np.isfinite(v).all() for v in g.values())
  for i in (1, 2):
    assert steps[i][0] == loss, (i, steps[i][0], loss)
    for k in g:
      assert np.array_equal(steps[i][1][k], g[k]), (k, i)
  masks = device_slope_masks(m, kw, B, T)
  dz_a = _dz_last(m, kw, B, T) if wide(name) else None
  xin = x[:, :-1]
  fwd_in = (xin, cond) if cond is not None else xin
  y_a = m(fwd_in).cpu().numpy()
  del m, steps

  # 3. stack forward == one fused launch per block: the same tile arithmetic, bit for bit
  m_f, steps_f, n_f = _train(name, {'WN_TC_STACK_FWD': '0'})
  assert n_f['stack_fwd'] == 0 and n_f['fused_fwd'] == L, n_f
  y_f = m_f(fwd_in).cpu().numpy()
  res['forward_max_abs_diff'] = float(np.abs(y_a - y_f).max())
  same = bool(np.array_equal(y_a, y_f))
  assert same, res
  assert steps_f[2][0] == loss
  for k in g:
    assert np.array_equal(steps_f[2][1][k], g[k]), k
  del m_f, steps_f, y_a, y_f

  if wide(name):
    # 4. stack backward vs the per-block chain: the same arithmetic in another fp32 summation order
    m_b, steps_b, n_b = _train(name, {'WN_TC_STACK_BWD': '0'})
    assert n_b['stack_fwd'] == L and n_b['stack_bwd'] == 0 and n_b['grouped'] > 0, n_b
    assert steps_b[2][0] == loss
    res['stack_bwd_dz_last'] = rel_l2(dz_a, _dz_last(m_b, kw, B, T))
    g_b = steps_b[2][1]
    e_b = errors(g, g_b)                                     # (a gradient that is zero on the chain must be zero here too)
    res['stack_bwd_worst'] = e_b[0]
    assert res['stack_bwd_dz_last'] <= TOL_DZ_STACK_BWD, res
    assert e_b[0][0] <= TOL_GRAD_STACK_BWD, res
    del m_b, steps_b

    # 5. grouped vs per-block weight gradients on the same (per-block) backward chain
    m_p, steps_p, n_p = _train(name, {'WN_TC_STACK_BWD': '0', 'WN_TC_GROUP_WGRAD': '0'})
    assert n_p['stack_bwd'] == 0 and n_p['grouped'] == 0, n_p
    assert steps_p[2][0] == loss
    g_p = steps_p[2][1]
    e_p = max((rel_err(g_b[k], g_p[k]), k) for k in g_p)
    res['grouped_worst'] = e_p
    assert e_p[0] <= TOL_GROUPED, res
    del m_p, steps_p, g_b, g_p

  # 6. every gradient against the bf16-faithful oracle, with the device's relu / leaky_relu slope masks and the same keep-masks
  p32 = {k: v.astype(np.float32).astype(np.float64) for k, v in p.items()}
  l_f, g_f = faithful.train_step(p32, cfg, x, cond, faithful=True, slope_masks=masks, keep_masks=keep)
  e_f = errors(g, g_f)
  glob = math.sqrt(sum(float(np.sum((g[k].astype(np.float64) - g_f[k]) ** 2)) for k in g_f) / sum(float(np.sum(g_f[k] ** 2)) for k in g_f))
  # and against float64 with the stated bf16 tolerance (this bounds bf16 storage, not the kernels)
  l_64, g_64 = faithful.train_step(p32, cfg, x, cond, faithful=False, keep_masks=keep)
  e_64 = errors(g, g_64)
  res.update(loss=loss, loss_faithful=l_f, worst_faithful=e_f[0], global_faithful=glob, loss_fp64=l_64, worst_fp64=e_64[0])
  print(json.dumps(res))
  tol_grad, tol_glob = (TOL_GRAD_FAITHFUL_DROPOUT, TOL_GLOBAL_FAITHFUL_DROPOUT) if keep is not None else (TOL_GRAD_FAITHFUL, TOL_GLOBAL_FAITHFUL)
  assert abs(loss - l_f) <= TOL_LOSS_FAITHFUL * abs(l_f), res
  assert e_f[0][0] <= tol_grad, res
  assert glob <= tol_glob, res
  assert abs(loss - l_64) <= TOL_LOSS_BF16 * abs(l_64), res
  assert e_64[0][0] <= (TOL_GRAD_BF16_PWL if kw.get('activation') in ('relu', 'leaky_relu') else TOL_GRAD_BF16), res


@pytest.mark.gpu
@pytest.mark.parametrize('name', CAUSALITY_CASES)
def test_causality_at_tile_edges(name):
  """Perturb input row t0 on either side of a tile boundary: outputs before t0 and from t0 + reach on are bit-identical, rows t0 and
  t0 + reach - 1 change, other sequences are bit-identical.  Perturb the last (ragged-tile) sample of sequence 0: sequence 1 is
  bit-identical, its causal taps read zeros, not sequence 0's tail."""
  import torch
  kw, cfg, p, x, cond, keep, B, T = _setup(name)
  m = _model(kw, p, B, T, cond)
  n = reach(kw)
  xin = torch.from_numpy(np.ascontiguousarray(x[:, :-1])).cuda()
  y0 = m(xin)
  assert int(m.handle.lib.wn_stack_forward_layers(m.handle.h)) == kw['blocks']
  t_edge = edge(name, T)
  b = B // 2
  others = [i for i in range(B) if i != b]
  for t0 in (t_edge, t_edge + 1):
    x2 = xin.clone()
    x2[b, t0, 0] += 0.25
    d = (m(x2) != y0).any(dim=-1)                          # (B, T): which outputs changed at all
    assert not bool(d[others].any()), t0
    assert not bool(d[b, :t0].any()), t0
    assert bool(d[b, t0]) and bool(d[b, t0 + n - 1]), t0
    assert not bool(d[b, t0 + n:].any()), t0
  if B > 1:
    x2 = xin.clone()
    x2[0, T - 1, 0] += 0.25                                # the last sample of sequence 0, inside its ragged last tile
    d = (m(x2) != y0).any(dim=-1)
    assert bool(d[0, T - 1]) and not bool(d[0, :T - 1].any())
    assert not bool(d[1:].any())
  print(f'{name}: B={B} T={T} reach={n} perturbed rows {t_edge}, {t_edge + 1}: exact')
