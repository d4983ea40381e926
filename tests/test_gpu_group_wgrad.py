"""Grouped weight-gradient launch (csrc/gemm_tc_wgroup.cuh) against the per-block launches (WN_TC_GROUP_WGRAD=0).

Both are this repo's CUDA paths; the oracle parity of each is covered by test_gpu_parity_bf16.py (models `group256_*`
take the grouped path) and test_gpu_golden.py.  Here: same model, weights and inputs through both schedules — the loss
is bit-equal (same forward), every gradient agrees to fp32 summation order (the row splits differ), and the grouped
path is bit-reproducible across eager calls and CUDA-graph replays (no atomics).  `side_launches` has enough 256-row
tiles (96 > 74 CTA pairs) for the side-stream launches beside the dgrad chain (reference: the filter gradients of
`tape.gradient`, model.py:335)."""

import numpy as np
import pytest

from tests.util import env_vars, make_inputs

pytestmark = pytest.mark.gpu

CASES = {
  'cond_skip_l2': (dict(channels=256, blocks=3, layers_per_block=1, dilation_bound=4, skip_channels=256, final_layers_channels=[256],
                        activation='tanh', conditioning='global', mapping_layers=[8], mapping_activation='tanh', l2_reg_factor=0.01), 3, 333),
  'noskip_k3': (dict(channels=256, blocks=2, layers_per_block=1, dilation_bound=9, kernel_size=3, use_skip=False, final_layers_channels=[128]), 2, 200),
  'multidil': (dict(channels=256, blocks=2, layers_per_block=2, dilation_bound=8, skip_channels=256, final_layers_channels=[128],
                    activation='leaky_relu'), 2, 257),
  # skip_channels=None: the skip is conv1's output (d x_out + d skip feeds conv1's gradient); three dilations per block
  'alias_multidil': (dict(channels=256, blocks=2, layers_per_block=3, dilation_bound=8, final_layers_channels=[128], activation='tanh'), 2, 300),
  'wide512': (dict(channels=256, dilation_channels=512, blocks=2, layers_per_block=1, dilation_bound=4, skip_channels=512,
                   final_layers_channels=[128]), 5, 130),
  'side_launches': (dict(channels=256, blocks=6, layers_per_block=1, dilation_bound=16, skip_channels=256, final_layers_channels=[256],
                         activation='tanh', conditioning='global', mapping_layers=[8], mapping_activation='tanh'), 3, 8000),
  'dropout': (dict(channels=256, blocks=2, layers_per_block=1, dilation_bound=4, skip_channels=256, final_layers_channels=[128], dropout=0.2), 2, 300),
  'logistic_head': (dict(channels=256, blocks=2, layers_per_block=1, dilation_bound=4, skip_channels=256, final_layers_channels=[256, 256],
                         num_mixtures=10, sampling_function='logistic', bits=16), 2, 150),
}


def _run(kw, B, T, group, env=None):
  from wavenets_b200 import WaveNet
  # (these tests hold the WEIGHT-GRADIENT schedules against each other on the same backward chain: the persistent
  # stack-backward launch, which replaces the chain and the side launches, is switched off unless a test asks for it)
  env = dict({'WN_TC_STACK_BWD': '0', 'WN_TC_GROUP_WGRAD': '1' if group else '0'}, **(env or {}))
  with env_vars(env):
    cond_in = 9 if kw.get('conditioning') else 0
    m = WaveNet(**kw, precision='bf16')   # the switches are read at wn_create
    x, cond = make_inputs(B, T, cond_in)
    m.build((x[:, :-1].shape, cond.shape) if cond is not None else x[:, :-1].shape)
    m.handle.glorot_init(seed=3, bias_std=0.05)
    if kw.get('dropout'):
      rng = np.random.default_rng(5)
      m.set_dropout_masks([(rng.random((B, T, kw['channels'])) > kw['dropout']).astype(np.uint8) for _ in range(kw['blocks'])])
    outs = []
    for _ in range(3):   # eager (plan built), eager (side launches), graph replay
      out = m.train_step((x, cond) if cond is not None else x)
      outs.append((out['loss'], m.get_grads(), int(m.handle.lib.wn_stack_backward_layers(m.handle.h))))
    return outs


@pytest.mark.parametrize('name', sorted(CASES))
def test_grouped_equals_per_block(name):
  kw, B, T = CASES[name]
  a = _run(kw, B, T, True)
  b = _run(kw, B, T, False)
  assert a[0][0] == b[0][0]
  for k in b[0][1]:
    ref = b[0][1][k]
    err = float(np.abs(a[0][1][k] - ref).max() / (np.abs(ref).max() + 1e-30))
    assert err < 2e-5, (k, err)
  for i in (1, 2):
    assert a[i][0] == a[0][0]
    for k in a[0][1]:
      assert np.array_equal(a[0][1][k], a[i][1][k]), (k, i)


@pytest.mark.parametrize('env', [{'WN_TC_GROUP_NH2': '0'}, {'WN_TC_GROUP_SPLIT': '1'}, {'WN_TC_GROUP_SPLIT': '7'}, {'WN_TC_GROUP_SIDE_EVERY': '2'},
                                 {'WN_TC_GROUP_SIDE_EVERY': '0'}])
def test_grouped_schedules_agree(env):
  """single 256x256 tiles, no row split, 7 row splits, side launch for every second block, no side launches"""
  kw, B, T = CASES['side_launches']
  a = _run(kw, B, T, True, env)
  b = _run(kw, B, T, True)
  for k in b[0][1]:
    ref = b[0][1][k]
    err = float(np.abs(a[2][1][k] - ref).max() / (np.abs(ref).max() + 1e-30))
    # 24,000 rows accumulated in fp32 by the tensor core in one chain (no row split) or in up to 7 chains: measured <= 1.0e-4
    assert err < 3e-4, (k, err)


def test_stack_forward_equals_per_block_launches():
  """The whole residual stack as ONE persistent launch (csrc/gemm_tc_stack.cuh: tiles of layer l wait for the x_out tiles
  of layer l-1 written by other CTA pairs of the same launch) against one fused launch per block: the same tile
  arithmetic, so the loss, every gradient and the forward output are bit-equal (block loop of WaveNet.call, model.py:229-234)."""
  kw, B, T = CASES['side_launches']
  a = _run(kw, B, T, True)
  b = _run(kw, B, T, True, {'WN_TC_STACK_FWD': '0'})
  for i in range(3):
    assert a[i][0] == b[i][0]
    for k in b[i][1]:
      assert np.array_equal(a[i][1][k], b[i][1][k]), (k, i)


def test_stack_backward_vs_per_block_chain():
  """The backward chain of all blocks as ONE persistent launch (csrc/gemm_tc_stack_bwd.cuh) against one gate-adjoint + one
  dgrad launch per block.  Same arithmetic in another fp32 summation order (taps, residual add): a sum landing on the other
  side of a bf16 rounding boundary flips a stored d z / d x_out element by one ulp, so the gradients agree to the bf16 storage
  error, not bit for bit; the fused launch itself is bit-reproducible (eager calls and graph replay)."""
  kw, B, T = CASES['side_launches']
  a = _run(kw, B, T, True, {'WN_TC_STACK_BWD': '1'})
  b = _run(kw, B, T, True)
  assert a[0][2] > 0 and b[0][2] == 0, 'the stack-backward launch must be held against the per-block chain'
  assert a[0][0] == b[0][0]
  for i in (1, 2):
    assert a[i][0] == a[0][0]
    for k in a[0][1]:
      assert np.array_equal(a[0][1][k], a[i][1][k]), (k, i)
  worst = 0.0
  for k in b[0][1]:
    ref = b[0][1][k]
    err = float(np.linalg.norm(a[0][1][k] - ref) / (np.linalg.norm(ref) + 1e-30))
    worst = max(worst, err)
    assert err < 5e-3, (k, err)
  print(f'stack backward vs per-block chain (6 blocks): worst gradient tensor rel-L2 {worst:.2e}')


def test_stack_forward_multi_dilation_equals_per_block_launches():
  """Blocks with several dilated convs (layers.py:64-88): the convs in front of the gated conv run as PLAIN layers of the same
  persistent launch (one 256 x 256 tile per m tile, bias + activation epilogue, tile flags towards the next conv).  Same tile
  arithmetic as the separate conv launches: loss and gradients bit-equal."""
  kw = dict(channels=256, blocks=3, layers_per_block=3, dilation_bound=32, skip_channels=256, final_layers_channels=[128], activation='leaky_relu')
  B, T = 3, 6500
  a = _run(kw, B, T, True)
  b = _run(kw, B, T, True, {'WN_TC_STACK_FWD': '0'})
  for i in range(3):
    assert a[i][0] == b[i][0]
    for k in b[i][1]:
      assert np.array_equal(a[i][1][k], b[i][1][k]), (k, i)


def test_stack_backward_multi_dilation_vs_per_block_chain_and_oracle():
  """Blocks with several dilated convs in the persistent stack-BACKWARD launch: the convs in front of the gated conv are plain
  layers (one OUT-type tile, all taps from L2, activation adjoint from the cached output of the conv in front; the residual
  gradient joins at the block's first conv).  Against the per-block chain (bf16 storage error: different fp32 summation order)
  and against the bf16-faithful oracle (every gradient tensor)."""
  from oracle import faithful
  from oracle import wavenet_oracle as wo
  from tests.util import device_slope_masks, oracle_config, rel_l2
  from wavenets_b200 import WaveNet
  kw = dict(channels=256, blocks=3, layers_per_block=3, dilation_bound=32, skip_channels=256, final_layers_channels=[128], activation='leaky_relu')
  B, T = 3, 6500
  cfg = oracle_config(kw, 0)
  p = wo.init_params(cfg, seed=1)
  x, _ = make_inputs(B, T, 0)

  def run(env):
    with env_vars(env):
      m = WaveNet(**kw, precision='bf16')
      m.build(x[:, :-1].shape)
      m.set_weights({k: v.astype(np.float32) for k, v in p.items()})
      for _ in range(3):
        out = m.train_step(x)
      return m, out['loss'], m.get_grads(), int(m.handle.lib.wn_stack_backward_layers(m.handle.h))

  m_a, l_a, g_a, n_a = run({})
  m_b, l_b, g_b, n_b = run({'WN_TC_STACK_BWD': '0'})
  assert n_a == 3 and n_b == 0
  assert l_a == l_b
  worst = max(rel_l2(g_a[k], g_b[k]) for k in g_b if np.linalg.norm(g_b[k]) > 0)
  print(f'multi-dilation stack backward vs per-block chain: worst gradient tensor rel-L2 {worst:.2e}')
  assert worst < 5e-3
  p32 = {k: v.astype(np.float32).astype(np.float64) for k, v in p.items()}
  l_f, g_f = faithful.train_step(p32, cfg, x, None, faithful=True, slope_masks=device_slope_masks(m_a, kw, B, T))
  assert abs(l_a - l_f) <= 5e-5 * abs(l_f)
  worst_f = max((rel_l2(g_a[k], g_f[k]), k) for k in g_f if np.linalg.norm(g_f[k]) > 0)
  print(f'multi-dilation stack backward vs bf16-faithful oracle: worst gradient tensor {worst_f}')
  assert worst_f[0] < 8e-3, worst_f


def test_plan_cache_eviction_keeps_results():
  """More (B, T) shapes than the handle caches plans for (4): the grouped-wgrad / stack-forward plans and the CUDA graphs that
  hold pointers into them are dropped and rebuilt; every shape reproduces its first result bit for bit."""
  from wavenets_b200 import WaveNet
  kw = dict(channels=256, blocks=2, layers_per_block=1, dilation_bound=4, skip_channels=256, final_layers_channels=[128])
  m = WaveNet(**kw, precision='bf16', max_batch=2, max_time=230)
  m.build((2, 230, 1))
  m.handle.glorot_init(seed=2, bias_std=0.05)
  first = {}
  for rnd in range(2):
    for T in (100, 120, 140, 160, 180, 200, 230):
      x, _ = make_inputs(2, T, 0, seed=T)
      for _ in range(3):      # eager, eager, graph replay
        out = m.train_step(x)
        g = m.get_grads()
        key = T
        if key not in first:
          first[key] = (out['loss'], {k: v.copy() for k, v in g.items()})
        else:
          assert out['loss'] == first[key][0], (T, rnd)
          for k in g:
            assert np.array_equal(g[k], first[key][1][k]), (T, rnd, k)
