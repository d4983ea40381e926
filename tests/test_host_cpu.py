"""CPU tests of the host side: the C-ABI library loads and exports every symbol the header
declares; constructor validation mirrors the reference's exceptions; config loader accepts
reference YAMLs.  No compute calls (no GPU here)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
  from wavenets_b200 import _lib
  lib = _lib.load()
  hdr = open(os.path.join(ROOT, 'include', 'wavenet_b200.h')).read()
  hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
  declared = sorted(set(re.findall(r'\b(wn_[a-z_0-9]+)\s*\(', hdr)))
  assert len(declared) >= 20
  for name in declared:
    assert hasattr(lib, name), f'{name} declared in include/wavenet_b200.h but not exported'
  assert sorted(_lib.EXPORTS) == declared
  assert b'sm_100a' in lib.wn_build_info()


def test_config_struct_matches_header_size():
  from wavenets_b200 import _lib
  import ctypes as C
  n_i32 = 4 + 3 + 8 + 2 + 4 + 4 + 1 + 8 + 2 + 1 + 512 + 3 + 3
  assert C.sizeof(_lib.WnConfig) == 4 * n_i32


def test_constructor_validation_matches_reference():
  from wavenets_b200 import WaveNet
  ok = dict(final_layers_channels=[8])
  with pytest.raises(ValueError, match="Conditioning must be"):
    WaveNet(conditioning='speaker', **ok)
  with pytest.raises(ValueError, match='Kernel size'):
    WaveNet(kernel_size=1, **ok)
  with pytest.raises(ValueError, match='dilation bound'):
    WaveNet(dilation_bound=100, **ok)
  with pytest.raises(ValueError, match='Layers per block'):
    WaveNet(layers_per_block=0, **ok)
  with pytest.raises(ValueError, match='Blocks'):
    WaveNet(blocks=0, **ok)
  with pytest.raises(ValueError, match='mixtures'):
    WaveNet(num_mixtures=0, sampling_function='gaussian', **ok)
  with pytest.raises(ValueError, match='Dropout'):
    WaveNet(dropout=1.5, **ok)
  with pytest.raises(ValueError, match='Sampling function'):
    WaveNet(sampling_function='laplace', **ok)
  with pytest.raises(ValueError, match='Categorical'):
    WaveNet(num_mixtures=3, **ok)
  with pytest.raises(ValueError, match='Mapping layers'):
    WaveNet(mapping_layers='8', **ok)
  with pytest.raises(NotImplementedError):
    WaveNet(conditioning='local', **ok)
  with pytest.raises(NotImplementedError):
    WaveNet(activation='gelu', **ok)
  m = WaveNet(kernel_size=2, channels=32, blocks=5, layers_per_block=5, dilation_bound=256, final_layers_channels=[128, 256])
  assert m.receptive_field == 768
  assert m.compute_receptive_field(16000) == 768 / 16000
  with pytest.raises(ValueError, match='Loss must be set'):
    m.compile(loss='mse')


def test_compiled_model_reports_keras_running_means():
  """model.py:166-168,340-360: a compiled model's logs are the running means of loss_tracker / reg_loss / compiled metrics
  since the last reset_metrics(); test_step carries no reg_loss; the step's own values stay in last_step_logs."""
  from wavenets_b200 import WaveNet
  from wavenets_b200.metrics import MeanSquaredError
  m = WaveNet(channels=8, blocks=2, final_layers_channels=[8], dilation_bound=2, l2_reg_factor=0.1)
  raw = m._logs_from_values([4.0, 0.5, 0.0], train=True)
  assert raw == {'loss': 4.0, 'reg_loss': 0.5}                       # not compiled: the step's own values
  m.compile(metrics=[MeanSquaredError()])
  assert [t.name for t in m.metrics] == ['mean_squared_error', 'loss', 'reg_loss'] and len(m.metrics) == 3
  a = m._logs_from_values([4.0, 0.5, 1.0], train=True)
  b = m._logs_from_values([2.0, 0.25, 3.0], train=True)
  assert a == {'loss': 4.0, 'reg_loss': 0.5, 'mean_squared_error': 1.0}
  assert b == {'loss': 3.0, 'reg_loss': 0.375, 'mean_squared_error': 2.0}
  assert m.last_step_logs == {'loss': 2.0, 'reg_loss': 0.25, 'mean_squared_error': 3.0}
  t = m._logs_from_values([1.0, 0.0, 5.0], train=False)              # test_step: the regulariser tracker is not fed
  assert t['loss'] == 7.0 / 3 and t['reg_loss'] == 0.375 and m.reg_loss.count == 2
  m.reset_metrics()
  assert m._logs_from_values([6.0, 1.0, 2.0], train=True) == {'loss': 6.0, 'reg_loss': 1.0, 'mean_squared_error': 2.0}
  m.compile()                                                        # fresh trackers, like Keras
  assert m.loss_tracker.count == 0 and m.metrics[0].name == 'loss'


def test_layer_attributes_and_errors():
  from wavenets_b200 import WaveNetLayer
  lay = WaveNetLayer(kernel=2, dilation_rate=[1, 2, 4], activation='leaky_relu', channels=16, skip_channels=None)
  assert lay.input_dilation == 1 and lay.depth == 3 and lay.kernel_size == 2 and lay.channels == 16
  assert len(lay.dilated_stack) == 3 and lay.dilated_stack[-1].filters == 32 and lay.conv_skip is None
  with pytest.raises(ValueError, match='not built'):
    lay.compute_output_shape((1, 8, 16))


def test_reference_yaml_loads():
  """tests/golden/defaults.yaml restates the reference's configfiles/defaults.yaml in its 27-line layout: train.py's key
  names (the `use_resiudal` typo included) and the file's dataset path, which differs from train.py's default."""
  from wavenets_b200 import load_config, model_kwargs, CONFIGS
  cfg = load_config(os.path.join(ROOT, 'tests', 'golden', 'defaults.yaml'))
  assert cfg['dataset'] == './datasets/svd8000'
  kw = model_kwargs(cfg)
  assert kw['use_residual'] is True and kw['channels'] == 32 and kw['final_layers_channels'] == [128, 256]
  assert set(CONFIGS) == {'c1', 'c2', 'c3', 'c4', 'c5'}


def test_no_gpu_fails_loudly():
  import torch
  if torch.cuda.is_available():
    pytest.skip('GPU present')
  from wavenets_b200 import WaveNet
  import numpy as np
  m = WaveNet(channels=8, blocks=2, final_layers_channels=[8], dilation_bound=4)
  with pytest.raises(RuntimeError, match='no CPU fallback'):
    m(np.zeros((1, 16, 1), np.float32))


def test_checkpoint_names_and_resume_parse(tmp_path):
  """train.py:68-86,149-154: file pattern and resume-by-filename."""
  from wavenets_b200 import checkpoint as ck
  assert ck.checkpoint_name(7, 0.0005) == 'weights-e0007-lr0.0005.weights.npz'
  assert ck.find_last_checkpoint(str(tmp_path / 'nope')) is None
  for e, lr in [(1, 0.0005), (12, 0.00025), (3, 0.0005)]:
    (tmp_path / ck.checkpoint_name(e, lr)).write_bytes(b'')
  # a reference run's Keras file in the same directory sorts last but cannot be read here: it is not picked
  (tmp_path / 'weights-e0099-lr0.0001.weights.h5').write_bytes(b'')
  path, epoch, lr = ck.find_last_checkpoint(str(tmp_path))
  assert path.endswith('weights-e0012-lr0.00025.weights.npz') and epoch == 12 and lr == 0.00025
  import pytest
  with pytest.raises(ValueError):
    ck.load_weights(None, str(tmp_path / 'weights-e0099-lr0.0001.weights.h5'))
