"""Time WaveNet.call(training=True) + WaveNet.backward (a caller-computed loss: forward, the adjoint of the predictions, the
backward pass) against the training step with the built-in loss, at the full C2 / C4 sizes (CONFIGS: batch 8, T = 8000).

Both sides run eagerly on the caller's stream (WN_CUDA_GRAPH=0 for the train_step handle: backward is not replayed from a CUDA
graph, so the fair comparison is the eager step); the graph-replayed train_step is printed too.  The C entry points are timed
with CUDA events around each call; the rounds alternate the order of the variants after a warm-up.  The workload (8 x 8000 rows
of 256-channel bf16 activations per block, 30 blocks) is far larger than the 126 MB L2.  The `pred_vjp` kernel time (the
softmax / mixture adjoint that starts wn_backward) comes from wn_profile_get in a separate profiled pass.  Prints the card name
and power limit next to the numbers; writes nothing."""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tests.util import env_vars  # noqa: E402
from wavenets_b200 import CONFIGS, WaveNet, _lib, model_kwargs, synth  # noqa: E402


def card():
  try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', str(torch.cuda.current_device())],
                       capture_output=True, text=True, timeout=30)
    return q.stdout.strip() or torch.cuda.get_device_name()
  except (OSError, subprocess.SubprocessError):
    return torch.cuda.get_device_name() + ', power limit unknown'


def _model(name, graphs):
  cfg = dict(CONFIGS[name])
  kw = model_kwargs(cfg)
  B, T = cfg['batch_size'], cfg['recording_length']
  cond_in = cfg.get('n_speakers', 109) if kw['conditioning'] == 'global' else 0
  with env_vars({'WN_CUDA_GRAPH': '1' if graphs else '0'}):
    m = WaveNet(**kw, precision=cfg['precision'], max_batch=B, max_time=T)
    m.build(((B, T, 1), (B, cond_in)) if cond_in else (B, T, 1))
  m.handle.glorot_init(seed=1, bias_std=0.02)
  return m, B, T, cond_in


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--configs', nargs='+', default=['c2', 'c4'])
  ap.add_argument('--reps', type=int, default=30)
  ap.add_argument('--warmup', type=int, default=5)
  a = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('no CUDA device: this script measures the B200 kernels and has no CPU mode')
  print(f'card: {card()}')
  dev = torch.device('cuda', 0)
  for name in a.configs:
    m, B, T, cond_in = _model(name, graphs=False)
    mg, _, _, _ = _model(name, graphs=True)
    mg.set_weights(m.get_weights())
    h, hg = m.handle, mg.handle
    frames = torch.as_tensor(synth.frames(B, T, seed=3)).reshape(B, T + 1).to(dev)
    x = frames[:, :-1].contiguous()
    cond = torch.as_tensor(synth.speakers_onehot(B, cond_in, seed=3)).to(dev) if cond_in else None
    cout = 3 * m.num_mixtures if m.num_mixtures is not None else 2 ** m.bits
    out = torch.empty((B, T, cout), dtype=torch.float32, device=dev)
    dpred = (torch.randn((B, T, cout), generator=torch.Generator().manual_seed(0)) / (B * T)).to(dev)
    dcond = torch.empty((B, cond_in), dtype=torch.float32, device=dev) if cond_in else None
    st = h.stream_ptr()

    def step(hh):
      _lib.check(hh.lib.wn_train_step(hh.h, hh.ptr(frames), hh.ptr(cond), B, T, 1, hh.ptr(hh._loss), st))

    def call_backward():
      _lib.check(h.lib.wn_forward_ex(h.h, h.ptr(x), h.ptr(cond), B, T, 1, h.ptr(out), st))
      _lib.check(h.lib.wn_backward(h.h, h.ptr(dpred), h.ptr(dcond), st))

    variants = {'train_step (eager)': lambda: step(h), 'train_step (graph replay)': lambda: step(hg), 'call(training=True) + backward': call_backward}
    for _ in range(a.warmup):
      for f in variants.values():
        f()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    keys = list(variants)
    for i in range(a.reps):
      for k in (keys if i % 2 == 0 else keys[::-1]):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        variants[k]()
        e1.record()
        e1.synchronize()
        times[k].append(e0.elapsed_time(e1))
    # the adjoint of the predictions alone, from the per-launch records of a profiled pass (tag 3: loss / head reductions)
    vjp = []
    for _ in range(5):
      _lib.check(h.lib.wn_forward_ex(h.h, h.ptr(x), h.ptr(cond), B, T, 1, h.ptr(out), st))
      _lib.check(h.lib.wn_profile_begin(h.h, 3))
      _lib.check(h.lib.wn_backward(h.h, h.ptr(dpred), h.ptr(dcond), st))
      _lib.check(h.lib.wn_profile_end(h.h, None, None))
      ms, lab = C.c_double(), C.create_string_buffer(64)
      n = h.lib.wn_profile_get(h.h, 0, None, None, 0)
      for i in range(n):
        h.lib.wn_profile_get(h.h, i, C.byref(ms), lab, 64)
        if lab.value.decode() == 'pred_vjp':
          vjp.append(ms.value)
    med = {k: statistics.median(v) for k, v in times.items()}
    print(f'{name}: B={B} T={T} {cfg_desc(m)}; {a.reps} alternating rounds after {a.warmup} warm-up')
    for k, v in times.items():
      print(f'  {k:32s} {med[k]:8.3f} ms  (p10-p90 {np.percentile(v, 10):.3f}-{np.percentile(v, 90):.3f})')
    print(f'  pred_vjp kernel                  {statistics.median(vjp) * 1e3:8.1f} us  (median of {len(vjp)})')
    print(f'  call + backward / eager train_step: x{med[keys[2]] / med[keys[0]]:.3f}')
    del m, mg
    torch.cuda.empty_cache()


def cfg_desc(m):
  head = f'{m.num_mixtures}-component {m.sampling_function} mixture' if m.num_mixtures else f'{2 ** m.bits}-way softmax'
  return f'{m.blocks} blocks x {m.layers_per_block}, {m.channels} channels, {m.precision}, {head}'


if __name__ == '__main__':
  main()
