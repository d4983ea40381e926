"""Time WaveNet.backward(input_grad=True, param_grads=False) — d loss / d x of a frozen model — against the full backward, at
the bench sizes of C2, C3 and C5 (CONFIGS: batch 8 x 8000, 8 x 8000, 4 x 16384).

Both variants run eagerly on the caller's stream behind the same call(training=True) (WN_CUDA_GRAPH=0): the call + backward pair
is timed with CUDA events, the rounds alternate the order of the variants after a warm-up.  Every block's activations (256-channel
bf16 rows, 30-40 blocks) are far larger than the 126 MB L2.  The `input_dgrad` kernel time comes from wn_profile_get in separate
profiled passes, with its achieved bandwidth: the bytes it must move (every d h0 row once, the K-1 halo rows of each 64-row tile
again, dx written once) over its time, against the data-sheet 7.7 TB/s.  Prints the card name and power limit next to the
numbers; writes nothing."""
import argparse
import ctypes as C
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from scripts.call_backward_time import _model, card, cfg_desc  # noqa: E402
from wavenets_b200 import _lib, synth  # noqa: E402

HBM_TBS = 7.7        # HGX B200 data sheet, one GPU
ICD_ROWS = 64        # rows per CTA of input_conv_dgrad (kernels_misc.cuh)


def dgrad_bytes(B, T, R, K, elem):
  rows = sum(min(ICD_ROWS + K - 1, T - t0) for t0 in range(0, T, ICD_ROWS))
  return B * rows * R * elem + B * T * 4


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--configs', nargs='+', default=['c2', 'c3', 'c5'])
  ap.add_argument('--reps', type=int, default=30)
  ap.add_argument('--warmup', type=int, default=5)
  a = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('no CUDA device: this script measures the B200 kernels and has no CPU mode')
  print(f'card: {card()}')
  dev = torch.device('cuda', 0)
  for name in a.configs:
    m, B, T, cond_in = _model(name, graphs=False)
    h = m.handle
    x = torch.as_tensor(synth.frames(B, T, seed=3)).reshape(B, T + 1)[:, :-1].contiguous().to(dev)
    cond = torch.as_tensor(synth.speakers_onehot(B, cond_in, seed=3)).to(dev) if cond_in else None
    cout = 3 * m.num_mixtures if m.num_mixtures is not None else 2 ** m.bits
    out = torch.empty((B, T, cout), dtype=torch.float32, device=dev)
    dpred = (torch.randn((B, T, cout), generator=torch.Generator().manual_seed(0)) / (B * T)).to(dev)
    dcond = torch.empty((B, cond_in), dtype=torch.float32, device=dev) if cond_in else None
    dx = torch.empty((B, T), dtype=torch.float32, device=dev)
    st = h.stream_ptr()

    def call():
      _lib.check(h.lib.wn_forward_ex(h.h, h.ptr(x), h.ptr(cond), B, T, 1, h.ptr(out), st))

    def full():
      call()
      _lib.check(h.lib.wn_backward(h.h, h.ptr(dpred), h.ptr(dcond), st))

    def input_only():
      call()
      _lib.check(h.lib.wn_backward_ex(h.h, h.ptr(dpred), h.ptr(dcond), h.ptr(dx), 0, st))

    variants = {'call + backward (parameter gradients)': full, 'call + backward(input_grad, no params)': input_only}
    launches = {}
    for k, f in variants.items():
      for _ in range(a.warmup):
        f()
      launches[k] = int(h.lib.wn_last_launch_count(h.h))
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
    # the dgrad kernel alone, from the per-launch records of profiled passes (tag 4: every launch)
    kern = []
    for _ in range(10):
      call()
      _lib.check(h.lib.wn_profile_begin(h.h, 4))
      _lib.check(h.lib.wn_backward_ex(h.h, h.ptr(dpred), h.ptr(dcond), h.ptr(dx), 0, st))
      _lib.check(h.lib.wn_profile_end(h.h, None, None))
      ms, lab = C.c_double(), C.create_string_buffer(64)
      n = h.lib.wn_profile_get(h.h, 0, None, None, 0)
      for i in range(n):
        h.lib.wn_profile_get(h.h, i, C.byref(ms), lab, 64)
        if lab.value.decode() == 'input_dgrad':
          kern.append(ms.value)
    med = {k: statistics.median(v) for k, v in times.items()}
    print(f'{name}: B={B} T={T} {cfg_desc(m)}; {a.reps} alternating rounds after {a.warmup} warm-up')
    for k, v in times.items():
      print(f'  {k:40s} {med[k]:8.3f} ms  (p10-p90 {np.percentile(v, 10):.3f}-{np.percentile(v, 90):.3f})  {launches[k]} launches')
    print(f'  input-only / full: x{med[keys[1]] / med[keys[0]]:.3f}')
    elem = 2 if m.precision == 'bf16' else 4
    nbytes = dgrad_bytes(B, T, m.channels, m.kernel_size, elem)
    t_us = statistics.median(kern) * 1e3
    gbs = nbytes / (t_us * 1e-6) / 1e9
    print(f'  input_dgrad kernel {t_us:8.1f} us (median of {len(kern)}), {nbytes / 1e6:.1f} MB -> {gbs:.0f} GB/s = '
          f'{gbs / (HBM_TBS * 1e3) * 100:.0f} % of {HBM_TBS} TB/s (HBM-bound: {nbytes / (HBM_TBS * 1e12) * 1e6:.1f} us at that rate)')
    del m
    torch.cuda.empty_cache()


if __name__ == '__main__':
  main()
