"""Time one bf16 WaveNetLayer called with time-constant conditioning (per-batch bias of the gated conv) against the same layer
called with a time-varying conditioning sequence (wn_layer_forward_seq: conv_cond as one more contraction segment, separate
gate / conv1 launches instead of the fused block kernel).

Shape: B = 8, T = 8000, R = D = S = 256, K = 2, Cc in {80, 256}.  The C entry points are timed directly with CUDA events on
the caller's stream, so the Python layer's input checks are not part of the numbers.  Each repetition runs both variants
back to back (order alternating), after a warm-up.  The block's activations (8*8000 rows x 256 channels, bf16 ~ 33 MB per
tensor) and the fp32 inputs and outputs exceed the 126 MB L2 together, so every pass streams from HBM.  Prints the card
name and power limit next to the numbers; writes nothing."""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from wavenets_b200 import WaveNetLayer, _lib  # noqa: E402


def card():
  try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', str(torch.cuda.current_device())],
                       capture_output=True, text=True, timeout=30)
    return q.stdout.strip() or torch.cuda.get_device_name()
  except (OSError, subprocess.SubprocessError):
    return torch.cuda.get_device_name() + ', power limit unknown'


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--reps', type=int, default=100)
  ap.add_argument('--warmup', type=int, default=10)
  ap.add_argument('--B', type=int, default=8)
  ap.add_argument('--T', type=int, default=8000)
  ap.add_argument('--channels', type=int, default=256)
  ap.add_argument('--cc', type=int, nargs='+', default=[80, 256])
  a = ap.parse_args()
  if not torch.cuda.is_available():
    raise SystemExit('no CUDA device: this script measures the B200 kernels and has no CPU mode')
  B, T, R = a.B, a.T, a.channels
  print(f'card: {card()}')
  print(f'layer: B={B} T={T} R=D=S={R} K=2 dilation 1, bf16; {a.reps} reps after {a.warmup} warm-up, alternating order')
  dev = torch.device('cuda', 0)
  g = torch.Generator(device='cpu').manual_seed(0)
  for Cc in a.cc:
    lay = WaveNetLayer(kernel=2, dilation_rate=1, channels=R, skip_channels=R, condition=True, precision='bf16')
    lay.build(((B, T, R), (B, T, Cc)))
    h = lay._handle
    x = torch.randn((B, T, R), generator=g).to(dev)
    c2 = torch.randn((B, Cc), generator=g).to(dev)
    c3 = torch.randn((B, T, Cc), generator=g).to(dev)
    xo, sk = torch.empty_like(x), torch.empty_like(x)
    dxo, dsk = torch.randn((B, T, R), generator=g).to(dev), torch.randn((B, T, R), generator=g).to(dev)
    dx, dc2, dc3 = torch.empty_like(x), torch.empty_like(c2), torch.empty_like(c3)
    st = h.stream_ptr()

    def fwd(seq):
      if seq:
        _lib.check(h.lib.wn_layer_forward_seq(h.h, 0, h.ptr(x), h.ptr(c3), B, T, 0, h.ptr(xo), h.ptr(sk), st))
      else:
        _lib.check(h.lib.wn_layer_forward_ex(h.h, 0, h.ptr(x), h.ptr(c2), B, T, 0, h.ptr(xo), h.ptr(sk), st))

    def bwd(seq):
      _lib.check(h.lib.wn_layer_backward(h.h, 0, h.ptr(dxo), h.ptr(dsk), h.ptr(dx), h.ptr(dc3 if seq else dc2), st))

    for i in range(a.warmup):
      for seq in (False, True):
        fwd(seq)
        bwd(seq)
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(2 * a.reps)]
    order = []
    for i in range(a.reps):
      pair = (False, True) if i % 2 == 0 else (True, False)
      for seq in pair:
        e = ev[len(order)]
        e[0].record()
        fwd(seq)
        e[1].record()
        bwd(seq)
        e[2].record()
        order.append(seq)
    torch.cuda.synchronize()
    res = {False: ([], []), True: ([], [])}
    for seq, e in zip(order, ev):
      res[seq][0].append(e[0].elapsed_time(e[1]))
      res[seq][1].append(e[0].elapsed_time(e[2]))
    med = {k: (statistics.median(v[0]), statistics.median(v[1])) for k, v in res.items()}
    q = {k: (np.percentile(v[0], [10, 90]), np.percentile(v[1], [10, 90])) for k, v in res.items()}
    for seq, name in ((False, 'time-constant (B,Cc)'), (True, 'sequence (B,T,Cc)')):
      f, fb = med[seq]
      print(f'Cc={Cc:4d} {name:22s} forward {f:7.3f} ms (p10-p90 {q[seq][0][0]:.3f}-{q[seq][0][1]:.3f})   '
            f'forward+backward {fb:7.3f} ms (p10-p90 {q[seq][1][0]:.3f}-{q[seq][1][1]:.3f})')
    print(f'Cc={Cc:4d} sequence / constant: forward x{med[True][0] / med[False][0]:.3f}, forward+backward x{med[True][1] / med[False][1]:.3f}')
    del lay
    torch.cuda.empty_cache()


if __name__ == '__main__':
  main()
