"""Multi-GPU correctness of WaveNet.backward (tf.GradientTape over WaveNet.call under MirroredStrategy, train.py:203): every replica
runs call + backward on its batch shard with d loss / d pred already divided by the GLOBAL batch, backward clips nothing here and
SUM-all-reduces the gradients; the result equals ONE GPU's backward over the concatenated batch.  Launch like
scripts/dp_grad_check.py: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P
scripts/dp_backward_check.py [--native 0|1]; rank 0 prints one JSON line per case and exits non-zero when a case misses its tolerance."""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
from wavenets_b200 import WaveNet, parallel, synth

CASES = {
  # fp32 tier: reduction-order differences only
  'fp32_cond_skip': (dict(channels=32, blocks=4, layers_per_block=2, activation='leaky_relu', dilation_bound=16, skip_channels=48,
                          final_layers_channels=[64, 64], conditioning='global', mapping_layers=[8, 16], mapping_activation='leaky_relu'), 'fp32', 2, 1500, 1e-5),
  # bf16 tier, persistent stack launches (75 row tiles per replica > 74 CTA pairs) and grouped weight gradients, mixture head
  'bf16_stack_logistic': (dict(channels=256, blocks=6, layers_per_block=1, dilation_bound=16, skip_channels=256, final_layers_channels=[256],
                               conditioning='global', mapping_layers=[8], mapping_activation='tanh', num_mixtures=10,
                               sampling_function='logistic', bits=16), 'bf16', 3, 6400, 3e-5),
}


def run_case(name, rank, local, world, native):
  kw, precision, b_local, T, tol = CASES[name]
  cond_in = 11 if kw.get('conditioning') else 0
  B = b_local * world
  dev = torch.device('cuda', local)
  x = synth.frames(B, T, seed=7)[:, :-1]
  cond = synth.speakers_onehot(B, cond_in, seed=7) if cond_in else None
  cout = 3 * kw['num_mixtures'] if kw.get('num_mixtures') else 256
  dpred = np.random.default_rng(5).standard_normal((B, T, cout)).astype(np.float32) / B
  lo, hi = parallel.shard_bounds(B, rank, world)
  m = WaveNet(**kw, precision=precision, device=local, max_batch=b_local, max_time=T)
  m.build(((b_local, T, 1), (b_local, cond_in)) if cond_in else (b_local, T, 1))
  m.handle.glorot_init(seed=1, bias_std=0.02)
  parallel.attach(m, native=native)
  m((x[lo:hi], cond[lo:hi]) if cond is not None else x[lo:hi])
  m.backward(dpred[lo:hi])
  g_dp = m.handle.flat_grads.clone()
  res = None
  if rank == 0:
    m1 = WaveNet(**kw, precision=precision, device=local, max_batch=B, max_time=T)
    m1.build(((B, T, 1), (B, cond_in)) if cond_in else (B, T, 1))
    m1.set_weights(m.get_weights())
    m1((x, cond) if cond is not None else x)
    m1.backward(dpred)
    g1 = m1.handle.flat_grads
    worst, who = 0.0, None
    hh = m.handle
    for nm, shape, off in zip(hh.names, hh.shapes, hh.offsets):
      n = int(np.prod(shape))
      a, b = g_dp[off:off + n].double(), g1[off:off + n].double()
      if float(b.norm()) == 0.0:
        assert float(a.abs().max()) == 0.0, nm
        continue
      e = float((a - b).norm() / b.norm())
      if e > worst:
        worst, who = e, nm
    res = {'case': name, 'n_replicas': world, 'precision': precision, 'global_batch': B, 'T': T, 'worst_rel_l2': worst, 'tensor': who, 'tol': tol,
           'allreduce': 'C ABI (wn_allreduce_grads, NCCL)' if m._comm is not None else 'torch.distributed',
           'stack_backward_layers': int(hh.lib.wn_stack_backward_layers(hh.h)), 'ok': bool(worst <= tol)}
    print(json.dumps(res), flush=True)
  dist.barrier()
  return res


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--native', type=int, default=1)
  ap.add_argument('--cases', default=','.join(CASES))
  args = ap.parse_args()
  rank, local, world = parallel.init_from_env()
  torch.cuda.set_device(local)
  ok = True
  for name in args.cases.split(','):
    r = run_case(name, rank, local, world, bool(args.native))
    if rank == 0 and not r['ok']:
      ok = False
  dist.barrier()
  dist.destroy_process_group()
  sys.exit(0 if ok else 1)


if __name__ == '__main__':
  main()
