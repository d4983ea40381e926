#!/usr/bin/env python
"""bench.py — audio samples/s of one fwd+bwd WaveNet training pass (forward, loss, backward,
gradient all-reduce; optimizer and metrics excluded) on N B200s of one node.

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
  python bench.py --impl reference ...                   # the reference path on the host CPU cores
  torchrun --nproc-per-node N bench.py --gpus N ...      # N > 1: one rank per GPU, NCCL

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.  Inputs and weights are seeded, so two builds
run with the same arguments and `--dump-outputs DIR` can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

METRIC = 'audio samples/sec fwd+bwd WaveNet stack'
UNIT = 'samples/s'
# label of wn_profile_get -> the kernel it names (for the JSON line)
HBM_PHASES = {
  'loss': 'softmax_ce_reg_kernel / softmax_ce_kernel / mixture_loss_kernel (loss + d logits, one pass)',
  'skip_sum': 'tc_conv_gemm_staged_kernel<bias_act_res>: skip accumulation as ONE K = L*D GEMM over the cached gate outputs',
  'head_fwd': 'tc_conv_gemm_staged_kernel<bias_act_res> x head convs (last one writes fp32 logits)',
  'head_bwd': 'tc_conv_gemm_staged_kernel<dgrad> x head convs (+ their weight gradients when not in the grouped launch)',
  'input_conv_fwd': 'input_conv_fwd_rows',
  'input_conv_bwd': 'input_conv_bwd_stage1_wide + reduce_parts_tall x2',
  'wgrad_group_finish': 'tc_wgrad_group_finish (sums the row splits of every 256x256 gradient tile, L2 term, bias column sums)',
}


def load_peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      pk = json.load(f)
    return dict(hbm=pk['hbm_gbs'], tensor=pk['bf16_tflops_sustained'], tensor_burst=pk['bf16_tflops'], source='measured')
  return dict(hbm=6650.0, tensor=1400.0, tensor_burst=1590.0, source='fallback')


class ClockSampler:
  """SM clock + throttle reasons DURING the timed region (B200_PROFILING.md recipe: `nvidia-smi --query-gpu=clocks.sm,
  clocks.max.sm,clocks_event_reasons.*`).  The same counters are read through NVML (pynvml) from a thread every 5 ms — the
  timed region of a default run is ~60 ms, less than nvidia-smi needs to start up; nvidia-smi -lms is the fallback."""
  Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
       'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
  BITS = {0x4: 'sw_power_cap', 0x8: 'hw_slowdown', 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown'}

  def __init__(self, index):
    self.index, self.proc, self.lines = index, None, []
    self.nvml, self.handle, self.samples, self.stop_flag = None, None, [], False
    try:
      import pynvml
      pynvml.nvmlInit()
      h = None
      try:
        import torch
        uuid = str(torch.cuda.get_device_properties(index).uuid)
        if not uuid.startswith('GPU-'):
          uuid = 'GPU-' + uuid
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, 'encode') else uuid)
      except Exception:
        h = None
      if h is None:
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        phys = index
        if vis:
          try:
            phys = int(vis.split(',')[index])
          except Exception:
            phys = index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
      self.nvml, self.handle = pynvml, h
      self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
    except Exception:
      self.nvml = None

  def _poll(self):
    n = self.nvml
    while not self.stop_flag:
      try:
        mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        try:
          mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
          mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        self.samples.append((mhz, mask))
      except Exception:
        pass
      time.sleep(0.005)

  def start(self):
    if self.nvml is not None:
      self.stop_flag = False
      self.thread = threading.Thread(target=self._poll, daemon=True)
      self.thread.start()
      return
    try:
      self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '100'],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._pump, daemon=True)
      self.thread.start()
    except Exception:
      self.proc = None

  def _pump(self):
    for line in self.proc.stdout:
      self.lines.append(line.strip())

  def stop(self):
    if self.nvml is not None:
      self.stop_flag = True
      self.thread.join(timeout=1.0)
      sm = [m for m, _ in self.samples]
      reasons = set()
      for _, mask in self.samples:
        for bit, name in self.BITS.items():
          if mask & bit:
            reasons.add(name)
      return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': self.sm_max, 'reasons': sorted(reasons), 'samples': len(sm),
              'source': 'nvml'}
    if self.proc is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    time.sleep(0.12)
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except Exception:
      self.proc.kill()
    sm, mx, reasons = [], [], set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for ln in self.lines:
      f = [x.strip() for x in ln.split(',')]
      if len(f) < 9:
        continue
      try:
        sm.append(float(f[1])); mx.append(float(f[2]))
      except ValueError:
        continue
      for name, v in zip(names, f[5:9]):
        if v.lower().startswith('active'):
          reasons.add(name)
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': sorted(reasons), 'samples': len(sm), 'source': 'nvidia-smi'}


def load_dram_profile(config, precision):
  """Per-kernel DRAM bytes of ONE step from the committed ncu launch list of this workload (profiles/dram_<cfg>.json, written
  by scripts/ncu_dram_summary.py from `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum`):
  {kernel: {launches, dram_read, dram_write, ms}}; None when no capture of this config is committed."""
  path = os.path.join(ROOT, 'profiles', f'dram_{config}.json')
  if not os.path.exists(path):
    return None
  with open(path) as f:
    d = json.load(f)
  return d if d.get('precision', precision) == precision else None


def cpu_reference_run(cfg, kw, cond_in, steps, warmup, budget_s, threads=None):
  """The reference path restated on torch CPU ops (oracle/torch_ref.py; TF is not installable):
  fwd+bwd, fp32, all host threads, on a bounded sample (B=1, T_sample) of the same workload."""
  import torch
  from oracle import wavenet_oracle as wo
  from oracle import torch_ref
  from wavenets_b200 import synth, workmodel
  threads = threads or os.cpu_count()
  torch.set_num_threads(threads)
  ocfg = wo.config_from_kwargs(kw, cond_in)
  flops = 3 * workmodel.flops_fwd_per_sample(kw)['total']
  # size the sample for a few seconds per step (~4e11 FLOP), within [512, recording_length]
  T_full = cfg['recording_length']
  T_s = int(min(T_full, max(512, 4.0e11 / flops)))
  p = wo.init_params(ocfg, seed=1, dtype=np.float32)
  stepper = torch_ref.CpuStepper(ocfg, p, threads=threads)
  x = synth.frames(1, T_s, seed=0, apply_mulaw=cfg.get('apply_mulaw', True))
  cond = synth.speakers_onehot(1, cond_in, seed=0) if cond_in else None
  for _ in range(warmup):
    stepper.step(x, cond)
  times = []
  t_begin = time.perf_counter()
  for _ in range(steps):
    t0 = time.perf_counter()
    stepper.step(x, cond)
    times.append(time.perf_counter() - t0)
    if time.perf_counter() - t_begin > budget_s:
      break
  dt = float(np.median(times))
  return {'value': T_s / dt, 'unit': UNIT, 'cores': threads, 'kind': 'port',
          'sample': f'B=1 x T={T_s} of the {cfg["recording_length"]}-sample segments, fp32, {len(times)} timed steps (median), '
                    'torch-CPU restatement of the reference path (TensorFlow not installable)',
          'ms_per_step': dt * 1e3, 'steps': len(times)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, loss, grads):
  """What one training step hands its caller, as float32 .npy files: loss.npy = [loss, reg_loss] and grads.npy = the
  gradients of every variable, flattened and concatenated in variable order.  When the gradients exceed the size limit,
  grads.npy holds a fixed, seeded sample of their entries (in index order), the same for every run of the same workload."""
  os.makedirs(out_dir, exist_ok=True)
  g = np.concatenate([v.ravel() for v in grads.values()]).astype(np.float32)
  budget = (DUMP_LIMIT_BYTES - (1 << 12)) // g.itemsize - loss.size   # (1 << 12): the two .npy headers
  if g.size > budget:
    g = g[np.sort(np.random.default_rng(0).choice(g.size, budget, replace=False))]
  np.save(os.path.join(out_dir, 'loss.npy'), loss.astype(np.float32))
  np.save(os.path.join(out_dir, 'grads.npy'), g)


def model_allreduce_kind(model):
  if model.n_replicas <= 1:
    return 'none (1 replica)'
  if model._comm is not None:
    return 'ncclAllReduce(SUM, fp32) over the flat gradient buffer behind the C ABI (wn_allreduce_grads), ' + (
      'enqueued by wn_train_step inside the step graph' if model._ar_fused else 'after per-replica clipnorm')
  return 'torch.distributed.all_reduce(SUM) on the flat gradient buffer'


def check_grads(model, kw, precision, local, rank, world, frames_np, cond_np, B_local, T, cond_in):
  """SURVEY.md 8e scaling check: the all-reduced gradients of the N shards == the 1-GPU gradients of the concatenated batch
  (compute_average_loss divides by the GLOBAL batch, model.py:328, so the replicas' gradients are summed)."""
  import torch
  import torch.distributed as dist
  from wavenets_b200 import WaveNet
  dev = torch.device('cuda', local)
  data = (torch.from_numpy(frames_np).to(dev), torch.from_numpy(cond_np).to(dev)) if cond_np is not None else torch.from_numpy(frames_np).to(dev)
  model.train_step_async(data)
  g_dp = model.handle.flat_grads.clone()
  # gather every rank's shard on rank 0 (plumbing) and run the whole batch on ONE GPU
  fr = torch.from_numpy(frames_np).to(dev)
  parts = [torch.empty_like(fr) for _ in range(world)] if world > 1 else [fr]
  if world > 1:
    dist.all_gather(parts, fr)
  allx = torch.cat(parts, 0)
  allc = None
  if cond_np is not None:
    cd = torch.from_numpy(cond_np).to(dev)
    cparts = [torch.empty_like(cd) for _ in range(world)] if world > 1 else [cd]
    if world > 1:
      dist.all_gather(cparts, cd)
    allc = torch.cat(cparts, 0)
  res = None
  if rank == 0:
    m1 = WaveNet(**kw, precision=precision, device=local, max_batch=B_local * world, max_time=T)
    m1.build(((B_local * world, T, 1), (B_local * world, cond_in)) if cond_in else (B_local * world, T, 1))
    m1.set_weights(model.get_weights())
    m1.train_step_async((allx, allc) if allc is not None else allx)
    g1 = m1.handle.flat_grads
    hh = model.handle
    worst, who = 0.0, None
    for name, shape, off in zip(hh.names, hh.shapes, hh.offsets):
      n = int(np.prod(shape))
      a, b = g_dp[off:off + n].double(), g1[off:off + n].double()
      den = float(b.norm())
      if den == 0.0:
        continue
      e = float((a - b).norm()) / den
      if e > worst:
        worst, who = e, name
    res = {'worst_rel_l2': worst, 'tensor': who, 'global_rel_l2': float((g_dp.double() - g1.double()).norm() / g1.double().norm()),
           'n_replicas': world, 'global_batch': B_local * world}
    del m1
  if world > 1:
    dist.barrier()
  return res


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=10)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--config', default='c2')
  ap.add_argument('--precision', default=None)
  ap.add_argument('--batch', type=int, default=None, help='sequences per GPU')
  ap.add_argument('--time', type=int, default=None, help='recording_length override')
  ap.add_argument('--channels', type=int, default=None)
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--profile-steps', type=int, default=3)
  ap.add_argument('--sustain-seconds', type=float, default=3.0, help='length of the additional seconds-long timed region (0 = off)')
  ap.add_argument('--dropout', type=float, default=None, help="override the config's dropout (defaults.yaml:17 trains with 0.1)")
  ap.add_argument('--check-grads', action='store_true', help='compare the all-reduced N-GPU gradients with a 1-GPU step on the concatenated batch')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='write the loss and gradients of the last timed step to DIR/loss.npy and DIR/grads.npy (float32, at most 64 MB)')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl != 'b200':
    ap.error('--dump-outputs writes the outputs of the CUDA path (--impl b200)')
  if args.warmup < 3 and args.impl == 'b200':
    args.warmup = 3   # timing rule: W >= 3

  from wavenets_b200 import CONFIGS, model_kwargs, synth
  cfg = dict(CONFIGS[args.config])
  if args.time:
    cfg['recording_length'] = args.time
  if args.channels:
    cfg['channels'] = args.channels
    if cfg.get('skip_channels'):
      cfg['skip_channels'] = args.channels
  if args.dropout is not None:
    cfg['dropout'] = args.dropout
  precision = args.precision or cfg.get('precision', 'bf16')
  B_local = args.batch or cfg['batch_size']
  T = cfg['recording_length']
  kw = model_kwargs(cfg)
  cond_in = cfg.get('n_speakers', 109) if kw['conditioning'] == 'global' else 0
  rank = int(os.environ.get('RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  workload = (f'{args.config}: WaveNet {kw["blocks"]}x{kw["layers_per_block"]} R={kw["channels"]} S={kw["skip_channels"]} '
              f'{"global-cond(" + str(cond_in) + ")" if cond_in else "uncond"} '
              f'{kw["sampling_function"]}{"-" + str(kw["num_mixtures"]) if kw["num_mixtures"] else "-" + str(2 ** kw["bits"])} '
              f'T={T} B={B_local}/GPU')

  # ------------------------------------------------------------------ reference arm (host CPU)
  if args.impl == 'reference':
    if rank != 0:
      return 0
    r = cpu_reference_run(cfg, kw, cond_in, max(1, args.steps), max(1, min(args.warmup, 2)), budget_s=120.0)
    line = {'impl': 'reference', 'metric': METRIC, 'value': r['value'], 'unit': UNIT, 'n_gpus': args.gpus, 'steps': r['steps'],
            'warmup': max(1, min(args.warmup, 2)), 'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': workload, 'sample': r['sample']},
            'cpu_baseline': {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
            'e2e': {'value': r['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))
    return 0

  # ------------------------------------------------------------------ this repo's CUDA path
  # stdout carries ONE JSON line: NCCL writes its version banner there when NCCL_DEBUG is VERSION or INFO
  # (it does on this image even without NCCL_DEBUG in the environment): until the line is printed, file descriptor 1
  # points at stderr
  sys.stdout.flush()
  saved_stdout = os.dup(1)
  os.dup2(2, 1)
  import torch
  import torch.distributed as dist
  from wavenets_b200 import WaveNet, parallel
  if not torch.cuda.is_available():
    raise RuntimeError('bench.py needs a B200 (no CPU fallback); use --impl reference for the host baseline')
  rank, local, world = parallel.init_from_env()
  torch.cuda.set_device(local)
  dev = torch.device('cuda', local)
  if world != args.gpus and rank == 0:
    print(f'# note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE', file=sys.stderr)

  model = WaveNet(**kw, precision=precision, device=local, max_batch=B_local, max_time=T)
  x_shape = (B_local, T, 1)
  model.build((x_shape, (B_local, cond_in)) if cond_in else x_shape)
  model.handle.glorot_init(seed=1, bias_std=0.0)
  parallel.attach(model)
  h = model.handle

  # synthetic mu-law audio + speaker ids; every rank gets its own shard of the global batch
  frames_np = synth.frames(B_local, T, seed=rank, apply_mulaw=cfg.get('apply_mulaw', True))
  cond_np = synth.speakers_onehot(B_local, cond_in, seed=rank) if cond_in else None
  frames_pin = torch.from_numpy(frames_np).pin_memory()
  cond_pin = torch.from_numpy(cond_np).pin_memory() if cond_np is not None else None
  frames_dev = frames_pin.to(dev)
  cond_dev = cond_pin.to(dev) if cond_pin is not None else None
  data_dev = (frames_dev, cond_dev) if cond_dev is not None else frames_dev
  data_host = (frames_pin, cond_pin) if cond_pin is not None else frames_pin

  def sync_all():
    torch.cuda.synchronize(dev)
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize(dev)

  def max_over_ranks(ms):
    if world == 1:
      return ms
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())

  # ---- warm-up (also builds tensor maps, NCCL channels)
  for _ in range(args.warmup):
    model.train_step_async(data_dev)
  # W steps are ~20 ms of work: 40 more untimed steps (a quarter of a second; the same count on every rank, each step
  # holds an all-reduce) so that the timed regions do not start on clocks that are still ramping up from idle
  for i in range(40):
    model.train_step_async(data_dev)
    if i % 8 == 7:
      torch.cuda.synchronize(dev)
  # (the host-buffer path stages into its own device buffers = its own CUDA graph: warm it up as well)
  for _ in range(max(1, args.warmup)):
    loss0 = float(model.train_step(data_host)['loss'])

  # ---- timed region 1: inputs resident in HBM
  sampler = ClockSampler(local) if (rank == 0 and not os.environ.get('WN_BENCH_NO_CLOCKS')) else None
  sync_all()
  if sampler:
    sampler.start()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(args.steps):
    loss_t = model.train_step_async(data_dev)
  e1.record()
  sync_all()
  ms_total = max_over_ranks(e0.elapsed_time(e1))
  launches = int(h.lib.wn_last_launch_count(h.h)) * args.steps
  side_l = C.c_int(0)
  wg_tiles = int(h.lib.wn_grouped_wgrad_tiles(h.h, C.byref(side_l)))   # of the timed (graph-replayed) step
  stack_layers = int(h.lib.wn_stack_forward_layers(h.h))
  stack_bwd_layers = int(h.lib.wn_stack_backward_layers(h.h))
  ar_early = int(h.lib.wn_allreduce_buckets(h.h))
  clocks = sampler.stop() if sampler else None
  loss_last = float(loss_t[0].item())
  # the steps below overwrite the gradient buffer: keep what the last timed step returned
  last_outputs = (loss_t.cpu().numpy(), model.get_grads()) if args.dump_outputs and rank == 0 else None

  # ---- timed region 2: end to end through the public API with HOST buffers
  sync_all()
  e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e2.record()
  pending = None
  for _ in range(args.steps):
    # pinned H2D of frames (+cond), step, all-reduce, D2H of the loss floats into pinned memory — EVERY step; the host
    # reads step k's loss after it has enqueued step k+1 (the way Keras `fit` fetches its logs), so the GPU never idles
    nxt = model.train_step_deferred(data_host)
    if pending is not None:
      out = pending.result()
    pending = nxt
  out = pending.result()
  e3.record()
  sync_all()
  ms_e2e = max_over_ranks(e2.elapsed_time(e3))
  # ---- (transparency) the strictly synchronous public call: H2D, step, D2H, host sync every step
  sync_all()
  es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  es0.record()
  for _ in range(args.steps):
    model.train_step(data_host)
  es1.record()
  sync_all()
  ms_e2e_sync = max_over_ranks(es0.elapsed_time(es1))

  h2d = frames_pin.numel() * 4 + (cond_pin.numel() * 4 if cond_pin is not None else 0)
  rows = B_local * T
  step_ms = ms_total / args.steps

  # ---- timed region 3: a seconds-long run (clocks settled under the power cap): the number the SUSTAINED tensor peak of
  # MEASURED_PEAKS.json is the matching denominator for (the K-step region above is a fraction of a second: burst peak)
  sustained = None
  if args.sustain_seconds > 0:
    n_sus = max(args.steps, int(np.ceil(args.sustain_seconds * 1e3 / step_ms)))
    sync_all()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler2 = ClockSampler(local) if (rank == 0 and not os.environ.get('WN_BENCH_NO_CLOCKS')) else None
    if sampler2:
      sampler2.start()
    s0.record()
    for i in range(n_sus):
      model.train_step_async(data_dev)      # (no host sync inside the region: one graph launch per step)
    s1.record()
    sync_all()
    ms_sus = max_over_ranks(s0.elapsed_time(s1))
    clocks2 = sampler2.stop() if sampler2 else None
    sustained = {'steps': n_sus, 'seconds': ms_sus * 1e-3, 'ms_per_step': ms_sus / n_sus, 'value': world * rows * n_sus / (ms_sus * 1e-3), 'unit': UNIT,
                 'clocks': clocks2}

  # ---- per-launch CUDA-event records (eager, single stream): kernel classes and phases
  from wavenets_b200 import workmodel
  flops = workmodel.flops_fwd_per_sample(kw)
  peaks = load_peaks()
  prof = {}
  by_label = {}
  # (one discarded eager step first: the passes below follow seconds of graph replays; every pass = one step, the fastest of
  # `profile_steps` repeats counts — a single slow outlier of the eager pass would otherwise scale the whole class)
  h.lib.wn_profile_begin(h.h, 4)
  model.train_step_async(data_dev)
  h.lib.wn_profile_end(h.h, None, None)
  for tag, name in ((1, 'dilated'), (2, 'gemm_all'), (4, 'all')):
    best = None
    for _ in range(max(1, args.profile_steps)):
      h.lib.wn_profile_begin(h.h, tag)
      model.train_step_async(data_dev)
      ms = C.c_double()
      n = C.c_int64()
      h.lib.wn_profile_end(h.h, C.byref(ms), C.byref(n))
      if best is None or ms.value < best[0]:
        best = (ms.value, n.value)
        if tag == 4:
          by_label = {}
          lab = C.create_string_buffer(64)
          d = C.c_double()
          nrec = int(h.lib.wn_profile_get(h.h, 0, C.byref(d), lab, 64))
          for i in range(nrec):
            h.lib.wn_profile_get(h.h, i, C.byref(d), lab, 64)
            e = by_label.setdefault(lab.value.decode(), [0.0, 0])
            e[0] += d.value
            e[1] += 1
    prof[name] = best
  kernels = {k: {'ms_per_step': v[0], 'launches_per_step': v[1]} for k, v in sorted(by_label.items(), key=lambda kv: -kv[1][0])}
  tiles_c, parts_c, side_c = C.c_int(0), C.c_int(0), C.c_int(0)
  h.lib.wn_grouped_wgrad_info(h.h, C.byref(tiles_c), C.byref(parts_c), C.byref(side_c))
  e_bytes = 2 if precision == 'bf16' else 4
  dram = load_dram_profile(args.config, precision) if (not args.time and not args.channels and not args.batch) else None

  # ---- roofline of the dominant kernel class
  # The timed region replays the step as a CUDA graph (two streams), where single kernels cannot be bracketed by events.
  # Each launch is therefore timed with an event pair in an eager, single-stream pass over the same inputs; that pass pays
  # a few microseconds of launch gap per kernel, so a class is charged its SHARE of the eager pass times the measured
  # graph-replay step (the ncu launch list under profiles/ shows the same share).
  fused_blocks = int(h.lib.wn_fused_forward_blocks(h.h))
  dmodel = kw['dilation_channels'] or kw['channels']
  dil_ms_eager, dil_launches = prof['dilated']
  share = dil_ms_eager / prof['all'][0] if prof['all'][0] > 0 else 0.0
  total_flops_step = 3.0 * flops['total'] * rows
  alg_bytes_step = workmodel.alg_bytes_per_sample(kw, e_bytes) * rows
  narrow = kw['channels'] < 128      # reference default width: AI of the un-fused layers is below the ridge (SURVEY.md 8d) -> HBM roofline
  if precision == 'bf16' and not narrow:
    # grouped weight gradients: ONE launch (+ side launches) computes the gated-conv, conv1, conv_skip and head filter
    # gradients as 256 x 256 tiles; the launch is timed in this class, so all of its products count as the class's work;
    # the fused forward kernels' conv1 products likewise (forward only; their adjoints run in other kernels)
    dil_flops_step = (2.0 * flops['dilated'] + (wg_tiles * 2.0 * 256 * 256 if wg_tiles else flops['dilated'])) * rows
    dil_flops_step += fused_blocks * 2.0 * dmodel * kw['channels'] * rows
    if stack_bwd_layers:
      # the stack-backward launch also holds the adjoints of conv1 / conv_skip (the DG tile: d g = [d x_out | d skip] . [Wr^T ; Ws^T]);
      # like the fused forward's conv1 products they cannot be separated from the launch's time, so they count as its work.
      # Last block under use_skip: conv1's output is unused, only the skip term exists.
      use_skip = kw.get('use_skip', True)
      s_w = (kw['skip_channels'] or kw['channels']) if use_skip else 0      # skip_channels=None: d skip meets Wr^T (a second R-wide segment)
      per_block = [((kw['channels'] if (l < kw['blocks'] - 1 or not use_skip) else 0) + s_w) for l in range(kw['blocks'])]
      dil_flops_step += sum(2.0 * dmodel * k for k in per_block) * rows
    dil_ms = share * step_ms
    achieved = dil_flops_step / (dil_ms * 1e-3) / 1e12 if dil_ms > 0 else 0.0
    top = None
    if dram:
      top = max(dram['kernels'].items(), key=lambda kv: kv[1]['ms'])
    roofline = {'bound': 'tensor', 'achieved': achieved, 'peak': peaks['tensor_burst'], 'unit': 'TFLOP/s', 'frac': achieved / peaks['tensor_burst'],
                'peak_source': f'{peaks["source"]} bf16 BURST (cuBLAS 8192^3 best of 10, MEASURED_PEAKS.json): the timed region is {ms_total * 1e-3:.2f} s long',
                # dram bytes (read + write) of the class's dominant kernel, per launch, from the committed ncu capture
                'traffic': (top[1]['dram_read'] + top[1]['dram_write']) / max(1, top[1]['launches']) if top else None,
                'traffic_kernel': top[0] if top else None,
                'kernel': ('tc_stack_fwd_kernel (gated conv + gate + conv1 + residual of ALL layers, one persistent launch, CTA pairs) + ' if stack_layers else
                           ('tc_block_fwd_kernel (gated conv + gate + conv1 + residual, CTA pairs) + ' if fused_blocks else 'tc_conv_gemm_staged_kernel<gate> + '))
                + ('tc_stack_bwd_kernel (gate adjoint + dgrad of ALL layers, one persistent launch, CTA pairs) + ' if stack_bwd_layers else 'tc_conv_gemm_staged_kernel<dgrad, cta_group::2> + ')
                + ('tc_wgrad_group_kernel (+ finish): gated-conv, conv1, conv_skip and head filter gradients of all blocks in one launch'
                   if wg_tiles else 'tc_wgrad_pair_kernel (+ tc_wgrad_finish) on the dilated convs'),
                'class': 'dilated-conv GEMMs (fwd + dgrad + wgrad) and the 1x1 products fused into the same launches (conv1 forward, conv1 / conv_skip adjoints, conv1 / conv_skip / head weight gradients)', 'launches_per_step': dil_launches, 'grouped_wgrad_tiles': wg_tiles,
                'stack_forward_layers': stack_layers, 'wgrad_side_launches': int(side_l.value), 'fused_forward_blocks': fused_blocks,
                'ms_per_step_in_kernel': dil_ms, 'ms_per_step_in_kernel_eager_events': dil_ms_eager,
                'ms_per_step_all_launches_eager_events': prof['all'][0], 'share_of_step': share, 'flops_per_step': dil_flops_step}
    if sustained:
      a_s = dil_flops_step / (share * sustained['ms_per_step'] * 1e-3) / 1e12 if share > 0 else 0.0
      roofline['sustained'] = {'achieved': a_s, 'peak': peaks['tensor'], 'frac': a_s / peaks['tensor'],
                               'peak_source': f'{peaks["source"]} bf16 SUSTAINED (cuBLAS back to back for 4 s): region of {sustained["seconds"]:.1f} s'}
  else:
    # fp32 tier at the reference's default width (R = 32): AI of the whole block is below the ridge (SURVEY.md 8d) -> HBM roofline
    # over the block-fused algorithmic bytes of the WHOLE step
    achieved = alg_bytes_step / (step_ms * 1e-3) / 1e9
    roofline = {'bound': 'hbm', 'achieved': achieved, 'peak': peaks['hbm'], 'unit': 'GB/s', 'frac': achieved / peaks['hbm'],
                'peak_source': f'{peaks["source"]} HBM copy bandwidth (MEASURED_PEAKS.json)', 'traffic': None,
                'kernel': ('whole step (tc_conv_gemm_staged_kernel + tc_wgrad_kernel, tcgen05 tier; 64-channel k-blocks padded in shared memory by TMA zero fill)'
                           if precision == 'bf16' else 'whole step (conv_gemm_simt + wgrad_simt FFMA tier)') + ': block-fused algorithmic bytes / step time',
                'alg_bytes_per_step': alg_bytes_step, 'launches_per_step': prof['all'][1],
                'tensor_equivalent_tflops': total_flops_step / (step_ms * 1e-3) / 1e12}
  if dram:
    roofline['traffic_by_kernel'] = {k: {'launches_per_step': v['launches'], 'dram_bytes_per_step': v['dram_read'] + v['dram_write'], 'ncu_ms_per_step': v['ms']}
                                     for k, v in dram['kernels'].items()}
    roofline['dram_bytes_per_step'] = sum(v['dram_read'] + v['dram_write'] for v in dram['kernels'].values())
    roofline['alg_bytes_per_step'] = alg_bytes_step
    roofline['traffic_source'] = dram.get('source')

  # ---- HBM-bound phases (north star item 3): achieved GB/s = bytes the phase must move as launched / its CUDA-event time
  head_grouped = bool(wg_tiles) and len(kw['final_layers_channels']) <= 2 and all(w % 256 == 0 for w in workmodel.head_widths(kw))
  phase_bytes = workmodel.hbm_phase_bytes_per_sample(kw, e_bytes, head_grouped)
  roofline_hbm = {}
  for lab, what in HBM_PHASES.items():
    if lab not in by_label or by_label[lab][0] <= 0:
      continue
    ms_l, n_l = by_label[lab]
    if lab == 'wgrad_group_finish':
      nbytes = (parts_c.value + tiles_c.value) * 65536 * 4
    else:
      nbytes = phase_bytes.get(lab, 0) * rows
    if nbytes <= 0:
      continue
    gbs = nbytes / (ms_l * 1e-3) / 1e9
    roofline_hbm[lab] = {'kernel': what, 'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm'], 'unit': 'GB/s', 'frac': gbs / peaks['hbm'],
                         'bytes_per_step': nbytes, 'ms_per_step': ms_l, 'launches_per_step': n_l}
  whole = {'tflops_all_gemms_whole_step': total_flops_step / (step_ms * 1e-3) / 1e12,
           'frac_of_burst_tensor_peak': total_flops_step / (step_ms * 1e-3) / 1e12 / peaks['tensor_burst'],
           'alg_bytes_per_step': alg_bytes_step, 'alg_gbs_whole_step': alg_bytes_step / (step_ms * 1e-3) / 1e9,
           'gemm_ms_per_step_eager_events': prof['gemm_all'][0]}
  if sustained:
    whole['frac_of_sustained_tensor_peak_sustained_region'] = total_flops_step / (sustained['ms_per_step'] * 1e-3) / 1e12 / peaks['tensor']

  line = {
    'metric': METRIC, 'value': world * rows * args.steps / (ms_total * 1e-3), 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
    'warmup': args.warmup, 'ms_per_step': step_ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
    'dtype': 'bf16' if precision == 'bf16' else 'f32', 'data': 'synthetic',
    'config': {'workload': workload, 'global_batch': B_local * world, 'segment': T, 'receptive_field': model.receptive_field,
               'params': int(h.n_scalars), 'parallelism': f'dp{world}', 'dropout': float(kw['dropout']),
               'l2': 'per-step working set (activations cached for backward) is GBs >> 126 MB L2; no explicit flush needed'
                     if rows * kw['channels'] * kw['blocks'] * e_bytes > 2.5e8 else 'per-step working set fits L2: steps run back to back on a warm L2 (as in training)',
               'flops_per_sample_fwd_bwd': 3 * flops['total'], 'allreduce': model_allreduce_kind(model),
               # gradient slices all-reduced EARLY on the communication stream, beside the next weight-gradient bucket's kernels
               'allreduce_early_buckets': ar_early, 'stack_backward_layers': stack_bwd_layers},
    'e2e': {'value': world * rows * args.steps / (ms_e2e * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 16,
            'ms_per_step': ms_e2e / args.steps, 'api': 'WaveNet.train_step_deferred(host buffers) + .result(): logs of step k read after step k+1 is enqueued',
            'sync_per_step_ms': ms_e2e_sync / args.steps},
    'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline, 'roofline_hbm': roofline_hbm, 'sustained': sustained, 'kernels': kernels,
    'whole_step': whole, 'loss': {'first': loss0, 'last': loss_last, 'e2e_last': out['loss']},
  }
  if args.check_grads:
    line['grad_check'] = check_grads(model, kw, precision, local, rank, world, frames_np, cond_np, B_local, T, cond_in)
  # ---- informational: one FULL training iteration as the reference runs it (model.py:309-348): the step above plus
  # per-variable clipnorm, Adam on the fp32 master weights, weight re-pack and the sampled-waveform MSE metric
  if world == 1:
    from wavenets_b200.optimizers import Adam
    from wavenets_b200.metrics import MeanSquaredError
    model.compile(optimizer=Adam(learning_rate=5e-4, clipnorm=1.0), metrics=[MeanSquaredError()])
    for _ in range(2):
      model.train_step(data_dev)
    sync_all()
    t0 = time.perf_counter()
    n_it = max(3, min(10, args.steps))
    for _ in range(n_it):
      logs = model.train_step(data_dev)
    sync_all()
    line['full_iteration'] = {'ms': (time.perf_counter() - t0) / n_it * 1e3, 'includes': 'fwd+loss+bwd, clipnorm, Adam, re-pack, sampled-waveform MSE',
                              'loss': model.last_step_logs['loss'], 'mean_squared_error': logs.get('mean_squared_error')}
  sys.stdout.flush()
  os.dup2(saved_stdout, 1)
  os.close(saved_stdout)
  if rank == 0:
    if world == 1 and not args.no_cpu_baseline:
      r = cpu_reference_run(cfg, kw, cond_in, steps=5, warmup=1, budget_s=25.0)
      line['cpu_baseline'] = {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}
    if last_outputs is not None:
      dump_outputs(args.dump_outputs, *last_outputs)
    print(json.dumps(line))
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()
  return 0


if __name__ == '__main__':
  sys.exit(main())
