#!/usr/bin/env python
"""bench.py — images/sec of the SqueezeDet inference hot path on N B200s of one node.

  python bench.py --gpus 1 --steps 20 --warmup 5
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
      --master-port P bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...     # the CPU restatement of the reference's path
  python bench.py ... --dump-outputs DIR   # also write the last timed step's results as .npy

One "step" = one pass of the hot path (backbone + ConvDet + interpret_output +
filter_prediction/NMS) over one batch of synthetic 1242x375 images.  Headline line: SqueezeDet,
b=20 PER GPU (weak scaling: the batch shards over GPUs with no data-path exchange; ONE
ncclAllGather of the filtered records per step, captured inside the forward's CUDA graph when
N > 1).  The same JSON line also carries
  * `strong_scaling` (N > 1): global b=20 sharded 3,3,3,3,2,2,2,2-style, padded per rank;
  * `other_configs`: BASELINE.json configs 3-5 (SqueezeDet+ b=20, ResNet50+ConvDet b=8,
    VGG16+ConvDet b=8 at N=1; SqueezeDet+ and VGG16 sharded at N>1).
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
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

METRIC = 'images/sec (1242x375, b=20)'
NETS = {'squeezeDet': ('SqueezeDet', 'kitti_squeezeDet_config'),
        'squeezeDet+': ('SqueezeDetPlus', 'kitti_squeezeDetPlus_config'),
        'vgg16': ('VGG16ConvDet', 'kitti_vgg16_config'),
        'resnet50': ('ResNet50ConvDet', 'kitti_res50_config')}
BASELINE_BATCH = {'squeezeDet': 20, 'squeezeDet+': 20, 'resnet50': 8, 'vgg16': 8}


def parse_args():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=20)
  ap.add_argument('--warmup', type=int, default=5)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--net', default='squeezeDet', choices=sorted(NETS))
  ap.add_argument('--batch', type=int, default=20, help='images per GPU per step')
  ap.add_argument('--width', type=int, default=1242)
  ap.add_argument('--height', type=int, default=375)
  ap.add_argument('--math', default='tc', choices=['tc', 'simt'])
  ap.add_argument('--cpu-sample', type=int, default=20,
                  help='images in the cpu_baseline sample (N=1, rank 0)')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-other-configs', action='store_true',
                  help='skip BASELINE configs 3-5 and the strong-scaling leg')
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='write what the last timed step of the headline run computed (rank 0) '
                       'as DIR/<name>.npy, float32/float64, at most 64 MB in all')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.dump_outputs and args.impl == 'reference':
    ap.error('--dump-outputs writes what the GPU path computed; --impl reference has no such output')
  return args


def measured_peaks():
  """HBM GB/s and bf16 TF/s from the driver-written MEASURED_PEAKS.json; TF32 dense peak from
  the tcgen05.mma issue-rate microbenchmark of this repo (profiles/r2_tf32_peak.json)."""
  out = dict(hbm_gbs=6650.0, tflops=1590.0, tflops_sustained=1400.0, source='fallback',
             tf32_tflops=1191.4, tf32_source='profiles/r2_tf32_peak.json missing: 4096 flop/clk/SM '
                                             'x 148 SMs x 1.965 GHz')
  try:
    with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
      p = json.load(f)
    out.update(hbm_gbs=float(p['hbm_gbs']), tflops=float(p['bf16_tflops']),
               tflops_sustained=float(p.get('bf16_tflops_sustained', p['bf16_tflops'])),
               source='measured')
  except Exception:
    pass                      # fallback stated in /opt/skills/guides/B200_PROFILING.md
  try:
    with open(os.path.join(ROOT, 'profiles', 'r2_tf32_peak.json')) as f:
      t = json.load(f)
    out.update(tf32_tflops=float(t['tf32_dense_tflops']), tf32_source='profiles/r2_tf32_peak.json')
  except Exception:
    pass
  return out


class ClockSampler:
  """Samples nvidia-smi clocks / throttle reasons DURING the timed region."""
  Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
       'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
       'clocks_event_reasons.sw_power_cap')

  def __init__(self, index):
    self.index = index
    self.rows = []
    self.proc = None
    self.thread = None

  def start(self):
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
           '--format=csv,noheader,nounits', '-lms', '100'],
          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except OSError:
      self.proc = None
      return
    self.thread = threading.Thread(target=self._read, daemon=True)
    self.thread.start()

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append(line.strip())

  def stop(self):
    if not self.proc:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    time.sleep(0.12)
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except Exception:
      self.proc.kill()
    sm, smax, reasons = [], [], set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for r in self.rows:
      parts = [p.strip() for p in r.split(',')]
      if len(parts) < 6:
        continue
      try:
        sm.append(float(parts[0]))
        smax.append(float(parts[1]))
      except ValueError:
        continue
      for nm, v in zip(names, parts[2:6]):
        if v.lower().startswith('active'):
          reasons.add(nm)
    return {'sm_mhz': float(np.median(sm)) if sm else None,
            'sm_max_mhz': max(smax) if smax else None, 'reasons': sorted(reasons),
            'samples': len(sm)}


def host_threads():
  """Host threads this process may actually use (cgroup/affinity aware; os.cpu_count()
  over-reports on shared GPU hosts and oversubscribed torch is 50x slower)."""
  try:
    n = len(os.sched_getaffinity(0))
  except AttributeError:
    n = os.cpu_count() or 1
  try:   # cgroup v2 cpu.max quota
    with open('/sys/fs/cgroup/cpu.max') as f:
      quota, period = f.read().split()
    if quota != 'max':
      n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
  except Exception:
    pass
  return n


def build_mc(net, batch, width, height):
  from squeezedet_b200 import config as cfg
  mc = getattr(cfg, NETS[net][1])()
  mc.IMAGE_WIDTH, mc.IMAGE_HEIGHT, mc.BATCH_SIZE = width, height, batch
  mc.ANCHOR_BOX = cfg.set_anchors(mc)
  mc.ANCHORS = len(mc.ANCHOR_BOX)
  return mc


# ------------------------------------------------------------------------------------------
def cpu_port_rate(args, n_images, threads=None):
  """The CPU arm: the oracle's torch-CPU restatement of the conv half (TF 1.0 is not
  installable) + numpy interpret_output + filter_prediction — the reference's OWN
  `ModelSkeleton.filter_prediction` / `util.nms` imported from /root/reference when that tree is
  present (this container), the pinned restatement of them otherwise (the GPU box).  (The ONLY
  place bench.py touches oracle/: the checker used as a baseline.)"""
  import oracle
  from oracle import ref_import
  from oracle.torch_port import TorchForward
  from squeezedet_b200.utils import synth
  mc = build_mc(args.net, args.batch, args.width, args.height)
  weights = synth.synthetic_weights(oracle.param_specs(args.net), seed=0)
  if threads is None:
    # all the host threads it can use -- but measured, not assumed: on shared GPU hosts the
    # visible CPU count exceeds the usable one and oversubscribed torch collapses.
    probe = synth.synthetic_images(1, args.height, args.width, seed=1)
    best, threads = None, 1
    nmax = host_threads()
    for cand in sorted({nmax, min(nmax, 64), min(nmax, 32), min(nmax, 16), min(nmax, 8)},
                       reverse=True):
      f = TorchForward(args.net, weights, threads=cand)
      f(probe)
      t0 = time.perf_counter()
      f(probe)
      dt = time.perf_counter() - t0
      if best is None or dt < best:
        best, threads = dt, cand
  fwd = TorchForward(args.net, weights, threads=threads)
  images = synth.synthetic_images(n_images, args.height, args.width, seed=1234)
  ref_ns = ref_import.load() if ref_import.available() else None
  filt = ('reference ModelSkeleton.filter_prediction (imported from /root/reference/src)'
          if ref_ns else 'oracle.filter_prediction (pinned restatement; /root/reference absent)')

  def one_pass():
    chunk = 4
    for i in range(0, n_images, chunk):
      preds = fwd(images[i:i + chunk])
      boxes, probs, cls = oracle.interpret_output(
          preds, mc.ANCHOR_BOX, mc.CLASSES, mc.ANCHOR_PER_GRID, mc.IMAGE_WIDTH,
          mc.IMAGE_HEIGHT, mc.EXP_THRESH)
      for j in range(len(probs)):
        if ref_ns:
          ref_import.ref_filter_prediction(ref_ns, boxes[j], probs[j], cls[j], mc.CLASSES,
                                           mc.TOP_N_DETECTION, mc.PROB_THRESH, mc.NMS_THRESH)
        else:
          oracle.filter_prediction(boxes[j], probs[j], cls[j], mc.CLASSES, mc.TOP_N_DETECTION,
                                   mc.PROB_THRESH, mc.NMS_THRESH)
  return one_pass, threads, filt


def run_reference(args):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return            # other ranks exit 0 without work
  sample = args.batch   # the SAME configuration as the main arm: one step = one batch of b images
  one_pass, threads, filt = cpu_port_rate(args, sample)
  for _ in range(max(min(args.warmup, 2), 1)):
    one_pass()
  t0 = time.perf_counter()
  for _ in range(args.steps):
    one_pass()
  dt = time.perf_counter() - t0
  value = sample * args.steps / dt
  what = ('%d synthetic %dx%d images/step: oracle restatement of the conv half on torch-CPU '
          '(TF-1.0 itself is not installable) + numpy interpret_output + %s'
          % (sample, args.width, args.height, filt))
  print(json.dumps({
      'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'images/sec',
      'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak',
      'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': config_dict(args, 1),
      'arithmetic': 'cpu f32 (torch-CPU convs + numpy post-processing)',
      'cpu_baseline': {'value': value, 'unit': 'images/sec', 'cores': threads, 'kind': 'port',
                       'sample': what, 'filter_impl': filt},
      'e2e': {'value': value, 'unit': 'images/sec', 'h2d_bytes_per_step': 0,
              'd2h_bytes_per_step': 0},
      'gpu_launches': 0}))


def config_dict(args, world):
  """The workload description; IDENTICAL in both arms (the reference arm runs "your arm's
  config" on the host cores)."""
  return {'workload': workload_name(args.net, args.width, args.height, args.batch),
          'net': args.net, 'global_batch': world * args.batch,
          'image': [args.height, args.width],
          'parallelism': 'batch-sharded x%d, one ncclAllGather of detections per step inside '
                         'the forward CUDA graph' % world,
          'l2': 'no flush: the activations of one step (GBs) stream through the 126 MB L2',
          'math': args.math}


def workload_name(net, width, height, batch):
  return '%s inference, synthetic %dx%d, batch %d per GPU, random (calibrated) weights' % (
      net, width, height, batch)


# ------------------------------------------------------------------------------------------
class Runner:
  """One engine of `net` at `batch` images on this rank's GPU, plus the buffers of the
  device-resident path (`value`) and of the host-buffer path (`e2e`)."""

  def __init__(self, args, net, batch, rank, world, local, stream, ident=None):
    import torch
    from squeezedet_b200 import _lib, nets
    from squeezedet_b200.utils import synth
    self.torch, self._lib = torch, _lib
    self.args, self.net, self.B = args, net, batch
    self.rank, self.world, self.local = rank, world, local
    self.stream = stream
    self.sptr = stream.cuda_stream
    mc = build_mc(net, batch, args.width, args.height)
    math_mode = _lib.MATH_TF32X3_TC if args.math == 'tc' else _lib.MATH_FP32_SIMT
    self.model = getattr(nets, NETS[net][0])(mc, local, math_mode=math_mode)
    self.model.load_weights(synth.synthetic_weights(synth.model_param_specs(self.model), seed=0))
    H, W = args.height, args.width
    # host inputs in pinned memory (e2e path) and a device-resident copy (`value` path)
    self.pinned = _lib.PinnedArray((batch, H, W, 3), np.float32)
    self.pinned.array[...] = synth.synthetic_images(batch, H, W, seed=1234 + rank)
    self.x_dev = torch.from_numpy(self.pinned.array).cuda(local)
    self.pinned_u8 = _lib.PinnedArray((batch, H, W, 3), np.uint8)
    self.pinned_u8.array[...] = np.random.default_rng(99 + rank).integers(
        0, 256, self.pinned_u8.array.shape, dtype=np.uint8)
    md = self.model.max_dets
    self.dets_host = [_lib.PinnedArray((batch, md), _lib.DET_DTYPE) for _ in range(2)]
    self.counts_host = [_lib.PinnedArray((batch,), np.int32) for _ in range(2)]
    self.lib = _lib.load()
    self.e2e_i = 0
    if world > 1:
      # the ONE collective of the path: ncclAllGather of the result blob, issued by the engine
      # on the compute stream inside the forward's CUDA graph (no torch on the data path)
      self.model.comm_init(world, rank, ident, in_forward=True)

  # ---- the two step functions -----------------------------------------------------------
  def step_device(self):
    self.model.forward_device(self.x_dev.data_ptr(), self.sptr)

  def step_e2e(self, kind, src):
    i = self.e2e_i
    self._lib.check(self.lib.sqdet_submit(self.model._engine, src, kind,
                                          self.dets_host[i & 1].ptr, self.counts_host[i & 1].ptr))
    if i >= 1:
      self._lib.check(self.lib.sqdet_wait(self.model._engine))   # step i-1 is on the host
    self.e2e_i = i + 1

  def drain_e2e(self):
    while True:
      try:
        self._lib.check(self.lib.sqdet_wait(self.model._engine))
      except self._lib.SqdetError:
        break
    self.e2e_i = 0
    self.torch.cuda.synchronize()

  def barrier(self):
    import torch.distributed as dist
    if self.world > 1:
      dist.barrier()
    self.torch.cuda.synchronize()

  def max_over_ranks(self, ms):
    import torch.distributed as dist
    t = self.torch.tensor([ms], device=self.x_dev.device)
    if self.world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())

  def timed_device(self, steps):
    torch = self.torch
    self.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(self.stream)
    for _ in range(steps):
      self.step_device()
    e1.record(self.stream)
    self.stream.synchronize()
    self.barrier()
    return self.max_over_ranks(e0.elapsed_time(e1))

  def timed_e2e(self, kind, src, steps):
    for _ in range(3):
      self.step_e2e(kind, src)
    self.drain_e2e()
    self.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
      self.step_e2e(kind, src)
    self.drain_e2e()                                   # last step's results delivered
    dt = time.perf_counter() - t0
    self.barrier()
    return self.max_over_ranks(dt * 1e3) / steps

  def fetch_outputs(self, budget=64 << 20):
    """The results of the last forward, as a caller of the device-resident path reads them:
    det_boxes [B,A,4], det_probs [B,A], det_class [B,A] (float32) and the filtered records
    [B,max_dets,7] (anchor, cls, prob, cx, cy, w, h; float64) with their counts [B].  Over
    `budget` bytes, the det_* arrays keep a fixed seeded sample of anchors, listed in
    anchor_sample.npy."""
    self.stream.synchronize()
    r = self.model.results_device()
    B, A, md = self.B, int(self.model.det_probs.shape[1]), r['max_dets']

    def fetch(ptr, dtype, shape):
      out = np.empty(shape, dtype)
      self._lib.check(self.lib.sqdet_memcpy_d2h(out.ctypes.data, ptr, out.nbytes, None))
      self._lib.check(self.lib.sqdet_stream_sync(self.local, None))
      return out
    dets = fetch(r['dets'], self._lib.DET_DTYPE, (B, md))
    arrays = {
        'det_boxes': fetch(r['det_boxes'], np.float32, (B, A, 4)),
        'det_probs': fetch(r['det_probs'], np.float32, (B, A)),
        'det_class': fetch(r['det_class'], np.int64, (B, A)).astype(np.float32),
        'records': np.stack([dets[f].astype(np.float64) for f in dets.dtype.names], axis=-1),
        'counts': fetch(r['counts'], np.int32, (B,)).astype(np.float64)}
    det_bytes = B * A * 6 * 4
    rest = arrays['records'].nbytes + arrays['counts'].nbytes
    if det_bytes + rest > budget:
      k = max(1, (budget - rest - 8 * A) // (B * 6 * 4))
      keep = np.sort(np.random.default_rng(0).choice(A, size=min(k, A), replace=False))
      for name in ('det_boxes', 'det_probs', 'det_class'):
        arrays[name] = np.ascontiguousarray(arrays[name][:, keep])
      arrays['anchor_sample'] = keep.astype(np.float64)
    return arrays

  def measure(self, steps, warmup, global_images, want_f32_feed=False, fetch=False):
    """-> dict(value, ms_per_step, e2e...).  `global_images` = images the whole job processes
    per step (world * B for weak scaling, the real global batch for strong scaling).  fetch=True
    adds 'outputs': fetch_outputs() of the last timed step (rank 0)."""
    _lib = self._lib
    for _ in range(max(warmup, 3)):
      self.step_device()
    ms = self.timed_device(steps) / steps
    out = {'ms_per_step': ms, 'value': global_images / (ms * 1e-3)}
    if fetch and self.rank == 0:
      out['outputs'] = self.fetch_outputs()       # before the e2e steps overwrite the results
    ms_e2e = self.timed_e2e(_lib.IMG_U8, self.pinned_u8.ptr, steps)
    out['e2e'] = {'value': global_images / (ms_e2e * 1e-3), 'unit': 'images/sec',
                  'h2d_bytes_per_step': int(self.pinned_u8.array.nbytes),
                  'd2h_bytes_per_step': int(self.dets_host[0].array.nbytes +
                                            self.counts_host[0].array.nbytes),
                  'ms_per_step': ms_e2e}
    if want_f32_feed:
      ms_f32 = self.timed_e2e(_lib.IMG_F32, self.pinned.ptr, steps)
      out['e2e_f32_feed'] = {'value': global_images / (ms_f32 * 1e-3), 'unit': 'images/sec',
                             'h2d_bytes_per_step': int(self.pinned.array.nbytes),
                             'd2h_bytes_per_step': out['e2e']['d2h_bytes_per_step'],
                             'ms_per_step': ms_f32,
                             'input': 'float32 mean-subtracted images (the reference feed_dict '
                                      'payload), PCIe-bound'}
    return out

  def check_gather(self):
    """N > 1: the gathered buffer must hold every rank's records (this rank's slice must equal
    its own blob, and every rank's counts must be valid)."""
    from squeezedet_b200 import shard
    dets, counts = self.model.detect_records(self.pinned.array)   # forward + in-graph gather
    g = self.model.read_gathered()
    mine_d, mine_c = shard.unpack_blob(g[self.rank], self.B, self.model.max_dets)
    ok = bool(np.array_equal(mine_c, counts) and np.array_equal(mine_d, dets))
    for r in range(self.world):
      _, c = shard.unpack_blob(g[r], self.B, self.model.max_dets)
      ok = ok and bool((c >= 0).all() and (c <= self.model.max_dets).all())
    return ok

  def per_op_table(self, peaks, reps=5):
    """Per-op CUDA-event times (un-graphed run of the same launches) with the HBM fraction of
    the op's algorithmic bytes and the tensor fraction of its issued (3xTF32) flops."""
    acc = None
    for _ in range(reps):
      rows = self.model.forward_profiled(self.x_dev.data_ptr(), self.sptr)
      t = np.array([ms for _, ms in rows])
      acc = t if acc is None else acc + t
    acc /= reps
    table = self.model.op_table()
    issue = 3.0 if self.args.math == 'tc' else 1.0
    per_op = []
    for (nm, fl, pa, by), ms in zip(table, acc):
      sec = max(float(ms), 1e-6) * 1e-3
      per_op.append({'op': nm, 'ms': round(float(ms), 4), 'gflop': round(fl / 1e9, 3),
                     'mbytes': round(by / 1e6, 2),
                     'hbm_frac': round(by / sec / 1e9 / peaks['hbm_gbs'], 4),
                     'tensor_frac': round(issue * fl / sec / 1e12 / peaks['tf32_tflops'], 4)})
    return table, acc, per_op

  def close(self):
    if self.world > 1:
      self.model.comm_destroy()
    self.model = None


def roofline_of(table, acc, peaks, clocks, math, traffic_file=None):
  top = int(np.argmax(acc))
  nm, fl, pa, by = table[top]
  ridge = peaks['tf32_tflops'] / 3.0 * 1e12 / (peaks['hbm_gbs'] * 1e9)   # algorithmic flop/B
  sec = float(acc[top]) * 1e-3
  if fl / max(by, 1) >= ridge:
    # tensor-bound: achieved = ALGORITHMIC flops / time against the measured dense TF32 issue
    # peak; 3xTF32 issues 3 MMAs per algorithmic MAC, so this tops out at 1/3 (`issued_frac`
    # below is the tensor-pipe view of the same number)
    ach, peak, unit, bound = fl / sec / 1e12, peaks['tf32_tflops'], 'TFLOP/s', 'tensor'
  else:
    ach, peak, unit, bound = by / sec / 1e9, peaks['hbm_gbs'], 'GB/s', 'hbm'
  traffic = None
  if traffic_file:
    try:
      with open(os.path.join(ROOT, 'profiles', traffic_file)) as f:
        traffic = json.load(f)['bytes_per_op'].get(nm)
    except Exception:
      pass
  sm_mhz = clocks['sm_mhz'] if clocks and clocks.get('sm_mhz') else 1965.0
  return {'kernel': nm, 'bound': bound, 'achieved': ach, 'peak': peak, 'unit': unit,
          'frac': ach / peak, 'traffic': traffic,
          'traffic_source': ('profiles/%s (ncu dram bytes, same workload)' % traffic_file)
                            if traffic else None,
          'peak_source': peaks['source'] if bound == 'hbm' else peaks['tf32_source'],
          'kernel_ms': float(acc[top]), 'kernel_share_of_step': float(acc[top] / acc.sum()),
          'achieved_tflops': fl / sec / 1e12,
          'issued_frac': (3.0 if math == 'tc' else 1.0) * fl / sec / 1e12 / peaks['tf32_tflops'],
          'hbm_frac': by / sec / 1e9 / peaks['hbm_gbs'],
          'fp32_simt_peak_tflops': 148 * 128 * 2 * sm_mhz * 1e6 / 1e12,
          'algorithmic_bytes_per_launch': by, 'algorithmic_flops_per_launch': fl}


def run_ours(args):
  import torch
  import torch.distributed as dist
  from squeezedet_b200 import _lib, shard

  rank = int(os.environ.get('RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  local = int(os.environ.get('LOCAL_RANK', '0'))
  if world != args.gpus and world > 1:
    raise SystemExit('--gpus %d but WORLD_SIZE=%d' % (args.gpus, world))
  if _lib.device_count() < 1:
    raise SystemExit('bench.py: no CUDA device visible; the engine has no CPU fallback')
  torch.cuda.set_device(local)
  if world > 1:
    # stdout carries exactly one JSON line: NCCL prints its version banner (and everything else) to
    # stdout at any NCCL_DEBUG level >= VERSION, so leave the level unset unless the caller asked for
    # more, and send whatever it prints to stderr
    if os.environ.get('NCCL_DEBUG', '').upper() in ('VERSION', 'WARN'):
      del os.environ['NCCL_DEBUG']
    os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
    dist.init_process_group('nccl', rank=rank, world_size=world,
                            device_id=torch.device('cuda', local))
  stream = torch.cuda.Stream(device=local)

  def new_ident():
    """ncclUniqueId of a fresh engine-owned communicator (torch.distributed is only the host
    channel that carries the 128 bytes, plus barriers and the max-over-ranks of the timings)."""
    if world == 1:
      return None
    box = [_lib.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    return box[0]

  peaks = measured_peaks()
  W = max(args.warmup, 3)
  B = args.batch

  # ---- headline: args.net, b per GPU (weak scaling) ----------------------------------------
  main = Runner(args, args.net, B, rank, world, local, stream, new_ident())
  sampler = ClockSampler(local)
  if rank == 0:
    sampler.start()
  res = main.measure(args.steps, W, world * B, want_f32_feed=True, fetch=bool(args.dump_outputs))
  gather_ok = main.check_gather() if world > 1 else None
  if world > 1:
    main.model.set_gather_in_forward(False)     # what follows is rank-local (no collective)
  if rank == 0:
    # extra loaded steps so the 100 ms nvidia-smi sampler sees the GPU under this workload
    t_end = time.perf_counter() + 0.6
    while time.perf_counter() < t_end:
      main.step_device()
      stream.synchronize()
  clocks = sampler.stop() if rank == 0 else None
  if 'outputs' in res:
    os.makedirs(args.dump_outputs, exist_ok=True)
    for name, a in res.pop('outputs').items():
      np.save(os.path.join(args.dump_outputs, name + '.npy'), a)

  roofline = per_op = None
  if rank == 0:
    table, acc, per_op = main.per_op_table(peaks)
    roofline = roofline_of(table, acc, peaks, clocks, args.math, 'r2_traffic.json')
    tot_by = sum(r[3] for r in table)
    tot_fl = sum(r[1] for r in table)
    sec = res['ms_per_step'] * 1e-3
    roofline['whole_step'] = {
        'algorithmic_gbytes': tot_by / 1e9, 'gflop': tot_fl / 1e9,
        'hbm_gbs': tot_by / sec / 1e9, 'hbm_frac': tot_by / sec / 1e9 / peaks['hbm_gbs'],
        'tflops': tot_fl / sec / 1e12,
        'tensor_frac_issued': (3.0 if args.math == 'tc' else 1.0) * tot_fl / sec / 1e12 /
                              peaks['tf32_tflops']}
  launches = main.model.launches_per_forward()
  op_bytes = sum(r[3] for r in main.model.op_table())
  main.close()
  main = None

  # ---- strong scaling: the SAME global batch over N GPUs ---------------------------------
  strong = None
  other = []
  if not args.no_other_configs and world > 1:
    gb = BASELINE_BATCH[args.net]
    bmax = max(shard.shard_sizes(gb, world))
    r = Runner(args, args.net, bmax, rank, world, local, stream, new_ident())
    m = r.measure(args.steps, W, gb)
    strong = {'scaling': 'strong', 'global_batch': gb, 'shards': shard.shard_sizes(gb, world),
              'batch_per_gpu_padded': bmax, 'value': m['value'], 'unit': 'images/sec',
              'ms_per_step': m['ms_per_step'], 'e2e': m['e2e'],
              'limit': 'per-GPU work shrinks to %d images: the persistent one-CTA-per-SM grids '
                       'run out of tiles (fire6-11 / ConvDet: %d tiles of 128 px for 148 SMs), '
                       'so the step approaches the sum of ~27 launch-latency-bound kernels'
                       % (bmax, bmax * 15)}
    r.close()

  # ---- BASELINE.json configs 3-5 -----------------------------------------------------------
  if not args.no_other_configs and args.net == 'squeezeDet':
    if world == 1:
      plans = [('squeezeDet+', 20, 20, 'weak'), ('resnet50', 8, 8, 'weak'), ('vgg16', 8, 8, 'weak')]
    else:
      gb_v = BASELINE_BATCH['vgg16']
      plans = [('squeezeDet+', 20, world * 20, 'weak'),
               ('squeezeDet+', max(shard.shard_sizes(20, world)), 20, 'strong'),
               ('vgg16', max(shard.shard_sizes(gb_v, world)), gb_v, 'strong')]
    for net, b, gimg, mode in plans:
      r = Runner(args, net, b, rank, world, local, stream, new_ident())
      m = r.measure(args.steps, 3, gimg)
      row = {'net': net, 'workload': workload_name(net, args.width, args.height, b),
             'n_gpus': world, 'scaling': mode, 'global_batch': gimg, 'batch_per_gpu': b,
             'value': m['value'], 'unit': 'images/sec', 'ms_per_step': m['ms_per_step'],
             'steps': args.steps, 'e2e': m['e2e']}
      if world > 1:
        r.model.set_gather_in_forward(False)
      if rank == 0:
        table, acc, pop = r.per_op_table(peaks, reps=3)
        row['roofline'] = roofline_of(table, acc, peaks, clocks, args.math)
        tot_fl = sum(x[1] for x in table)
        tot_by = sum(x[3] for x in table)
        sec = m['ms_per_step'] * 1e-3
        row['whole_step'] = {'gflop': tot_fl / 1e9, 'algorithmic_gbytes': tot_by / 1e9,
                             'tflops': tot_fl / sec / 1e12,
                             'tensor_frac_issued': (3.0 if args.math == 'tc' else 1.0) * tot_fl /
                                                   sec / 1e12 / peaks['tf32_tflops'],
                             'hbm_frac': tot_by / sec / 1e9 / peaks['hbm_gbs']}
        row['launches_per_step'] = r.model.launches_per_forward()
        row['top_ops'] = sorted(pop, key=lambda x: -x['ms'])[:4]
      r.close()
      other.append(row)

  cpu_baseline = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    n = args.cpu_sample
    one_pass, threads, filt = cpu_port_rate(args, n)
    one_pass()                                   # warm-up
    t0 = time.perf_counter()
    reps = 0
    while reps < 3 or (time.perf_counter() - t0 < 10.0 and reps < 50):
      one_pass()
      reps += 1
    dt = time.perf_counter() - t0
    cpu_baseline = {'value': n * reps / dt, 'unit': 'images/sec', 'cores': threads,
                    'kind': 'port', 'filter_impl': filt,
                    'sample': '%d passes over %d synthetic %dx%d images: oracle restatement '
                              '(torch-CPU convs, all host threads) + numpy interpret + %s'
                              % (reps, n, args.width, args.height, filt)}

  if rank == 0:
    out = {
        'metric': METRIC, 'value': res['value'], 'unit': 'images/sec', 'n_gpus': world,
        'steps': args.steps, 'warmup': W, 'ms_per_step': res['ms_per_step'],
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32 (3xTF32 tcgen05, fp32 accumulate)' if args.math == 'tc' else 'f32',
        'data': 'synthetic',
        'config': config_dict(args, world),
        'algorithmic_gbytes_per_step': op_bytes / 1e9,
        'e2e': dict(res['e2e'],
                    input='uint8 BGR images in pinned host memory; `- mc.BGR_MEANS` '
                          '(demo.py:190) runs on the GPU; sqdet_submit/sqdet_wait, 2 in flight',
                    timer='host wall clock around K submits + final wait (covers H2D, kernels, '
                          'D2H), max over ranks'),
        'e2e_f32_feed': res.get('e2e_f32_feed'),
        'gpu_launches': launches * args.steps,
        'launches_per_step': launches,
        'gather_verified': gather_ok,
        'clocks': clocks, 'roofline': roofline, 'cpu_baseline': cpu_baseline,
        'strong_scaling': strong, 'other_configs': other,
        'per_op': per_op,
    }
    print(json.dumps(out))
  if world > 1:
    dist.destroy_process_group()


def main():
  args = parse_args()
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_ours(args)


if __name__ == '__main__':
  main()
