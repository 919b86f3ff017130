"""Images/sec of the B200 EfficientDet path on N GPUs of one box (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config d0|d4|d7x|v2s]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--config picks the BASELINE.json configuration (default d0 = configs[1], the one the metric is
quoted on):
  d0   EfficientDet-D0  640x640   batch 32/GPU   (headline)
  d4   EfficientDet-D4  1024x1024 batch 8/GPU    (configs[3])
  d7x  EfficientDet-D7x 1536x1536 batch 2/GPU    (configs[4])
  v2s  EfficientNetV2-S 384x384   batch 128, backbone + head conv only (configs[2])

A "step" = one pass of the hot path (stem .. heads .. pre-NMS .. NMS) over one batch of synthetic
images per GPU.  `value` is whole-job images/s with inputs already resident in HBM; `e2e` is the
same metric through the public serving call with HOST buffers (pinned uint8 images copied H2D and
the [B,100,7] detections copied D2H inside the timed region, three requests in flight).  Inputs
and the activations written between kernels (GBs per step) exceed the 126 MB L2, so every timed
iteration starts with a flushed L2.

--dump-outputs DIR writes, after the timed steps, what the last step of each timed path returned
(DIR/<name>.npy, float32, at most 64 MB in all).  Inputs and weights are seeded, so two builds run
with the same arguments can be compared output for output.

--impl reference times the reference's CPU implementation of the path.  TensorFlow is probed at
run time (it is not installable offline); without it the arm runs the oracle port
(oracle/efficientdet_oracle.py + oracle/postprocess_oracle.py) on the host cores, each step a
bounded sample of the same batch.
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

CONFIGS = {
    'd0': dict(kind='det', model='efficientdet-d0', image_size=640, batch=32, raw_hw=(480, 640),
               blocks='16 MBConv, 3 BiFPN cells'),
    'd4': dict(kind='det', model='efficientdet-d4', image_size=1024, batch=8, raw_hw=(768, 1024),
               blocks='32 MBConv, 7 BiFPN cells'),
    'd7x': dict(kind='det', model='efficientdet-d7x', image_size=1536, batch=2, raw_hw=(1152, 1536),
                blocks='55 MBConv, 8 BiFPN cells (levels 3-8)'),
    'v2s': dict(kind='cls', model='efficientnetv2-s', image_size=384, batch=128,
                blocks='40 (Fused-)MBConv blocks + head conv'),
}


def metric_name(cfg):
  if cfg['kind'] == 'det':
    name = cfg['model'].replace('efficientdet-', 'EfficientDet-').replace('-d', '-D')
    return '%s images/sec @ batch %d/GPU (%dx%d, forward + post-process)' % (
        name, cfg['batch'], cfg['image_size'], cfg['image_size'])
  return 'EfficientNetV2-S images/sec @ batch %d/GPU (%dx%d, backbone + head conv)' % (
      cfg['batch'], cfg['image_size'], cfg['image_size'])


def build_config(cfg):
  from automl_b200 import hparams_config
  c = hparams_config.get_efficientdet_config(cfg['model'])
  c.override(dict(image_size=cfg['image_size']))
  return c


def workload_config(cfg, world):
  """The `config` object of the JSON line: identical for our arm and the reference arm."""
  s = cfg['image_size']
  if cfg['kind'] == 'det':
    what = '%s %dx%d batch %d/GPU: stem, %s, class/box heads, pre-NMS, NMS-V5 (gaussian)' % (
        cfg['model'], s, s, cfg['batch'], cfg['blocks'])
  else:
    what = '%s %dx%d batch %d/GPU: stem, %s' % (cfg['model'], s, s, cfg['batch'], cfg['blocks'])
  return {'workload': what, 'global_batch': world * cfg['batch'],
          'parallelism': 'batch-shard x%d' % world,
          'l2': 'inputs and per-step activations (GBs) exceed the 126 MB L2, so every timed '
                'iteration starts with a flushed L2'}


class ClockSampler(object):
  """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
  Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
       'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
       'clocks_event_reasons.sw_power_cap')

  def __init__(self, index=0):
    self.index, self.samples, self.proc = index, [], None

  def start(self):
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
           '--format=csv,noheader,nounits', '-lms', '100'],
          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      threading.Thread(target=self._read, daemon=True).start()
    except OSError:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.samples.append(line.strip())

  def stop(self):
    if self.proc is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    time.sleep(0.15)
    self.proc.terminate()
    sm, mx, reasons = [], [], set()
    for s in self.samples:
      parts = [p.strip() for p in s.split(',')]
      if len(parts) < 6:
        continue
      try:
        sm.append(float(parts[0])); mx.append(float(parts[1]))
      except ValueError:
        continue
      for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                            'sw_power_cap'), parts[2:6]):
        if val.lower().startswith('active'):
          reasons.add(name)
    sm.sort()
    return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': sorted(reasons), 'samples': len(sm)}


DUMP_BYTES = 64 << 20   # --dump-outputs: every array together


def dump_outputs(out_dir, outputs):
  """Writes each output (name -> array) as out_dir/<name>.npy in float32.  One larger than its
  share of DUMP_BYTES is stored as a sample of its elements, flattened: the same seeded positions,
  in index order, on every run."""
  import numpy as np
  os.makedirs(out_dir, exist_ok=True)
  share = DUMP_BYTES // len(outputs) - 1024     # room for the .npy header
  for name, a in outputs.items():
    a = np.asarray(a, np.float32)
    if a.nbytes > share:
      idx = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
      a = a.reshape(-1)[np.sort(idx)]
    np.save(os.path.join(out_dir, name + '.npy'), a)


def measured_peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      d = json.load(f)
    return d['hbm_gbs'], d.get('bf16_tflops_sustained', d.get('bf16_tflops')), 'measured'
  return 6650.0, 1400.0, 'fallback'


# ---- the reference's CPU implementation -----------------------------------------------------------
def probe_tensorflow():
  """The reference's own path needs TensorFlow (requirements.txt:8).  Probed at run time on the
  box; not installable offline, so normally absent."""
  for extra in (os.path.join(ROOT, 'baseline', '_ref'),):
    if os.path.isdir(extra) and extra not in sys.path:
      sys.path.append(extra)
  try:
    import tensorflow as tf  # pylint: disable=g-import-not-at-top
    return getattr(tf, '__version__', 'unknown')
  except Exception:  # pylint: disable=broad-except
    return None


class CpuPath(object):
  """The oracle port of the path on the host cores (`kind: "port"`), built once, timed per call."""

  def __init__(self, cfg):
    import torch
    self.cfg = cfg
    self.cores = min(os.cpu_count() or 1, 32)   # more threads than this slow the small convs down
    torch.set_num_threads(self.cores)
    if cfg['kind'] == 'det':
      from automl_b200 import arch, weights as weights_lib
      from oracle import efficientdet_oracle as eo
      self.config = build_config(cfg)
      w = weights_lib.synthetic_weights(arch.DetArch(self.config), 0)
      self.oracle = eo.Oracle(self.config, w, torch.float32)
      self.params = self.config.as_dict()
    else:
      from automl_b200.efficientnetv2 import effnetv2_model
      from oracle import effnetv2_oracle
      a = effnetv2_model.EffNetV2Arch(cfg['model'])
      w = effnetv2_model.synthetic_weights(a, 0)
      self.oracle = effnetv2_oracle.EffNetV2Oracle(a, w, torch.float32)

  def run(self, images):
    """Seconds for one pass over `images` (float32 [n,S,S,3])."""
    import numpy as np
    t0 = time.perf_counter()
    if self.cfg['kind'] == 'det':
      from oracle import postprocess_oracle as po
      cls_o, box_o = self.oracle(images)
      po.det_post_process(self.params, {l: v.numpy() for l, v in cls_o.items()},
                          {l: v.numpy() for l, v in box_o.items()},
                          np.ones(len(images), np.float32))
    else:
      self.oracle(images)
    return time.perf_counter() - t0


def cpu_images(cfg, n, seed=0):
  import numpy as np
  s = cfg['image_size']
  lo = -1.0 if cfg['kind'] == 'cls' else 0.0
  return np.random.default_rng(seed).uniform(lo, 1.0, size=(n, s, s, 3)).astype(np.float32)


def cpu_baseline(cfg, seconds_budget=25.0):
  """Reported baseline inside our arm (rank 0, N=1 only): a bounded sample of the batch."""
  path = CpuPath(cfg)
  one = path.run(cpu_images(cfg, 1))
  nimg = int(max(1, min(cfg['batch'], seconds_budget // max(one, 1e-3))))
  dt = path.run(cpu_images(cfg, nimg))
  return {'value': nimg / dt, 'unit': 'images/s', 'cores': path.cores, 'kind': 'port',
          'tensorflow': probe_tensorflow(),
          'sample': '%d image(s) of the %dx%d batch through the oracle port (PyTorch-CPU network '
                    '+ numpy post-process), %.1f s' % (nimg, cfg['image_size'], cfg['image_size'], dt)}


def run_reference(args, cfg, rank, world):
  """--impl reference: every step is one measured pass of the CPU path over a bounded sample of
  the batch, sized so that warmup + steps end within ~150 s; ms_per_step is the measured mean."""
  if rank != 0:
    return
  tf_version = probe_tensorflow()
  path = CpuPath(cfg)
  total = max(1, args.steps + args.warmup)
  per_step = max(1.5, 150.0 / total)
  one = path.run(cpu_images(cfg, 1))
  nimg = int(max(1, min(cfg['batch'], per_step // max(one, 1e-3))))
  x = cpu_images(cfg, nimg)
  times = []
  for i in range(args.warmup + args.steps):
    dt = path.run(x)
    if i >= args.warmup:
      times.append(dt)
  mean_s = sum(times) / len(times)
  v = nimg / mean_s
  base = {'value': v, 'unit': 'images/s', 'cores': path.cores, 'kind': 'port',
          'tensorflow': tf_version,
          'sample': 'each step = %d image(s) of the %d-image batch through the oracle port of the '
                    'reference path (PyTorch-CPU network + numpy post-process) on %d host threads; '
                    'TensorFlow %s' % (nimg, cfg['batch'], path.cores,
                                       tf_version or 'not importable on this box')}
  line = {
      'impl': 'reference', 'metric': metric_name(cfg), 'value': v, 'unit': 'images/s',
      'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
      'ms_per_step': 1000.0 * mean_s, 'higher_is_better': True, 'scaling': 'weak',
      'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
      'config': workload_config(cfg, world), 'cpu_baseline': base,
      'e2e': {'value': v, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
  }
  print(json.dumps(line))


# ---- roofline ------------------------------------------------------------------------------------
def family_of(kind):
  """Kernel family of an op kind (all (k, stride) depthwise instantiations are one family)."""
  if kind.startswith('depthwise'):
    return 'depthwise_kernel'
  return {'pointwise_tc': 'pointwise_tc_kernel', 'pointwise_simt': 'pointwise_kernel',
          'sepconv_tc': 'sepconv_direct_kernel', 'bifpn_fuse_dw': 'fuse_dw_kernel',
          'mbconv_expand_dw': 'mbconv_front_kernel', 'conv_tc': 'conv_tc_kernel',
          'nms_v5': 'nms_v5_fast_kernel'}.get(kind, kind + '_kernel')


def roofline_from_rows(rows, exclude=('nms_v5',)):
  """Dominant kernel family by summed CUDA-event time of its launches; NMS runs on its own stream
  overlapped with the next step, so it is not a candidate for the step's dominant kernel."""
  hbm_peak, tf_peak, peak_src = measured_peaks()
  kinds, fams = {}, {}
  for r in rows:
    k = kinds.setdefault(r['kind'], {'ms': 0.0, 'bytes': 0, 'flops': 0, 'launches': 0})
    f = fams.setdefault(family_of(r['kind']), {'ms': 0.0, 'bytes': 0, 'flops': 0, 'launches': 0})
    for d in (k, f):
      d['ms'] += r['ms']; d['bytes'] += r['bytes']; d['flops'] += r['flops']; d['launches'] += 1
  total_ms = sum(k['ms'] for k in kinds.values())
  cand = {n: f for n, f in fams.items() if not any(n.startswith(family_of(e)) for e in exclude)}
  name = max(cand, key=lambda n: cand[n]['ms'])
  fam = cand[name]
  gbs = fam['bytes'] / (fam['ms'] / 1e3) / 1e9
  tfs = fam['flops'] / (fam['ms'] / 1e3) / 1e12
  # the bound is whichever roofline the family sits closer to
  if tfs / tf_peak > gbs / hbm_peak:
    roof = {'bound': 'tensor', 'achieved': tfs, 'peak': tf_peak, 'unit': 'TFLOP/s', 'frac': tfs / tf_peak}
  else:
    roof = {'bound': 'hbm', 'achieved': gbs, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': gbs / hbm_peak}
  roof.update({'kernel': name, 'traffic': None, 'peak_source': peak_src,
               'share_of_step': fam['ms'] / total_ms, 'launches': fam['launches'],
               'per_kind': {n: {'ms': round(k['ms'], 4),
                                'GBps': round(k['bytes'] / max(k['ms'], 1e-9) / 1e6, 1),
                                'TFLOPs': round(k['flops'] / max(k['ms'], 1e-9) / 1e9, 2),
                                'launches': k['launches']} for n, k in sorted(kinds.items())}})
  return roof, kinds, total_ms


def attach_traffic(roof, cfg_name):
  """DRAM bytes of the dominant family per forward from the committed ncu capture of this same
  command (profiles/r2_traffic_<config>.json, written by scripts/make_profiles.py)."""
  for rnd in ('r2', 'r1'):
    path = os.path.join(ROOT, 'profiles', '%s_traffic_%s.json' % (rnd, cfg_name))
    if not os.path.exists(path) and cfg_name == 'd0':
      path = os.path.join(ROOT, 'profiles', '%s_traffic.json' % rnd)
    if not os.path.exists(path):
      continue
    with open(path) as f:
      t = json.load(f).get('per_forward', {}).get(roof['kernel'])
    if t:
      roof['traffic'] = int((t['dram_read_MB'] + t['dram_write_MB']) * 1e6)
      roof['traffic_source'] = ('%s (ncu dram__bytes_read.sum + dram__bytes_write.sum, family sum '
                                'per forward)' % os.path.relpath(path, ROOT))
      return


# ---- our arm ---------------------------------------------------------------------------------------
def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=20)
  ap.add_argument('--warmup', type=int, default=5)
  ap.add_argument('--impl', default='ours')
  ap.add_argument('--config', default='d0', choices=sorted(CONFIGS))
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--profile-out', default='')
  ap.add_argument('--dump-outputs', default='', metavar='DIR')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  cfg = CONFIGS[args.config]

  rank = int(os.environ.get('RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  if args.impl == 'reference':
    run_reference(args, cfg, rank, world)
    return

  import numpy as np
  import torch
  import torch.distributed as dist
  import __graft_entry__
  __graft_entry__.build()

  torch.cuda.set_device(local_rank)
  dev = 'cuda:%d' % local_rank
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device(dev))
  batch = cfg['batch']
  warmup = max(3, args.warmup)
  rng = np.random.default_rng(rank)
  e2e_last = {}   # what the last e2e step returned to its caller

  if cfg['kind'] == 'det':
    from automl_b200 import inference, parallel
    # COCO-shaped raw input (4:3 uint8 images) in pinned host memory
    host_raw = torch.from_numpy(
        rng.integers(0, 256, size=(batch,) + cfg['raw_hw'] + (3,), dtype=np.uint8)).pin_memory()
    driver = inference.ServingDriver(cfg['model'], '_', batch_size=batch,
                                     model_params={'image_size': cfg['image_size']}, device=dev,
                                     image_id_base=rank * batch)
    driver.build()
    eng = driver.engine
    gathered = torch.empty(world * batch, eng.max_output_size, 7, device=dev) if world > 1 else None
    gather_hook = (lambda det: parallel.gather_detections(det, gathered)) if world > 1 else None

    def resident_step():
      # network + pre-NMS on the main stream; NMS (+ the single collective of the path, the
      # all-gather of per-image detections) on the engine's NMS stream, overlapping the next step
      eng.run(postprocess=True, after_nms=gather_hook)

    def resident_finish():
      eng.wait_detections()      # the last step's NMS / all-gather is inside the timed region

    def resident_outputs():
      return {'detections': eng.detections.cpu().numpy()}

    def e2e_loop(steps):
      # the public serving call, three requests in flight: every step copies its uint8 batch H2D
      # and its detections D2H; results are collected in order
      pending = collections.deque()
      for _ in range(steps):
        pending.append(driver.submit(host_raw))
        if len(pending) >= driver.MAX_IN_FLIGHT:
          pending.popleft().result()
      while pending:
        det = pending.popleft().result()
      e2e_last['e2e_detections'] = det

    driver.serve_images(host_raw)   # builds the graphs and leaves a pre-processed batch in HBM
    h2d = int(host_raw.numel()) + 4 * batch
    d2h = int(world * batch * eng.max_output_size * 7 * 4)
    api = ('inference.ServingDriver.submit(uint8 [%d,%d,%d,3] pinned host).result() -> numpy '
           'detections, three requests in flight (H2D, device pre-process, network, NMS, all-gather, '
           'D2H per step)' % ((batch,) + cfg['raw_hw']))
    profile = lambda: eng.profile_ops(iters=3)
    launches = eng.launches_per_forward
    extra = lambda: {'nms_full_queue_images': eng.nms_fallback_count()}
  else:
    from automl_b200.efficientnetv2 import effnetv2_model
    s = cfg['image_size']
    model = effnetv2_model.get_model(cfg['model'], weights=None, batch_size=batch, image_size=s,
                                     device=dev)
    host_x = torch.from_numpy(rng.uniform(-1, 1, size=(batch, s, s, 3)).astype(np.float32)).pin_memory()
    host_out = torch.empty(tuple(model(host_x).shape), dtype=torch.float16).pin_memory()

    def resident_step():
      model.run()

    def resident_finish():
      pass

    def resident_outputs():
      return {'head_1x1': model.endpoints['head_1x1'].float().cpu().numpy()}

    def e2e_loop(steps):
      # public pipelined call: H2D of batch i+1 / D2H of the feature map of batch i-1 overlap the
      # network of batch i; every step copies its float32 batch H2D and its feature map D2H
      for out in model.serve_stream(host_x for _ in range(steps)):
        pass
      e2e_last['e2e_head_1x1'] = out   # pinned host buffer, valid until the next serve_stream

    h2d = int(host_x.numel() * 4)
    d2h = int(host_out.numel() * 2)
    api = ('effnetv2_model.get_model(...).serve_stream(float32 [%d,%d,%d,3] pinned host batches) '
           '-> head feature maps in pinned host memory, two batches in flight' % (batch, s, s))

    def profile():
      evs = []
      for nm, fn in model._ops:  # pylint: disable=protected-access
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); evs.append((e0, e1))
      torch.cuda.synchronize()
      return [dict(info, ms=e0.elapsed_time(e1)) for (e0, e1), info in zip(evs, model.op_info)]
    launches = len(model._ops)  # pylint: disable=protected-access
    extra = lambda: {}

  def timed(loop, steps, warm):
    loop(warm)
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loop(steps)
    e1.record()
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
      dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())

  def resident_loop(steps):
    for _ in range(steps):
      resident_step()
    resident_finish()

  torch.cuda.synchronize()
  sampler = ClockSampler(local_rank)
  if rank == 0:
    sampler.start()
  ms_dev = timed(resident_loop, args.steps, warmup)
  # the e2e steps run on the same engine buffers, so the resident outputs are read before them
  outputs = resident_outputs() if args.dump_outputs and rank == 0 else None
  ms_e2e = timed(e2e_loop, args.steps, 3)
  clocks = sampler.stop() if rank == 0 else None
  if outputs is not None:
    outputs.update({k: torch.as_tensor(v).float().numpy() for k, v in e2e_last.items()})
    dump_outputs(args.dump_outputs, outputs)

  value = world * batch * args.steps / (ms_dev / 1000.0)
  e2e_value = world * batch * args.steps / (ms_e2e / 1000.0)

  line = None
  if rank == 0:
    rows = profile()
    roofline, kinds, total_ms = roofline_from_rows(rows)
    attach_traffic(roofline, args.config)
    if args.profile_out:
      with open(args.profile_out, 'w') as f:
        json.dump({'ops': rows, 'kinds': roofline['per_kind'], 'sum_ms': total_ms}, f, indent=1)
    line = {
        'metric': metric_name(cfg), 'value': value, 'unit': 'images/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': warmup,
        'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f16 storage / f32 accumulate', 'data': 'synthetic',
        'config': workload_config(cfg, world),
        'e2e': {'value': e2e_value, 'unit': 'images/s', 'ms_per_step': ms_e2e / args.steps,
                'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'api': api},
        'gpu_launches': launches * args.steps,
        'clocks': clocks, 'roofline': roofline, 'cpu_baseline': None,
    }
    line.update(extra())
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()
  if rank == 0:
    # the CPU baseline runs on rank 0 at N=1 only, after the process group is gone, so no other
    # rank ever spins in a collective while the host cores are busy
    if world == 1 and not args.no_cpu_baseline:
      line['cpu_baseline'] = cpu_baseline(cfg)
    print(json.dumps(line))


if __name__ == '__main__':
  main()
