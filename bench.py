"""FoV-steps/s and segmented-voxels/s benchmark of the B200 flood-fill engine (contract: DESIGN.md "Measurement").

  python bench.py --gpus 1 --steps K --warmup W            # our arm, N = 1
  python bench.py --impl reference --steps K --warmup W    # reference arm (CPU restatement, rank 0 only)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workloads (BASELINE.json):

  N = 1   configs[0] — the configuration the metric is quoted on: the README run
          `run_inference.py configs/inference_training_sample2.pbtxt` on a 250^3 bounding box, i.e.
          Canvas.segment_all with PolicyPeaks seeds and the pbtxt's inference options, ConvStack3DFFNModel depth 12,
          fov 33^3, deltas 8, FIB-25 weights, on the synthetic stand-in for training_sample2 (Voronoi phantom,
          seed 0; SURVEY.md 8d).  ONE timed step = the whole canvas (~25.6 k FoV steps, ~585 objects) on a fresh
          canvas: a flood fill has no meaningful K-FoV-step prefix (seed policy, object commits and the last objects
          are part of the metric), so --steps K times K such steps (profiler runs cap the seed list with
          --max-seeds); `steps` in the output line is K, `fov_steps` the FoV steps done in them.
          `value` = FoV steps / wall clock of segment_all (device PolicyPeaks included) with the volume resident
          in HBM, summed over the K steps; `e2e` = the same metric through one Runner.run (volume file -> pinned
          H2D -> segment_all -> D2H -> seg-*.npz / .prob written), which is what a user of run_inference.py gets.
          --dump-outputs DIR writes what the last timed step returned (see dump_outputs); the inputs (volume,
          weights, PolicyPeaks tie-break noise) are seeded, so two builds can be compared output for output.
  N > 1   configs[3] — a 1024^3 volume as 8 slabs of 512^3 (2x2x2), slabs_of_rank(8, rank, N) per GPU, every slab an
          independent canvas (the reference's subvolume semantics, doc/manual.md:107-127), then the merge inside the
          timed region: all_gather of the id counts, id offsets on the device, NCCL gather of the label AND
          probability slabs to rank 0.  Strong scaling over the same 8 slabs for N = 2, 4, 8.  (At N = 1 the driver's
          line is configs[0]; both are FoV steps/s of the same kernel on canvases of the same statistics.)

A "FoV step" is one network evaluation + merge + paste + movement-policy update of the persistent kernel
(= the reference's 'inference-calls' counter); steps of objects that were started ahead of their turn and
then discarded are NOT counted (they are reported as `steps_executed`).
"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

FOV = (33, 33, 33)
DELTAS = (8, 8, 8)
DEPTH = 12
WEIGHTS = os.path.join(REPO, 'tests', 'golden', 'fib25_convstack.npz')
WORKLOAD_N1 = ('configs[0]: Runner.run / Canvas.segment_all with PolicyPeaks on a synthetic 250^3 volume (seed 0), '
               'ConvStack3DFFNModel depth 12 fov 33^3 deltas 8, FIB-25 weights, options of inference_training_sample2.pbtxt')
WORKLOAD_MULTI = ('configs[3]: synthetic 1024^3 as 8 slabs of 512^3 (seeds 300..307), slabs_of_rank(8, rank, N), '
                  'Canvas.segment_all with PolicyPeaks per slab, NCCL merge of labels + probability maps on rank 0')


def flops_per_step():
  v = FOV[0] * FOV[1] * FOV[2]
  return 2 * v * (27 * 2 * 32 + (2 * DEPTH - 1) * 27 * 32 * 32 + 32)


def load_weights():
  from ffn_b200 import tf_checkpoint
  if os.path.exists(WEIGHTS):
    return tf_checkpoint.load_convstack_npz(WEIGHTS), 'FIB-25 checkpoint (fixture)'
  rng = np.random.RandomState(0)
  ws = [rng.randn(3, 3, 3, 2 if i == 0 else 32, 32).astype(np.float32) * 0.05 for i in range(2 * DEPTH)]
  ws.append(rng.randn(1, 1, 1, 32, 1).astype(np.float32) * 0.05)
  bs = [np.zeros(32, np.float32) for _ in range(2 * DEPTH)] + [np.zeros(1, np.float32)]
  return (ws, bs), 'random-init'


def make_volume(shape, seed):
  from ffn_b200.synthetic import voronoi_phantom
  cache = os.path.join(os.environ.get('FFN_BENCH_CACHE', '/tmp/ffn_bench_cache'), 'vol_%d_%d.npy' % (shape[0], seed))
  if os.path.exists(cache):
    return np.load(cache)
  vol = voronoi_phantom(shape, seed)
  try:
    os.makedirs(os.path.dirname(cache), exist_ok=True)
    np.save(cache, vol)
  except OSError:
    pass
  return vol


class ClockSampler:
  """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

  QUERY = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
           'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
           'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, index):
    self.index = index
    self.lines = []
    self.proc = None

  def start(self):
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.QUERY, '--format=csv,noheader,nounits',
           '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      threading.Thread(target=self._pump, daemon=True).start()
    except OSError:
      self.proc = None

  def _pump(self):
    for line in self.proc.stdout:
      self.lines.append(line.strip())

  def wait_ready(self, timeout=5.0):
    """Blocks until the first sample has arrived.  nvidia-smi's start-up (NVML initialisation) holds driver locks
    for a few hundred ms: inside the timed region it stalled the first allocation / launch of segment_all by
    ~0.5 s (round 2: wall 2.29 s against 1.70 s of kernel time); the periodic samples afterwards do not."""
    t0 = time.time()
    while self.proc is not None and not self.lines and time.time() - t0 < timeout and self.proc.poll() is None:
      time.sleep(0.02)

  def stop(self):
    if self.proc is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    time.sleep(0.15)
    self.proc.terminate()
    sm, mx, reasons = [], [], set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for ln in self.lines:
      parts = [p.strip() for p in ln.split(',')]
      if len(parts) < 8:
        continue
      try:
        sm.append(float(parts[0])); mx.append(float(parts[1]))
      except ValueError:
        continue
      for n, v in zip(names, parts[4:8]):
        if v.lower().startswith('active'):
          reasons.add(n)
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': sorted(reasons), 'samples': len(sm)}


def ncu_dram_traffic():
  """DRAM bytes (read + write) per launch of the flood kernel from the newest committed `ncu --set full`
  summary under profiles/ (file name carries the FoV steps of the captured launch), or None."""
  import glob
  import re
  scale = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
  for path in sorted(glob.glob(os.path.join(REPO, 'profiles', 'r*_ncu_full_flood_kernel_steps*.txt')), reverse=True):
    m = re.search(r'steps(\d+)', os.path.basename(path))
    total, seen = 0.0, 0
    try:
      with open(path) as f:
        for line in f:
          for key in ('dram__bytes_read.sum [', 'dram__bytes_write.sum ['):
            if line.startswith(key):
              unit = line[len(key):line.index(']')]
              total += float(line.split('=')[1]) * scale[unit]
              seen += 1
    except (OSError, ValueError, KeyError):
      continue
    if seen == 2 and m:
      n = int(m.group(1))
      return {'bytes_per_launch': total, 'steps_per_launch': n, 'bytes_per_step': total / n,
              'source': os.path.relpath(path, REPO)}
  return None


def measured_peaks():
  path = os.path.join(REPO, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      d = json.load(f)
    return d.get('bf16_tflops', 1590.0), d.get('bf16_tflops_sustained', 1400.0), 'measured (MEASURED_PEAKS.json)'
  return 1590.0, 1400.0, 'fallback (B200_PROFILING.md)'


def best_cpu_threads():
  """torch's conv3d on one 33^3 patch stops scaling (and then collapses) well below the core count
  of a big host: pick the thread count that maximises steps/s, like a user of the reference would."""
  import torch
  from oracle.network import ConvStackOracle
  (w, b), _ = load_weights()
  net = ConvStackOracle(w, b)
  rng = np.random.RandomState(0)
  seed = np.full(FOV, -2.9444, np.float32)
  img = rng.randn(*FOV).astype(np.float32)
  ncpu = os.cpu_count() or 1
  best, best_t = None, 1e30
  for n in sorted({min(ncpu, c) for c in (4, 8, 16, 32, 64, ncpu)}):
    torch.set_num_threads(n)
    net(seed, img)
    dt = 1e30
    for _ in range(3):                      # best of three: a single sample is too noisy on a shared host
      t0 = time.time()
      net(seed, img)
      dt = min(dt, time.time() - t0)
    if dt < best_t:
      best, best_t = n, dt
  torch.set_num_threads(best)
  return best


def run_cpu_sample(vol, n_steps, threads):
  """The reference's path restated on the CPU (oracle/): PolicyPeaks seeds + Canvas.segment_all on the same
  volume, stopped after n_steps FoV steps.  Returns (steps, voxels labelled so far, seconds of the flood fill,
  seconds of the seed policy)."""
  import torch
  from oracle import flood_fill as ff
  from oracle import seed_peaks
  from oracle.network import ConvStackOracle
  torch.set_num_threads(threads)
  (w, b), _ = load_weights()
  net = ConvStackOracle(w, b)
  image = (vol.astype(np.float32) - np.float32(128.0)) / np.float32(33.0)
  t0 = time.time()
  seeds = seed_peaks.policy_peaks(image, margin_zyx=(16, 16, 16))
  t_seed = time.time() - t0
  cv = ff.Canvas(net, image, FOV, DELTAS, ff.Options())

  class _Stop(Exception):
    pass
  orig = cv.update_at

  def limited(pos):
    if len(cv.trace) >= n_steps:
      raise _Stop()
    return orig(pos)
  cv.update_at = limited
  t0 = time.time()
  try:
    cv.segment_all(seeds)
  except _Stop:
    pass
  secs = time.time() - t0
  return len(cv.trace), int((cv.segmentation > 0).sum()), secs, t_seed


def device_seeds(cv, margin=(16, 16, 16)):
  """PolicyPeaks on the device + the border filter of BaseSeedPolicy.__next__ (seed.py:81-88)."""
  from ffn_b200.inference import seed as seed_mod
  noise = seed_mod._tie_break_noise(tuple(cv.shape))   # RandomState(42).rand(*shape), seed.py:133-139
  coords = cv.seed_peaks((1, 1, 1), noise)
  m = np.asarray(margin)[None]
  keep = np.all((coords - m >= 0) & (coords + m < np.asarray(cv.shape)[None]), axis=1)
  return np.ascontiguousarray(coords[keep], dtype=np.int32), noise.nbytes


def request_for(vol_path, out_dir):
  from google.protobuf import text_format
  from ffn.inference import inference_pb2
  req = inference_pb2.InferenceRequest()
  # configs/inference_training_sample2.pbtxt with the volume / checkpoint paths of this box
  text_format.Parse('''image { hdf5: "%s:raw" } image_mean: 128 image_stddev: 33 checkpoint_interval: 1800
    seed_policy: "PolicyPeaks" model_checkpoint_path: "%s" model_name: "convstack_3d.ConvStack3DFFNModel"
    model_args: "{\\"depth\\": 12, \\"fov_size\\": [33, 33, 33], \\"deltas\\": [8, 8, 8]}"
    segmentation_output_dir: "%s"
    inference_options { init_activation: 0.95 pad_value: 0.05 move_threshold: 0.9 min_boundary_dist { x: 1 y: 1 z: 1}
                        segment_threshold: 0.6 min_segment_size: 1000 }''' % (vol_path, WEIGHTS, out_dir), req)
  return req


def reference_arm(args, rank):
  """The reference's own CPU implementation of the path: TensorFlow cannot be installed offline, so this times
  the CPU restatement in oracle/ (kind 'port') with the host threads torch's conv3d can use, on a bounded
  sample of the same workload: the first FoV steps of the same segment_all on the same volume and seeds."""
  if rank != 0:
    return
  n1 = args.gpus == 1
  vol = make_volume((250, 250, 250), 0) if n1 else make_volume((512, 512, 512), 300)
  if not n1:
    vol = vol[:256, :256, :256]     # bounded sample: a corner of slab 0 (the CPU seed policy alone is minutes on 512^3)
  threads = best_cpu_threads()
  budget = args.steps if 0 < args.steps < 1000 else 24     # a bounded sample: ~1 s of CPU per FoV step on 8 cores
  steps, vox, secs, t_seed = run_cpu_sample(vol, budget, threads)
  value = steps / secs
  line = {
      'impl': 'reference', 'metric': 'fov_steps_per_sec', 'value': value, 'unit': 'FoV steps/s',
      'n_gpus': args.gpus, 'steps': steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * secs / max(steps, 1),
      'higher_is_better': True, 'scaling': 'weak' if n1 else 'strong', 'vs_baseline': None, 'dtype': 'f32',
      'data': 'synthetic',
      'config': {'workload': WORKLOAD_N1 if n1 else WORKLOAD_MULTI,
                 'note': 'CPU restatement of the reference path (TensorFlow not installable offline); '
                         'published P100 run of the reference: 65.5 FoV steps/s, 35.2 k voxels/s (README)'},
      'cpu_baseline': {'value': value, 'unit': 'FoV steps/s', 'cores': threads, 'kind': 'port',
                       'sample': 'first %d FoV steps of the same segment_all%s; CPU PolicyPeaks took %.1f s (not in value)' % (
                           steps, '' if n1 else ' on a 256^3 corner of slab 0', t_seed),
                       'voxels_per_sec': vox / secs},
      'e2e': {'value': value, 'unit': 'FoV steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
  }
  print(json.dumps(line), flush=True)


def extras_n1(engine, eng, _lib, args):
  """Secondary numbers: the single-seed latency case (configs[1]) and the batched conv stack alone."""
  from ffn_b200.synthetic import interior_seed
  out = {}
  vol1 = make_volume((256, 256, 256), 1)
  cv = eng.DeviceCanvas(engine, vol1, eng.make_options(), 128.0, 33.0)
  start = interior_seed(vol1, (128, 128, 128))
  cv.segment_at(start)
  c0 = cv.counters(); st = cv.segment_at(start); c1 = cv.counters()
  dev = c1.device_seconds - c0.device_seconds
  out['configs1_single_seed_256'] = {'steps': int(st.iters), 'steps_per_s': st.iters / dev, 'us_per_step': 1e6 * dev / st.iters,
                                     'note': 'one object = a strictly sequential chain of FoV steps: latency-bound'}
  cv.close()
  rng = np.random.RandomState(0)
  batch = 48
  seed = np.where(rng.rand(batch, *FOV) < 0.3, rng.randn(batch, *FOV) * 2, -2.9444).astype(np.float32)
  img = rng.randn(batch, *FOV).astype(np.float32)
  engine.predict(seed, img)
  engine.predict(seed, img)
  ns = engine.info()['last_kernel_ns']
  rate = batch / (ns * 1e-9)
  out['predict_batch48'] = {'patches_per_s': rate, 'kernel_us': ns / 1e3,
                            'roofline_frac': rate * flops_per_step() / 1e12 / measured_peaks()[0],
                            'note': 'ffn_predict(batch=48): the conv stack alone, four patches per round'}
  return out


def _raster_relabel(seg):
  """Labels > 0 -> rank of first occurrence in C order (the canonical relabelling of SURVEY.md 8c)."""
  flat = np.asarray(seg).ravel()
  ids, first = np.unique(flat, return_index=True)
  keep = ids > 0
  ids, first = ids[keep], first[keep]
  rank = np.empty(len(ids), dtype=np.int64)
  rank[np.argsort(first, kind='stable')] = np.arange(1, len(ids) + 1)
  out = np.zeros(flat.shape, dtype=np.int64)
  pos = flat > 0
  out[pos] = rank[np.searchsorted(ids, flat[pos])]
  return out.reshape(np.asarray(seg).shape)


def parity_fields(engine, eng, _lib):
  """How far the benchmarked arithmetic is from the fp32 reference, from the committed fixtures (tests/golden):
  logits of the reference network on recorded patches, and Canvas.segment_all on the 64x72x80 volume whose labels
  the reference's own unmodified modules produced (make_golden.py)."""
  gdir = os.path.join(REPO, 'tests', 'golden')
  out = {}
  pat = np.load(os.path.join(gdir, 'net_patches.npz'))
  got = engine.predict(pat['seed'], pat['image'])
  out['max_abs_logit_err_vs_fp32'] = float(np.abs(got - pat['logits_fp32']).max())
  g = np.load(os.path.join(gdir, 'flood_fill_64.npz'))
  cv = eng.DeviceCanvas(engine, g['volume'], eng.make_options(), 128.0, 33.0)
  origins, _, ctr = cv.segment_all(g['seeds'])
  seg = cv.read(_lib.ARRAY_SEGMENTATION)
  cv.close()
  a, b = _raster_relabel(np.maximum(seg, 0)), _raster_relabel(np.maximum(g['segmentation'], 0))
  fg = (a > 0) | (b > 0)
  out['label_iou_vs_fp32_reference'] = float(((a == b) & fg).sum()) / float(max(fg.sum(), 1))
  out['labels_bit_exact'] = bool(np.array_equal(np.maximum(seg, 0), np.maximum(g['segmentation'], 0)))
  out['segments'] = [len(origins), int(g['origins'].shape[0])]
  out['fov_steps'] = [int(ctr.inference_calls), int(json.loads(str(g['counters']))['inference-calls'])]
  out['note'] = ('golden 64x72x80 canvas, reference labels from the unmodified ffn.inference modules (fp32); '
                 '--compute x2 (split fp16 on the tensor cores) and fp32 are label-exact, see tests/test_gpu_parity.py')
  return out


DUMP_SAMPLE_VOXELS = 1 << 20


def dump_outputs(out_dir, canvas, _lib, seeds, origins, overlaps):
  """Writes what the last timed segment_all returned to its caller, as float32 / float64 .npy files (~17 MB):
  the seeds it was given, origins (id, z, y, x, iters) and overlaps (id, other_id, count) sorted by row, and the
  labels and quantized probabilities at a fixed sample of voxels (RandomState(0), flat C-order indices)."""
  os.makedirs(out_dir, exist_ok=True)
  seg = canvas.read(_lib.ARRAY_SEGMENTATION).ravel()
  qprob = canvas.read(_lib.ARRAY_QPROB).ravel()
  index = np.sort(np.random.RandomState(0).choice(seg.size, min(DUMP_SAMPLE_VOXELS, seg.size), replace=False))

  def rows(a, width):
    a = np.asarray(a, dtype=np.float64).reshape(-1, width)
    return a[np.lexsort(a.T[::-1])]
  arrays = {
      'seeds': np.asarray(seeds, dtype=np.float32).reshape(-1, 3),
      'origins': rows([(o.id, *o.start_zyx, o.iters) for o in origins], 5),
      'overlaps': rows([(v.id, v.other_id, v.count) for v in overlaps], 3),
      'sample_index': index.astype(np.float64),
      'segmentation': seg[index].astype(np.float32),
      'qprob': qprob[index].astype(np.float32),
  }
  for name, a in arrays.items():
    np.save(os.path.join(out_dir, name + '.npy'), a)


def run_n1(args, rank, local_rank):
  import torch
  from ffn_b200 import _lib
  from ffn_b200 import engine as eng
  (w, b), wdesc = load_weights()
  mode = {'fp16': _lib.COMPUTE_FP16_TC, 'fp32': _lib.COMPUTE_FP32, 'x2': _lib.COMPUTE_FP16X2_TC}[args.compute]
  engine = eng.Engine(w, b, FOV, DELTAS, device=local_rank, compute_mode=mode)
  if args.chains:
    engine.set_chains(args.chains)
  shape = (250, 250, 250)
  vol = make_volume(shape, 0)
  pinned = torch.empty(shape, dtype=torch.uint8, pin_memory=True)
  pinned.numpy()[...] = vol
  opts = eng.make_options()
  seed_cap = args.max_seeds

  # ---- warm-up: W short flood fills on a scratch canvas (allocator, instruction cache, weights in L2)
  warm = eng.DeviceCanvas(engine, pinned.numpy(), opts, 128.0, 33.0)
  wseeds, _ = device_seeds(warm)
  warm.segment_all(wseeds[:max(8 * max(args.warmup, 3), 24)])
  warm.close()

  # ---- device-resident leg: --steps timed steps, each one whole segment_all on a fresh canvas whose volume is
  # in HBM before its step starts; the wall clock sums the steps
  sampler = ClockSampler(local_rank)
  sampler.start()
  sampler.wait_ready()
  launches0 = engine.info()['launches']
  wall = t_seed = dev_seconds = 0.0
  steps = vox = 0
  spec = {}
  canvas = None
  for _ in range(args.steps):
    if canvas is not None:
      canvas.close()
    canvas = eng.DeviceCanvas(engine, pinned.numpy(), opts, 128.0, 33.0, keep_probability_maps=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    seeds, _ = device_seeds(canvas)
    t_seed += time.perf_counter() - t0
    if seed_cap:
      seeds = seeds[:seed_cap]
    origins, overlaps, ctr = canvas.segment_all(seeds, overlaps_cap=max(64 * len(seeds), 1 << 16))
    torch.cuda.synchronize()
    wall += time.perf_counter() - t0
    steps += int(ctr.inference_calls)
    vox += int(ctr.voxels_segmented)
    dev_seconds += float(ctr.device_seconds)
    for k, v in canvas.spec_stats().items():
      spec[k] = v if k == 'chains' else spec.get(k, 0) + v
  clocks = sampler.stop()
  launches = engine.info()['launches'] - launches0 + 10 * args.steps        # + the ten seed-policy kernels per step
  if args.dump_outputs:
    dump_outputs(args.dump_outputs, canvas, _lib, seeds, origins, overlaps)
  canvas.close()

  # ---- end-to-end leg: what run_inference.py does — Runner.start + Runner.run on a volume file
  if args.skip_e2e:
    e2e_seconds, e2e_steps, e2e_vox = wall, steps, vox
  else:
    from ffn.inference import runner as runner_mod
    tmp = tempfile.mkdtemp(prefix='ffn_bench_')
    vol_path = os.path.join(tmp, 'vol.npy')
    np.save(vol_path, vol)
    runner = runner_mod.Runner(device=local_rank, compute_mode=mode)
    runner.start(request_for(vol_path, os.path.join(tmp, 'out')))
    if args.chains:
      runner.executor.engine.set_chains(args.chains)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rc = runner.run((0, 0, 0), shape)
    e2e_seconds = time.perf_counter() - t0
    cnt = {k: c.value for k, c in rc.counters}
    e2e_steps = int(cnt.get('inference-calls', 0))
    e2e_vox = int(cnt.get('voxels-segmented', 0))
    runner.stop_executor()
    del rc

  value = steps / wall
  burst, sustained, src = measured_peaks()
  kernel_rate = steps / dev_seconds                                  # counted steps over the flood kernel's own time
  achieved = kernel_rate * flops_per_step() / 1e12
  executed = spec['steps_executed'] / dev_seconds * flops_per_step() / 1e12
  line = {
      'metric': 'fov_steps_per_sec', 'value': value, 'unit': 'FoV steps/s', 'n_gpus': 1,
      'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': 1e3 * wall / args.steps,
      'fov_steps': steps, 'ms_per_fov_step': 1e3 * wall / max(steps, 1),
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
      'dtype': {'fp16': 'f16', 'fp32': 'f32', 'x2': 'f16x2 (hi+lo split, ~f32)'}[args.compute], 'data': 'synthetic',
      'config': {
          'workload': WORKLOAD_N1,
          'weights': wdesc, 'accumulate': 'f32', 'timed_pass': 'each step is one whole segment_all (device PolicyPeaks + flood fill + commits) '
          'on a fresh canvas' + (' — capped at %d seeds' % seed_cap if seed_cap else ''),
          'l2': 'canvas state (image u8 + 4 seed f32 arrays + segmentation i32 + qprob u8 = 330 MB) exceeds L2; '
                'the ~25 MB activation working set of four chains is L2-resident by design',
          'published_reference_p100': {'fov_steps_per_sec': 65.5, 'voxels_per_sec': 35216},
      },
      'voxels_per_sec': vox / wall,
      'segments': int(ctr.segments), 'objects_run': int(ctr.segment_at_calls), 'seeds': int(len(seeds)),
      'seed_policy_seconds': t_seed,
      'device_only': {'value': kernel_rate, 'unit': 'FoV steps/s', 'seconds': dev_seconds,
                      'note': 'CUDA events around the flood-kernel launches only'},
      'chains': {'max': args.chains or 4, **spec},
      'gpu_launches': int(launches),
      'clocks': clocks,
      'e2e': {'value': e2e_steps / e2e_seconds, 'unit': 'FoV steps/s', 'voxels_per_sec': e2e_vox / e2e_seconds,
              'seconds': e2e_seconds,
              'h2d_bytes_per_step': int((vol.nbytes + 8 * vol.size) / max(e2e_steps, 1)),
              'd2h_bytes_per_step': int((4 * vol.size + vol.size) / max(e2e_steps, 1)),
              'path': 'Runner.run: volume file -> H2D (uint8 volume + float64 PolicyPeaks tie-break noise) -> '
                      'segment_all -> D2H (int32 labels + uint8 probabilities) -> seg-*.npz + .prob written'},
      'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': burst, 'unit': 'TFLOP/s',
                   'frac': achieved / burst, 'frac_of_sustained': achieved / sustained, 'peak_source': src,
                   'flops_per_step': flops_per_step(), 'executed_frac': executed / burst,
                   'note': 'achieved = counted FoV steps x FLOP/step / flood-kernel seconds (CUDA events around its '
                           'launches); executed_frac also counts the steps of discarded early runs',
                   'traffic': ncu_dram_traffic()},
  }
  if not args.skip_extras and args.compute == 'fp16':
    try:
      line.update(extras_n1(engine, eng, _lib, args))
    except Exception as e:  # pylint: disable=broad-except
      line['extras_error'] = repr(e)
  if not args.skip_extras:
    try:
      line['parity'] = parity_fields(engine, eng, _lib)
    except Exception as e:  # pylint: disable=broad-except
      line['parity'] = {'error': repr(e)}
  if not args.skip_extras:
    try:
      threads = best_cpu_threads()
      csteps, cvox, csecs, ct_seed = run_cpu_sample(vol, args.cpu_baseline_steps, threads)
      line['cpu_baseline'] = {'value': csteps / csecs, 'unit': 'FoV steps/s', 'cores': threads, 'kind': 'port',
                              'sample': 'first %d FoV steps of the same segment_all; CPU PolicyPeaks took %.1f s (not in value)' % (
                                  csteps, ct_seed),
                              'voxels_per_sec': cvox / csecs}
    except Exception as e:  # pylint: disable=broad-except
      line['cpu_baseline'] = {'error': repr(e)}
  print(json.dumps(line), flush=True)
  engine.close()


def run_multi(args, rank, local_rank, world):
  import torch
  import torch.distributed as dist
  from ffn_b200 import _lib, distributed as D
  from ffn_b200 import engine as eng
  (w, b), wdesc = load_weights()
  engine = eng.Engine(w, b, FOV, DELTAS, device=local_rank)
  if args.chains:
    engine.set_chains(args.chains)
  n_slabs, slab = 8, (512, 512, 512)
  if args.slab:
    slab = (args.slab,) * 3
  mine = D.slabs_of_rank(n_slabs, rank, world)
  vols = []
  for k in mine:                                           # untimed: synthetic data generation
    v = make_volume(slab, 300 + k)
    p = torch.empty(slab, dtype=torch.uint8, pin_memory=True)
    p.numpy()[...] = v
    vols.append(p)
  opts = eng.make_options()
  dev = torch.device('cuda', local_rank)

  def barrier():
    dist.barrier()
    torch.cuda.synchronize()

  # warm-up: NCCL connections (the first collective sets them up), allocator, kernels
  wt = torch.zeros(1 << 20, dtype=torch.int32, device=dev)
  dist.all_reduce(wt)
  dist.gather(wt, [torch.empty_like(wt) for _ in range(world)] if rank == 0 else None, dst=0)
  D.gather_max_ids(0, device=dev)
  torch.cuda.synchronize()
  warm = eng.DeviceCanvas(engine, vols[0].numpy()[:160, :160, :160].copy(), opts, 128.0, 33.0)
  wseeds, _ = device_seeds(warm)
  warm.segment_all(wseeds[:max(8 * max(args.warmup, 3), 24)])
  warm.close()
  # PolicyPeaks' tie-break table RandomState(42).rand(*shape) (seed.py:133-139) is a constant of the algorithm, like the
  # weights: drawn once per process for the slab shape, before the timed region (its H2D copy per slab stays inside)
  from ffn_b200.inference import seed as seed_mod
  seed_mod._tie_break_noise(tuple(slab))

  sampler = ClockSampler(local_rank)
  sampler.start()
  sampler.wait_ready()
  barrier()
  t0 = time.perf_counter()
  canvases, steps, vox, dev_s, executed, h2d = [], 0, 0, 0.0, 0, 0
  launches0 = engine.info()['launches']
  for p in vols:                                           # each slab: upload, device PolicyPeaks, segment_all
    cv = eng.DeviceCanvas(engine, p.numpy(), opts, 128.0, 33.0, keep_probability_maps=True)
    seeds, nbytes = device_seeds(cv)
    h2d += p.numpy().nbytes + nbytes
    _, _, ctr = cv.segment_all(seeds, overlaps_cap=max(64 * len(seeds), 1 << 16))
    steps += int(ctr.inference_calls)
    vox += int(ctr.voxels_segmented)
    dev_s += float(ctr.device_seconds)
    executed += cv.spec_stats()['steps_executed']
    canvases.append((cv, int(ctr.max_id)))
  torch.cuda.synchronize()
  t_work = time.perf_counter() - t0
  # ---- the one exchange step: ids made globally unique, label + probability slabs gathered on rank 0
  tm = time.perf_counter()
  labs = [D.canvas_tensor(cv, _lib.ARRAY_SEGMENTATION, slab, '<i4', dev) for cv, _ in canvases]     # alias engine memory
  probs = [D.canvas_tensor(cv, _lib.ARRAY_QPROB, slab, '|u1', dev) for cv, _ in canvases]
  gl, gp, _, total_ids = D.merge_slabs(labs, probs, [m for _, m in canvases], dst=0,
                                       add_offset=lambda i, o: canvases[i][0].add_id_offset(o))    # HBM-bound relabel kernel
  gathered_vox = 0
  if rank == 0:
    gathered_vox = int(sum(int((t > 0).sum()) for row in gl for t in row))
    assert sum(t.numel() for row in gp for t in row) == n_slabs * slab[0] * slab[1] * slab[2]
  del gp
  torch.cuda.synchronize()
  t_merge = time.perf_counter() - tm
  barrier()
  total = time.perf_counter() - t0
  clocks = sampler.stop()
  # ---- OUTSIDE the timed region, rank 0 only, on the gathered labels in its HBM (no collectives from here to `del gl`)
  merge_check, stitch_info = None, None
  if rank == 0:
    try:
      # the merge must leave every slab with its own id range: (min id, max id) intervals pairwise disjoint, all within
      # 1..total_ids — what `per-slab results with offsets` means for the reference's private id spaces (manual.md:107-127)
      spans = []
      for row in gl:
        for t in row:
          pos = t[t > 0]
          if pos.numel():
            spans.append((int(pos.min()), int(pos.max())))
      spans.sort()
      disjoint = all(spans[i][1] < spans[i + 1][0] for i in range(len(spans) - 1))
      merge_check = {'slabs_with_labels': len(spans), 'id_ranges_disjoint': bool(disjoint),
                     'max_id_seen': max([b for _, b in spans] or [0]), 'total_ids': int(total_ids),
                     'ok': bool(disjoint and max([b for _, b in spans] or [0]) <= int(total_ids))}
    except Exception as e:  # pylint: disable=broad-except
      merge_check = {'error': repr(e)}
    if args.stitch:
      # optional: reconcile ids across the touching slab faces (the reference leaves this to the user, doc/manual.md:119-127)
      try:
        from ffn_b200 import stitch
        ts = time.perf_counter()
        mapping, n_pairs = stitch.stitch_slabs(stitch.grid_of(gl, world, n_slabs))
        torch.cuda.synchronize()
        stitch_info = {'seconds': time.perf_counter() - ts, 'joined_pairs': int(n_pairs), 'ids_renamed': len(mapping)}
      except Exception as e:  # pylint: disable=broad-except
        stitch_info = {'error': repr(e)}
  del gl
  launches = engine.info()['launches'] - launches0 + 10 * len(vols)

  stats = torch.tensor([steps, vox, dev_s, t_work, t_merge, total, executed, launches, h2d], dtype=torch.float64, device=dev)
  smax = stats.clone(); dist.all_reduce(smax, op=dist.ReduceOp.MAX)
  smin = stats.clone(); dist.all_reduce(smin, op=dist.ReduceOp.MIN)
  ssum = stats.clone(); dist.all_reduce(ssum, op=dist.ReduceOp.SUM)
  if rank == 0:
    wall = float(smax[5])
    value = float(ssum[0]) / wall
    burst, sustained, src = measured_peaks()
    achieved = float(ssum[0]) / float(smax[2]) / world * flops_per_step() / 1e12     # per GPU, busiest rank's kernel time
    line = {
        'metric': 'fov_steps_per_sec', 'value': value, 'unit': 'FoV steps/s', 'n_gpus': world,
        'steps': int(ssum[0]), 'warmup': max(args.warmup, 3), 'ms_per_step': 1e3 * wall / max(float(ssum[0]), 1.0),
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic',
        'config': {'workload': WORKLOAD_MULTI, 'weights': wdesc, 'accumulate': 'f32', 'slab': list(slab),
                   'timed_pass': 'per rank: upload + device PolicyPeaks + segment_all of its slabs, then the NCCL merge; '
                                 'barrier to barrier, max over ranks; --steps is ignored',
                   'l2': 'every slab canvas (3.1 GB) exceeds L2'},
        'voxels_per_sec': float(ssum[1]) / wall,
        'merge_seconds': float(smax[4]), 'work_seconds_max': float(smax[3]), 'work_seconds_min': float(smin[3]),
        'imbalance': float(smax[3]) / max(float(smin[3]), 1e-9),
        'labelled_voxels_on_rank0_after_merge': gathered_vox, 'total_ids': int(total_ids),
        'steps_executed': int(ssum[6]),
        'merge_check': merge_check, 'stitch': stitch_info,
        'gpu_launches': int(ssum[7]),
        'clocks': clocks,
        'e2e': {'value': value, 'unit': 'FoV steps/s', 'voxels_per_sec': float(ssum[1]) / wall,
                'h2d_bytes_per_step': int(float(ssum[8]) / max(float(ssum[0]), 1.0)),
                'd2h_bytes_per_step': 0,
                'path': 'the timed region IS the end-to-end path: pinned uint8 slabs + PolicyPeaks noise H2D, '
                        'segment_all, merged labels / probabilities left in rank 0 HBM (NCCL gather, no D2H)'},
        'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': burst, 'unit': 'TFLOP/s', 'frac': achieved / burst,
                     'frac_of_sustained': achieved / sustained, 'peak_source': src, 'flops_per_step': flops_per_step(),
                     'note': 'per GPU: counted steps x FLOP/step / (busiest rank flood-kernel seconds x N)',
                     'traffic': ncu_dram_traffic()},
    }
    print(json.dumps(line), flush=True)
  for cv, _ in canvases:
    cv.close()
  engine.close()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=0,
                  help='timed steps: N = 1, whole segment_all passes (0 = one); --impl reference, FoV steps (0 = 24)')
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--compute', default='fp16', choices=['fp16', 'fp32', 'x2'])
  ap.add_argument('--chains', type=int, default=0, help='objects in flight per GPU (1..4, 0 = default 4)')
  ap.add_argument('--slab', type=int, default=0, help='N > 1: slab edge instead of 512 (tests)')
  ap.add_argument('--stitch', action='store_true', help='N > 1: after the timed region, reconcile ids across slab faces on rank 0')
  ap.add_argument('--max-seeds', type=int, default=0, help='N = 1: only the first K PolicyPeaks seeds (profiler runs)')
  ap.add_argument('--cpu-baseline-steps', type=int, default=24)
  ap.add_argument('--skip-extras', action='store_true', help='no single-seed / predict / cpu_baseline legs (profiler runs)')
  ap.add_argument('--skip-e2e', action='store_true', help='no Runner.run leg (profiler runs; the line then repeats the device-resident value)')
  ap.add_argument('--dump-outputs', metavar='DIR', help='N = 1: write what the last timed step computed to DIR/<name>.npy')
  args = ap.parse_args()
  rank = int(os.environ.get('RANK', '0'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  if args.steps < 0:
    ap.error('--steps must be >= 0')
  if args.dump_outputs and (args.impl == 'reference' or world > 1):
    ap.error('--dump-outputs is only supported by the N = 1 GPU arm')

  if args.impl == 'reference':
    reference_arm(args, rank)
    return
  args.steps = args.steps or 1

  import torch
  import torch.distributed as dist
  if not torch.cuda.is_available():
    raise SystemExit('bench.py needs a CUDA device: the engine has no CPU fallback')
  torch.cuda.set_device(local_rank)
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    run_multi(args, rank, local_rank, world)
    dist.destroy_process_group()
  else:
    run_n1(args, rank, local_rank)


if __name__ == '__main__':
  main()
