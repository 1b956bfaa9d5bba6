"""CPU-only checks of the host package: wire formats, file layout, counters, seed policies, the
C-ABI surface, and the 'no CPU fallback' guarantees."""

import json
import os
import re

import numpy as np
import pytest
from google.protobuf import text_format

from ffn.inference import inference_pb2, inference_utils, movement, seed, storage
from ffn.utils import bounding_box_pb2
from ffn_b200 import _lib, distributed
from oracle import flood_fill as ff

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SAMPLE_REQUEST = """
image { hdf5: "third_party/neuroproof_examples/training_sample2/grayscale_maps.h5:raw" }
image_mean: 128
image_stddev: 33
checkpoint_interval: 1800
seed_policy: "PolicyPeaks"
model_checkpoint_path: "models/fib25/model.ckpt-27465036"
model_name: "convstack_3d.ConvStack3DFFNModel"
model_args: "{\\"depth\\": 12, \\"fov_size\\": [33, 33, 33], \\"deltas\\": [8, 8, 8]}"
segmentation_output_dir: "results/fib25/training2"
inference_options {
  init_activation: 0.95
  pad_value: 0.05
  move_threshold: 0.9
  min_boundary_dist { x: 1 y: 1 z: 1}
  segment_threshold: 0.6
  min_segment_size: 1000
}
"""


def test_request_text_format_and_wire_roundtrip():
  req = inference_pb2.InferenceRequest()
  text_format.Parse(SAMPLE_REQUEST, req)
  assert req.model_name == 'convstack_3d.ConvStack3DFFNModel'
  assert json.loads(req.model_args)['depth'] == 12
  assert req.batch_size == 1 and req.concurrent_requests == 1          # proto2 defaults
  assert req.inference_options.disco_seed_threshold == 0.0
  assert req.image.WhichOneof('volume_path') == 'hdf5'
  assert req.alignment_options.type == inference_pb2.AlignmentOptions.NO_ALIGNMENT
  again = inference_pb2.InferenceRequest()
  again.ParseFromString(req.SerializeToString())
  assert again == req
  box = bounding_box_pb2.BoundingBox()
  text_format.Parse('start { x:0 y:0 z:0 } size { x:250 y:250 z:250 }', box)
  assert (box.size.x, box.size.y, box.size.z) == (250, 250, 250)


def test_field_numbers_match_reference_schema():
  """Spot-check of tags that matter for reading files written by the reference."""
  d = inference_pb2.InferenceRequest.DESCRIPTOR.fields_by_name
  assert {n: d[n].number for n in ('image', 'image_mean', 'model_name', 'model_args', 'batch_size',
                                   'inference_options', 'segmentation_output_dir', 'seed_policy',
                                   'init_segmentation', 'seed_masks')} == {
      'image': 24, 'image_mean': 2, 'model_name': 11, 'model_args': 12, 'batch_size': 27,
      'inference_options': 14, 'segmentation_output_dir': 15, 'seed_policy': 17, 'init_segmentation': 25,
      'seed_masks': 30}
  o = inference_pb2.InferenceOptions.DESCRIPTOR.fields_by_name
  assert [o[n].number for n in ('init_activation', 'pad_value', 'move_threshold', 'disco_seed_threshold',
                                'min_boundary_dist', 'segment_threshold', 'min_segment_size')] == [1, 2, 3, 5, 6, 7, 8]


def test_storage_paths_and_quantisation(tmp_path, golden_dir):
  corner = (10, 20, 30)   # z, y, x
  assert storage.segmentation_path('/o', corner) == '/o/30/20/seg-30_20_10.npz'
  assert storage.object_prob_path('/o', corner) == '/o/30/20/seg-30_20_10.prob'
  assert storage.checkpoint_path('/o', corner) == '/o/30/20/seg-30_20_10.cpoint'
  assert storage.get_corner_from_path('/o/30/20/seg-30_20_10.npz') == corner
  g = np.load(os.path.join(golden_dir, 'qprob.npz'))
  np.testing.assert_array_equal(storage.quantize_probability(g['prob']), g['q'])
  dq = storage.dequantize_probability(np.array([0, 1, 128, 255], np.uint8))
  assert np.isnan(dq[0]) and abs(dq[2] - 127.5 / 255) < 1e-6
  labels = np.zeros((4, 4, 4), np.int32)
  labels[1:3] = 300
  origins = {300: storage.OriginInfo((1, 2, 3), 7, 0.5)}
  path = str(tmp_path / '3' / '2' / 'seg-3_2_1.npz')
  storage.save_subvolume(labels, origins, path, counters='{}')
  seg, org = storage.load_segmentation(str(tmp_path), (1, 2, 3))
  assert seg.dtype == np.uint64 and seg.max() == 300 and org[300].iters == 7
  with np.load(path, allow_pickle=True) as z:
    assert z['segmentation'].dtype == np.uint16


def test_savez_deflate_is_a_plain_npz(tmp_path):
  """The seg-*.npz / .prob writer (deflate pieces compressed on a thread pool, stitched into one stream per
  member): np.load and zipfile read it back, large members included, object members pickled as numpy does."""
  import io
  import zipfile
  rng = np.random.RandomState(3)
  big = (rng.rand(96, 128, 130) < 0.2).astype(np.uint8) * rng.randint(1, 200, (96, 128, 130)).astype(np.uint8)
  assert big.nbytes > (1 << 20)
  old_chunk = storage._DEFLATE_CHUNK
  storage._DEFLATE_CHUNK = 1 << 18                      # several pieces per member
  try:
    bio = io.BytesIO()
    storage.savez_deflate(bio, segmentation=big, origins={7: (1, 2, 3)}, request=b'\x00\x01', counters='{}',
                          overlaps=np.zeros((0, 3), np.int64), fortran=np.asfortranarray(rng.rand(40, 50, 60)),
                          empty=np.zeros((0,), np.float32))
  finally:
    storage._DEFLATE_CHUNK = old_chunk
  bio.seek(0)
  assert zipfile.ZipFile(bio).testzip() is None         # CRCs and sizes of every member
  bio.seek(0)
  with np.load(bio, allow_pickle=True) as z:
    np.testing.assert_array_equal(z['segmentation'], big)
    assert z['origins'].item() == {7: (1, 2, 3)} and z['request'].item() == b'\x00\x01' and z['counters'].item() == '{}'
    assert z['overlaps'].shape == (0, 3) and z['empty'].shape == (0,)
    assert z['fortran'].shape == (40, 50, 60)
  assert len(bio.getvalue()) < big.nbytes // 2 + 40 * 50 * 60 * 8 + 4096     # the label member really is deflated


def test_counters_and_timer():
  c = inference_utils.Counters()
  sub = c.get_sub_counters()
  with inference_utils.timer_counter(sub, 'inference'):
    pass
  sub['voxels-segmented'].IncrementBy(5)
  assert sub['inference-calls'].value == 1 and c['voxels-segmented'].value == 5
  state = sub.dumps()
  other = inference_utils.Counters()
  other.loads(state)
  assert other['voxels-segmented'].value == 5


class _FakeCanvas:
  def __init__(self, shape, image=None):
    self.shape = shape
    self.margin = np.array([16, 16, 16])
    self.image = image if image is not None else np.zeros(shape, np.float32)
    self.segmentation = np.zeros(shape, np.int32)
    self.restrictor = None
    self.voxel_size_zyx = (1, 1, 1)


def test_grid_seed_policy_matches_oracle_and_border_filter():
  cv = _FakeCanvas((48, 56, 64))
  pol = seed.PolicyGrid3d(cv)
  got = np.array(list(pol))
  want = ff.grid_seeds(cv.shape)
  keep = np.all((want - 16 >= 0) & (want + 16 < np.array(cv.shape)), axis=1)
  np.testing.assert_array_equal(got, want[keep])
  pol2 = seed.PolicyGrid3d(cv)
  first = next(pol2)
  assert pol2.remaining().shape[0] == got.shape[0] - 1 and first == tuple(got[0])
  coords, idx = pol2.get_state(previous=True)
  assert idx == 0 and coords.shape == got.shape


def test_policy_peaks_runs_and_is_sorted():
  from ffn_b200.synthetic import voronoi_phantom
  vol = voronoi_phantom((48, 64, 64), seed=2, cell_volume=20000.0)
  cv = _FakeCanvas(vol.shape, (vol.astype(np.float32) - 128) / 33)
  coords = seed.PolicyPeaks(cv).remaining()
  assert coords.shape[0] > 3
  assert [tuple(c) for c in coords] == sorted(tuple(c) for c in coords)


def test_host_scored_moves_match_oracle(golden_dir):
  g = np.load(os.path.join(golden_dir, 'moves.npz'))
  for i in range(0, int(g['n']), 5):
    got = sorted(movement.get_scored_move_offsets(g['deltas_%d' % i], g['logits_%d' % i], float(g['threshold'])),
                 reverse=True)
    arr = np.asarray([(float(s),) + r for s, r in got], dtype=np.float64).reshape(-1, 4)
    np.testing.assert_array_equal(arr, g['moves_%d' % i])


def test_c_abi_exports_every_declared_symbol():
  header = open(os.path.join(REPO, 'include', 'ffn_b200.h')).read()
  declared = set(re.findall(r'\b(ffn_[a-z0-9_]+)\s*\(', header))
  assert declared, 'no declarations found'
  lib = _lib.load()
  missing = [n for n in sorted(declared) if not hasattr(lib, n)]
  assert not missing, missing
  assert declared == set(_lib.EXPORTS)


def test_no_cpu_fallback_without_gpu():
  import torch
  if torch.cuda.is_available():
    pytest.skip('GPU present')
  from ffn_b200 import engine as eng, tf_checkpoint
  w, b = tf_checkpoint.load_convstack_npz(os.path.join(REPO, 'tests', 'golden', 'fib25_convstack.npz'))
  with pytest.raises(RuntimeError):
    eng.Engine(w, b)


def test_canvas_rejects_foreign_executor_clients():
  from ffn.inference import executor, inference
  from ffn.training import model as ffn_model
  info = ffn_model.ModelInfo([8, 8, 8], [33, 33, 33], [33, 33, 33], [33, 33, 33])

  class Other(executor.ExecutorClient):
    pass
  with pytest.raises(TypeError):
    inference.Canvas(info, Other(inference_utils.Counters(), executor.ExecutorInterface()),
                     np.zeros((40, 40, 40), np.float32), inference_pb2.InferenceOptions())


def test_product_never_imports_oracle():
  bad = []
  for root in ('ffn_b200', 'ffn'):
    for d, _, files in os.walk(os.path.join(REPO, root)):
      for f in files:
        if f.endswith('.py'):
          src = open(os.path.join(d, f)).read()
          if re.search(r'^\s*(from|import)\s+oracle\b', src, re.M):
            bad.append(os.path.join(d, f))
  assert not bad, bad


def test_slab_partition_and_offsets():
  boxes = distributed.slab_boxes((1024, 1024, 1024), 8)
  assert len(boxes) == 8 and all(b[1] == (512, 512, 512) for b in boxes)
  cover = np.zeros((4, 4, 4), int)
  for (lo, sz) in distributed.slab_boxes((4, 4, 4), 8):
    cover[lo[0]:lo[0] + sz[0], lo[1]:lo[1] + sz[1], lo[2]:lo[2] + sz[2]] += 1
  assert (cover == 1).all()
  assert distributed.exclusive_offsets([3, 0, 5]) == [0, 3, 3]
  assert distributed.slabs_of_rank(8, 1, 2) == [4, 5, 6, 7]


def test_resegmentation_helpers(tmp_path):
  """get_starting_location / get_target_path (resegmentation.py:37-80)."""
  from ffn.inference import inference_pb2, resegmentation
  req = inference_pb2.ResegmentationRequest()
  req.output_directory = str(tmp_path / 'out')
  req.exclusion_radius.x, req.exclusion_radius.y, req.exclusion_radius.z = 2, 1, 1
  pt = req.points.add()
  pt.id_a, pt.id_b = 7, 11
  pt.point.x, pt.point.y, pt.point.z = 30, 20, 10
  d = np.zeros((8, 9, 10))
  d[4, 5, 6], d[4, 5, 8], d[4, 5, 9], d[1, 1, 1] = 5.0, 4.0, 3.5, 1.0
  assert resegmentation.get_starting_location(d, req.exclusion_radius) == (4, 5, 6)
  assert d[4, 5, 6] == 0 and d[4, 5, 8] == 0 and d[4, 5, 9] == 3.5      # x radius 2 cleared, 3 kept
  assert resegmentation.get_starting_location(d, req.exclusion_radius) == (4, 5, 9)
  path = resegmentation.get_target_path(req, 0)
  assert path == os.path.join(req.output_directory, '7-11_at_30_20_10.npz')
  open(path, 'wb').close()
  assert resegmentation.get_target_path(req, 0) is None                  # finished points are skipped
  req.subdir_digits = 3
  sharded = resegmentation.get_target_path(req, 0)
  assert os.path.basename(os.path.dirname(sharded)) == __import__('hashlib').md5(b'711').hexdigest()[:3]


def test_resegmentation_process_point_host_logic(tmp_path):
  """process_point (resegmentation.py:114-293) with a stand-in canvas: segment clearing, EDT seeding with
  margins and retries, recovery test, result file keys (ragged histories as object arrays)."""
  from ffn.inference import align, inference_pb2, inference_utils, resegmentation
  from ffn_b200 import synthetic
  _, cells = synthetic.voronoi_phantom((96, 96, 96), seed=7, cell_volume=45000.0, return_cells=True)
  z, y, x, a, b = 40, 40, 49, 14, 18
  made = []

  class FakeCanvas:
    def __init__(self, corner, size):
      self.corner_zyx = np.asarray(corner)
      sel = tuple(slice(c, c + s) for c, s in zip(corner, size))
      self.segmentation = cells[sel].astype(np.int32).copy()
      self.seg_prob = np.full(size, 255, np.uint8)
      self.seed = np.full(size, np.nan, np.float32)
      self.margin = np.array([16, 16, 16])
      self.restrictor = None
      self.counters = inference_utils.Counters()
      self.history, self.history_deleted, self.calls = [], [], []

    def local_id(self, i):
      return i

    def log_info(self, *args, **kwargs):
      pass

    def _deregister_client(self):
      pass

    def segment_at(self, pos):
      assert self.segmentation[pos] == 0                      # the segment in question was cleared first
      self.calls.append(pos)
      self.seed[...] = np.nan
      self.seed[tuple(slice(p - 10, p + 11) for p in pos)] = 3.0
      n = 3 + len(self.calls)
      self.history, self.history_deleted = [pos] * n, [0] * n

  class FakeRunner:
    counters = inference_utils.Counters()
    init_seg_volume = cells[np.newaxis]

    def make_canvas(self, corner, size, **kwargs):
      assert kwargs == {'keep_history': True}
      made.append(FakeCanvas(corner, size))
      return made[-1], align.Alignment(corner, size)

  req = inference_pb2.ResegmentationRequest()
  req.radius.x = req.radius.y = req.radius.z = 40
  req.output_directory = str(tmp_path)
  req.max_retry_iters = 2
  req.exclusion_radius.x = req.exclusion_radius.y = req.exclusion_radius.z = 4
  req.analysis_radius.x = req.analysis_radius.y = req.analysis_radius.z = 24
  req.inference.inference_options.segment_threshold = 0.6
  req.inference.inference_options.min_segment_size = 100000     # never recovered: every retry is used
  for ids in ((a, b), (a,), (a, 999)):
    pt = req.points.add()
    pt.id_a = ids[0]
    if len(ids) > 1:
      pt.id_b = ids[1]
    pt.point.x, pt.point.y, pt.point.z = x, y, z
  resegmentation.process(req, FakeRunner())

  pair = np.load(tmp_path / ('%d-%d_at_%d_%d_%d.npz' % (a, b, x, y, z)), allow_pickle=True)
  assert pair['probs'].shape == (2, 81, 81, 81) and pair['raw_probs'].dtype == np.uint8
  assert [len(h) for h in pair['histories']] == [5, 7] and [len(d) for d in pair['deletes']] == [5, 7]
  assert [len(s) for s in pair['start_points']] == [2, 2]
  assert len(made[0].calls) == 4 and tuple(pair['corner_zyx']) == (0, 0, 9)
  # context is kept: other labels untouched, the two segments and their probabilities cleared
  sub = cells[0:81, 0:81, 9:90]
  keep = (sub != a) & (sub != b)
  np.testing.assert_array_equal(made[0].segmentation[keep], sub[keep])
  assert not made[0].segmentation[~keep].any() and not made[0].seg_prob[~keep].any()
  assert inference_pb2.ResegmentationRequest.FromString(pair['request'].tobytes()).max_retry_iters == 2
  end = np.load(tmp_path / ('%d-0_at_%d_%d_%d.npz' % (a, x, y, z)), allow_pickle=True)
  assert end['probs'].shape == (1, 81, 81, 81) and not made[1].segmentation.any()     # endpoint: everything cleared
  assert not os.path.exists(tmp_path / ('%d-999_at_%d_%d_%d.npz' % (a, x, y, z)))      # id not present: skipped


def test_shift_mask_restriction_matches_reference(golden_dir):
  """MovementRestrictor with a shift mask: the per-voxel movement mask handed to the device equals the
  reference's own is_valid_pos at every position (fixture: tests/golden/make_golden_restrictor.py;
  movement.py:247-336), for scales 1 / 2 / 4 and boxes that start outside the volume."""
  from ffn.inference import movement
  from ffn.utils import bounding_box
  g = np.load(os.path.join(golden_dir, 'restrictor_shift.npz'))
  informative = 0
  for i in range(int(g['n'])):
    fov = bounding_box.BoundingBox(start=g['fov_start_%d' % i], size=g['fov_size_%d' % i])
    r = movement.MovementRestrictor(mask=g['mask_%d' % i], shift_mask=g['shift_%d' % i], shift_mask_fov=fov,
                                    shift_mask_threshold=int(g['threshold_%d' % i]),
                                    shift_mask_scale=int(g['scale_%d' % i]))
    valid = g['valid_%d' % i]
    np.testing.assert_array_equal(r.movement_mask(valid.shape), ~valid)
    rng = np.random.RandomState(i)
    for _ in range(50):
      pos = tuple(int(rng.randint(0, d)) for d in valid.shape)
      assert r.is_valid_pos(pos) == bool(valid[pos])
    informative += 0.05 < valid.mean() < 0.95
  assert informative >= 6
  # without a shift mask the movement mask is the position mask itself
  plain = movement.MovementRestrictor(mask=g['mask_0'])
  np.testing.assert_array_equal(plain.movement_mask(g['mask_0'].shape), g['mask_0'])
  assert movement.MovementRestrictor().movement_mask((3, 4, 5)) is None


def test_runner_make_restrictor_with_shift_mask(tmp_path):
  """Runner.make_restrictor (runner.py:218-305) crops the shift field of the subvolume at
  `shift_mask_scale` resolution and the resulting movement mask blocks exactly the positions whose
  default FoV box (the model's input size) contains a large shift."""
  from ffn.inference import align, inference_pb2, inference_utils, runner as runner_mod
  from ffn.training import model as ffn_model
  vol_shape = (40, 64, 72)
  scale = 2
  shift = np.zeros((2, vol_shape[0], vol_shape[1] // scale, vol_shape[2] // scale), dtype=np.float32)
  shift[1, 20, 12, 20] = 9.0                                  # one distorted patch: section 20, y ~ 24, x ~ 40
  np.save(tmp_path / 'shift.npy', shift)
  r = runner_mod.Runner()
  r.request = inference_pb2.InferenceRequest()
  r.request.shift_mask.hdf5 = '%s:shift' % (tmp_path / 'shift.npy')
  r.request.shift_mask_scale = scale
  r.request.shift_mask_threshold = 4
  from ffn.inference import storage
  r._shift_mask_volume = storage.decorated_volume(r.request.shift_mask)
  r._model_info = ffn_model.ModelInfo(np.array([4, 4, 2]), np.array([17, 17, 9]), np.array([17, 17, 9]),
                                      np.array([17, 17, 9]))
  r.counters = inference_utils.Counters()
  corner, size = np.array([8, 10, 14]), np.array([24, 40, 44])
  restrictor = r.make_restrictor(corner, size, None, align.Alignment(corner, size))
  assert restrictor.shift_mask.shape == (24, 20, 22) and restrictor.shift_mask.sum() == 1
  mm = restrictor.movement_mask(tuple(size))
  # blocked <=> the (9, 17, 17) box around the position covers section 20 and shift-mask pixel (12, 20)
  z, y, x = np.indices(tuple(size))
  gz, gy, gx = z + corner[0], y + corner[1], x + corner[2]
  want = ((np.abs(gz - 20) <= 4) & ((np.maximum(y - 8, 0)) // scale + corner[1] // scale <= 12) &
          ((y + 8) // scale + corner[1] // scale >= 12) &
          ((np.maximum(x - 8, 0)) // scale + corner[2] // scale <= 20) & ((x + 8) // scale + corner[2] // scale >= 20))
  np.testing.assert_array_equal(mm, want)
  assert 0 < mm.sum() < mm.size


def test_bench_reference_arm_contract():
  """`bench.py --impl reference` (the CPU restatement timed on the host cores) prints ONE JSON line with the
  contract's keys; the GPU arm's extra objects are checked on the GPU box by the driver."""
  import json
  import subprocess
  import sys
  repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  res = subprocess.run([sys.executable, os.path.join(repo, 'bench.py'), '--impl', 'reference', '--steps', '1',
                        '--warmup', '1'], capture_output=True, text=True, timeout=600, cwd=repo)
  assert res.returncode == 0, res.stderr[-2000:]
  lines = [ln for ln in res.stdout.splitlines() if ln.startswith('{')]
  assert len(lines) == 1
  d = json.loads(lines[0])
  assert d['impl'] == 'reference' and d['metric'] == 'fov_steps_per_sec' and d['higher_is_better'] is True
  assert d['n_gpus'] == 1 and d['steps'] == 1 and d['warmup'] == 1 and d['value'] > 0
  assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
  assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
  assert 'workload' in d['config'] and d['data'] == 'synthetic' and d['vs_baseline'] is None


def test_bench_traffic_comes_from_committed_ncu_capture():
  import bench
  t = bench.ncu_dram_traffic()
  assert t is not None and t['steps_per_launch'] >= 16
  # at most about the compulsory 431 KB/step (u8 image); far less when the touched part of the canvas stays in the
  # 126 MB L2 between steps (250^3 bench canvas: 55 KB/step)
  assert 1e4 < t['bytes_per_step'] < 431244 * 2


def test_load_segmentation_reads_the_reference_shipped_result(tmp_path, golden_dir):
  """results/fib25/sample-training2.npz of the reference checkout: a Python-2 pickle of OriginInfo under the
  original module path — storage.load_segmentation reads it (latin1 + module mapping).  The file is rebuilt from
  sample_training2_ref.npz (tests/golden/make_golden_reference_files.py): its `origins` member verbatim, and its
  labels at a seeded sample of voxels and at every origin's start (0 elsewhere)."""
  import io
  import zipfile
  from ffn.inference import storage
  r = np.load(os.path.join(golden_dir, 'sample_training2_ref.npz'))
  labels = np.zeros(tuple(r['shape']), dtype=np.dtype(str(r['dtype'])))
  labels.ravel()[r['sample_index']] = r['sample_labels']
  buf = io.BytesIO()
  np.save(buf, labels)
  d = tmp_path / '0' / '0'
  d.mkdir(parents=True)
  with zipfile.ZipFile(str(d / 'seg-0_0_0.npz'), 'w', zipfile.ZIP_DEFLATED) as z:
    z.writestr('segmentation.npy', buf.getvalue())
    z.writestr('origins.npy', r['origins_npy'].tobytes())
  seg, origins = storage.load_segmentation(str(tmp_path), (0, 0, 0))
  assert seg.shape == (250, 250, 250) and seg.dtype == np.uint64
  np.testing.assert_array_equal(seg.ravel()[r['sample_index']], r['sample_labels'])
  assert len(origins) == 254 and origins[1].iters == 1884
  assert all(seg[tuple(int(v) for v in o.start_zyx)] == sid for sid, o in origins.items())   # every origin carries its own id


def test_stitch_slabs_recovers_objects_cut_by_slab_borders():
  """ffn_b200.stitch: a volume of known objects is cut into 2x2x2 touching slabs, every slab labelled in a private
  id space (connected pieces of the objects, ids from 1), ids made globally unique by the slab offsets of
  distributed.exclusive_offsets — then the union-find reconciliation over the shared faces must give back exactly
  the partition of the uncut volume (doc/manual.md:119-127 describes this step and leaves it unimplemented)."""
  import torch
  from scipy import ndimage
  from ffn_b200 import distributed as D, stitch
  from ffn_b200.synthetic import voronoi_phantom
  _, cells = voronoi_phantom((64, 72, 80), seed=5, return_cells=True, cell_volume=9000.0)
  # ground truth = connected components of the cells (membranes are 0)
  truth = np.zeros(cells.shape, dtype=np.int64)
  nxt = 0
  for cid in np.unique(cells[cells > 0]):
    comp, n = ndimage.label(cells == cid)
    truth[comp > 0] = comp[comp > 0] + nxt
    nxt += n
  boxes = D.slab_boxes(cells.shape, 8)
  grid = D.slab_grid(8)
  local, max_ids = [], []
  for lo, size in boxes:
    sub = cells[lo[0]:lo[0] + size[0], lo[1]:lo[1] + size[1], lo[2]:lo[2] + size[2]]
    lab = np.zeros(sub.shape, dtype=np.int32)
    nxt_local = 0
    for cid in np.unique(sub[sub > 0]):
      comp, n = ndimage.label(sub == cid)
      lab[comp > 0] = comp[comp > 0] + nxt_local
      nxt_local += n
    local.append(lab)
    max_ids.append(nxt_local)
  offsets = D.exclusive_offsets(max_ids)
  slabs = {}
  for k, (lab, off) in enumerate(zip(local, offsets)):
    lab = lab.copy()
    lab[lab > 0] += off
    iz, rem = divmod(k, grid[1] * grid[2])
    iy, ix = divmod(rem, grid[2])
    slabs[(iz, iy, ix)] = torch.from_numpy(lab)
  before = sum(max_ids)
  mapping, n_pairs = stitch.stitch_slabs(slabs, min_contact=4, min_fraction=0.5)
  assert n_pairs > 0 and len(mapping) > 0
  # reassemble
  out = np.zeros(cells.shape, dtype=np.int64)
  for k, (lo, size) in enumerate(boxes):
    iz, rem = divmod(k, grid[1] * grid[2])
    iy, ix = divmod(rem, grid[2])
    out[lo[0]:lo[0] + size[0], lo[1]:lo[1] + size[1], lo[2]:lo[2] + size[2]] = slabs[(iz, iy, ix)].numpy()
  assert len(np.unique(out[out > 0])) < before
  # partition agreement: every stitched object lies inside ONE true object, and nearly every true object is ONE
  # stitched object (pieces touching the cut through fewer than min_contact voxels legitimately stay separate)
  fg = truth > 0
  assert np.array_equal(out > 0, fg)
  pair = np.unique(np.stack([out[fg], truth[fg]], axis=1), axis=0)
  assert len(np.unique(pair[:, 0])) == len(pair), 'a stitched object spans two true objects (false merge)'
  n_true, n_out = len(np.unique(pair[:, 1])), len(pair)
  assert n_true <= n_out <= n_true + max(2, n_true // 8), (n_true, n_out)
  # voxels in true objects that ended up as exactly one stitched object
  pieces = np.bincount(np.unique(pair[:, 1], return_inverse=True)[1])
  whole = np.unique(pair[:, 1])[pieces == 1]
  assert np.isin(truth[fg], whole).mean() >= 0.85, float(np.isin(truth[fg], whole).mean())
  # union-find basics: representative = smallest id, idempotent
  uf = stitch.UnionFind()
  uf.union(7, 3); uf.union(9, 7); uf.union(5, 5)
  assert uf.mapping() == {7: 3, 9: 3}
  m2, n2 = stitch.stitch_slabs(slabs, min_contact=4, min_fraction=0.5)
  assert all(uf2 == m2[k] for k, uf2 in m2.items()) and not m2   # second pass: nothing left to join


def test_resegmentation_process_point_equals_reference_golden_with_oracle_canvas(tmp_path, golden_dir):
  """The host side of resegmentation.process_point against the REFERENCE's own process_point (fixture reseg_64.npz,
  tests/golden/make_golden_reseg.py): with the oracle canvas standing in for the device canvas (same fp32 network as
  the fixture), seeding, attempts, histories, history_deleted, start points and the saved probability arrays must be
  the reference's, bit for bit.  (-m gpu has the same comparison through Runner and the device canvas.)"""
  from ffn.inference import align, inference_pb2, inference_utils, resegmentation
  from ffn_b200 import tf_checkpoint
  from oracle import flood_fill as ff
  from oracle.network import ConvStackOracle
  r = np.load(os.path.join(golden_dir, 'reseg_64.npz'))
  g = np.load(os.path.join(golden_dir, 'flood_fill_64.npz'))
  w, b = tf_checkpoint.load_convstack_npz(os.path.join(golden_dir, 'fib25_convstack.npz'))
  net = ConvStackOracle(w, b)
  seg_all = np.maximum(g['segmentation'], 0).astype(np.uint64)

  class OracleCanvas:
    def __init__(self, corner, size):
      self.corner_zyx = np.asarray(corner)
      sel = tuple(slice(int(c), int(c + s)) for c, s in zip(corner, size))
      image = (g['volume'][sel].astype(np.float32) - np.float32(128.0)) / np.float32(33.0)
      self._cv = ff.Canvas(net, image, (33, 33, 33), (8, 8, 8), ff.Options())
      sub = seg_all[sel]
      ids = np.unique(sub[sub > 0])                              # make_contiguous: ascending ids -> 1..n
      self._g2l = {int(v): i + 1 for i, v in enumerate(ids)}
      local = np.zeros(sub.shape, np.int32)
      for gid, lid in self._g2l.items():
        local[sub == gid] = lid
      self._cv.segmentation[...] = local
      self.segmentation = self._cv.segmentation
      self.seg_prob = np.where(local > 0, 255, 0).astype(np.uint8)
      self.margin = np.array([16, 16, 16])
      self.restrictor = None
      self.counters = inference_utils.Counters()

    seed = property(lambda self: self._cv.seed)
    history = property(lambda self: self._cv.history)
    history_deleted = property(lambda self: self._cv.history_deleted)

    def local_id(self, gid):
      return self._g2l.get(int(gid), gid)

    def log_info(self, *args, **kwargs):
      pass

    def _deregister_client(self):
      pass

    def segment_at(self, pos):
      return self._cv.segment_at(tuple(int(p) for p in pos))

  class OracleRunner:
    counters = inference_utils.Counters()
    init_seg_volume = seg_all[np.newaxis]

    def make_canvas(self, corner, size, **kwargs):
      assert kwargs == {'keep_history': True}
      return OracleCanvas(corner, size), align.Alignment(corner, size)

  pz, py, px = (int(v) for v in r['point_zyx'])
  id_a, id_b = int(r['id_a']), int(r['id_b'])
  req = inference_pb2.ResegmentationRequest()
  req.radius.z, req.radius.y, req.radius.x = (int(v) for v in r['radius_zyx'])
  req.output_directory = str(tmp_path)
  req.max_retry_iters = int(r['max_retry_iters'])
  req.exclusion_radius.x = req.exclusion_radius.y = req.exclusion_radius.z = int(r['exclusion_radius'])
  req.init_exclusion_radius.x = req.init_exclusion_radius.y = req.init_exclusion_radius.z = int(r['init_exclusion_radius'])
  req.analysis_radius.z, req.analysis_radius.y, req.analysis_radius.x = (int(v) for v in r['analysis_radius_zyx'])
  req.segment_recovery_fraction = float(r['segment_recovery_fraction'])
  req.inference.inference_options.segment_threshold = 0.6
  req.inference.inference_options.min_segment_size = 1000
  for ids in ((id_a, id_b), (id_a,)):
    pt = req.points.add()
    pt.id_a = ids[0]
    if len(ids) > 1:
      pt.id_b = ids[1]
    pt.point.x, pt.point.y, pt.point.z = px, py, pz
  resegmentation.process(req, OracleRunner())
  for tag, ids in (('pair', (id_a, id_b)), ('endpoint', (id_a,))):
    out = np.load(tmp_path / ('%d-%d_at_%d_%d_%d.npz' % (ids[0], ids[1] if len(ids) > 1 else 0, px, py, pz)), allow_pickle=True)
    np.testing.assert_array_equal(np.asarray(out['corner_zyx']), r[tag + '_corner_zyx'])
    n_obj = int(r[tag + '_n_objects'])
    assert len(out['histories']) == n_obj
    for k in range(2):
      np.testing.assert_array_equal(np.asarray(out['start_points'][k], dtype=np.int64).reshape(-1, 3), r['%s_starts_%d' % (tag, k)])
    for k in range(n_obj):
      np.testing.assert_array_equal(np.asarray(out['histories'][k], dtype=np.int32).reshape(-1, 3), r['%s_history_%d' % (tag, k)])
      np.testing.assert_array_equal(np.asarray(out['deletes'][k], dtype=np.int64), r['%s_deletes_%d' % (tag, k)])
    np.testing.assert_array_equal(out['raw_probs'], r[tag + '_raw_probs'])
    np.testing.assert_array_equal(out['probs'], r[tag + '_probs'])


def test_subvolume_files_interoperate_with_the_reference_writer_and_reader(tmp_path, golden_dir):
  """seg-*.npz both ways (fixtures from tests/golden/make_golden_storage.py): files written by the reference's own
  `storage.save_subvolume` (ids <= 255 -> uint8, > 255 -> uint16) are read by this package's `load_segmentation` /
  `load_origins`; and this package's writer produces, key by key, the arrays the reference wrote — the same file,
  read by the reference's own `load_segmentation`, gave `*_read_by_reference` when the fixture was made."""
  import shutil
  from ffn.inference import storage
  r = np.load(os.path.join(golden_dir, 'storage_roundtrip.npz'))
  for tag, dtype in (('u8', np.uint8), ('u16', np.uint16)):
    labels = r[tag + '_labels']
    ids = r[tag + '_origin_ids'].tolist()
    origins = {sid: storage.OriginInfo(tuple(int(v) for v in r[tag + '_origin_start'][k]), int(r[tag + '_origin_iters'][k]),
                                       float(r[tag + '_origin_wall'][k])) for k, sid in enumerate(ids)}
    # the reference's file -> our reader
    ref_dir = tmp_path / ('ref_' + tag)
    path = storage.segmentation_path(str(ref_dir), (0, 0, 0))
    os.makedirs(os.path.dirname(path))
    shutil.copy(os.path.join(golden_dir, 'ref_subvolume_%s.npz' % tag), path)
    seg, got = storage.load_segmentation(str(ref_dir), (0, 0, 0), split_cc=False)
    assert seg.dtype == np.uint64
    np.testing.assert_array_equal(seg, labels.astype(np.uint64))
    np.testing.assert_array_equal(seg, r[tag + '_read_by_reference'])
    assert {k: (tuple(v.start_zyx), v.iters, v.walltime_sec) for k, v in got.items()} == {
        k: (tuple(v.start_zyx), v.iters, v.walltime_sec) for k, v in origins.items()}
    assert storage.load_origins(str(ref_dir), (0, 0, 0)).keys() == origins.keys()
    # our writer == the reference's writer, array by array
    ours = tmp_path / ('ours_' + tag) / 'seg.npz'
    overlaps = {sid: np.array([[1, 2], [k, 3 * k]], dtype=np.int64) for k, sid in enumerate(ids)}
    storage.save_subvolume(labels.copy(), origins, str(ours), request=b'request-bytes', counters='{"a": 1}', overlaps=overlaps)
    a = np.load(ours, allow_pickle=True)
    b = np.load(os.path.join(golden_dir, 'ref_subvolume_%s.npz' % tag), allow_pickle=True)
    assert sorted(a.files) == sorted(b.files)
    assert a['segmentation'].dtype == dtype == b['segmentation'].dtype
    np.testing.assert_array_equal(a['segmentation'], b['segmentation'])
    assert a['request'].tobytes() == b['request'].tobytes() and str(a['counters']) == str(b['counters'])
    oa, ob = a['origins'].item(), b['origins'].item()
    assert {k: tuple(v) for k, v in oa.items()} == {k: tuple(v) for k, v in ob.items()}
    va, vb = a['overlaps'].item(), b['overlaps'].item()
    assert va.keys() == vb.keys() and all(np.array_equal(va[k], vb[k]) for k in va)


def test_seed_policies_and_counters_equal_the_reference_modules(golden_dir):
  """The simple seed policies (PolicyMax, PolicyGrid2d / 3d with custom steps and offsets, PolicyDenseSeeds with
  erosions / invert, ReverseCoords, SequentialPolicies — seed.py:307-313,411-544 behind the border filter of
  BaseSeedPolicy.__next__, :63-95) and `Counters.dumps / loads` (inference_utils.py:90-150) against the outputs of the
  reference's own modules (tests/golden/make_golden_policies.py)."""
  import importlib.util
  from ffn.inference import inference_utils, seed
  spec = importlib.util.spec_from_file_location('make_golden_policies', os.path.join(golden_dir, 'make_golden_policies.py'))
  r = np.load(os.path.join(golden_dir, 'seed_policies_ref.npz'))

  class FakeCanvas:
    image = r['image']
    shape = tuple(r['image'].shape)
    margin = r['margin']
    restrictor = None
    segmentation = np.zeros(r['image'].shape, np.int32)

  cases = [
      ('max', 'PolicyMax', {}),
      ('grid2d', 'PolicyGrid2d', {'step': 6, 'offsets': (0, 3, 1)}),
      ('grid3d', 'PolicyGrid3d', {'step': 5, 'offsets': (0, 2, 4)}),
      ('dense', 'PolicyDenseSeeds', {'threshold': 0.5, 'num_erosions': 1}),
      ('dense_inv', 'PolicyDenseSeeds', {'threshold': 0.55, 'num_erosions': 2, 'invert': True}),
      ('reverse', 'ReverseCoords', {'policy_to_reverse': 'PolicyGrid3d', 'step': 6}),
      ('sequential', 'SequentialPolicies', {'policies': [('PolicyGrid3d', {'step': 7}), ('PolicyGrid2d', {'step': 9})]}),
  ]
  del spec
  for name, cls, kwargs in cases:
    canvas = FakeCanvas()
    got = np.array([tuple(int(v) for v in c) for c in getattr(seed, cls)(canvas, **kwargs)], dtype=np.int64).reshape(-1, 3)
    np.testing.assert_array_equal(got, r['coords_' + name], err_msg=name)

  c = inference_utils.Counters()
  c['inference-calls'].IncrementBy(144)
  c['voxels-segmented'].Set(123456)
  c['inference-time-ms'].IncrementBy(2500)
  sub = c.get_sub_counters()
  sub['skip_invalid_pos'].IncrementBy(7)
  sub['voxels-segmented'].IncrementBy(44)
  assert json.loads(sub.dumps()) == json.loads(str(r['sub_counters_dumps']))
  # Deliberate, documented difference (inference_utils.py here): sub-counters FEED their parent — the reference's
  # get_sub_counters (inference_utils.py:133-134) builds children whose updates never reach the parent, so its
  # Runner.counters / counters.txt miss everything the canvases counted.  Own values must agree:
  ref = json.loads(str(r['counters_dumps']))
  ours = json.loads(c.dumps())
  assert ours == dict(ref, **{'voxels-segmented': ref['voxels-segmented'] + 44, 'skip_invalid_pos': 7})
  d = inference_utils.Counters()
  d.loads(str(r['counters_dumps']))
  assert json.loads(d.dumps()) == json.loads(str(r['counters_after_loads']))


def test_build_mask_equals_reference(golden_dir):
  """storage.build_mask (MaskConfig lists: coordinate expressions, image channels, volume channels with value lists,
  per-channel and per-config invert, OR of several configs) against the reference's own build_mask
  (storage.py:323-411; fixture from tests/golden/make_golden_build_mask.py) — the `request.masks` / `seed_masks` path
  of Runner.make_restrictor."""
  import importlib.util
  from google.protobuf import text_format
  from ffn.inference import inference_pb2, storage
  spec = importlib.util.spec_from_file_location('make_golden_build_mask', os.path.join(golden_dir, 'make_golden_build_mask.py'))
  gen = importlib.util.module_from_spec(spec)
  sys_path = list(__import__('sys').path)
  try:
    spec.loader.exec_module(gen)             # only for its CASES table (no reference import happens at module level)
  finally:
    __import__('sys').path[:] = sys_path
  r = np.load(os.path.join(golden_dir, 'build_mask_ref.npz'))
  corner, size = tuple(int(v) for v in r['corner']), tuple(int(v) for v in r['size'])
  for name, texts in gen.CASES.items():
    configs = [text_format.Parse(t, inference_pb2.MaskConfig()) for t in texts]
    cache = {c.volume.mask.SerializeToString(): r['volume'] for c in configs if c.WhichOneof('source') == 'volume'}
    got = storage.build_mask(configs, corner, size, mask_volume_map=cache, image=r['image'])
    assert got.dtype == bool
    np.testing.assert_array_equal(got, r['mask_' + name], err_msg=name)


def test_small_host_helpers_equal_the_reference(tmp_path, golden_dir):
  """align.Alignment / Aligner, storage.clip_subvolume_to_bounds / dequantize_probability / threshold_segmentation /
  path helpers / get_existing_subvolume_path / get_existing_corners, segmentation.reduce_id_bits / clear_dust against
  the outputs of the reference's own functions (tests/golden/make_golden_helpers.py -> helpers_ref.npz)."""
  import importlib.util
  import sys
  from ffn.inference import align, segmentation, storage
  saved = list(sys.path)
  try:
    spec = importlib.util.spec_from_file_location('make_golden_helpers', os.path.join(golden_dir, 'make_golden_helpers.py'))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)                         # only its CROPS / CLIPS / CORNERS tables
  finally:
    sys.path[:] = saved
  r = np.load(os.path.join(golden_dir, 'helpers_ref.npz'))
  # ---- align
  for i, (sc, ss, dc, ds, fill) in enumerate(gen.CROPS):
    a = align.Alignment(dc, ds)
    got = a.align_and_crop(np.array(sc), r['crop_src_%d' % i], np.array(dc), np.array(ds), fill=fill)
    np.testing.assert_array_equal(got, r['crop_out_%d' % i], err_msg='crop %d' % i)
    assert got.dtype == r['crop_out_%d' % i].dtype
  a = align.Aligner().generate_alignment((4, 5, 6), (10, 20, 30))
  np.testing.assert_array_equal(a.corner, r['align_corner'])
  np.testing.assert_array_equal(a.size, r['align_size'])
  for fwd in (True, False):
    c, s = a.expand_bounds(np.array((1, 2, 3)), np.array((7, 8, 9)), forward=fwd)
    np.testing.assert_array_equal(np.stack([c, s]), r['expand_%d' % fwd])
  pts = np.array([[1, 2, 3], [4, 5, 6]]).T
  np.testing.assert_array_equal(a.transform(pts), r['transform'])
  rs = a.rescaled(np.array((1.0, 0.5, 0.5)))
  np.testing.assert_array_equal(np.stack([rs.corner, rs.size]).astype(np.float64), r['rescaled'])
  np.testing.assert_array_equal(a.transform_shift_mask(np.array((4, 5, 6)), 2, r['shift_in']), r['shift_out'])
  # ---- clip
  vol3, vol4 = np.zeros((20, 24, 28)), np.zeros((2, 20, 24, 28))
  k = 0
  for corner, size in gen.CLIPS:
    for vol in (vol3, vol4):
      want = r['clips'][k]
      k += 1
      if want[0] == -1 and want[3] == -1:
        continue                                                   # disjoint boxes: the reference raises
      c, s = storage.clip_subvolume_to_bounds(np.array(corner), np.array(size), vol)
      assert list(np.asarray(c).astype(int)) + list(np.asarray(s).astype(int)) == want.tolist(), (corner, size)
  # ---- probabilities
  got = storage.dequantize_probability(np.arange(256, dtype=np.uint8))
  np.testing.assert_array_equal(np.isnan(got), np.isnan(r['dequantized']))
  np.testing.assert_array_equal(got[1:], r['dequantized'][1:])
  assert got.dtype == r['dequantized'].dtype
  corner = (5, 6, 7)
  prob_path = storage.object_prob_path(str(tmp_path), corner)
  os.makedirs(os.path.dirname(prob_path), exist_ok=True)
  with open(prob_path, 'wb') as f:
    np.savez_compressed(f, qprob=r['thr_qprob'])
  labels = r['thr_labels'].copy()
  storage.threshold_segmentation(str(tmp_path), corner, labels, 0.7)
  np.testing.assert_array_equal(labels, r['thr_out'])
  # ---- paths
  paths = json.loads(str(r['paths_json']))
  for c in gen.CORNERS:
    ours = [storage.subvolume_path('/out', c, 'npz'), storage.legacy_subvolume_path('/out', c, 'npz'),
            storage.segmentation_path('/out', c), storage.object_prob_path('/out', c), storage.checkpoint_path('/out', c),
            storage.legacy_segmentation_path('/out', c), storage.legacy_object_prob_path('/out', c)]
    assert ours == paths[str(tuple(c))]
    assert storage.get_corner_from_path(ours[0]) == tuple(c)
  d2 = tmp_path / 'existing'
  for c, legacy, suffix in (((1, 2, 3), False, 'npz'), ((4, 5, 6), True, 'npz'), ((7, 8, 9), False, 'cpoint')):
    p = storage.legacy_subvolume_path(str(d2), c, suffix) if legacy else storage.subvolume_path(str(d2), c, suffix)
    os.makedirs(os.path.dirname(p), exist_ok=True)
    open(p, 'wb').close()
  existing = json.loads(str(r['existing_json']))
  for c in ((1, 2, 3), (4, 5, 6), (7, 8, 9), (9, 9, 9)):
    for allow in (False, True):
      got = storage.get_existing_subvolume_path(str(d2), c, allow)
      assert (None if got is None else os.path.relpath(got, str(d2))) == existing['%r/%d' % (c, allow)]
  assert sorted(storage.get_existing_corners(str(d2))) == [tuple(v) for v in r['existing_corners'].tolist()]
  # ---- segmentation helpers
  for top in (200, 300, 70000):
    assert str(segmentation.reduce_id_bits(r['reduce_in_%d' % top]).dtype) == str(r['reduce_dtype_%d' % top])
  np.testing.assert_array_equal(segmentation.clear_dust(r['dust_in'].copy(), min_size=9), r['dust_out'])


def test_every_proto_field_matches_the_reference_proto_sources(golden_dir):
  """The runtime-built descriptors (ffn_b200/inference/protos.py) against the reference's .proto SOURCES, field by
  field: name, number, label, type (scalar / message / enum), default, oneof membership; enum values too (fixture:
  tests/golden/make_golden_schema.py parses inference.proto, bounding_box.proto, vector.proto)."""
  from google.protobuf import descriptor
  from ffn.inference import inference_pb2
  from ffn.utils import bounding_box_pb2, vector_pb2
  schema = json.load(open(os.path.join(golden_dir, 'proto_schema_ref.json')))
  pool = inference_pb2.InferenceRequest.DESCRIPTOR.file.pool
  del bounding_box_pb2, vector_pb2
  scalar = {descriptor.FieldDescriptor.TYPE_DOUBLE: 'double', descriptor.FieldDescriptor.TYPE_FLOAT: 'float',
            descriptor.FieldDescriptor.TYPE_INT64: 'int64', descriptor.FieldDescriptor.TYPE_UINT64: 'uint64',
            descriptor.FieldDescriptor.TYPE_INT32: 'int32', descriptor.FieldDescriptor.TYPE_BOOL: 'bool',
            descriptor.FieldDescriptor.TYPE_STRING: 'string', descriptor.FieldDescriptor.TYPE_BYTES: 'bytes',
            descriptor.FieldDescriptor.TYPE_UINT32: 'uint32'}
  checked = 0
  for full, ref in schema.items():
    if full.endswith('.<file>'):
      continue
    d = pool.FindMessageTypeByName(full)
    assert sorted(f.name for f in d.fields) == sorted(ref['fields']), full
    for name, (number, label, ftype, default, oneof) in ref['fields'].items():
      f = d.fields_by_name[name]
      where = '%s.%s' % (full, name)
      assert f.number == number, where
      repeated = getattr(f, 'is_repeated', None)          # property (protobuf >= 6), method, or absent
      if repeated is None:
        repeated = f.label == f.LABEL_REPEATED
      elif callable(repeated):
        repeated = repeated()
      assert repeated == (label == 'repeated'), where
      if f.type == f.TYPE_MESSAGE:
        assert f.message_type.full_name.split('.')[-1] == ftype.split('.')[-1], where
      elif f.type == f.TYPE_ENUM:
        assert f.enum_type.name == ftype.split('.')[-1], where
      else:
        assert scalar[f.type] == ftype, where
      if default is not None:
        assert f.has_default_value, where
        got = f.default_value
        if f.type == f.TYPE_ENUM:
          got = f.enum_type.values_by_number[got].name
        elif f.type == f.TYPE_BOOL:
          got = 'true' if got else 'false'
        assert (float(got) == float(default)) if f.type in (f.TYPE_FLOAT, f.TYPE_DOUBLE, f.TYPE_INT32, f.TYPE_INT64) \
            else (str(got) == default), (where, got, default)
      assert (f.containing_oneof.name if f.containing_oneof else None) == oneof, where
      checked += 1
    for ename, values in ref['enums'].items():
      e = d.enum_types_by_name[ename]
      assert {v.name: v.number for v in e.values} == values, (full, ename)
  assert checked >= 95
