"""The CPU oracle against fixtures produced by the reference's own Python modules.

Fixtures come from tests/golden/make_golden.py, which imports the unmodified
ffn/inference/{inference,movement,seed,storage}.py from the reference checkout.
"""

import json
import os

import numpy as np
import pytest

from oracle import flood_fill as ff
from oracle.toy_net import toy_image, toy_net


def _load(golden_dir, name):
  return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def test_thresholds_match_reference(golden_dir):
  g = _load(golden_dir, 'flood_fill_64.npz')
  init, pad, move, seg = g['thresholds']
  assert float(ff.f32_logit(0.95)) == init
  assert float(ff.f32_logit(0.05)) == pad
  assert float(ff.f32_logit(0.9)) == move
  assert float(ff.f32_logit(0.6)) == seg
  assert ff.policy_threshold(0.9) == float(g['policy_threshold'])
  # SURVEY 8a row 6: the f64 policy threshold and the f32 canvas threshold select the same scores.
  assert np.float32(move).view(np.uint32) == 0x400c9f53
  assert np.nextafter(np.float32(move), np.float32(0)) < g['policy_threshold'] <= move


def test_quantize_probability(golden_dir):
  g = _load(golden_dir, 'qprob.npz')
  np.testing.assert_array_equal(ff.quantize_probability(g['prob']), g['q'])
  np.testing.assert_array_equal(
      ff.quantize_probability(np.array([0, .003, .5, .6, .999, 1.0])), [1, 1, 128, 153, 254, 255])


def test_scored_moves(golden_dir):
  g = _load(golden_dir, 'moves.npz')
  th = float(g['threshold'])
  for i in range(int(g['n'])):
    deltas, logits, want = g['deltas_%d' % i], g['logits_%d' % i], g['moves_%d' % i]
    got = ff.scored_moves(deltas, logits, th)
    got.sort(reverse=True)
    arr = np.asarray([(float(s),) + r for s, r in got], dtype=np.float64).reshape(-1, 4)
    np.testing.assert_array_equal(arr, want)


def test_grid_seeds_match_policy_grid3d(golden_dir):
  g = _load(golden_dir, 'toy_flood_fill.npz')
  shape = g['cells'].shape
  seeds = ff.grid_seeds(shape)
  margin = np.array([16, 16, 16])
  keep = np.all((seeds - margin >= 0) & (seeds + margin < np.array(shape)), axis=1)
  np.testing.assert_array_equal(seeds[keep], g['seeds'])   # after the border filter seed.py:81-88


def _check_canvas(canvas, g, exact_seed=True):
  np.testing.assert_array_equal(np.asarray(canvas.trace, dtype=np.int32).reshape(-1, 3), g['trace'])
  np.testing.assert_array_equal(canvas.segmentation, g['segmentation'])
  if exact_seed:
    np.testing.assert_array_equal(canvas.seed, g['seed_canvas'])
    np.testing.assert_array_equal(canvas.seg_prob, g['seg_prob'])
  else:
    np.testing.assert_allclose(canvas.seed, g['seed_canvas'], atol=2e-3, rtol=0, equal_nan=True)
    assert np.abs(canvas.seg_prob.astype(int) - g['seg_prob'].astype(int)).max() <= 1
  origins = np.array([(k,) + v[0] + (v[1],) for k, v in sorted(canvas.origins.items())],
                     dtype=np.int64).reshape(-1, 5)
  np.testing.assert_array_equal(origins, g['origins'])
  owner, ids, cnt = [], [], []
  for k, v in sorted(canvas.overlaps.items()):
    for i, c in zip(v[0], v[1]):
      owner.append(k); ids.append(int(i)); cnt.append(int(c))
  np.testing.assert_array_equal(np.asarray([owner, ids, cnt], dtype=np.int64).reshape(3, -1),
                                g['overlaps'].reshape(3, -1))
  want = json.loads(str(g['counters']))
  for name in ('skip_threshold', 'skip_invalid_pos', 'voxels-segmented', 'voxels-overlapping',
               'inference-calls', 'seed_got_too_weak'):
    assert canvas.counters.get(name, 0) == want.get(name, 0), name
  assert canvas.counters['segment_at-calls'] == want['segment_at-loop-calls']


def test_toy_flood_fill_bit_exact(golden_dir):
  """Loop logic pinned machine-independently (elementwise-only toy network)."""
  g = _load(golden_dir, 'toy_flood_fill.npz')
  image = toy_image(g['cells'])
  opts = ff.Options(min_segment_size=int(g['min_segment_size']),
                    min_boundary_dist=tuple(int(v) for v in g['min_boundary_dist']))
  canvas = ff.Canvas(toy_net, image, (33, 33, 33), (8, 8, 8), opts)
  canvas.segment_all(g['seeds'])
  _check_canvas(canvas, g, exact_seed=True)


def _rebuild_fib25_checkpoint(golden_dir, out_dir):
  """The reference's FIB-25 TF checkpoint, byte for byte: its `.index` and non-weight tensor bytes from fib25_ckpt.npz,
  the seed_update weights from fib25_convstack.npz placed where the index says (make_golden_reference_files.py)."""
  import hashlib
  from ffn_b200 import tf_checkpoint
  c = _load(golden_dir, 'fib25_ckpt.npz')
  prefix = os.path.join(str(out_dir), 'model.ckpt-27465036')
  with open(prefix + '.index', 'wb') as f:
    f.write(c['index'].tobytes())
  data = bytearray(int(c['data_size']))
  pos = 0
  for lo, hi in c['other_offsets']:
    data[lo:hi] = c['other_bytes'][pos:pos + hi - lo].tobytes()
    pos += hi - lo
  w, b = tf_checkpoint.load_convstack_npz(os.path.join(golden_dir, 'fib25_convstack.npz'))
  names = ['conv%d_%s' % (i, s) for i in range(12) for s in 'ab'] + ['conv_lom']
  entries = tf_checkpoint.list_variables(prefix)
  for name, wi, bi in zip(names, w, b):
    for kind, arr in (('weights', wi), ('biases', bi)):
      e = entries['seed_update/%s/%s' % (name, kind)]
      assert tuple(e['shape']) == arr.shape and e['size'] == arr.nbytes, (name, kind)
      data[e['offset']:e['offset'] + e['size']] = arr.astype('<f4').tobytes()
  assert hashlib.sha256(data).hexdigest() == str(c['data_sha256'])
  with open(prefix + '.data-00000-of-00001', 'wb') as f:
    f.write(data)
  return prefix


@pytest.mark.slow
def test_real_net_flood_fill(golden_dir, tmp_path):
  """Same loop with the FIB-25 conv stack (torch CPU), weights read from the TF checkpoint.  Exactness is
  qualified by the decision margin because conv3d rounding may differ between CPUs."""
  from ffn_b200 import tf_checkpoint
  from oracle.network import ConvStackOracle
  ckpt = _rebuild_fib25_checkpoint(golden_dir, tmp_path)
  g = _load(golden_dir, 'flood_fill_64.npz')
  w, b = tf_checkpoint.load_convstack_weights(ckpt, 12)
  image = (g['volume'].astype(np.float32) - 128.0) / 33.0
  canvas = ff.Canvas(ConvStackOracle(w, b), image, (33, 33, 33), (8, 8, 8), ff.Options())
  canvas.segment_all(g['seeds'])
  if canvas.min_margin < 1e-4:
    pytest.skip('knife-edge decision (margin %g): trajectory not comparable across CPUs' % canvas.min_margin)
  _check_canvas(canvas, g, exact_seed=False)


def test_canonical_relabel():
  seg = np.array([[0, 7, 7], [3, 3, -1], [7, 9, 0]])
  np.testing.assert_array_equal(ff.canonical_relabel(seg), [[0, 1, 1], [2, 2, 0], [1, 3, 0]])


def test_golden_sample_summary(golden_dir):
  """Sanity ranges of the reference's shipped 250^3 result (input volume is not available)."""
  with open(os.path.join(golden_dir, 'sample_training2_summary.json')) as f:
    s = json.load(f)
  assert s['shape'] == [250, 250, 250]
  assert s['num_segments'] == 254 == s['num_origins'] == s['origins_carry_own_id']
  assert s['counters']['inference-calls'] == 25799
  assert s['counters']['voxels-segmented'] == 13867123


def test_oracle_history_matches_reference_keep_history(golden_dir):
  """Canvas.history / history_deleted (keep_history=True) of the reference's own segment_at,
  recorded by tests/golden/make_golden_history.py, for two objects on the 64x72x80 phantom."""
  from oracle import flood_fill as ff
  from oracle.network import ConvStackOracle
  from ffn_b200 import tf_checkpoint
  g = np.load(os.path.join(golden_dir, 'flood_fill_64.npz'))
  h = np.load(os.path.join(golden_dir, 'segment_at_history_64.npz'))
  w, b = tf_checkpoint.load_convstack_npz(os.path.join(golden_dir, 'fib25_convstack.npz'))
  image = (g['volume'].astype(np.float32) - 128.0) / 33.0
  cv = ff.Canvas(ConvStackOracle(w, b), image, (33, 33, 33), (8, 8, 8), ff.Options())
  cv.segment_at(tuple(int(v) for v in h['start']))
  np.testing.assert_array_equal(np.asarray(cv.history, np.int32).reshape(-1, 3), h['history'])
  np.testing.assert_array_equal(np.asarray(cv.history_deleted, np.int64), h['history_deleted'])
  assert h['history_deleted'].sum() > 0
  cv.segment_at(tuple(int(v) for v in h['second_start']))
  np.testing.assert_array_equal(np.asarray(cv.history, np.int32).reshape(-1, 3), h['second_history'])
  np.testing.assert_array_equal(np.asarray(cv.history_deleted, np.int64), h['second_history_deleted'])


def test_toy_masked_flood_fill_bit_exact(golden_dir):
  """segment_all behind a MovementRestrictor with mask, seed_mask and a shift mask — the reference's own
  run (tests/golden/make_golden_masks.py).  The oracle (like the device) gets the shift rule folded into
  the movement mask by ffn_b200's MovementRestrictor.movement_mask."""
  from ffn_b200.inference import movement
  from ffn_b200.utils import bounding_box
  g = _load(golden_dir, 'toy_masks_flood_fill.npz')
  restrictor = movement.MovementRestrictor(
      mask=g['mask'], seed_mask=g['seed_mask'], shift_mask=g['shift'],
      shift_mask_fov=bounding_box.BoundingBox(start=g['fov_start'], size=g['fov_size']),
      shift_mask_threshold=int(g['shift_threshold']), shift_mask_scale=int(g['shift_scale']))
  opts = ff.Options(min_segment_size=int(g['min_segment_size']),
                    min_boundary_dist=tuple(int(v) for v in g['min_boundary_dist']))
  canvas = ff.Canvas(toy_net, toy_image(g['cells']), (33, 33, 33), (8, 8, 8), opts,
                     mask=restrictor.movement_mask(g['cells'].shape), seed_mask=g['seed_mask'])
  canvas.segment_all(g['seeds'])
  _check_canvas(canvas, g, exact_seed=True)
  want = json.loads(str(g['counters']))
  assert want['skip_restriced_pos'] > 0 and canvas.counters['skip_restriced_pos'] == want['skip_restriced_pos']


def test_toy_anisotropic_flood_fill_bit_exact(golden_dir):
  """fov (17, 33, 33), deltas (4, 8, 8) — the geometry of BASELINE configs[4] — against the reference."""
  g = _load(golden_dir, 'toy_aniso_flood_fill.npz')
  opts = ff.Options(min_segment_size=int(g['min_segment_size']),
                    min_boundary_dist=tuple(int(v) for v in g['min_boundary_dist']))
  canvas = ff.Canvas(toy_net, toy_image(g['cells']), (17, 33, 33), (4, 8, 8), opts)
  canvas.segment_all(g['seeds'])
  _check_canvas(canvas, g, exact_seed=True)
  assert g['trace'].shape[0] > 100


def test_seed_peaks_edt_restatement_equals_the_definition():
  """oracle/seed_peaks.py restates edt.edt with scipy's exact EDT: pinned against the O(n^2) definition
  (distance to the nearest background voxel in physical units), isotropic and anisotropic."""
  from scipy import ndimage
  from oracle import seed_peaks
  rng = np.random.RandomState(0)
  fg = rng.rand(9, 11, 13) > 0.25
  for voxel in ((1.0, 1.0, 1.0), (2.0, 1.0, 1.0), (3.0, 1.5, 1.0)):
    want = seed_peaks.brute_force_edt(fg, voxel)
    got = ndimage.distance_transform_edt(fg, sampling=voxel)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-12)


def test_seed_peaks_oracle_properties():
  """Lexicographic order, border filter, exclusions, spacing > min_distance (Chebyshev) and determinism."""
  from ffn_b200.synthetic import voronoi_phantom
  from oracle import seed_peaks
  vol = voronoi_phantom((48, 56, 64), seed=9, cell_volume=9000.0)
  image = (vol.astype(np.float32) - np.float32(128)) / np.float32(33)
  seg = np.zeros(vol.shape, np.int32)
  seg[10:30, 10:30, 10:30] = 3
  mask = np.zeros(vol.shape, bool)
  mask[:, :6, :] = True
  c = seed_peaks.policy_peaks(image, (1, 1, 1), segmentation=seg, mask=mask, margin_zyx=(4, 4, 4))
  assert c.shape[0] > 10
  assert [tuple(r) for r in c.tolist()] == sorted(tuple(r) for r in c.tolist())
  assert np.all(c >= 4) and np.all(c + 4 < np.asarray(vol.shape)[None])
  assert not any(seg[z, y, x] > 0 or mask[z, y, x] for z, y, x in c)
  d = np.abs(c[:, None, :] - c[None, :, :]).max(axis=2)
  np.fill_diagonal(d, 99)
  assert d.min() > 3
  np.testing.assert_array_equal(c, seed_peaks.policy_peaks(image, (1, 1, 1), segmentation=seg, mask=mask, margin_zyx=(4, 4, 4)))
  full = seed_peaks.policy_peaks(image, (2, 1, 1))
  assert full.shape[0] > 10 and not np.array_equal(full, seed_peaks.policy_peaks(image, (1, 1, 1)))


def test_seed_peaks_oracle_equals_reference_policy_peaks(golden_dir):
  """oracle/seed_peaks.py against the reference's OWN PolicyPeaks (seed.py:36-199, run unmodified by
  tests/golden/make_golden_peaks.py with only the two un-vendored third-party calls — edt.edt and
  skimage.feature.peak_local_max — injected by definition): isotropic, anisotropic voxel size, and a canvas with a
  movement mask, a seed mask, existing labels and -1 markers.  The seed LIST (order included) must be equal."""
  from oracle import seed_peaks
  r = np.load(os.path.join(golden_dir, 'policy_peaks_ref.npz'))
  for case in ('iso', 'aniso', 'masked'):
    vol = r[case + '_volume']
    image = (vol.astype(np.float32) - np.float32(128.0)) / np.float32(33.0)
    kw = {}
    if case == 'masked':
      kw = dict(mask=r['masked_mask'], seed_mask=r['masked_seed_mask'])
    got = seed_peaks.policy_peaks(image, voxel_size_zyx=tuple(float(v) for v in r[case + '_voxel']),
                                  segmentation=r[case + '_segmentation'], margin_zyx=tuple(int(v) for v in r[case + '_margin']), **kw)
    want = r[case + '_coords']
    assert want.shape[0] >= 8, (case, want.shape)
    np.testing.assert_array_equal(got, want, err_msg=case)


def test_network_oracle_equals_an_independent_correlation_restatement(golden_dir):
  """The torch-based network oracle against a second, torch-free restatement of the same TensorFlow semantics
  (convstack_3d.py:26-56,83-95; model.py:168-183): every Conv3D as a sum of scipy.ndimage.correlate calls — one per
  (input, output) channel pair, zero padding ('SAME'), kernel NOT flipped (cross-correlation), DHWIO weights indexed
  directly — BiasAdd, ReLU placement (tf_slim: `_a` convolutions activated, `_b` linear), pre-activation residual
  modules, 1x1x1 conv_lom, logits = seed + update.  Full FIB-25 depth on a small patch, float64 on both sides."""
  import torch
  from scipy import ndimage
  from ffn_b200 import tf_checkpoint
  from oracle.network import ConvStackOracle
  w, b = tf_checkpoint.load_convstack_npz(os.path.join(golden_dir, 'fib25_convstack.npz'))
  rng = np.random.RandomState(2)
  shape = (7, 9, 10)
  image = rng.randn(*shape).astype(np.float32)
  seed = np.where(rng.rand(*shape) < 0.4, rng.randn(*shape) * 2, -2.9444).astype(np.float32)

  def conv(x, wk, bias):                                   # x [C_in, Z, Y, X], wk [3, 3, 3, C_in, C_out]
    out = np.empty((wk.shape[4],) + x.shape[1:], dtype=np.float64)
    for co in range(wk.shape[4]):
      acc = np.zeros(x.shape[1:], dtype=np.float64)
      for ci in range(wk.shape[3]):
        acc += ndimage.correlate(x[ci], wk[:, :, :, ci, co].astype(np.float64), mode='constant', cval=0.0)
      out[co] = acc + np.float64(bias[co])
    return out

  relu = lambda t: np.maximum(t, 0.0)
  depth = (len(w) - 1) // 2
  net = np.stack([image, seed]).astype(np.float64)         # channel 0 = image, 1 = seed (convstack_3d.py:86)
  net = relu(conv(net, w[0], b[0]))
  net = conv(net, w[1], b[1])
  for m in range(1, depth):
    skip = net
    net = relu(net)
    net = relu(conv(net, w[2 * m], b[2 * m]))
    net = conv(net, w[2 * m + 1], b[2 * m + 1])
    net = net + skip
  net = relu(net)
  update = np.tensordot(w[-1][0, 0, 0, :, 0].astype(np.float64), net, axes=(0, 0)) + np.float64(b[-1][0])
  want = seed.astype(np.float64) + update
  orc = ConvStackOracle(w, b, dtype=torch.float64)
  got64 = seed.astype(np.float64) + orc.update(seed, image)
  assert np.abs(got64 - want).max() <= 1e-9 * max(1.0, np.abs(want).max())
  got32 = ConvStackOracle(w, b)(seed, image)
  assert np.abs(got32 - want).max() <= 2e-4
