"""The conv stack and the device flood loop at the fields of view, depths, grids and chain counts the engine
accepts, not only at the 33^3 / depth-12 product geometry.

What depends on the geometry is where a tiled tensor-core kernel goes wrong: the row space (pitches xp = fx and
pp = (fy + 1) * fx, guard rows, tiles of 126 output rows), the float row decode, the SAME padding in x that is
applied after the dx taps were stacked along N (the m_up / m_dn masks of the tensor-core epilogue, the tap skip of
the fp32 path), the partial sums that cross warp boundaries at accumulator rows 32 / 64 / 96, the tiles a CTA
owns and the TMEM column of every (chain, tile) residual, and in the flood loop the FoV-dependent staging
offsets, faces and lookahead clearance.

  1. Locality (exact, every mode): each logit depends only on the inputs within Chebyshev distance 2 * depth of
     its voxel, and a voxel's arithmetic does not depend on the rest of the patch, so changing one input voxel
     p must leave every logit outside p +- 2 * depth bit-identical.  A line-wrap or tile-boundary error shows up
     as a non-zero difference outside that box.
  2. Parity with a float64 oracle at every accepted geometry of a matrix (random He-scaled weights).
  3. Grid / chain invariance (exact): grid and chain count only decide which CTA computes a tile and in what
     order, so predict is bit-identical across them, up to 10 tiles per CTA (TMEM full).
  4. The flood loop away from 33^3: chains vs the sequential loop (bit for bit) and vs the oracle loop driven by
     the same device network.
  5. Clean rejection of the geometries the engine cannot run.
"""

import json
import os

import numpy as np
import pytest
import torch

from oracle import flood_fill as ff
from oracle.network import ConvStackOracle

# Every test here needs the device except test_oracle_locality_impulse, so the mark is per test, not per module.
gpu = pytest.mark.gpu

TILE_OUT = 126          # FoV rows one tensor-core tile outputs (device_types.cuh: kTileOut)
MAX_TILES_PER_CTA = 10  # TMEM-resident residual stream: 512 columns = 2 * 96 accumulators + 10 * 32
MODES = ('fp32', 'x2', 'tc')
PAD = float(np.float32(ff.f32_logit(0.05)))
INIT = float(np.float32(ff.f32_logit(0.95)))

# Relative bounds of the fast fp16 mode (max error / max(1, max |oracle|)).  Measured on a B200 (1000 W) by
# test_parity_with_float64_oracle: at most 1.0e-3 against the float64 oracle and 7.8e-4 against the fp16-operand
# oracle (17x33x33, depth 9); the bounds leave a margin of about 3x.  The FIB-25 bounds of test_gpu_parity.py
# (4e-2 / 1.5e-2 absolute at max |logit| 6.15) are 6.5e-3 / 2.4e-3 relative: these are no looser.
TC_TOL_F64_ORACLE = 3e-3
TC_TOL_FP16_ORACLE = 2.4e-3
PARITY_TOL = 1e-4       # fp32 and split-fp16 (x2) against the float64 oracle


def _mode_id(mode):
  from ffn_b200 import _lib
  return {'fp32': _lib.COMPUTE_FP32, 'x2': _lib.COMPUTE_FP16X2_TC, 'tc': _lib.COMPUTE_FP16_TC}[mode]


def random_stack(depth, seed, scale=1.0, b_scale=0.5):
  """Seeded He-scaled DHWIO weights and non-zero biases (conv0_a, conv0_b, ..., conv_lom); the `_b` convolutions
  of the residual modules are scaled by `b_scale` so that logits stay O(1-10) up to depth 16."""
  rng = np.random.RandomState(seed)
  w, b = [], []
  for l in range(2 * depth):
    cin = 2 if l == 0 else 32
    s = np.sqrt(2.0 / (27 * cin)) * scale * (b_scale if (l % 2 == 1 and l > 1) else 1.0)
    w.append((rng.randn(3, 3, 3, cin, 32) * s).astype(np.float32))
    b.append((rng.randn(32) * 0.1).astype(np.float32))
  w.append((rng.randn(1, 1, 1, 32, 1) * np.sqrt(1.0 / 32)).astype(np.float32))
  b.append((rng.randn(1) * 0.1).astype(np.float32))
  return w, b


def oracle_logits(w, b, seed, image, operand_round=None):
  """float64 logits (seed + update), not rounded to float32."""
  upd = ConvStackOracle(w, b, dtype=torch.float64, operand_round=operand_round).update(seed, image)
  return np.asarray(seed, np.float64) + upd


def make_patches(fov, n_distinct, rng):
  """(seed, image) pairs: seeds mix pad, init_activation and random logits; pair 3 (mod 4) has its image at the
  u8-normalised extremes +-3.9."""
  seeds, imgs = [], []
  c = tuple(s // 2 for s in fov)
  for i in range(n_distinct):
    kind = i % 4
    img = rng.randn(*fov).astype(np.float32)
    if kind == 0:                                   # a fresh object: pad everywhere, init_activation at the centre
      seed = np.full(fov, PAD, np.float32)
      seed[c] = INIT
    elif kind == 1:                                 # an object in flight: random logits in places, pad elsewhere
      seed = np.where(rng.rand(*fov) < 0.4, rng.randn(*fov) * 3.0, PAD).astype(np.float32)
    elif kind == 2:
      seed = (rng.randn(*fov) * 4.0).astype(np.float32)
    else:
      img = np.where(rng.rand(*fov) < 0.5, -3.9, 3.9).astype(np.float32)
      seed = np.where(rng.rand(*fov) < 0.5, INIT, PAD).astype(np.float32)
    seeds.append(seed)
    imgs.append(img)
  return np.stack(seeds), np.stack(imgs)


def geom(fov):
  fz, fy, fx = fov
  pp = (fy + 1) * fx
  nr = (fz - 1) * pp + (fy - 1) * fx + fx
  return pp, nr, (nr + TILE_OUT - 1) // TILE_OUT


def row_voxel(fov, r):
  """FoV voxel of row r of the kernels' row space, or None for a pad line / a row past the FoV."""
  pp, nr, _ = geom(fov)
  if r < 0 or r >= nr:
    return None
  z, rem = divmod(r, pp)
  y, x = divmod(rem, fov[2])
  return (z, y, x) if y < fov[1] else None


def probe_voxels(fov):
  """Corners, both row ends, the y / z faces, the rows around tile boundaries and the warp-exchange rows."""
  fz, fy, fx = fov
  zc, yc, xc = fz // 2, fy // 2, fx // 2
  pts = [(z, y, x) for z in (0, fz - 1) for y in (0, fy - 1) for x in (0, fx - 1)]
  pts += [(zc, yc, 0), (zc, yc, fx - 1), (zc, 0, xc), (zc, fy - 1, xc), (0, yc, xc), (fz - 1, yc, xc)]
  pts += [(zc, yc, xc), (zc - 1, yc + 1, 0), (zc + 1, yc - 1, fx - 1)]
  _, _, nt = geom(fov)
  for t in sorted({0, 1, nt // 2, nt - 1}):
    offs = (-1, 0, 1) if t > 0 else ()
    # accumulator row m of tile t holds FoV row t * 126 - 1 + m; warps exchange at m = 31|32, 63|64, 95|96
    offs += (30, 31, 32, 62, 63, 64, 94, 95, 96)
    for off in offs:
      v = row_voxel(fov, t * TILE_OUT + off)
      if v is not None:
        pts.append(v)
  out = []
  for p in pts:
    if p not in out:
      out.append(p)
  return out


def box_mask(fov, p, radius):
  """True inside the Chebyshev box p +- radius, clipped to the FoV."""
  m = np.zeros(fov, bool)
  m[tuple(slice(max(c - radius, 0), c + radius + 1) for c in p)] = True
  return m


def shell_mask(fov, p, radius):
  """True at Chebyshev distance exactly `radius` from p."""
  idx = np.indices(fov)
  d = np.max(np.abs(idx - np.asarray(p).reshape(3, 1, 1, 1)), axis=0)
  return d == radius


# ----------------------------------------------------------------------------------------------------------------
# CPU: the locality claim on the oracle itself
# ----------------------------------------------------------------------------------------------------------------
def test_oracle_locality_impulse():
  """An impulse diff through a random depth-2 stack at (9,9,11): zero outside p +- 4 and non-zero on the box
  boundary — the receptive field the GPU locality test relies on is exactly 2 * depth."""
  fov, depth = (9, 9, 11), 2
  w, b = random_stack(depth, 11)
  rng = np.random.RandomState(5)
  seed, img = make_patches(fov, 2, rng)
  seed, img = seed[1], img[1]
  p = (4, 4, 5)
  base = oracle_logits(w, b, seed, img)
  for channel in ('image', 'seed'):
    s2, i2 = seed.copy(), img.copy()
    (i2 if channel == 'image' else s2)[p] += np.float32(2.5)
    d = oracle_logits(w, b, s2, i2) - base
    assert (d[~box_mask(fov, p, 2 * depth)] == 0).all(), channel
    assert (d[shell_mask(fov, p, 2 * depth)] != 0).any(), channel


# ----------------------------------------------------------------------------------------------------------------
# 1. Locality
# ----------------------------------------------------------------------------------------------------------------
LOCALITY = [((9, 11, 13), 1), ((9, 11, 13), 2), ((9, 11, 33), 2)]


@gpu
@pytest.mark.parametrize('fov,depth', LOCALITY, ids=['9x11x13-d1', '9x11x13-d2', '9x11x33-d2'])
def test_locality_is_exact(fov, depth):
  """d = predict(perturbed) - predict(base), one input voxel changed (image and seed channel separately): d is
  bit-exactly zero outside p +- 2 * depth in every mode; inside, fp32 and x2 match the float64 oracle's d; and
  the box is tight (d != 0 at distance exactly 2 * depth for an interior p)."""
  from ffn_b200 import engine as eng
  w, b = random_stack(depth, 100 + depth)
  rng = np.random.RandomState(7)
  s0, i0 = make_patches(fov, 2, rng)
  seed, img = s0[1], i0[1]
  pts = probe_voxels(fov)
  seeds, imgs, tags = [seed], [img], [None]
  for p in pts:
    for channel in ('image', 'seed'):
      s2, i2 = seed.copy(), img.copy()
      (i2 if channel == 'image' else s2)[p] += np.float32(2.5)
      seeds.append(s2)
      imgs.append(i2)
      tags.append((p, channel))
  seeds, imgs = np.stack(seeds), np.stack(imgs)
  want = oracle_logits(w, b, seeds, imgs)
  scale = max(1.0, float(np.abs(want).max()))
  radius = 2 * depth
  e = eng.Engine(w, b, fov, (1, 1, 1), compute_mode=_mode_id('fp32'))
  print('locality %r depth %d: %d tiles, %d probe voxels x 2 channels' % (fov, depth, geom(fov)[2], len(pts)))
  for mode in MODES:
    e.set_compute_mode(_mode_id(mode))
    got = e.predict(seeds, imgs)
    assert np.isfinite(got).all()
    leaks, max_err, tight = [], 0.0, False
    for i in range(1, len(tags)):
      p, channel = tags[i]
      d = got[i] - got[0]
      inside = box_mask(fov, p, radius)
      out = np.argwhere((d != 0) & ~inside)
      if out.size:
        leaks.append((p, channel, tuple(int(v) for v in out[0]), float(d[tuple(out[0])]), len(out)))
      if mode != 'tc':
        max_err = max(max_err, float(np.abs(d - (want[i] - want[0]))[inside].max()))
      if all(radius <= c < s - radius for c, s in zip(p, fov)):
        tight = tight or bool((d[shell_mask(fov, p, radius)] != 0).any())
    print('  %-4s leaks outside the box: %d cases; max |d - d_oracle| inside = %.3g (scale %.3g); tight: %s' % (
        mode, len(leaks), max_err, scale, tight))
    assert not leaks, (mode, leaks[:5])
    if mode != 'tc':
      assert max_err <= 2 * PARITY_TOL * scale, (mode, max_err)
      assert tight, mode
  e.close()


# ----------------------------------------------------------------------------------------------------------------
# 2. Parity with the float64 oracle across the geometry matrix
# ----------------------------------------------------------------------------------------------------------------
# (fov, depth, weight scale, distinct patches)
PARITY = [
    ((3, 3, 3), 1, 1.0, 4), ((3, 3, 3), 2, 1.0, 4),            # 1 tile: a 1-CTA grid, the leader is the only worker
    ((5, 7, 9), 1, 1.0, 4), ((5, 7, 9), 3, 1.0, 4),            # 3 tiles, unequal axes both ways
    ((9, 7, 5), 1, 1.0, 4), ((9, 7, 5), 3, 1.0, 4),
    ((33, 3, 3), 2, 1.0, 4), ((3, 33, 33), 2, 1.0, 4),         # degenerate planes / lines
    ((31, 29, 27), 2, 1.0, 4),                                 # every pitch different from 33
    ((17, 33, 33), 9, 1.0, 4),                                 # BASELINE configs[4]
    ((33, 33, 33), 1, 1.0, 4), ((33, 33, 33), 16, 1.0, 1),     # depth limits (depth 16: one patch, the oracle is slow)
    ((49, 49, 33), 2, 1.0, 4), ((65, 65, 33), 2, 1.0, 4),      # 5 and 8 tiles per CTA at 148 SMs: chain limit 2 and 1
    ((33, 33, 33), 2, 0.25, 4), ((33, 33, 33), 2, 4.0, 4),     # split-fp16 (w * 2^10 = hi + lo) is not range-limited
]


def _parity_id(case):
  fov, depth, scale, _ = case
  return '%s-d%d%s' % ('x'.join(map(str, fov)), depth, '' if scale == 1.0 else '-w%g' % scale)


@gpu
@pytest.mark.parametrize('case', PARITY, ids=[_parity_id(c) for c in PARITY])
def test_parity_with_float64_oracle(case):
  """max |got - oracle64| <= tol * max(1, max |oracle64|) in all three modes; the fast fp16 mode is bounded
  against the oracle with fp16-rounded conv operands as well.  A repeated patch in the batch gives identical
  logits."""
  from ffn_b200 import engine as eng
  fov, depth, scale, n = case
  # at depth 16 the residual convolutions are scaled down further (x0.25, max |logit| 9 instead of 23): at x0.5 two
  # correct fp16-operand evaluations that differ only in accumulation order already disagree by 2.5e-3 relative
  w, b = random_stack(depth, 1000 + depth * 7 + sum(fov), scale=scale, b_scale=0.25 if depth >= 16 else 0.5)
  rng = np.random.RandomState(sum(fov) + depth)
  seeds, imgs = make_patches(fov, n, rng)
  if n > 1:                                         # batch of n + 1: the first pair again
    seeds, imgs = np.concatenate([seeds, seeds[:1]]), np.concatenate([imgs, imgs[:1]])
  want = oracle_logits(w, b, seeds, imgs)
  want16 = oracle_logits(w, b, seeds, imgs, operand_round='fp16')
  norm = max(1.0, float(np.abs(want).max()))
  e = eng.Engine(w, b, fov, tuple(s // 2 for s in fov), compute_mode=_mode_id('fp32'))
  info = e.info()
  for mode in MODES:
    e.set_compute_mode(_mode_id(mode))
    got = e.predict(seeds, imgs)
    assert np.isfinite(got).all()
    err = float(np.abs(got - want).max())
    line = 'parity %-14s depth %2d w x%-4g %-4s grid %3d tiles %4d: max err %.3g, rel %.3g (max |oracle| %.3g)' % (
        'x'.join(map(str, fov)), depth, scale, mode, info['grid'], info['tiles'], err, err / norm, norm)
    if mode == 'tc':
      err16 = float(np.abs(got - want16).max())
      line += '; vs fp16-operand oracle %.3g, rel %.3g' % (err16, err16 / norm)
    print(line)
    if n > 1:
      np.testing.assert_array_equal(got[-1], got[0])
    if mode == 'tc':
      assert err16 <= TC_TOL_FP16_ORACLE * norm, (mode, err16)
      assert err <= TC_TOL_F64_ORACLE * norm, (mode, err)
    else:
      assert err <= PARITY_TOL * norm, (mode, err)
  e.close()


# ----------------------------------------------------------------------------------------------------------------
# 3. Grid, tiles-per-CTA and chain invariance
# ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def fib25(golden_dir):
  from ffn_b200 import tf_checkpoint
  return tf_checkpoint.load_convstack_npz(os.path.join(golden_dir, 'fib25_convstack.npz'))


def _grid_sweep(e, seeds, imgs, grids, label):
  ref = e.predict(seeds, imgs)                      # default grid, default chains
  for grid in grids:
    e.set_grid(grid)
    tiles = -(-e.info()['tiles'] // grid)
    for chains in (1, 0):
      e.set_chains(chains)
      got = e.predict(seeds, imgs)
      same = np.array_equal(got, ref)
      print('%s grid %3d (%2d tiles/CTA) chains %s: %s' % (label, grid, tiles, chains or 'default',
                                                          'identical' if same else 'DIFFERS by %.3g' %
                                                          float(np.abs(got - ref).max())))
      assert same, (label, grid, chains)
  e.set_grid(0)
  e.set_chains(0)


@gpu
@pytest.mark.parametrize('mode', ['tc', 'x2'])
def test_grid_and_chains_do_not_change_predict(fib25, golden_dir, mode):
  """33^3 (294 tiles), FIB-25 depth 12, a 9-patch batch: bit-identical from 148 CTAs down to 30 (10 tiles per
  CTA: TMEM full), with one chain and with the default; a grid of 29 is refused."""
  from ffn_b200 import engine as eng
  w, b = fib25
  pat = np.load(os.path.join(golden_dir, 'net_patches.npz'))
  seeds = np.concatenate([pat['seed'], pat['seed'][:4][::-1]])
  imgs = np.concatenate([pat['image'], pat['image'][1:5]])
  e = eng.Engine(w, b, (33, 33, 33), (8, 8, 8), compute_mode=_mode_id(mode))
  info = e.info()
  assert info['tiles'] == 294
  grids = [g for g in (148, 147, 98, 74, 59, 49, 42, 37, 33, 30) if g <= info['sm_count']]
  _grid_sweep(e, seeds, imgs, grids, '33^3 %s' % mode)
  with pytest.raises(RuntimeError, match='tiles per CTA'):
    e.set_grid(29)
  np.testing.assert_array_equal(e.predict(seeds[:2], imgs[:2]), e.predict(seeds, imgs)[:2])
  e.close()


@gpu
@pytest.mark.parametrize('mode', ['tc', 'x2'])
def test_grid_and_chains_do_not_change_predict_65(mode):
  """(65,65,33): 1124 tiles, 8 per CTA at the default grid; the smallest legal grid runs 10."""
  from ffn_b200 import engine as eng
  fov = (65, 65, 33)
  w, b = random_stack(2, 65)
  seeds, imgs = make_patches(fov, 9, np.random.RandomState(65))
  e = eng.Engine(w, b, fov, (8, 8, 8), compute_mode=_mode_id(mode))
  nt = e.info()['tiles']
  assert nt == geom(fov)[2]
  smallest = -(-nt // MAX_TILES_PER_CTA)
  _grid_sweep(e, seeds, imgs, [smallest], '65x65x33 %s' % mode)
  with pytest.raises(RuntimeError, match='tiles per CTA'):
    e.set_grid(smallest - 1)
  e.close()


# ----------------------------------------------------------------------------------------------------------------
# 4. The flood loop away from 33^3
# ----------------------------------------------------------------------------------------------------------------
def _image(vol):
  return (vol.astype(np.float32) - np.float32(128.0)) / np.float32(33.0)


def _run_segment_all(e, vol, seeds, chains, **opts):
  from ffn_b200 import _lib, engine as eng
  e.set_chains(chains)
  cv = eng.DeviceCanvas(e, vol, eng.make_options(**opts), 128.0, 33.0)
  origins, overlaps, ctr = cv.segment_all(seeds)
  out = dict(seg=cv.read(_lib.ARRAY_SEGMENTATION), seed=cv.read(_lib.ARRAY_SEED), qprob=cv.read(_lib.ARRAY_QPROB),
             origins=[(o.id, tuple(o.start_zyx), o.iters) for o in origins],
             overlaps=sorted((o.id, o.other_id, o.count) for o in overlaps),
             ctr={n: getattr(ctr, n) for n, _ in ctr._fields_ if n not in ('device_seconds', 'kernel_launches')})
  cv.close()
  e.set_chains(0)
  return out


def _flood_case(e, vol, seeds, fov, deltas, chains, min_steps, min_objects, min_segment_size=1000):
  """Device segment_all with 2.. chains == the sequential device loop (bit for bit) == the oracle loop driven by
  the same device network (labels, seed, origins, overlaps, counters; qprob within the expf / expit bin edge)."""
  one = _run_segment_all(e, vol, seeds, 1, min_segment_size=min_segment_size)
  for k in chains:
    if k == 1:
      continue
    many = _run_segment_all(e, vol, seeds, k, min_segment_size=min_segment_size)
    for key in ('seg', 'qprob', 'seed'):
      np.testing.assert_array_equal(many[key], one[key], err_msg='%d chains: %s' % (k, key))
    assert many['origins'] == one['origins'] and many['overlaps'] == one['overlaps'] and many['ctr'] == one['ctr'], k
  hyb = ff.Canvas(lambda s, im: e.predict(s, im), _image(vol), fov, deltas, ff.Options(min_segment_size=min_segment_size))
  hyb.segment_all(seeds)
  np.testing.assert_array_equal(one['seg'], hyb.segmentation)
  np.testing.assert_array_equal(one['seed'], hyb.seed)
  qd = np.abs(one['qprob'].astype(int) - hyb.seg_prob.astype(int))
  assert qd.max() <= 1 and (qd > 0).mean() < 1e-3
  assert one['origins'] == [(k, v[0], v[1]) for k, v in sorted(hyb.origins.items())]
  want_ov = sorted((k, int(o), int(n)) for k, v in hyb.overlaps.items() for o, n in zip(v[0].tolist(), v[1].tolist()))
  assert one['overlaps'] == want_ov
  c = one['ctr']
  assert c['inference_calls'] == len(hyb.trace)
  assert c['skip_threshold'] == hyb.counters['skip_threshold']
  assert c['skip_invalid_pos'] == hyb.counters['skip_invalid_pos']
  print('flood %r deltas %r: %d FoV steps, %d objects, %d overlaps, %d voxels labelled; chains %r bit-exact' % (
      fov, deltas, c['inference_calls'], len(one['origins']), len(one['overlaps']), int((one['seg'] > 0).sum()),
      list(chains)))
  assert c['inference_calls'] >= min_steps and len(one['origins']) >= min_objects
  return one


def _cut(w, b, depth, lom_shift):
  """FIB-25 cut to its first `depth` modules.  The cut network was never trained at that depth and on the phantoms
  rejects nearly every object; raising its conv_lom bias by `lom_shift` makes it grow objects (accepted, too small
  and overlapping ones), which is what the loop comparisons need."""
  return w[:2 * depth] + [w[-1]], b[:2 * depth] + [b[-1] + np.float32(lom_shift)]


@gpu
def test_flood_configs4_geometry_with_chains(fib25):
  """BASELINE configs[4]: fov (17,33,33), deltas (4,8,8), depth 9, whole-canvas segment_all with 1-4 chains."""
  from ffn_b200 import _lib, engine as eng
  from ffn_b200.synthetic import voronoi_phantom
  w, b = _cut(*fib25, 9, 2.0)
  fov, deltas = (17, 33, 33), (4, 8, 8)
  vol = voronoi_phantom((40, 80, 80), seed=4, sigma=(0.5, 1.0, 1.0), voxel_size_zyx=(2.0, 1.0, 1.0), cell_volume=25000.0)
  seeds = ff.grid_seeds(vol.shape, step=12, offsets=(0, 6))
  e = eng.Engine(w, b, fov, deltas, compute_mode=_lib.COMPUTE_FP16_TC)
  _flood_case(e, vol, seeds, fov, deltas, (1, 2, 3, 4), min_steps=30, min_objects=3)
  e.close()


@gpu
@pytest.mark.parametrize('deltas', [(4, 4, 4), (0, 2, 2)], ids=['d444', 'd022'])
def test_flood_small_fov(fib25, deltas):
  """fov 9^3: deltas 4 put the faces on the FoV boundary; delta 0 means no z faces, and the done-lattice
  quantisation divides by max(delta, 1)."""
  from ffn_b200 import _lib, engine as eng
  from ffn_b200.synthetic import voronoi_phantom
  w, b = _cut(*fib25, 4, 5.0)
  fov = (9, 9, 9)
  vol = voronoi_phantom((36, 44, 52), seed=9, cell_volume=6000.0)
  seeds = ff.grid_seeds(vol.shape, step=7, offsets=(0, 3))
  e = eng.Engine(w, b, fov, deltas, compute_mode=_lib.COMPUTE_FP16_TC)
  _flood_case(e, vol, seeds, fov, deltas, (1, 4), min_steps=300, min_objects=3, min_segment_size=50)
  e.close()


@gpu
def test_flood_65x65x33_sequential_at_8_tiles_per_cta(fib25):
  """fov (65,65,33), deltas 8, depth 2: 8 tiles per CTA at 148 SMs, chain limit 1 (the sequential path)."""
  from ffn_b200 import _lib, engine as eng
  from ffn_b200.synthetic import voronoi_phantom
  w, b = _cut(*fib25, 2, 3.0)
  fov, deltas = (65, 65, 33), (8, 8, 8)
  vol = voronoi_phantom((84, 96, 64), seed=12, cell_volume=40000.0)
  seeds = ff.grid_seeds(vol.shape, step=16, offsets=(0, 8))
  e = eng.Engine(w, b, fov, deltas, compute_mode=_lib.COMPUTE_FP16_TC)
  print('65x65x33: %r' % e.info())
  _flood_case(e, vol, seeds, fov, deltas, (1, 4), min_steps=5, min_objects=3)
  e.close()


@gpu
def test_flood_golden64_at_10_tiles_per_cta(fib25, golden_dir):
  """33^3 with a 30-CTA grid (10 tiles per CTA, TMEM full) in the split-fp16 mode == the reference's own
  segment_all on the golden 64^3 volume."""
  from ffn_b200 import _lib, engine as eng
  g = np.load(os.path.join(golden_dir, 'flood_fill_64.npz'))
  w, b = fib25
  e = eng.Engine(w, b, (33, 33, 33), (8, 8, 8), compute_mode=_lib.COMPUTE_FP16X2_TC, num_ctas=30)
  assert e.info()['grid'] == 30
  cv = eng.DeviceCanvas(e, g['volume'], eng.make_options(), 128.0, 33.0)
  origins, overlaps, ctr = cv.segment_all(g['seeds'])
  seg = cv.read(_lib.ARRAY_SEGMENTATION)
  np.testing.assert_array_equal(seg, g['segmentation'])
  diff = np.abs(cv.read(_lib.ARRAY_QPROB).astype(int) - g['seg_prob'].astype(int))
  assert diff.max() <= 1 and (diff > 0).mean() < 1e-3
  got = np.array([[o.id] + list(o.start_zyx) + [o.iters] for o in origins], dtype=np.int64).reshape(-1, 5)
  np.testing.assert_array_equal(got, g['origins'])
  want_ov = sorted(zip(*g['overlaps'].tolist())) if g['overlaps'].size else []
  assert sorted((o.id, o.other_id, o.count) for o in overlaps) == [tuple(int(v) for v in t) for t in want_ov]
  gc = json.loads(str(g['counters']))
  assert ctr.inference_calls == gc['inference-calls']
  assert ctr.segment_at_calls == gc['segment_at-loop-calls']
  assert ctr.skip_threshold == gc.get('skip_threshold', 0)
  assert ctr.skip_invalid_pos == gc.get('skip_invalid_pos', 0)
  assert ctr.voxels_segmented == gc['voxels-segmented']
  assert ctr.voxels_overlapping == gc['voxels-overlapping']
  cv.close()
  e.close()


# ----------------------------------------------------------------------------------------------------------------
# 5. Clean rejection
# ----------------------------------------------------------------------------------------------------------------
@gpu
def test_rejected_geometries_raise_cleanly():
  """Geometries outside the engine's limits raise with the engine's message; a fresh engine works afterwards."""
  from ffn_b200 import _lib, engine as eng
  w1, b1 = random_stack(1, 3)
  cases = [
      ((3, 3, 35), (1, 1, 1), w1, b1, 'shared-memory'),          # x extent 35: 233 072 B of shared memory
      ((3, 3, 4), (1, 1, 1), w1, b1, 'odd'),
      ((1, 3, 3), (0, 1, 1), w1, b1, 'odd and >= 3'),
      ((5, 5, 5), (1, 3, 1), w1, b1, r'deltas must lie in \[0, fov // 2\]'),
  ]
  for fov, deltas, w, b, msg in cases:
    with pytest.raises(RuntimeError, match=msg):
      eng.Engine(w, b, fov, deltas)
  w17, b17 = random_stack(17, 3)
  with pytest.raises(RuntimeError, match='unsupported depth'):
    eng.Engine(w17, b17, (5, 5, 5), (1, 1, 1))
  with pytest.raises(RuntimeError, match='unsupported depth'):
    eng.Engine(w1[-1:], b1[-1:], (5, 5, 5), (1, 1, 1))             # depth 0: conv_lom only
  e = eng.Engine(w1, b1, (5, 5, 5), (1, 1, 1), compute_mode=_lib.COMPUTE_FP32)
  with pytest.raises(RuntimeError, match='at most 4 chains'):
    e.set_chains(5)
  seeds, imgs = make_patches((5, 5, 5), 2, np.random.RandomState(0))
  got = e.predict(seeds, imgs)
  assert np.abs(got - oracle_logits(w1, b1, seeds, imgs)).max() <= PARITY_TOL * 10
  e.close()
