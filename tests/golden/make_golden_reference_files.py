"""Small stand-ins for two data files of the reference checkout, so that the tests reading them run anywhere:

    python tests/golden/make_golden_reference_files.py <reference checkout>

  fib25_ckpt.npz          models/fib25/model.ckpt-27465036: the `.index` file verbatim, the bytes of the data shard that
                          are not seed_update weights (fib25_convstack.npz holds those), the shard's size and SHA-256.
                          With fib25_convstack.npz this rebuilds the checkpoint byte for byte.
  sample_training2_ref.npz
                          results/fib25/sample-training2.npz: its `origins.npy` member verbatim (a Python-2 pickle of
                          OriginInfo under the original module path) and the segmentation labels at a fixed, seeded
                          sample of voxels plus every origin's start voxel (the whole 250^3 array is ~1 MB compressed).
"""
import hashlib
import os
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)

CKPT = 'models/fib25/model.ckpt-27465036'
RESULT = 'results/fib25/sample-training2.npz'
SAMPLE_VOXELS = 4096


def checkpoint_fixture(ref):
  from ffn_b200 import tf_checkpoint
  prefix = os.path.join(ref, CKPT)
  with open(prefix + '.index', 'rb') as f:
    index = f.read()
  with open(prefix + '.data-00000-of-00001', 'rb') as f:
    data = f.read()
  spans = sorted((e['offset'], e['offset'] + e['size'], name)
                 for name, e in tf_checkpoint.list_variables(prefix).items())
  other_offsets, other_bytes = [], []
  for lo, hi, name in spans:
    if not name.startswith('seed_update/'):
      other_offsets.append([lo, hi])
      other_bytes.append(np.frombuffer(data[lo:hi], np.uint8))
  np.savez_compressed(os.path.join(HERE, 'fib25_ckpt.npz'),
                      index=np.frombuffer(index, np.uint8),
                      other_offsets=np.asarray(other_offsets, np.int64),
                      other_bytes=np.concatenate(other_bytes),
                      data_size=np.int64(len(data)),
                      data_sha256=np.array(hashlib.sha256(data).hexdigest()))
  print('wrote fib25_ckpt.npz: %d index bytes, %d other tensor bytes' % (len(index), sum(map(len, other_bytes))))


def sample_result_fixture(ref):
  from ffn_b200.inference import storage
  path = os.path.join(ref, RESULT)
  with zipfile.ZipFile(path) as z:
    origins_npy = z.read('origins.npy')
  seg = np.load(path)['segmentation']
  origins = storage._load_origins(np.load(path, allow_pickle=True), path)
  starts = np.ravel_multi_index(np.asarray([o.start_zyx for o in origins.values()]).T, seg.shape)
  rng = np.random.RandomState(0)
  index = np.union1d(rng.choice(seg.size, SAMPLE_VOXELS, replace=False), starts).astype(np.int64)
  np.savez_compressed(os.path.join(HERE, 'sample_training2_ref.npz'),
                      origins_npy=np.frombuffer(origins_npy, np.uint8),
                      shape=np.asarray(seg.shape, np.int64), dtype=np.array(seg.dtype.str),
                      sample_index=index, sample_labels=seg.ravel()[index])
  print('wrote sample_training2_ref.npz: %d origins, %d sampled voxels' % (len(origins), index.size))


def main():
  if len(sys.argv) != 2:
    raise SystemExit(__doc__)
  checkpoint_fixture(sys.argv[1])
  sample_result_fixture(sys.argv[1])


if __name__ == '__main__':
  main()
