"""N2 (SURVEY.md 8f): the GPU test-time data preparation (harness.prepare_test_batch_gpu: rotation, scale, shift,
truncation, batch column, spatial shape, point->voxel hash; S3DIS x4 split) against what the reference's OWN dataset code
-- CustomDataset.transform_test / __getitem__ / collate_fn (softgroup/data/custom.py:162-256) and S3DISDataset
(softgroup/data/s3dis.py:46-115), run on the host -- returned for the same raw scans: tests/golden/ref_host.json
(digests of the collated tensors; tests/golden/make_reference_golden.py)."""
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from softgroup_b200 import harness, synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
from digest import digest  # noqa: E402

pytestmark = pytest.mark.gpu

COLLATE_SIZES = [2000, 150000]
TENSOR_KEYS = ('voxel_coords', 'v2p_map', 'p2v_map', 'coords_float', 'feats', 'batch_idxs', 'semantic_labels', 'coords')


def raw_scan(seed, n, shape='c2_scannet'):
    """raw, mean-centred float32 points like prepare_data_inst.py:55-56 (before any test transform)."""
    scan = synth.make_scan(shape, seed=seed, n_points=n)
    rng = np.random.RandomState(seed)
    xyz = (rng.rand(n, 3) * np.array([7, 5, 2.6])).astype(np.float32)
    xyz -= xyz.mean(0)
    rgb = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
    sem = scan['semantic_labels'].astype(np.int64)
    ins = scan['instance_labels'].astype(np.int64).copy()
    ins[ins < 0] = -100
    return xyz, rgb, sem, ins


def reference_collate(cls, raw, x4_split=None):
    """The reference dataloader's output for one raw scan: `cls` is the reference's CustomDataset or S3DISDataset."""
    ds = object.__new__(cls)
    ds.voxel_cfg = SimpleNamespace(scale=50, spatial_shape=[128, 512], max_npoint=250000, min_npoint=5000)
    ds.training = False
    ds.filenames = ['scene0000_00_inst_nostuff.pth']
    ds.suffix = '_inst_nostuff.pth'
    ds.load = lambda filename: tuple(a.copy() for a in raw)
    if x4_split is not None:
        ds.x4_split = x4_split
    return ds.collate_fn([ds[0]])


def batch_record(batch):
    """Digests of the collated tensors (dtype, shape and bytes; labels and raw coordinates by value, as int64), spatial
    shape and batch size."""
    rec = {}
    for k in TENSOR_KEYS:
        if k in batch:
            a = batch[k].cpu().numpy()
            rec[k] = digest(a.astype(np.int64) if k in ('semantic_labels', 'coords') else a)
    rec['spatial_shape'] = np.asarray(batch['spatial_shape']).tolist()
    rec['batch_size'] = int(batch['batch_size'])
    return rec


def _check(want, batch_gpu):
    got = batch_record(batch_gpu)
    assert sorted(got) == sorted(want)
    for k in want:
        assert got[k] == want[k], k


@pytest.mark.parametrize('n', COLLATE_SIZES)
def test_transform_collate_matches_reference_dataset(host_gold, n):
    raw = raw_scan(1, n)
    got = harness.prepare_test_batch_gpu(raw[0], raw[1], raw[2], raw[3], scale=50, min_spatial_shape=128)
    _check(host_gold['collate_%d' % n], got)


def test_x4_split_matches_reference_s3dis_dataset(host_gold):
    raw = raw_scan(2, 40003, shape='c3_s3dis')  # not a multiple of 4: the pieces have different lengths
    got = harness.prepare_test_batch_gpu(raw[0], raw[1], raw[2], raw[3], scale=50, min_spatial_shape=128, x4_split=True)
    want = dict(host_gold['collate_x4'])
    want.pop('coords', None)  # the x4 test compared the collated tensors without the raw coords
    got.pop('coords', None)
    _check(want, got)
