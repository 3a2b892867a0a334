"""Host-side methods of the model against what the REFERENCE'S OWN methods returned on the same inputs: the unmodified
reference SoftGroup class, instantiated on this repo's shims on CPU, had its CUDA-free methods called directly --
panoptic_fusion (softgroup.py:606-639), get_gt_instances (:641-653), merge_4_parts (:397-409), pyramid_inverse_map
(:500-507, dense matrix), get_level (:482-489). Results: tests/golden/ref_host.{npz,json}
(tests/golden/make_reference_golden.py)."""
import numpy as np
import pytest
import torch

from softgroup_b200.configs import model_cfg
from softgroup_b200.model import SoftGroup
from softgroup_b200.util import rle_encode

LEVEL_SIZES = (5, 100000, 100001, 1000000, 1000001)


def _ours(name):
    return SoftGroup(**model_cfg(name, channels=16, num_blocks=2)).eval()


def panoptic_inputs(seed):
    rng = np.random.RandomState(seed)
    n = 800
    sem = rng.randint(0, 19, n)
    insts = []
    for _ in range(15):
        lo = rng.randint(0, n - 60)
        m = np.zeros(n, np.int64)
        m[lo:lo + rng.randint(5, 60)] = rng.rand() < 0.9  # overlapping runs -> the skip rule triggers
        insts.append(dict(scan_id='s', label_id=int(rng.randint(1, 9)), conf=float(rng.rand()), pred_mask=rle_encode(m)))
    return sem, insts


def gt_instances_inputs():
    rng = np.random.RandomState(0)
    sem = torch.from_numpy(rng.randint(-1, 20, 500)).long()
    sem[sem == -1] = -100
    inst = torch.from_numpy(rng.randint(-1, 12, 500)).long()
    inst[inst == -1] = -100
    return sem, inst


def merge_inputs():
    return torch.arange(4 * 7 * 3, dtype=torch.float32).view(28, 3)


def pyramid_inputs():
    """-> (proposals_idx, proposals_offset, number of voxels, level-to-point map)."""
    rng = np.random.RandomState(1)
    n_vox, n_pts = 60, 400
    l2p = torch.from_numpy(rng.randint(0, n_vox, n_pts).astype(np.int32))
    members = rng.permutation(n_vox)[:45]  # a voxel belongs to at most one cluster
    cut = [0, 10, 11, 30, 45]
    pidx = torch.tensor([[c, int(v)] for c in range(4) for v in members[cut[c]:cut[c + 1]]], dtype=torch.int32)
    poff = torch.tensor(cut, dtype=torch.int32)
    return pidx, poff, n_vox, l2p


@pytest.mark.parametrize('seed', range(3))
def test_panoptic_fusion(host_arrays, seed):
    sem, insts = panoptic_inputs(seed)
    want = host_arrays['panoptic_fusion_%d' % seed]
    got = _ours('kitti').panoptic_fusion(sem.copy(), insts)
    assert got.dtype == want.dtype and np.array_equal(got, want)


def test_get_gt_instances(host_arrays):
    sem, inst = gt_instances_inputs()
    got = _ours('scannet').get_gt_instances(sem.clone(), inst.clone())
    assert np.array_equal(got, host_arrays['gt_instances'])


def test_merge_4_parts(host_arrays):
    assert torch.equal(_ours('s3dis').merge_4_parts(merge_inputs()), torch.from_numpy(host_arrays['merge_4_parts']))


def test_pyramid_inverse_map_and_level(host_arrays, host_gold):
    ours = _ours('stpls3d++')
    for n in LEVEL_SIZES:
        assert ours.get_level(n) == host_gold['get_level'][str(n)]
    got_idx, got_off = ours.pyramid_inverse_map(*pyramid_inputs())
    assert np.array_equal(got_idx.numpy(), host_arrays['pyramid_inverse_idx'].astype(np.int32))
    assert np.array_equal(got_off.numpy(), host_arrays['pyramid_inverse_off'])
