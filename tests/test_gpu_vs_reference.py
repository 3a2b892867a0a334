"""This repo's kernels AND the oracle's restatements of the CUDA-only reference ops against what the reference's OWN CUDA
kernels (the unmodified reference ops, compiled for sm_100a by oracle/build_ref.py) returned on the same inputs on a B200:
tests/golden/ref_gpu_kernels.npz (tests/golden/make_reference_golden.py). Neighbour lists are stored as lengths + digest."""
import os
import sys

import numpy as np
import pytest
import torch

import oracle
from softgroup_b200 import ops

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, 'golden'))
from digest import digest, lists_digest  # noqa: E402

pytestmark = pytest.mark.gpu

BALLQUERY_CASES = [(3000, 0.03, 0.04), (2500, 0.006, 0.04), (4000, 0.2, 0.02)]


@pytest.fixture(scope='module')
def gold():
    return np.load(os.path.join(HERE, 'golden', 'ref_gpu_kernels.npz'))


def _c(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _lists(idx, sl):
    idx, sl = idx.cpu().numpy(), sl.cpu().numpy()
    return [idx[s:s + l] for s, l in sl]


def _assert_lists(got, gold, key):
    lens, dig = lists_digest(got)
    assert np.array_equal(lens, gold[key + '_lens']), key
    assert dig == str(gold[key + '_digest']), key


def ballquery_inputs(n, sigma):
    rng = np.random.RandomState(n)
    centers = rng.rand(6, 3)
    xyz = (centers[rng.randint(0, 6, n)] + rng.randn(n, 3) * sigma).astype(np.float32)
    cut = n // 3
    bo = np.array([0, cut, n], np.int32)
    bi = np.repeat(np.arange(2), np.diff(bo)).astype(np.int32)
    return xyz, bi, bo


def nonfinite_inputs():
    rng = np.random.RandomState(7)
    n = 3000
    xyz = (rng.rand(4, 3)[rng.randint(0, 4, n)] + rng.randn(n, 3) * 0.02).astype(np.float32)
    bad = rng.choice(n, 40, replace=False)
    xyz[bad[:15], rng.randint(0, 3, 15)] = np.nan
    xyz[bad[15:30], rng.randint(0, 3, 15)] = np.inf
    xyz[bad[30:], rng.randint(0, 3, 10)] = -np.inf
    return xyz, np.zeros(n, np.int32), np.array([0, n], np.int32), bad


def voxelize_inputs():
    rng = np.random.RandomState(1)
    coords = np.concatenate([np.zeros((20000, 1), np.int64), rng.randint(0, 30, (20000, 3))], 1)
    _, _, om = oracle.voxelization_idx(coords, 1, 4)
    feats = rng.randn(20000, 32).astype(np.float32)
    return feats, om


def segment_inputs():
    rng = np.random.RandomState(2)
    lens = rng.randint(1, 700, 40)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    x = rng.randn(off[-1], 32).astype(np.float32)
    return x, off


def mask_inputs():
    rng = np.random.RandomState(3)
    N, nI, nP = 4000, 17, 25
    labels = rng.randint(-1, nI, N).astype(np.int64)
    labels[labels < 0] = -100
    pointnum = np.bincount(labels[labels >= 0], minlength=nI).astype(np.int32)
    cls = rng.randint(0, 18, nI).astype(np.int64)
    cls[3] = -100
    lens = rng.randint(1, 300, nP)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    pidx = rng.randint(0, N, off[-1]).astype(np.int32)
    sig = rng.rand(off[-1]).astype(np.float32)
    return pidx, off, labels, pointnum, cls, sig


def octree_inputs():
    rng = np.random.RandomState(4)
    return (rng.rand(3000, 3) * np.array([3., 2., 1.])).astype(np.float32)


@pytest.mark.parametrize('n,sigma,r', BALLQUERY_CASES)
def test_ballquery_vs_reference_kernel(gold, n, sigma, r):
    xyz, bi, bo = ballquery_inputs(n, sigma)
    gidx, gsl = ops.ballquery_batch_p(_c(xyz), _c(bi), _c(bo), r, 100)
    oidx, osl = oracle.ballquery_batch_p(xyz, bi, bo, r)
    G = _lists(gidx, gsl)
    O = [oidx[s:s + l] for s, l in osl]
    _assert_lists(G, gold, 'bq%d' % n)  # ours == reference kernel
    for i in range(n):
        assert np.array_equal(G[i], O[i]), i  # oracle restatement == ours == reference kernel (pins the oracle)


def test_ballquery_nonfinite_points_vs_reference_kernel(gold):
    """NaN / Inf coordinates (a diverged offset head): the reference kernel gives such a point the empty list and nobody
    lists it, every comparison with it being false (bfs_cluster.cu:38-44). Same here, blocking AND asynchronous entry
    points (round-1 advice: the async path left start_len rows of dropped points uninitialised); the clustering
    downstream then sees isolated nodes."""
    from softgroup_b200.ops import ballquery_batch_p_nosync, bfs_cluster_segments
    xyz, bi, bo, bad = nonfinite_inputs()
    n = xyz.shape[0]
    gidx, gsl = ops.ballquery_batch_p(_c(xyz), _c(bi), _c(bo), 0.04, 100)
    oidx, osl = oracle.ballquery_batch_p(xyz, bi, bo, 0.04)
    G = _lists(gidx, gsl)
    O = [oidx[s:s + l] for s, l in osl]
    _assert_lists(G, gold, 'bq_nonfinite')
    for i in range(n):
        assert np.array_equal(G[i], O[i]), i
    assert all(len(G[i]) == 0 for i in bad)
    # asynchronous entry point used by the fused forward + clustering on its lists
    aidx, asl, tot = ballquery_batch_p_nosync(_c(xyz), _c(bi), _c(bo), 0.04)
    A = _lists(aidx, asl)
    for i in range(n):
        assert np.array_equal(A[i], O[i]), i
    assert int(tot[0]) == oidx.size and int(tot[1]) == 0
    cidx, coff = bfs_cluster_segments(aidx, asl, 10.0, nactive=tot[0:1], upstream_err=tot[1:2])
    mean = np.full(20, -1, np.float32)
    wi, wo = oracle.bfs_cluster(mean, oidx, osl, 10.0, 3)
    assert np.array_equal(cidx.cpu().numpy(), wi) and np.array_equal(coff.cpu().numpy(), wo)


def test_ballquery_out_of_range_is_reported():
    """A finite coordinate beyond the addressable cell range is a limit of this implementation: SGB_ERR_RANGE from the
    blocking call, and from the clustering call downstream of the asynchronous one (never silent garbage)."""
    from softgroup_b200.ops import ballquery_batch_p_nosync, bfs_cluster_segments
    from softgroup_b200.ops._lib import SgbError
    xyz = np.random.RandomState(0).rand(500, 3).astype(np.float32)
    xyz[17, 1] = 1e7
    bi, bo = np.zeros(500, np.int32), np.array([0, 500], np.int32)
    with pytest.raises(SgbError):
        ops.ballquery_batch_p(_c(xyz), _c(bi), _c(bo), 0.04, 100)
    aidx, asl, tot = ballquery_batch_p_nosync(_c(xyz), _c(bi), _c(bo), 0.04)
    with pytest.raises(SgbError):
        bfs_cluster_segments(aidx, asl, 10.0, nactive=tot[0:1], upstream_err=tot[1:2])


def test_voxelize_fp_vs_reference_kernel(gold):
    feats, om = voxelize_inputs()
    ours = ops.voxelization(_c(feats), _c(om), 4).cpu().numpy()
    assert digest(ours) == str(gold['voxelize_fp_digest'])
    assert np.array_equal(ours, oracle.voxelization(feats, om, 4))


def test_segment_ops_vs_reference_kernels(gold):
    x, off = segment_inputs()
    xc, oc = _c(x), _c(off)
    for name in ('sec_min', 'sec_max', 'sec_mean'):
        want = gold[name]
        assert np.array_equal(want, getattr(oracle, name)(x, off)), name  # oracle == reference kernel
        got = getattr(ops, name)(xc, oc).cpu().numpy()
        if name == 'sec_mean':
            np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-6)
        else:
            assert np.array_equal(got, want)
    want = gold['global_avg_pool_fp']
    assert np.array_equal(want, oracle.global_avg_pool(x, off))
    np.testing.assert_allclose(ops.global_avg_pool(xc, oc).cpu().numpy(), want, rtol=1e-5, atol=1e-6)


def test_mask_ops_vs_reference_kernels(gold):
    pidx, off, labels, pointnum, cls, sig = mask_inputs()
    iou = ops.get_mask_iou_on_cluster(_c(pidx), _c(off), _c(labels), _c(pointnum))
    assert np.array_equal(gold['mask_iou_on_cluster'], iou.cpu().numpy())
    assert np.array_equal(gold['mask_iou_on_cluster'], oracle.get_mask_iou_on_cluster(pidx, off, labels, pointnum))
    assert np.array_equal(gold['mask_iou_on_pred'],
                          ops.get_mask_iou_on_pred(_c(pidx), _c(off), _c(labels), _c(pointnum), _c(sig)).cpu().numpy())
    ours = ops.get_mask_label(_c(pidx), _c(off), _c(labels), _c(cls), _c(pointnum), iou, 0.02)
    assert np.array_equal(gold['mask_label'], ours.cpu().numpy())


def test_octree_oracle_vs_reference_kernel(gold):
    """Pins the oracle's octree ball query (leaf-major order, box/sphere test contraction) on the reference kernel."""
    pts = octree_inputs()
    oidx, osl = oracle.octree_ball_query(pts, 50, 0.15)
    _assert_lists([oidx[s:s + l] for s, l in osl], gold, 'octree')
