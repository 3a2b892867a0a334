"""CPU: the oracle (oracle/sg_oracle.c) against the golden vectors produced by the compiled reference, and against what
the compiled reference returned on the fresh inputs built below (tests/golden/ref_host.json, digests;
tests/golden/make_reference_golden.py)."""
import os
import sys

import numpy as np
import pytest

import oracle
from softgroup_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
from digest import digest  # noqa: E402

FRESH_BFS_THRESHOLDS = [(0.5, 5), (2.0, 5), (3.0, 0)]


def test_voxelize_idx_golden_c1(golden):
    oc, im, om = oracle.voxelization_idx(golden['vox_c1_coords'], 1, 4)
    assert np.array_equal(oc, golden['vox_c1_out_coords'])
    assert np.array_equal(im, golden['vox_c1_input_map'])
    assert np.array_equal(om, golden['vox_c1_output_map'])


@pytest.mark.parametrize('mode', [1, 2, 3, 4])
def test_voxelize_idx_golden_ragged(golden, mode):
    oc, im, om = oracle.voxelization_idx(golden['vox_rag_coords'], 2, mode)
    assert np.array_equal(oc, golden['vox_rag_m%d_out_coords' % mode])
    assert np.array_equal(im, golden['vox_rag_m%d_input_map' % mode])
    assert np.array_equal(om, golden['vox_rag_m%d_output_map' % mode])


def test_bfs_cluster_golden(golden):
    mean = golden['class_numpoint_mean']
    for k in range(int(golden['bfs_count'])):
        ci, co = oracle.bfs_cluster(mean, golden['bfs%d_idx' % k], golden['bfs%d_sl' % k], float(golden['bfs%d_thr' % k]),
                                    int(golden['bfs%d_cls' % k]))
        assert np.array_equal(ci, golden['bfs%d_cidx' % k]), k
        assert np.array_equal(co, golden['bfs%d_coff' % k]), k


def test_octree_build_golden(golden):
    boxes, pt_inds, psl = oracle.build_octree(golden['oct_pts'])
    assert np.array_equal(boxes, golden['oct_boxes'])
    assert np.array_equal(pt_inds, golden['oct_pt_inds'])
    assert np.array_equal(psl, golden['oct_psl'])


def test_ballquery_properties():
    """No CPU reference exists for ballquery_batch_p; check the restatement against a float64 brute force away
    from the boundary, plus ordering / cap / self-inclusion."""
    rng = np.random.RandomState(0)
    xyz = (rng.rand(600, 3) * 0.5).astype(np.float32)
    bi = np.concatenate([np.zeros(400, np.int32), np.ones(200, np.int32)])
    bo = np.array([0, 400, 600], np.int32)
    r = 0.06
    idx, sl = oracle.ballquery_batch_p(xyz, bi, bo, r)
    d = np.linalg.norm(xyz[:, None].astype(np.float64) - xyz[None].astype(np.float64), axis=2)
    for i in range(600):
        lst = idx[sl[i, 0]:sl[i, 0] + sl[i, 1]]
        assert np.all(np.diff(lst) > 0) and i in lst
        seg = np.arange(bo[bi[i]], bo[bi[i] + 1])
        sure = seg[d[i, seg] < r * (1 - 1e-5)]
        maybe = seg[d[i, seg] < r * (1 + 1e-5)]
        assert set(sure) <= set(lst) <= set(maybe)


def test_ballquery_cap():
    xyz = np.zeros((1500, 3), np.float32)
    idx, sl = oracle.ballquery_batch_p(xyz, np.zeros(1500, np.int32), np.array([0, 1500], np.int32), 0.1)
    assert np.all(sl[:, 1] == 1000)
    assert np.array_equal(idx[:1000], np.arange(1000))


def fresh_inputs():
    """A hashed scan and random asymmetric graphs incl. duplicates inside a list: (coords, class means, [(n, idx, sl)])."""
    scan = synth.make_scan('c1_plumbing', seed=3, n_points=5000)
    rng = np.random.RandomState(5)
    mean = np.full(20, -1, np.float32)
    graphs = []
    for t in range(20):
        n = rng.randint(5, 120)
        lens = rng.randint(0, 6, n)
        idx = rng.randint(0, n, int(lens.sum()) + 1).astype(np.int32)
        sl = np.stack([np.concatenate([[0], np.cumsum(lens)[:-1]]), lens], 1).astype(np.int32)
        graphs.append((n, idx, sl))
    return scan['coords'], mean, graphs


def fresh_more_inputs(seed):
    """-> (batched coords, (points, ball-query lists, start_len, class means), clustered cloud for the octree)."""
    rng = np.random.RandomState(100 + seed)
    # voxelize_idx: 3 batch items (one empty), heavy duplication
    n = 4000
    b = rng.choice([0, 2], n)  # batch item 1 stays empty
    xyz = rng.randint(0, 12, (n, 3))
    coords = np.concatenate([b[:, None], xyz], 1).astype(np.int64)
    coords = coords[np.argsort(b, kind='stable')]
    pts = (rng.rand(700, 3) * np.array([1.0, 1.0, 0.3])).astype(np.float32)
    idx, sl = oracle.ballquery_batch_p(pts, np.zeros(700, np.int32), np.array([0, 700], np.int32), 0.09)
    mean = np.full(20, -1, np.float32)
    mean[5] = 40.0
    cl = (rng.randn(3000, 3) * 0.2 + rng.randint(0, 4, (3000, 1))).astype(np.float32)
    return coords, (pts, idx, sl, mean), cl


def _digests(arrays):
    return [digest(a) for a in arrays]


def test_vs_reference_fresh(host_gold):
    coords, mean, graphs = fresh_inputs()
    assert _digests(oracle.voxelization_idx(coords, 1, 4)) == host_gold['fresh_vox']
    for (n, idx, sl), want in zip(graphs, host_gold['fresh_bfs']):
        assert _digests(oracle.bfs_cluster(mean, idx, sl, 2.0, 0)) == want
    assert len(graphs) == len(host_gold['fresh_bfs'])


@pytest.mark.parametrize('seed', range(4))
def test_vs_reference_fresh_more(host_gold, seed):
    """More fresh-input comparisons with the compiled reference: batched hashing with duplicates and empty batches,
    class-mean (relative) BFS thresholds, octree build on clustered points."""
    coords, (pts, idx, sl, mean), cl = fresh_more_inputs(seed)
    for mode, want in zip((1, 2, 3, 4), host_gold['more%d_vox' % seed]):
        assert _digests(oracle.voxelization_idx(coords, 3, mode)) == want, mode
    # bfs_cluster with relative thresholds (threshold * class mean, bfs_cluster.cpp:70-77) on ball-query graphs
    for (thr, cls), want in zip(FRESH_BFS_THRESHOLDS, host_gold['more%d_bfs' % seed]):
        assert _digests(oracle.bfs_cluster(mean, idx, sl, thr, cls)) == want, (thr, cls)
    # octree build (octree_ball_query.cpp:19-165)
    assert _digests(oracle.build_octree(cl)) == host_gold['more%d_octree' % seed]
