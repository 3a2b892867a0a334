"""forward_grouping host logic on CPU: the one-launch segmented restructure (softgroup_b200/model/softgroup.py) against
the reference's per-class loop (softgroup/model/softgroup.py:411-480). The two device ops it calls are replaced by
stand-ins built on the oracle (the CPU checker), so only the Python restructuring is under test here -- class-major
entry order, segment ids, per-segment thresholds in float32, index mapping back to points, proposal concatenation."""
import numpy as np
import pytest
import torch

import oracle
from softgroup_b200 import synth
from softgroup_b200.configs import model_cfg
from softgroup_b200.model import SoftGroup
from softgroup_b200.model import softgroup as sg_module


def _fake_ballquery_nosync(coords, batch_idxs, batch_offsets, radius):
    idx, sl = oracle.ballquery_batch_p(coords.numpy(), batch_idxs.numpy(), batch_offsets.numpy(), radius)
    return (torch.from_numpy(idx.astype(np.int32)), torch.from_numpy(sl.astype(np.int32)),
            torch.tensor([idx.size, 0], dtype=torch.int32))


def _fake_group_entries(scores, classes, score_thr, min_npoint, batch_idxs, batch_size, coords_float, pt_offsets):
    """CPU stand-in of csrc/grouping.cu written as the reference's own per-class loop (softgroup.py:430-446)."""
    pts, seg, counts = [], [], []
    for r, c in enumerate(classes):
        obj = (scores[:, c] > score_thr).nonzero().view(-1)
        if obj.size(0) < min_npoint:
            counts.append(0)
            continue
        counts.append(obj.size(0))
        pts.append(obj)
        seg.append(r * batch_size + batch_idxs[obj].long())
    pts = torch.cat(pts).int() if pts else torch.zeros(0, dtype=torch.int32)
    seg = torch.cat(seg).int() if seg else torch.zeros(0, dtype=torch.int32)
    shifted = coords_float[pts.long()] + pt_offsets[pts.long()]
    seg_offsets = torch.zeros(len(classes) * batch_size + 1, dtype=torch.int32)
    seg_offsets[1:] = torch.bincount(seg.long(), minlength=len(classes) * batch_size).cumsum(0).int()
    total = torch.tensor([pts.numel()] + counts, dtype=torch.int32)
    return pts, seg, shifted, seg_offsets, total


def _fake_bfs_segments(ball_query_idxs, start_len, thr, node_seg=None, seg_thr=None, nactive=None, upstream_err=None):
    """bfs_cluster.cpp:33-126 over the whole node set with a per-seed-segment threshold (what the library computes)."""
    idxs, sl = ball_query_idxs.numpy(), start_len.numpy()
    n = sl.shape[0]
    seen = np.zeros(n, bool)
    cl, offs = [], [0]
    for i in range(n):
        if seen[i]:
            continue
        seen[i] = True
        queue, comp = [i], []
        while queue:
            u = queue.pop(0)
            comp.append(u)
            for v in idxs[sl[u, 0]:sl[u, 0] + sl[u, 1]]:
                if not seen[v]:
                    seen[v] = True
                    queue.append(int(v))
        t = np.float32(thr) if node_seg is None else np.float32(seg_thr[node_seg[i]])
        if np.float32(len(comp)) >= t:
            cid = len(offs) - 1
            cl += [(cid, u) for u in comp]
            offs.append(offs[-1] + len(comp))
    return (torch.tensor(cl, dtype=torch.int32).reshape(-1, 2), torch.tensor(offs, dtype=torch.int32))


def reference_forward_grouping(model, semantic_scores, pt_offsets, batch_idxs, coords_float):
    """The reference's loop, ops taken from the oracle (ballquery_batch_p: bfs_cluster.cu:15-101 restatement,
    bfs_cluster: the compiled reference's algorithm)."""
    g = model.grouping_cfg
    get = model._cfg
    bs = int(batch_idxs.max()) + 1
    scores = torch.from_numpy(semantic_scores).softmax(-1).numpy()
    mean = np.asarray(get(g, 'class_numpoint_mean'), np.float32)
    idx_list, off_list = [], []
    for class_id in range(model.semantic_classes):
        if class_id in get(g, 'ignore_classes'):
            continue
        obj = np.nonzero(scores[:, class_id] > get(g, 'score_thr'))[0]
        if obj.size < get(model.test_cfg, 'min_npoint'):
            continue
        b = batch_idxs[obj].astype(np.int32)
        boff = np.zeros(bs + 1, np.int32)
        boff[1:] = np.cumsum(np.bincount(b, minlength=bs))
        xyz = (coords_float[obj] + pt_offsets[obj]).astype(np.float32)
        nb, sl = oracle.ballquery_batch_p(xyz, b, boff, get(g, 'radius'))
        pidx, poff = oracle.bfs_cluster(mean, nb, sl, get(g, 'npoint_thr'), class_id)
        pidx = pidx.copy()
        pidx[:, 1] = obj[pidx[:, 1]]
        if off_list:
            pidx[:, 0] += sum(len(x) for x in off_list) - 1
            poff = (poff + off_list[-1][-1])[1:]
        if pidx.shape[0] > 0:
            idx_list.append(pidx)
            off_list.append(poff)
    if not idx_list:
        return np.zeros((0, 2), np.int32), np.zeros((0, ), np.int32)
    return np.concatenate(idx_list), np.concatenate(off_list)


@pytest.mark.parametrize('seed,batch', [(0, 1), (1, 1), (2, 2)])
def test_forward_grouping_equals_reference_loop(monkeypatch, seed, batch):
    monkeypatch.setattr(sg_module, 'ballquery_batch_p_nosync', _fake_ballquery_nosync)
    monkeypatch.setattr(sg_module, 'bfs_cluster_segments', _fake_bfs_segments)
    monkeypatch.setattr(sg_module, 'group_entries', _fake_group_entries)
    model = SoftGroup(**model_cfg('scannet', channels=16, num_blocks=2, test_cfg=dict(min_npoint=30))).eval()
    parts = [synth.make_scan('c1_plumbing', seed=seed * 10 + b, n_points=1500) for b in range(batch)]
    scores, offs, coords, bidx = [], [], [], []
    for b, sc in enumerate(parts):
        s, o = synth.grouping_inputs(sc, sigma=0.03, seed=seed)
        # a few confused points so that some classes fall under min_npoint and some points pass two classes
        rng = np.random.RandomState(seed)
        flip = rng.choice(s.shape[0], 60, replace=False)
        s[flip, rng.randint(2, 20, 60)] += 9.0
        scores.append(s)
        offs.append(o)
        coords.append(sc['coords_float'])
        bidx.append(np.full(s.shape[0], b, np.int32))
    scores, offs, coords, bidx = map(np.concatenate, (scores, offs, coords, bidx))
    got_idx, got_off = model.forward_grouping(torch.from_numpy(scores), torch.from_numpy(offs), torch.from_numpy(bidx),
                                              torch.from_numpy(coords))
    want_idx, want_off = reference_forward_grouping(model, scores, offs, bidx, coords)
    assert want_off.size > 2, 'the case must produce several proposals'
    assert np.array_equal(got_idx.numpy(), want_idx)
    assert np.array_equal(got_off.numpy(), want_off)


# ---- SoftGroup++ grouping (pyramid re-voxelisation + octree ball query), with and without lvl_fusion ------------
def _fake_ball_query(coords, batch_idxs, batch_offsets, radius, mean_active, with_octree=False):
    if with_octree:
        idx, sl = oracle.octree_ball_query(coords.numpy(), mean_active, radius)
    else:
        idx, sl = oracle.ballquery_batch_p(coords.numpy(), batch_idxs.numpy(), batch_offsets.numpy(), radius)
    return torch.from_numpy(idx.astype(np.int32)), torch.from_numpy(sl.astype(np.int32))


def _fake_voxelization(feats, map_rule, mode=4):
    return torch.from_numpy(oracle.voxelization(feats.numpy(), map_rule.numpy(), mode))


def reference_forward_grouping_pp(model, semantic_scores, pt_offsets, batch_idxs, coords_float, lvl_fusion):
    """softgroup.py:411-507 with the dense [nCluster, n] inverse map of :500-507."""
    g = model.grouping_cfg
    get = model._cfg
    bs = int(batch_idxs.max()) + 1
    scores = torch.from_numpy(semantic_scores).softmax(-1).numpy()
    mean = np.asarray(get(g, 'class_numpoint_mean'), np.float32)
    base = get(g, 'pyramid_base_size')
    idx_list, off_list = [], []
    for class_id in range(model.semantic_classes):
        if class_id in get(g, 'ignore_classes'):
            continue
        obj = np.nonzero(scores[:, class_id] > get(g, 'score_thr'))[0]
        if obj.size < get(model.test_cfg, 'min_npoint'):
            continue
        b = batch_idxs[obj].astype(np.int32)
        xyz, off = coords_float[obj], pt_offsets[obj]
        level = model.get_level(obj.size)
        radius = get(g, 'radius') * level
        l2p = None
        if level > 1 or not lvl_fusion:
            vc = np.concatenate([b[:, None].astype(np.int64), (torch.from_numpy(xyz) / (base * level)).long().numpy()], 1)
            vcoords, l2p, p2l = oracle.voxelization_idx(vc, int(b[-1]) + 1, 4)
            n_before = obj.size
            xyz = oracle.voxelization(xyz, p2l, 4)
            off = oracle.voxelization(off, p2l, 4)
            b = vcoords[:, 0].astype(np.int32)
        boff = np.zeros(bs + 1, np.int32)
        boff[1:] = np.cumsum(np.bincount(b, minlength=bs))
        nb, sl = oracle.octree_ball_query((xyz + off).astype(np.float32), get(g, 'mean_active'), radius)
        pidx, poff = oracle.bfs_cluster(mean, nb, sl, get(g, 'npoint_thr'), class_id)
        if l2p is not None:
            dense = np.zeros((poff.size - 1, xyz.shape[0]), np.int32)
            dense[pidx[:, 0], pidx[:, 1]] = 1
            dense = dense[:, l2p.astype(np.int64)]
            assert dense.shape[1] == n_before
            pidx = np.stack(np.nonzero(dense), 1).astype(np.int32)
            poff = np.concatenate([[0], np.cumsum(dense.sum(1))]).astype(np.int32)
        pidx = pidx.copy()
        pidx[:, 1] = obj[pidx[:, 1]]
        if off_list:
            pidx[:, 0] += sum(len(x) for x in off_list) - 1
            poff = (poff + off_list[-1][-1])[1:]
        if pidx.shape[0] > 0:
            idx_list.append(pidx)
            off_list.append(poff)
    if not idx_list:
        return np.zeros((0, 2), np.int32), np.zeros((0, ), np.int32)
    return np.concatenate(idx_list), np.concatenate(off_list)


@pytest.mark.parametrize('lvl_fusion', [False, True])
def test_forward_grouping_pp_equals_reference_loop(monkeypatch, lvl_fusion):
    monkeypatch.setattr(sg_module, 'ball_query', _fake_ball_query)
    monkeypatch.setattr(sg_module, 'bfs_cluster_segments', _fake_bfs_segments)
    monkeypatch.setattr(sg_module, 'voxelization', _fake_voxelization)
    cfg = model_cfg('scannet++', channels=16, num_blocks=2, test_cfg=dict(min_npoint=30))
    cfg['grouping_cfg'].update(pyramid_base_size=0.02, radius=0.04)
    model = SoftGroup(**cfg).eval()
    model.get_level = lambda n: 2 if n > 250 else 1  # both levels at a size the CPU oracle handles
    sc = synth.make_scan('c1_plumbing', seed=5, n_points=2500)
    scores, offs = synth.grouping_inputs(sc, sigma=0.03, seed=5)
    coords, bidx = sc['coords_float'], np.zeros(scores.shape[0], np.int32)
    got_idx, got_off = model.forward_grouping(torch.from_numpy(scores), torch.from_numpy(offs), torch.from_numpy(bidx),
                                              torch.from_numpy(coords), lvl_fusion=lvl_fusion)
    want_idx, want_off = reference_forward_grouping_pp(model, scores, offs, bidx, coords, lvl_fusion)
    assert want_off.size > 2
    assert np.array_equal(got_idx.numpy(), want_idx)
    assert np.array_equal(got_off.numpy(), want_off)


# ---- clusters_voxelization (softgroup.py:655-709): per-cluster rescaling to the 20^3 grid + hashing -------------
def _fake_sec(fn):
    return lambda inp, offsets: torch.from_numpy(fn(inp.numpy(), offsets.numpy()))


def test_clusters_voxelization_equals_reference_steps(monkeypatch):
    monkeypatch.setattr(sg_module, 'sec_min', _fake_sec(oracle.sec_min))
    monkeypatch.setattr(sg_module, 'sec_max', _fake_sec(oracle.sec_max))
    monkeypatch.setattr(sg_module, 'voxelization', _fake_voxelization)
    model = SoftGroup(**model_cfg('scannet', channels=16, num_blocks=2)).eval()
    rng = np.random.RandomState(0)
    n, nprop, C = 2000, 9, 16
    coords = (rng.rand(n, 3) * np.array([4.0, 3.0, 2.0])).astype(np.float32)
    feats = rng.randn(n, C).astype(np.float32)
    lens = rng.randint(20, 300, nprop)
    lens[3] = 1  # a single-point cluster: zero extent -> scale clamps to the cap
    members = [rng.choice(n, ln, replace=False) for ln in lens]
    pidx = np.concatenate([np.stack([np.full(len(m), p), m], 1) for p, m in enumerate(members)]).astype(np.int32)
    poff = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    scale, S = 50, 20
    x, inp_map = model.clusters_voxelization(torch.from_numpy(pidx), torch.from_numpy(poff), torch.from_numpy(feats),
                                             torch.from_numpy(coords), scale=scale, spatial_shape=S)
    # the reference's steps, line by line, on torch CPU + oracle ops
    bi = torch.from_numpy(pidx[:, 0]).long()
    ci = torch.from_numpy(pidx[:, 1]).long()
    f = torch.from_numpy(feats)[ci]
    c = torch.from_numpy(coords)[ci]
    cmin = torch.from_numpy(oracle.sec_min(c.numpy(), poff))
    cmax = torch.from_numpy(oracle.sec_max(c.numpy(), poff))
    cs = 1 / ((cmax - cmin) / S).max(1)[0] - 0.01
    cs = torch.clamp(cs, min=None, max=scale)
    cmin = cmin * cs[:, None]
    cs = cs[bi]
    c = c * cs[:, None]
    c -= cmin[bi]
    assert c.shape.numel() == ((c >= 0) * (c < S)).sum()
    c = torch.cat([bi.view(-1, 1), c.long()], 1)
    oc, imap, omap = oracle.voxelization_idx(c.numpy(), nprop, 4)
    of = oracle.voxelization(f.numpy(), omap, 4)
    assert np.array_equal(x.indices.numpy(), oc.astype(np.int32)) and x.batch_size == nprop
    assert list(x.spatial_shape) == [S] * 3
    assert np.array_equal(inp_map.numpy(), imap)
    assert np.array_equal(x.features.numpy(), of)


# ---- the reference's OWN forward_grouping (unmodified class on our shims) as the golden -------------------------
def forward_grouping_inputs():
    """(semantic scores, offsets, batch_idxs, coords_float) of a 2000-point scan."""
    sc = synth.make_scan('c1_plumbing', seed=7, n_points=2000)
    scores, offs = synth.grouping_inputs(sc, sigma=0.03, seed=7)
    return [torch.from_numpy(scores), torch.from_numpy(offs), torch.zeros(scores.shape[0], dtype=torch.int32),
            torch.from_numpy(sc['coords_float'])]


def test_forward_grouping_equals_reference_method(monkeypatch, host_arrays):
    """softgroup/model/softgroup.py:411-480 itself ran on CPU once its three CUDA touch points (ball_query, bfs_cluster,
    get_batch_offsets' .cuda()) were replaced by oracle stand-ins (tests/golden/make_reference_golden.py); ours must
    return the same tensors."""
    cfg = model_cfg('scannet', channels=16, num_blocks=2, test_cfg=dict(min_npoint=30))
    ours = SoftGroup(**cfg).eval()
    monkeypatch.setattr(sg_module, 'ballquery_batch_p_nosync', _fake_ballquery_nosync)
    monkeypatch.setattr(sg_module, 'bfs_cluster_segments', _fake_bfs_segments)
    monkeypatch.setattr(sg_module, 'group_entries', _fake_group_entries)
    want_idx = torch.from_numpy(host_arrays['forward_grouping_idx'])
    want_off = torch.from_numpy(host_arrays['forward_grouping_off'])
    got_idx, got_off = ours.forward_grouping(*forward_grouping_inputs())
    assert want_off.numel() > 2
    assert torch.equal(got_idx, want_idx) and torch.equal(got_off, want_off)
