"""Host-side logic that needs no GPU: weight packing layout, RLE wire format (numpy path and the library's host
formatter), config values against the reference YAMLs, BatchNorm folding, synthetic-scan layout."""
import numpy as np
import pytest
import torch

from softgroup_b200 import configs, synth
from softgroup_b200.spconv import core
from softgroup_b200.util import rle as rle_util

# ---- tcgen05 weight packing (include/sgb200.h: Wp fp16 [K][nkc][4][2][N][8]) ------------------------------------
@pytest.mark.parametrize('K,Cin,Cout', [(1, 6, 32), (3, 40, 20), (8, 32, 64), (27, 96, 96)])
def test_pack_weight_tc_layout(K, Cin, Cout):
    g = torch.Generator().manual_seed(K * 1000 + Cin * 10 + Cout)
    W = torch.randn(K, Cin, Cout, generator=g) * torch.logspace(-3, 1, Cout)[None, None, :]
    packed = core.pack_weight_tc(W)
    N = (Cout + 15) // 16 * 16
    nkc = (Cin + 31) // 32
    assert packed.dtype == torch.float32 and packed.numel() == K * nkc * 4 * 2 * N * 4
    halves = packed.view(torch.float16).view(K, nkc, 4, 2, N, 8)
    hi, lo = halves[:, :, :, 0].float(), halves[:, :, :, 1].float()  # [K, nkc, 4, N, 8]
    # element (k, kc, q, n, e) <-> W[k][32*kc + 8*q + e][n]
    full = torch.zeros(K, nkc * 32, N)
    full[:, :Cin, :Cout] = W
    want = full.view(K, nkc, 4, 8, N).permute(0, 1, 2, 4, 3)
    assert torch.equal(hi, want.half().float())  # hi = fp16(x)
    from softgroup_b200.ops import _lib
    shift = _lib.lib().sgb_spconv_lo_shift()
    assert shift == 11  # remainders are carried scaled by 2^11: no fp16 subnormals for |x - hi| >= 2^-25
    assert torch.equal(lo, ((want - want.half().float()) * 2.0**shift).half().float())  # lo = fp16((x - hi) * 2^shift)
    # the split is fp32-grade: |x - hi - lo 2^-shift| <= 2^-22 |x| while the scaled remainder is a normal fp16 number,
    # 2^-36 absolute below that (|x - hi| < 2^-25) -- the bound written in spconv_tc.cu and DESIGN.md 3.2
    err = (want - hi - lo * 2.0**-shift).abs()
    assert (err <= torch.maximum(want.abs() * 2.0**-22, torch.tensor(2.0**-36))).all()
    # padding (channels past Cin, columns past Cout) is exactly zero
    assert (hi.permute(0, 1, 2, 4, 3).reshape(K, nkc * 32, N)[:, Cin:, :] == 0).all()
    assert (hi[..., Cout:, :] == 0).all() and (lo[..., Cout:, :] == 0).all()


# ---- RLE wire format (softgroup/util/rle.py:5-19) --------------------------------------------------------------
def _reference_rle(mask):
    """Independent restatement of the reference encoder on a dense mask."""
    out, n, i = [], len(mask), 0
    while i < n:
        if mask[i]:
            j = i
            while j < n and mask[j]:
                j += 1
            out += [i + 1, j - i]
            i = j
        else:
            i += 1
    return dict(length=n, counts=' '.join(map(str, out)))


@pytest.mark.parametrize('seed', range(4))
def test_rle_paths_agree(seed):
    rng = np.random.RandomState(seed)
    n = 3000
    masks = [(rng.rand(n) < p).astype(np.uint8) for p in (0.0, 0.02, 0.5, 0.98, 1.0)]
    masks.append(np.zeros(n, np.uint8))
    masks[-1][[0, n - 1]] = 1  # runs touching both ends
    ids = [np.nonzero(m)[0].astype(np.int32) for m in masks]
    offs = np.concatenate([[0], np.cumsum([len(i) for i in ids])]).astype(np.int64)
    many = rle_util.rle_encode_many(np.concatenate(ids), offs, n)  # libsgb200 host formatter (no GPU involved)
    for m, i, r in zip(masks, ids, many):
        want = _reference_rle(m)
        assert rle_util.rle_encode(m) == want
        assert rle_util.rle_encode_ids(i, n) == want
        assert r == want
        assert np.array_equal(rle_util.rle_decode(want), m)


def test_rle_encode_many_empty():
    assert rle_util.rle_encode_many(np.zeros(0, np.int32), np.zeros(1, np.int64), 10) == []


# ---- configs are restated data: pinned on the `model` sections of the reference YAMLs (tests/golden/ref_host.json) -----
CONFIG_FILES = [('scannet', 'configs/softgroup/softgroup_scannet.yaml'),
                ('s3dis', 'configs/softgroup/softgroup_s3dis_fold5.yaml'),
                ('kitti', 'configs/softgroup/softgroup_kitti.yaml'),
                ('stpls3d++', 'configs/softgroup++/softgroup++_stpls3d.yaml'),
                ('scannet++', 'configs/softgroup++/softgroup++_scannet.yaml')]


@pytest.mark.parametrize('name,path', CONFIG_FILES)
def test_configs_match_reference_yaml(host_gold, name, path):
    ref = host_gold['configs'][name]
    ours = configs.model_cfg(name)
    for key in ('channels', 'num_blocks', 'semantic_classes', 'instance_classes', 'sem2ins_classes', 'semantic_only',
                'ignore_label'):
        assert ours[key] == ref[key], key
    for key in ('in_channels', 'with_coords'):
        if key in ref:
            assert ours[key] == ref[key], key
    for key, val in ref['grouping_cfg'].items():
        got = ours['grouping_cfg'][key]
        if isinstance(val, list):
            assert [float(v) for v in got] == [float(v) for v in val], key
        else:
            assert got == val, key
    for key, val in ref['instance_voxel_cfg'].items():
        assert ours['instance_voxel_cfg'][key] == val, key
    for key, val in ref['test_cfg'].items():
        assert ours['test_cfg'][key] == val, key


# ---- BatchNorm1d(eval) folding (softgroup.py:54, eps = 1e-4) ---------------------------------------------------
def test_fold_bn_matches_batchnorm_eval():
    torch.manual_seed(0)
    bn = torch.nn.BatchNorm1d(48, eps=1e-4, momentum=0.1)
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.normal_()
        bn.running_mean.normal_()
        bn.running_var.uniform_(0.2, 3.0)
    bn.eval()
    scale, shift = core.fold_bn(bn)
    x = torch.randn(100, 48)
    assert torch.allclose(x * scale + shift, bn(x), rtol=1e-6, atol=1e-6)
    with torch.no_grad():
        bn.weight.mul_(2.0)  # the cache must notice in-place updates (load_state_dict)
    scale2, shift2 = core.fold_bn(bn)
    assert torch.allclose(x * scale2 + shift2, bn(x), rtol=1e-6, atol=1e-6)
    bn.train()
    with pytest.raises(RuntimeError):
        core.fold_bn(bn)


# ---- synthetic scans keep the reference collate layout (custom.py:191-256) -------------------------------------
@pytest.mark.parametrize('shape', ['c1_plumbing', 'c4_kitti'])
def test_synth_scan_layout(shape):
    n = 3000
    a = synth.make_scan(shape, seed=3, n_points=n)
    b = synth.make_scan(shape, seed=3, n_points=n)
    for k in ('coords', 'coords_float', 'feats', 'semantic_labels', 'instance_labels', 'pt_offset_labels'):
        assert np.array_equal(a[k], b[k]), k  # deterministic in the seed
    assert a['coords'].dtype == np.int64 and a['coords'].shape == (n, 4) and (a['coords'][:, 0] == 0).all()
    assert a['coords_float'].dtype == np.float32 and a['coords_float'].shape == (n, 3)
    assert (a['coords'][:, 1:] >= 0).all() and (a['coords'][:, 1:].max(0) < a['spatial_shape']).all()
    assert (a['spatial_shape'] >= 128).all()  # custom.py:248 clips at voxel_cfg.spatial_shape[0]
    inst = a['instance_labels']
    assert a['instance_pointnum'].sum() == (inst >= 0).sum()
    assert np.abs(a['pt_offset_labels'][inst < 0]).max() == 0
    x4 = synth.to_x4_split(a)
    assert x4['batch_size'] == 4 and np.array_equal(np.sort(x4['x4_order']), np.arange(n))
    assert set(np.unique(x4['coords'][:, 0])) == {0, 1, 2, 3}


# ---- bfs_cluster labelling: sequential emulation of the frontier iteration (bfs_cluster.cu) ---------------------
def _reference_seed_labels(lists):
    """bfs_cluster.cpp:33-126 semantics: seeds in index order, BFS over the DIRECTED out-lists, first claim wins."""
    n = len(lists)
    label = [-1] * n
    for i in range(n):
        if label[i] >= 0:
            continue
        label[i] = i
        queue = [i]
        while queue:
            u = queue.pop(0)
            for v in lists[u]:
                if label[v] < 0:
                    label[v] = i
                    queue.append(v)
    return label


@pytest.mark.parametrize('seed', range(6))
def test_frontier_label_iteration_reaches_reference_labels(seed):
    """label[v] = smallest index that can reach v; a node re-pushes only when its chased label dropped below the one
    it pushed last (`pushed`), and the pass without a push ends the loop -- in any processing order."""
    rng = np.random.RandomState(seed)
    n = 300
    pts = rng.rand(n, 2) * (1.0 if seed % 2 else 3.0)
    d = ((pts[:, None] - pts[None]) ** 2).sum(-1)
    cap = 6  # truncation to the first `cap` neighbours by index makes the graph asymmetric, like the 1000 cap
    lists = [list(np.nonzero(d[u] < 0.02)[0][:cap]) for u in range(n)]
    want = _reference_seed_labels(lists)
    label = list(range(n))
    pushed = [2**31 - 1] * n
    for _ in range(10 * n):
        any_push = False
        for u in rng.permutation(n):  # arbitrary order stands in for the GPU's scheduling
            lu = label[u]
            while label[lu] < lu:
                lu = label[lu]
            label[u] = min(label[u], lu)
            if lu >= pushed[u]:
                continue
            any_push = True
            for v in lists[u]:
                label[v] = min(label[v], lu)
            pushed[u] = lu
        if not any_push:
            break
    assert label == want


@pytest.mark.parametrize('seed', range(6))
def test_select_then_push_iteration_reaches_reference_labels(seed):
    """The two-kernel form of a pass (bfs_frontier_select_kernel / bfs_frontier_push_kernel): ALL nodes chase their label and
    decide first (the queue holds (node, label to push), `pushed` is updated at selection), then the queued entries push --
    the labels the selection saw are one pass old. Same fixed point, in any order inside either step."""
    rng = np.random.RandomState(100 + seed)
    n = 300
    pts = rng.rand(n, 2) * (1.0 if seed % 2 else 3.0)
    d = ((pts[:, None] - pts[None]) ** 2).sum(-1)
    cap = 6
    lists = [list(np.nonzero(d[u] < 0.02)[0][:cap]) for u in range(n)]
    want = _reference_seed_labels(lists)
    label = list(range(n))
    pushed = [2**31 - 1] * n
    for _ in range(10 * n):
        queue = []
        for u in rng.permutation(n):  # select
            lu = label[u]
            while label[lu] < lu:
                lu = label[lu]
            label[u] = min(label[u], lu)
            if lu < pushed[u]:
                queue.append((u, lu))
                pushed[u] = lu
        if not queue:
            break
        for k in rng.permutation(len(queue)):  # push
            u, lu = queue[k]
            for v in lists[u]:
                label[v] = min(label[v], lu)
    assert label == want


# ---- cooperative gather of spconv_tc_kernel<1> (round-2 candidate): index arithmetic emulated lane by lane --------
def test_coop_gather_tile_indexing_is_a_conflict_free_transpose():
    """Write side: instruction j, lane l -> row R = 4j + (l >> 3), logical 16-byte chunk i = l & 7, physical chunk
    i ^ (R & 7). Read side: lane r, register group c <- physical chunk c ^ (r & 7) of row r. Every lane must end up with
    its own row in logical chunk order, and every quarter-warp access must touch 8 different 16-byte bank groups."""
    rng = np.random.RandomState(0)
    rows = rng.randint(0, 1000, (32, 8))  # rows[r][i] = id of logical chunk i of the source row feeding tile row r
    tile = -np.ones((32, 8), np.int64)
    for j in range(8):
        for q in range(4):  # quarter-warp = one shared-memory wavefront of a 128-bit access
            banks = set()
            for l in range(8 * q, 8 * q + 8):
                R, i = 4 * j + (l >> 3), l & 7
                phys = i ^ (R & 7)
                assert tile[R, phys] == -1
                tile[R, phys] = rows[R, i]
                banks.add((R * 128 + phys * 16) // 16 % 8)
            assert len(banks) == 8
    assert (tile >= 0).all()
    for c in range(8):
        for q in range(4):
            banks = set()
            for r in range(8 * q, 8 * q + 8):
                phys = c ^ (r & 7)
                assert tile[r, phys] == rows[r, c]  # register group c of lane r = logical chunk c of row r
                banks.add((r * 128 + phys * 16) // 16 % 8)
            assert len(banks) == 8
