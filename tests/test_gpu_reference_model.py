"""Drop-in proof on hardware (SURVEY.md 8b, VERDICT round 1 row g1): the UNMODIFIED reference `SoftGroup` class
(softgroup/model/softgroup.py + blocks.py) was instantiated on `softgroup_b200.install_as_reference_backends()` -- this
repo's `spconv.pytorch` and `softgroup.ops` -- moved to a B200 and called exactly like tools/test.py:145-152 does
(`model(batch)` on the dataloader's collated batch). What it returned is stored in tests/golden/ref_gpu_model.npz
(tests/golden/make_reference_golden.py) and compared here with

  * this repo's restructured `softgroup_b200.model.SoftGroup` with the same weights on the same scan: proposals / masks
    (RLE strings, by digest) / labels identical, scores within 1e-4, point-wise outputs within 1e-4 relative (offsets on
    a fixed sample of 1024 points; the pass-through arrays by digest);
  * for the plain config also with the reference-generated fixture tests/golden/ref_forward_c1.npz (the reference's
    own forward_test on CPU stand-ins).

The `scannet++` case ran the reference's own lvl_fusion / pyramid / octree code path (softgroup.py:309-312, 332-334,
427-463, 560-561) on the GPU ops -- the reference-order procedure for this repo's sparse lvl_fusion implementation."""
import os
import sys

import numpy as np
import pytest
import torch

from softgroup_b200 import harness, synth
from softgroup_b200.configs import model_cfg
from softgroup_b200.model import SoftGroup

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, 'golden'))
from digest import digest  # noqa: E402
from seeded_weights import CFG_OVERRIDES, SCAN, WEIGHT_SEED, fill_seeded, load_calibrated  # noqa: E402

pytestmark = pytest.mark.gpu

PASSTHROUGH = ('semantic_labels', 'instance_labels', 'coords_float', 'color_feats', 'offset_labels', 'gt_instances')
N_OFFSET_SAMPLE = 1024


@pytest.fixture(scope='module')
def gold():
    return np.load(os.path.join(HERE, 'golden', 'ref_gpu_model.npz'))


def case(name, n_points=None):
    """-> (model config, scan, calibrated head weights or None); 'c1' is the configuration of ref_forward_c1.npz."""
    if name == 'c1':
        fixture = np.load(os.path.join(HERE, 'golden', 'ref_forward_c1.npz'), allow_pickle=True)
        return model_cfg('scannet', **CFG_OVERRIDES), synth.make_scan(SCAN['shape'], seed=SCAN['seed']), fixture['calibrated']
    # Full-size model (32 channels x 7 levels); 'scannet++' = pyramid + octree + lvl_fusion at test time. Grouping thresholds
    # that give proposals on a random-weight (calibrated-head) model: the yaml values (4 cm radius, thresholds relative to
    # ScanNet class sizes) select nothing there -- both models returned 0 instances
    cfg = model_cfg(name, grouping_cfg=dict(radius=0.15, class_numpoint_mean=[-1.] * 20, npoint_thr=100),
                    test_cfg=dict(min_npoint=50))
    return cfg, synth.make_scan('c2_scannet', seed=5, n_points=n_points), None


def our_model(cfg, scan, calibrated=None):
    ours = SoftGroup(**cfg).eval()
    fill_seeded(ours, WEIGHT_SEED)
    if calibrated is not None:
        load_calibrated(ours, calibrated)
    ours = ours.cuda()
    if calibrated is None:
        harness.calibrate_heads(ours, harness.to_host_batch(scan))
    return ours


def _canon(a):
    a = np.asarray(a)
    if np.issubdtype(a.dtype, np.integer):
        return a.astype(np.int64)
    if np.issubdtype(a.dtype, np.floating):
        return a.astype(np.float64)
    return a


def _str_digest(s):
    return digest(np.frombuffer(s.encode(), np.uint8))


def summarize(r, prefix):
    """The golden record of a forward_test result dict (a reference class result when the fixture is made)."""
    g = {prefix + 'keys': np.array(sorted(r.keys())), prefix + 'scan_id': np.array(str(r['scan_id']))}
    for k in PASSTHROUGH:
        g[prefix + k + '_digest'] = np.array(digest(_canon(r[k])))
    off = np.asarray(r['offset_preds'], np.float32)
    rows = np.sort(np.random.RandomState(0).permutation(off.shape[0])[:N_OFFSET_SAMPLE])
    g[prefix + 'offset_rows'] = rows
    g[prefix + 'offset_sample'] = off[rows]
    g[prefix + 'offset_absmax'] = np.abs(off).max()
    g[prefix + 'semantic_preds'] = np.asarray(r['semantic_preds']).astype(np.int16)
    inst = r['pred_instances']
    g[prefix + 'inst_scan_id'] = np.array([str(x['scan_id']) for x in inst])
    g[prefix + 'inst_label_id'] = np.array([int(x['label_id']) for x in inst], np.int64)
    g[prefix + 'inst_length'] = np.array([int(x['pred_mask']['length']) for x in inst], np.int64)
    g[prefix + 'inst_counts_digest'] = np.array([_str_digest(x['pred_mask']['counts']) for x in inst])
    g[prefix + 'inst_conf'] = np.array([float(x['conf']) for x in inst], np.float64)
    return g


def _compare(gold, prefix, b, n_points, rel=1e-4):
    """gold: the stored reference class result, b: this repo's result."""
    a = {k[len(prefix):]: gold[k] for k in gold.files if k.startswith(prefix)}
    assert [str(k) for k in a['keys']] == sorted(b.keys())
    assert str(a['scan_id']) == str(b['scan_id'])
    for k in PASSTHROUGH:
        assert digest(_canon(b[k])) == str(a[k + '_digest']), k
    off_b = np.asarray(b['offset_preds'])
    assert off_b.shape[0] == n_points
    assert np.abs(a['offset_sample'] - off_b[a['offset_rows']]).max() <= rel * max(float(a['offset_absmax']), 1e-6)
    sp_a, sp_b = a['semantic_preds'], np.asarray(b['semantic_preds'])
    assert sp_a.shape == sp_b.shape
    assert (sp_a != sp_b).mean() <= 1e-3  # argmax of scores that agree to 1e-4: ties may flip on a handful of points
    ib = b['pred_instances']
    assert len(a['inst_label_id']) == len(ib) and len(ib) > 0
    for i, y in enumerate(ib):
        assert str(a['inst_scan_id'][i]) == str(y['scan_id']) and int(a['inst_label_id'][i]) == y['label_id']
        assert int(a['inst_length'][i]) == n_points == y['pred_mask']['length']
        assert str(a['inst_counts_digest'][i]) == _str_digest(y['pred_mask']['counts'])
        assert abs(float(a['inst_conf'][i]) - float(y['conf'])) <= rel * max(1.0, abs(float(y['conf'])))
    return len(ib)


def run_ours(name, n_points=None):
    cfg, scan, calibrated = case(name, n_points)
    ours = our_model(cfg, scan, calibrated)
    with torch.no_grad():
        return ours(dict(harness.collate_like_reference(scan))), scan['coords'].shape[0]


def test_reference_class_runs_on_b200_and_matches(gold):
    fixture = np.load(os.path.join(HERE, 'golden', 'ref_forward_c1.npz'), allow_pickle=True)
    r_our, n_points = run_ours('c1')
    n = _compare(gold, 'c1/', r_our, n_points)
    # and the reference class on the B200 equals the reference's own CPU run (fixture): same instances, same masks
    assert n == len(fixture['inst_rle'])
    assert [str(x) for x in gold['c1/inst_counts_digest']] == [_str_digest(str(x)) for x in fixture['inst_rle']]
    assert [int(x) for x in gold['c1/inst_label_id']] == [int(x) for x in fixture['inst_label_id']]
    conf = gold['c1/inst_conf']
    assert np.abs(conf - fixture['inst_conf']).max() <= 2e-4 * max(1.0, np.abs(fixture['inst_conf']).max())


@pytest.mark.parametrize('name,n_points', [('scannet', 30000), ('scannet++', 20000)])
def test_reference_class_vs_restructured_forward(gold, name, n_points):
    r_our, n = run_ours(name, n_points)
    _compare(gold, name + '/', r_our, n)
