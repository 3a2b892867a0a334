"""tests/golden/ref_forward_c1.npz -- stage outputs of the REFERENCE'S OWN forward_test (unmodified
softgroup/model/{blocks,softgroup}.py run on CPU over oracle stand-ins, tests/golden/make_forward_golden.py).

CPU checks here (no GPU):
  * this repo's model gets bit-identical weights from the seeded filler (digest in the fixture);
  * this repo's host logic, fed with the fixture's intermediates, reproduces the reference's outputs:
    forward_grouping, clusters_voxelization, get_instances, get_gt_instances;
  * the oracle's U-Net composition (spconv_oracle.backbone) equals the reference's blocks.py composition."""
import os
import sys

import numpy as np
import pytest
import torch

import oracle
from oracle import spconv_oracle as so
from softgroup_b200 import synth
from softgroup_b200.configs import model_cfg
from softgroup_b200.model import SoftGroup
from softgroup_b200.model import softgroup as sg_module

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, 'golden'))
from seeded_weights import CFG_OVERRIDES, SCAN, WEIGHT_SEED, fill_seeded, load_calibrated, weights_digest  # noqa: E402
from test_host_grouping import (_fake_ballquery_nosync, _fake_bfs_segments, _fake_group_entries, _fake_sec,  # noqa: E402
                                _fake_voxelization)


@pytest.fixture(scope='module')
def gold():
    return np.load(os.path.join(HERE, 'golden', 'ref_forward_c1.npz'))


@pytest.fixture(scope='module')
def model(gold):
    m = SoftGroup(**model_cfg('scannet', **CFG_OVERRIDES)).eval()
    fill_seeded(m, WEIGHT_SEED)
    load_calibrated(m, gold['calibrated'])
    return m


def test_seeded_weights_are_identical(gold, model):
    assert weights_digest(model) == int(gold['weights_digest'])


def test_oracle_unet_composition_equals_reference_blocks(gold, model):
    sd = {k: v.detach().numpy() for k, v in model.state_dict().items()}
    cfg = model_cfg('scannet', **CFG_OVERRIDES)
    scan = synth.make_scan(SCAN['shape'], seed=SCAN['seed'])
    out = so.backbone(gold['voxel_feats'], gold['voxel_coords'].astype(np.int32), scan['spatial_shape'], sd,
                      cfg['channels'], cfg['num_blocks'], acc64=True)
    want = gold['output_feats']  # point rows = voxel rows gathered by v2p_map (softgroup.py:374)
    got = out[gold['v2p_map']]
    assert np.abs(got - want).max() <= 2e-5 * max(1.0, np.abs(want).max())


def test_forward_grouping_reproduces_reference_proposals(monkeypatch, gold, model):
    monkeypatch.setattr(sg_module, 'ballquery_batch_p_nosync', _fake_ballquery_nosync)
    monkeypatch.setattr(sg_module, 'bfs_cluster_segments', _fake_bfs_segments)
    monkeypatch.setattr(sg_module, 'group_entries', _fake_group_entries)
    n = gold['semantic_scores'].shape[0]
    scan = synth.make_scan(SCAN['shape'], seed=SCAN['seed'])
    pidx, poff = model.forward_grouping(torch.from_numpy(gold['semantic_scores']), torch.from_numpy(gold['pt_offsets']),
                                        torch.zeros(n, dtype=torch.int32), torch.from_numpy(scan['coords_float']))
    assert np.array_equal(pidx.numpy(), gold['proposals_idx'])
    assert np.array_equal(poff.numpy(), gold['proposals_offset'])


def test_clusters_voxelization_reproduces_reference(monkeypatch, gold, model):
    monkeypatch.setattr(sg_module, 'sec_min', _fake_sec(oracle.sec_min))
    monkeypatch.setattr(sg_module, 'sec_max', _fake_sec(oracle.sec_max))
    monkeypatch.setattr(sg_module, 'voxelization', _fake_voxelization)
    scan = synth.make_scan(SCAN['shape'], seed=SCAN['seed'])
    x, inp_map = model.clusters_voxelization(torch.from_numpy(gold['proposals_idx']),
                                             torch.from_numpy(gold['proposals_offset']),
                                             torch.from_numpy(gold['output_feats']),
                                             torch.from_numpy(scan['coords_float']), **model._voxel_cfg())
    assert np.array_equal(x.indices.numpy(), gold['inst_voxel_coords'])
    assert np.array_equal(inp_map.numpy(), gold['inst_map'])
    assert np.array_equal(x.features.numpy(), gold['inst_voxel_feats'])


def test_get_instances_reproduces_reference(host_instance_ops, gold, model):
    inst = model.get_instances('x', torch.from_numpy(gold['proposals_idx']), torch.from_numpy(gold['semantic_scores']),
                               torch.from_numpy(gold['cls_scores']), torch.from_numpy(gold['iou_scores']),
                               torch.from_numpy(gold['mask_scores']))
    assert len(inst) == gold['inst_conf'].size > 0
    assert [int(p['label_id']) for p in inst] == gold['inst_label_id'].tolist()
    assert np.array_equal(np.asarray([p['conf'] for p in inst], np.float32), gold['inst_conf'])
    assert [p['pred_mask']['counts'] for p in inst] == gold['inst_rle'].tolist()
    assert all(p['pred_mask']['length'] == gold['semantic_scores'].shape[0] for p in inst)


def test_get_gt_instances_reproduces_reference(gold, model):
    scan = synth.make_scan(SCAN['shape'], seed=SCAN['seed'])
    got = model.get_gt_instances(torch.from_numpy(scan['semantic_labels']), torch.from_numpy(scan['instance_labels']))
    assert np.array_equal(got, gold['gt_instances'])
