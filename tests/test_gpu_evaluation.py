"""N4 (SURVEY.md 8f): the GPU assignment step of the instance evaluation against what the reference's own
`ScanNetEval.assign_instances_for_scan` / `evaluate_matches` (softgroup/evaluation/instance_eval.py:39-309, run with the
numpy >= 1.24 aliases installed instead of editing it) returned on the same scans: tests/golden/ref_host.json
(digests of the match structures; tests/golden/make_reference_golden.py)."""
import json
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from softgroup_b200 import evaluation as sgb_eval
from softgroup_b200.util import rle_encode

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
from digest import digest  # noqa: E402

pytestmark = pytest.mark.gpu

CLASS_NAMES = ['c%d' % i for i in range(18)]


def evaluator(host_gold, use_label=True):
    """The attributes of the reference ScanNetEval(CLASS_NAMES, use_label) that the GPU assignment reads, as stored."""
    e = dict(host_gold['evaluator_use_label_%s' % use_label])
    e['id2label'] = {int(k): v for k, v in e['id2label']}
    e['valid_class_ids'] = np.asarray(e['valid_class_ids'])
    e['min_region_sizes'] = np.asarray(e['min_region_sizes'])
    return SimpleNamespace(**e)


class _MatchRecorder(SimpleNamespace):
    """Stands in for the reference evaluator's evaluate_matches / compute_averages, which are pure functions of the
    matches: it keeps what `evaluate` hands over and returns the averages the reference computed from its own matches."""
    def evaluate_matches(self, matches):
        self.matches = matches
        return None, None

    def compute_averages(self, ap, rc):
        return self.averages


def scan(seed, n=60000, n_gt=25, n_pred=120, n_classes=18):
    rng = np.random.RandomState(seed)
    gts = np.zeros(n, np.int64)
    # ground truth: contiguous-ish blobs with class*1000 + instance id; some void classes (0 and 19+)
    pos = rng.permutation(n)
    cuts = np.sort(rng.choice(np.arange(1, n), n_gt, replace=False))
    segs = np.split(pos, cuts)
    for k, seg in enumerate(segs):
        cls = rng.randint(0, n_classes + 3)  # 0 and > n_classes are void
        gts[seg] = cls * 1000 + k + 1 if cls > 0 else 0
    preds = []
    for k in range(n_pred):
        seg = segs[rng.randint(len(segs))]
        keep = seg[rng.rand(seg.size) < rng.uniform(0.2, 1.0)]
        extra = rng.choice(n, rng.randint(0, 300), replace=False)
        m = np.zeros(n, np.uint8)
        m[keep] = 1
        m[extra] = 1
        if k % 17 == 0:
            m[:] = 0
            m[rng.choice(n, 30, replace=False)] = 1  # below min_region_size: skipped
        label = int(rng.randint(1, n_classes + 2))  # n_classes + 1 is not a valid label: skipped
        mask = rle_encode(m) if k % 2 else m  # both wire formats
        preds.append(dict(scan_id='scan%d' % seed, label_id=label, conf=float(rng.rand()), pred_mask=mask))
    return preds, gts


def average_scans():
    return [scan(s, n=30000, n_pred=80) for s in (2, 3)]


def _plain(x):
    """The JSON form of a match structure (numpy scalars as Python numbers, string keys)."""
    return json.loads(json.dumps(x, default=lambda v: v.item() if isinstance(v, np.generic) else v.tolist()))


def matches_digest(x):
    """Digest of the canonical JSON text of a match structure (the golden file keeps these, not the structures)."""
    return digest(np.frombuffer(json.dumps(_plain(x), sort_keys=True).encode(), np.uint8))


@pytest.fixture(autouse=True)
def _numpy_aliases():
    sgb_eval.install_numpy_aliases()


@pytest.mark.parametrize('use_label', [True, False])
def test_assign_instances_matches_reference(host_gold, use_label):
    want = host_gold['assign_use_label_%s' % use_label]
    want_g2p, want_p2g = want['gt2pred'], want['pred2gt']  # label -> digest of the reference's list
    got_g2p, got_p2g = sgb_eval.assign_instances_for_scan(evaluator(host_gold, use_label), *scan(1))
    assert got_p2g.keys() == want_p2g.keys() and got_g2p.keys() == want_g2p.keys()
    for label in want_p2g:
        assert matches_digest(got_p2g[label]) == want_p2g[label], label
    for label in want_g2p:
        assert matches_digest(got_g2p[label]) == want_g2p[label], label
    assert sum(len(p['matched_gt']) for v in got_p2g.values() for p in v) == want['n_match'] > 30


def test_evaluate_matches_reference_averages(host_gold):
    """`evaluate` hands the reference's evaluate_matches exactly the matches the reference's own assignment made, so the
    reference computes the stored averages from them."""
    want = host_gold['averages']
    scans = average_scans()
    ev = _MatchRecorder(averages=want, **vars(evaluator(host_gold)))
    got = sgb_eval.evaluate(ev, [s[0] for s in scans], [s[1] for s in scans], verbose=False)
    assert got is want
    assert matches_digest(ev.matches) == host_gold['average_matches']
    assert np.isfinite(want['all_ap_50%'])
