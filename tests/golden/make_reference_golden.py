"""Generate the golden files of the tests that compare with the original SoftGroup project, by running its unmodified code
on the inputs those tests build:

    python tests/golden/make_reference_golden.py cpu OUT_DIR   the reference's CPU ops (oracle/_ref), its model class on this
                                                                repo's shims (CPU methods), dataset and evaluation code, and
                                                                the configuration files -> ref_host.npz, ref_host.json
    python tests/golden/make_reference_golden.py gpu OUT_DIR   on a B200: the reference's CUDA kernels and its model class on
                                                                this repo's GPU backends -> ref_gpu_kernels.npz, ref_gpu_model.npz

Needs the reference tree (SOFTGROUP_REFERENCE=<checkout of the original repository>) for the cpu part, and the reference
extension + staged model code that oracle/build_ref.py builds from it into oracle/_ref for both parts. The tests
themselves need neither. Copy the outputs into tests/golden/."""
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, 'tests'), HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import oracle  # noqa: E402
from oracle import build_ref  # noqa: E402
from digest import digest, lists_digest  # noqa: E402


class _Cfg(dict):
    """Attribute access on nested config dicts (the reference reads `self.test_cfg.x4_split`, `self.grouping_cfg.radius`:
    tools/test.py builds its configs with Munch)."""
    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError:
            raise AttributeError(name)

    @classmethod
    def wrap(cls, d):
        return cls({k: (cls.wrap(v) if isinstance(v, dict) else v) for k, v in d.items()})


def _ref_ops():
    ref = build_ref.load_ref()
    assert ref is not None, 'oracle/_ref not built (oracle/build_ref.py)'
    return ref


def _ref_model_module():
    m = build_ref.import_reference_model()
    assert m is not None, 'reference model code not staged (oracle/build_ref.py)'
    return m


# ---- GPU: the reference's CUDA kernels ---------------------------------------------------------------------------------
def _c(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _ref_ballquery(ref, xyz, bi, bo, r, mean_active):
    n = xyz.size(0)
    while True:  # functions.py:258-266
        idx = torch.zeros(n * mean_active, dtype=torch.int32, device='cuda')
        sl = torch.zeros((n, 2), dtype=torch.int32, device='cuda')
        na = ref.ballquery_batch_p(xyz, bi, bo, idx, sl, n, mean_active, r)
        if na <= n * mean_active:
            return idx[:na], sl
        mean_active = int(na // n + 1)


def _lists(idx, sl):
    idx, sl = idx.cpu().numpy(), sl.cpu().numpy()
    return [idx[s:s + l] for s, l in sl]


def gpu_kernels():
    import test_gpu_vs_reference as T
    ref = _ref_ops()
    g = {}

    def put_lists(key, lists):
        g[key + '_lens'], g[key + '_digest'] = lists_digest(lists)

    for n, sigma, r in T.BALLQUERY_CASES:
        xyz, bi, bo = T.ballquery_inputs(n, sigma)
        put_lists('bq%d' % n, _lists(*_ref_ballquery(ref, _c(xyz), _c(bi), _c(bo), r, 100)))
    xyz, bi, bo, _ = T.nonfinite_inputs()
    put_lists('bq_nonfinite', _lists(*_ref_ballquery(ref, _c(xyz), _c(bi), _c(bo), 0.04, 100)))
    feats, om = T.voxelize_inputs()
    M = om.shape[0]
    out = torch.zeros((M, 32), device='cuda')
    ref.voxelize_fp(_c(feats), out, _c(om), 4, M, om.shape[1] - 1, 32)
    g['voxelize_fp_digest'] = digest(out.cpu().numpy())
    x, off = T.segment_inputs()
    nP = off.shape[0] - 1
    for name in ('sec_min', 'sec_max', 'sec_mean', 'global_avg_pool_fp'):
        out = torch.zeros((nP, 32), device='cuda')
        getattr(ref, name)(_c(x), _c(off), out, nP, 32)
        g[name] = out.cpu().numpy()
    pidx, off, labels, pointnum, cls, sig = T.mask_inputs()
    nI, nP = pointnum.shape[0], off.shape[0] - 1
    iou = torch.zeros((nP, nI), device='cuda')
    ref.get_mask_iou_on_cluster(_c(pidx), _c(off), _c(labels), _c(pointnum), iou, nI, nP)
    g['mask_iou_on_cluster'] = iou.cpu().numpy()
    iou2 = torch.zeros((nP, nI), device='cuda')
    ref.get_mask_iou_on_pred(_c(pidx), _c(off), _c(labels), _c(pointnum), iou2, nI, nP, _c(sig))
    g['mask_iou_on_pred'] = iou2.cpu().numpy()
    ml = torch.full((int(off[-1]), ), -1.0, device='cuda')
    ref.get_mask_label(_c(pidx), _c(off), _c(labels), _c(cls), iou, nI, nP, 0.02, ml)
    g['mask_label'] = ml.cpu().numpy()
    pts = T.octree_inputs()
    boxes, pt_inds, psl = oracle.build_octree(pts)
    n, mean_active = pts.shape[0], 50
    while True:
        out_inds = torch.zeros(n * mean_active, dtype=torch.int32, device='cuda')
        out_sl = torch.zeros((n, 2), dtype=torch.int32, device='cuda')
        tot = ref.octree_ball_query(_c(pts), _c(boxes), _c(pt_inds), _c(psl), out_inds, out_sl, mean_active, 0.15)
        if tot <= n * mean_active:
            break
        mean_active = int(tot // n + 1)
    put_lists('octree', _lists(out_inds[:tot], out_sl))
    return g


def gpu_model():
    import test_gpu_reference_model as T
    from softgroup_b200 import harness
    from softgroup_b200.ops import functions as F
    ref_module = _ref_model_module()
    # softgroup.py:570 indexes a CPU tensor with a CUDA mask, which the PyTorch 1.x of the reference accepted and
    # PyTorch >= 2 does not
    F.TORCH2_COMPAT = True
    g = {}
    for name, n_points in (('c1', None), ('scannet', 30000), ('scannet++', 20000)):
        cfg, scan, calibrated = T.case(name, n_points)
        ours = T.our_model(cfg, scan, calibrated)
        ref = ref_module.SoftGroup(**_Cfg.wrap(cfg))
        ref.eval()  # the reference overrides train() without returning self (softgroup.py:98-104): no chaining
        ref.load_state_dict(ours.state_dict(), strict=True)
        ref = ref.cuda()
        with torch.no_grad():
            r = ref(dict(harness.collate_like_reference(scan)))  # tools/test.py:148 `result = model(batch)`
        g.update(T.summarize(r, name + '/'))
    F.TORCH2_COMPAT = False
    return g


# ---- CPU: the reference's CPU ops, model methods, dataset, evaluation and configs ---------------------------------------
def _ref_voxelize_idx(ref, coords, batch, mode):
    c = torch.from_numpy(coords)
    oc, im, om = c.new(), torch.IntTensor(c.size(0)).zero_(), torch.IntTensor()
    ref.voxelize_idx(c, oc, im, om, batch, mode)
    return oc.numpy(), im.numpy(), om.numpy()


def _ref_bfs(ref, mean, idx, sl, n, thr, cls):
    ci, co = torch.IntTensor(), torch.IntTensor()
    ref.bfs_cluster(torch.from_numpy(mean), torch.from_numpy(idx), torch.from_numpy(sl), ci, co, n, thr, cls)
    return ci.numpy().reshape(-1, 2), co.numpy()


def host_ops(g):
    import test_oracle as T
    ref = _ref_ops()
    coords, mean, graphs = T.fresh_inputs()
    g['fresh_vox'] = [digest(a) for a in _ref_voxelize_idx(ref, coords, 1, 4)]
    g['fresh_bfs'] = [[digest(a) for a in _ref_bfs(ref, mean, idx, sl, n, 2.0, 0)] for n, idx, sl in graphs]
    for seed in range(4):
        coords, (pts, idx, sl, mean), cl = T.fresh_more_inputs(seed)
        g['more%d_vox' % seed] = [[digest(a) for a in _ref_voxelize_idx(ref, coords, 3, mode)] for mode in (1, 2, 3, 4)]
        g['more%d_bfs' % seed] = [[digest(a) for a in _ref_bfs(ref, mean, idx, sl, pts.shape[0], thr, cls)]
                                  for thr, cls in T.FRESH_BFS_THRESHOLDS]
        rb, rp, rs = torch.zeros(585, 6), torch.zeros(cl.shape[0], dtype=torch.int32), torch.zeros(512, 2, dtype=torch.int32)
        mx, mn = cl.max(0), cl.min(0)  # the Python wrapper passes (centre, extent) of the cloud (functions.py:19-24)
        xyzwhl = torch.from_numpy(np.concatenate([(mx + mn) / np.float32(2), mx - mn]).astype(np.float32))
        ref.build_and_export_octree(torch.from_numpy(cl), xyzwhl, rb, rp, rs, 3)
        g['more%d_octree' % seed] = [digest(a.numpy()) for a in (rb, rp, rs)]


def host_model_methods(g, arrays):
    import test_host_grouping as TG
    import test_host_vs_reference_methods as T
    from softgroup_b200.configs import model_cfg
    from softgroup_b200.model import SoftGroup
    m = _ref_model_module()

    def ref_of(name, **kw):
        cfg = model_cfg(name, **kw)
        ref = m.SoftGroup(**cfg)
        ref.eval()  # the reference's train() override does not return self
        ref.test_cfg = types.SimpleNamespace(**cfg['test_cfg'])  # the reference reads attributes (Munch in tools/test.py)
        ref.grouping_cfg = types.SimpleNamespace(**cfg['grouping_cfg'])
        return ref, cfg

    ref, _ = ref_of('kitti', channels=16, num_blocks=2)
    for seed in range(3):
        sem, insts = T.panoptic_inputs(seed)
        arrays['panoptic_fusion_%d' % seed] = ref.panoptic_fusion(sem.copy(), insts)
    ref, _ = ref_of('scannet', channels=16, num_blocks=2)
    sem, inst = T.gt_instances_inputs()
    arrays['gt_instances'] = np.asarray(ref.get_gt_instances(sem.clone(), inst.clone()))
    ref, _ = ref_of('s3dis', channels=16, num_blocks=2)
    arrays['merge_4_parts'] = ref.merge_4_parts(T.merge_inputs()).numpy()
    ref, _ = ref_of('stpls3d++', channels=16, num_blocks=2)
    g['get_level'] = {str(n): int(ref.get_level(n)) for n in T.LEVEL_SIZES}
    idx, off = ref.pyramid_inverse_map(*T.pyramid_inputs())
    arrays['pyramid_inverse_idx'], arrays['pyramid_inverse_off'] = idx.numpy(), off.numpy()
    # forward_grouping (softgroup.py:411-480) on CPU with its CUDA touch points replaced by oracle stand-ins
    ref, cfg = ref_of('scannet', channels=16, num_blocks=2, test_cfg=dict(min_npoint=30))
    ref.get_batch_offsets = SoftGroup(**cfg).get_batch_offsets

    def ref_bfs(mean, idxs, start_len, thr, class_id):
        a, b = oracle.bfs_cluster(mean.numpy(), idxs.numpy(), start_len.numpy(), thr, class_id)
        return torch.from_numpy(a.astype(np.int32)), torch.from_numpy(b.astype(np.int32))

    m.ball_query, m.bfs_cluster = TG._fake_ball_query, ref_bfs
    want_idx, want_off = ref.forward_grouping(*TG.forward_grouping_inputs(), ref.grouping_cfg)
    arrays['forward_grouping_idx'], arrays['forward_grouping_off'] = want_idx.int().numpy(), want_off.int().numpy()
    # state_dict contract: names and shapes of the reference class (checkpoints load unchanged)
    sd = m.SoftGroup(**model_cfg('scannet')).state_dict()
    g['state_dict'] = [[k, list(v.shape)] for k, v in sd.items()]


def host_configs(g):
    import yaml
    import test_host_logic as T
    g['configs'] = {name: yaml.safe_load(open(os.path.join(build_ref.REF_ROOT, path)))['model']
                    for name, path in T.CONFIG_FILES}


def host_dataprep(g):
    import test_gpu_dataprep as T
    custom, s3dis = build_ref.import_reference_data()
    for n in T.COLLATE_SIZES:
        g['collate_%d' % n] = T.batch_record(T.reference_collate(custom.CustomDataset, T.raw_scan(1, n)))
    g['collate_x4'] = T.batch_record(T.reference_collate(s3dis.S3DISDataset, T.raw_scan(2, 40003, 'c3_s3dis'),
                                                         x4_split=True))


def _plain(x):
    if isinstance(x, dict):
        return {str(k): _plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    if isinstance(x, np.generic):
        return x.item()
    if isinstance(x, np.ndarray):
        return x.tolist()
    return x


def host_evaluation(g):
    import test_gpu_evaluation as T
    from softgroup_b200 import evaluation as sgb_eval
    m = build_ref.import_reference_eval()
    sgb_eval.install_numpy_aliases()
    for use_label in (True, False):
        ev = m.ScanNetEval(T.CLASS_NAMES, use_label=use_label)
        g['evaluator_use_label_%s' % use_label] = dict(
            valid_class_labels=list(ev.valid_class_labels), valid_class_ids=_plain(ev.valid_class_ids),
            id2label=[[int(k), v] for k, v in ev.id2label.items()], eval_class_labels=list(ev.eval_class_labels),
            min_region_sizes=_plain(ev.min_region_sizes), use_label=bool(ev.use_label))
        g2p, p2g = ev.assign_instances_for_scan(*T.scan(1))
        g['assign_use_label_%s' % use_label] = dict(
            gt2pred={k: T.matches_digest(v) for k, v in g2p.items()}, pred2gt={k: T.matches_digest(v) for k, v in p2g.items()},
            n_match=sum(len(p['matched_gt']) for v in p2g.values() for p in v))
    ev = m.ScanNetEval(T.CLASS_NAMES)
    matches = {}
    for i, (preds, gts) in enumerate(T.average_scans()):
        g2p, p2g = ev.assign_instances_for_scan(preds, gts)
        matches['gt_%d' % i] = dict(gt=g2p, pred=p2g)
    g['average_matches'] = T.matches_digest(matches)
    ap, rc = ev.evaluate_matches(matches)
    g['averages'] = _plain(ev.compute_averages(ap, rc))


def main():
    part, out = sys.argv[1], sys.argv[2]
    os.makedirs(out, exist_ok=True)
    if part == 'gpu':
        assert torch.cuda.is_available(), 'the gpu part runs the reference CUDA kernels'
        np.savez_compressed(os.path.join(out, 'ref_gpu_kernels.npz'), **gpu_kernels())
        np.savez_compressed(os.path.join(out, 'ref_gpu_model.npz'), **gpu_model())
    elif part == 'cpu':
        g, arrays = {}, {}
        host_ops(g)
        host_model_methods(g, arrays)
        host_configs(g)
        host_dataprep(g)
        host_evaluation(g)
        np.savez_compressed(os.path.join(out, 'ref_host.npz'), **arrays)
        with open(os.path.join(out, 'ref_host.json'), 'w') as f:
            json.dump(g, f, indent=0, sort_keys=True)
    else:
        raise SystemExit(__doc__)
    print('written to', out)


if __name__ == '__main__':
    main()
