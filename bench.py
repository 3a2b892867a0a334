#!/usr/bin/env python
"""bench.py -- scans/sec of the SoftGroup per-scan inference hot path on synthetic ScanNet-shape scans.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference ...                     (the reference's CPU path on the host cores)

A "step" is one pass of the hot path over one scan: GPU point->voxel hashing, voxel pooling, sparse U-Net,
point heads, segmented ball query + BFS clustering, cluster re-voxelisation, tiny U-Net + heads, instance
filtering. Workload = BASELINE.json configs[1] (ScanNet-shape, ~150k points, 18 instance classes), one scan
per GPU per step (weak scaling, scans are independent; NCCL only reduces the timing).
Prints ONE JSON line (see the contract in the task description / DESIGN.md section "Measurement").
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'scans/sec on 150k-pt ScanNet-shape synth'
WORKLOAD = 'c2_scannet'
N_POINTS = 150000
# BASELINE.json configs (index -> key). `c2` is the configuration the metric is quoted on and the default; the others are
# the same hot path at the other configs' full sizes (bench lines for context, selected with --workload).
WORKLOADS = {
    'c2': dict(cfg='scannet', shape='c2_scannet', n=150000, sigma=0.03, metric=METRIC,
               what='ScanNet-shape synthetic scan (~150k pts, 18 classes), full SoftGroup inference, one scan per GPU per step'),
    'c2frag': dict(cfg='scannet', shape='c2_scannet', n=150000, sigma=0.03, fragments=6, confusion=0.15,
                   metric=METRIC + ' (fragmented predictions: hundreds of proposals)',
                   what='ScanNet-shape scan as c2, point-wise predictions of a noisy checkpoint: objects split into up to 6 '
                        'fragments, 15 % of the instance points carry a second class'),
    'c3': dict(cfg='s3dis', shape='c3_s3dis', n=800000, sigma=0.03, x4=True, metric='rooms/sec on 800k-pt S3DIS-shape synth',
               what='S3DIS-Area5-shape synthetic room (~800k pts, 13 classes), x4_split backbone, grouping on all points'),
    'c4': dict(cfg='kitti', shape='c4_kitti', n=120000, sigma=0.05, intensity_only=True,
               metric='sweeps/sec on 120k-pt SemanticKITTI-shape synth',
               what='SemanticKITTI-shape synthetic sweep (~120k pts), panoptic config, one sweep per GPU per step'),
    'c5': dict(cfg='stpls3d++', shape='c5_stpls3d', n=1500000, sigma=0.3, no_coords=True,
               metric='tiles/sec on 1.5M-pt STPLS3D-shape synth',
               what='STPLS3D-shape synthetic tile (~1.5M pts), SoftGroup++ pyramid + octree path, one tile per GPU per step'),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--cpu-sample-points', type=int, default=20000)
    ap.add_argument('--workload', default='c2', choices=sorted(WORKLOADS))
    ap.add_argument('--inflight', type=int, default=3,
                    help='scans in flight per GPU in the timed legs (harness.ScanPipeline); 1 = strictly one after another')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the result of the last timed device step (rank 0) as DIR/<name>.npy, for comparing builds')
    return ap.parse_args()


DUMP_BUDGET = 64 << 20


def dump_outputs(out, path):
    """The arrays of a forward_test(device_only=True) result as float32 (floating point) or float64 (integers and masks,
    exact) .npy files. Above DUMP_BUDGET bytes in all, every array keeps a fixed, seeded sample of its rows."""
    flat = dict(out.get('device_instances') or {})
    flat = {'instance_' + k: v for k, v in flat.items()}
    for k in ('semantic_preds', 'pt_offsets', 'proposals_idx', 'proposals_offset'):
        flat[k] = out[k]
    arrs = {}
    for k, v in flat.items():
        a = v.detach().cpu().numpy()
        arrs[k] = a.astype(np.float32 if np.issubdtype(a.dtype, np.floating) else np.float64)
    total = sum(a.nbytes for a in arrs.values())
    if total > DUMP_BUDGET:
        frac = DUMP_BUDGET / float(total)
        for k, a in arrs.items():
            n = a.shape[0]
            rows = np.sort(np.random.RandomState(0).permutation(n)[:int(n * frac)])
            arrs[k] = a[rows]
    os.makedirs(path, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(path, k + '.npy'), a)


# ---------------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md "clocks DURING the timed region")
# ---------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.stop = False
        self.th = None

    def _run(self):
        while not self.stop:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5)
                if out.returncode == 0 and out.stdout.strip():
                    self.rows.append([x.strip() for x in out.stdout.strip().split(',')])
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit())
        mx = [float(r[1]) for r in self.rows if r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for j, n in enumerate(names) if any(r[3 + j].lower().startswith('active') for r in self.rows)]
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(self.rows))


# ---------------------------------------------------------------------------------------------------------
# CPU path (oracle / compiled reference): cpu_baseline leg and --impl reference
# ---------------------------------------------------------------------------------------------------------
def crop_scan(scan, n_keep):
    """Spatially contiguous crop (same point density) holding ~n_keep points; labels re-indexed."""
    from softgroup_b200 import synth  # noqa: F401
    xyz = scan['coords_float']
    n = xyz.shape[0]
    if n_keep >= n:
        return scan
    # grow a box from the x-min side until it holds n_keep points
    order = np.argsort(xyz[:, 0], kind='stable')
    sel = np.sort(order[:n_keep])
    out = {}
    for k, v in scan.items():
        if isinstance(v, np.ndarray) and v.shape[:1] == (n, ):
            out[k] = v[sel]
        else:
            out[k] = v
    c = out['coords'].copy()
    c[:, 1:] -= c[:, 1:].min(0)
    out['coords'] = c
    out['spatial_shape'] = np.clip(c[:, 1:].max(0) + 1, 128, None)
    return out


def cpu_path_once(scan, sd, cfg, use_ref):
    """One pass of the hot path on the host: reference CPU ops where the reference has them (voxelize_idx,
    bfs_cluster -- compiled from its own sources in oracle/_ref), oracle restatements for the ops that are
    CUDA-only in the reference (ball query, voxelize_fp, sec_*) and for the spconv-delegated sparse U-Net.
    Returns (seconds, stage dict)."""
    import torch
    import oracle
    from oracle import spconv_oracle as so
    st = {}
    t0 = time.perf_counter()
    if use_ref is not None:
        c = torch.from_numpy(scan['coords'])
        oc, im, om = c.new(), torch.IntTensor(c.size(0)).zero_(), torch.IntTensor()
        use_ref.voxelize_idx(c, oc, im, om, 1, 4)
        vc, v2p, p2v = oc.numpy(), im.numpy(), om.numpy()
    else:
        vc, v2p, p2v = oracle.voxelization_idx(scan['coords'], 1, 4)
    st['voxelize_idx'] = time.perf_counter() - t0
    t1 = time.perf_counter()
    feats = np.concatenate([scan['feats'], scan['coords_float']], 1).astype(np.float32)
    vfeats = oracle.voxelization(feats, p2v, 4)
    out = so.backbone(vfeats, vc.astype(np.int32), scan['spatial_shape'], sd, cfg['channels'], cfg['num_blocks'])
    pf = out[v2p]
    st['backbone'] = time.perf_counter() - t1
    t2 = time.perf_counter()

    def mlp(x, p):
        h = x @ sd[p + '.0.weight'].T + sd[p + '.0.bias']
        h = so._bn_relu(h, sd, p + '.1')
        return h @ sd[p + '.3.weight'].T + sd[p + '.3.bias']

    sem = mlp(pf, 'semantic_linear')
    off = mlp(pf, 'offset_linear')
    if 'inj_scores' in scan:  # same synthetic point-wise predictions as the GPU arm (computed heads are discarded)
        sem, off = scan['inj_scores'], scan['inj_offsets']
    e = np.exp(sem - sem.max(1, keepdims=True))
    prob = e / e.sum(1, keepdims=True)
    g = cfg['grouping_cfg']
    mean = np.asarray(g['class_numpoint_mean'], np.float32)
    nprop, nact = 0, 0
    st['heads'] = time.perf_counter() - t2
    tb = tq = 0.0
    for c in range(cfg['semantic_classes']):
        if c in g['ignore_classes']:
            continue
        sel = np.where(prob[:, c] > g['score_thr'])[0]
        if sel.size < cfg['test_cfg']['min_npoint']:
            continue
        xyz = (scan['coords_float'][sel] + off[sel]).astype(np.float32)
        t = time.perf_counter()
        idx, sl = oracle.ballquery_batch_p(xyz, np.zeros(sel.size, np.int32), np.array([0, sel.size], np.int32),
                                           g['radius'])
        tq += time.perf_counter() - t
        t = time.perf_counter()
        if use_ref is not None:
            ci, co = torch.IntTensor(), torch.IntTensor()
            use_ref.bfs_cluster(torch.from_numpy(mean), torch.from_numpy(idx if idx.size else np.zeros(1, np.int32)),
                                torch.from_numpy(sl), ci, co, int(sel.size), float(g['npoint_thr']), int(c))
            nprop += co.numel() - 1
        else:
            ci, co = oracle.bfs_cluster(mean, idx, sl, g['npoint_thr'], c)
            nprop += len(co) - 1
        tb += time.perf_counter() - t
        nact += idx.size
    st['ballquery'] = tq
    st['bfs_cluster'] = tb
    total = time.perf_counter() - t0
    st['nProposal'] = nprop
    st['nActive'] = nact
    return total, st


def cpu_leg(args, sd, cfg, scan, steps, warmup):
    import torch
    from oracle.build_ref import load_ref
    try:
        ref = load_ref()
    except Exception:
        ref = None
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    from softgroup_b200 import synth as _synth
    scan = dict(scan)
    scan['inj_scores'], scan['inj_offsets'] = _synth.grouping_inputs(scan, sigma=0.03, seed=args.seed)
    sub = crop_scan(scan, args.cpu_sample_points)
    frac = sub['coords'].shape[0] / float(scan['coords'].shape[0])
    times, stages = [], None
    for it in range(warmup + steps):
        t, st = cpu_path_once(sub, sd, cfg, ref)
        if it >= warmup:
            times.append(t)
            stages = st
    sec = float(np.mean(times))
    kind = 'reference' if ref is not None else 'port'
    sample = ('%d-point spatial crop (%.3f of a %d-point scan) through the CPU path: voxelize_idx + bfs_cluster = %s, '
              'ball query / voxelize_fp / sparse U-Net (spconv) = oracle restatements (CUDA-only or third-party in '
              'the reference); value = crop fraction / seconds; instance head not included' %
              (sub['coords'].shape[0], frac, scan['coords'].shape[0],
               'compiled reference (oracle/_ref)' if ref is not None else 'oracle port'))
    return dict(value=frac / sec, unit='scans/sec', cores=cores, kind=kind, sample=sample,
                ms_per_sample=sec * 1e3, stages_ms={k: (round(v * 1e3, 2) if isinstance(v, float) else v)
                                                    for k, v in stages.items()}), sec


def reference_gpu_ops_leg(scan, cfg, inj, out, reps=3):
    """The reference's OWN CUDA/CPU ops (oracle/_ref: the unmodified softgroup/ops/src compiled for sm_100a) timed on this
    B200 on the tensors of the same scan, called the way softgroup/ops/functions.py and softgroup/model/softgroup.py call
    them (per-class loop, relaunch when the index buffer overflows, lists copied to the host for the CPU BFS). CUDA events
    around each call sequence; median of `reps`. Reported beside `roofline.by_kernel` -- a like-for-like kernel baseline,
    not a target. Returns None when oracle/_ref is not on the box."""
    import torch
    from oracle.build_ref import load_ref
    try:
        ref = load_ref()
    except Exception:
        ref = None
    if ref is None:
        return None
    from softgroup_b200 import ops as our_ops
    g = cfg['grouping_cfg']
    dev = torch.device('cuda')

    def timed(fn):
        ts = []
        for _ in range(reps):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            r = fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append((e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))
        ts.sort()
        return r, ts[len(ts) // 2]

    res = {}
    # ---- voxelize_fp (functions.py:220) ---------------------------------------------------------------------------
    coords = torch.from_numpy(scan['coords']).to(dev)
    vc, v2p, p2v = our_ops.voxelization_idx(coords, 1)
    feats = torch.cat([torch.from_numpy(scan['feats']), torch.from_numpy(scan['coords_float'])], 1).to(dev).contiguous()
    M, C = vc.size(0), feats.size(1)

    def vfp():
        o = torch.zeros((M, C), device=dev)
        ref.voxelize_fp(feats, o, p2v, 4, M, p2v.size(1) - 1, C)
        return o

    _, (ms, wall) = timed(vfp)
    res['voxelize_fp'] = dict(ms=ms, wall_ms=wall)
    # ---- voxelize_idx (CPU hash, functions.py:189; the reference runs it in the dataloader and twice more in the forward)
    ccpu = torch.from_numpy(scan['coords'])

    def vidx():
        oc, im, om = ccpu.new(), torch.IntTensor(ccpu.size(0)).zero_(), torch.IntTensor()
        ref.voxelize_idx(ccpu, oc, im, om, 1, 4)

    _, (ms, wall) = timed(vidx)
    res['voxelize_idx_cpu'] = dict(ms=wall, wall_ms=wall)
    # ---- grouping: per-class ballquery_batch_p (GPU, relaunch loop) + bfs_cluster (CPU, after .cpu()) -------------------
    scores, offs = inj
    prob = scores.softmax(-1)
    cf = torch.from_numpy(scan['coords_float']).to(dev)
    mean = torch.tensor(g['class_numpoint_mean'], dtype=torch.float32)
    classes = [c for c in range(cfg['semantic_classes']) if c not in g['ignore_classes']]

    def grouping():
        t_bq = t_bfs = 0.0
        nact = nprop = 0
        for c in classes:
            obj = (prob[:, c] > g['score_thr']).nonzero().view(-1)
            if obj.size(0) < cfg['test_cfg']['min_npoint']:
                continue
            xyz = (cf[obj] + offs[obj]).contiguous()
            n = xyz.size(0)
            bi = torch.zeros(n, dtype=torch.int32, device=dev)
            bo = torch.tensor([0, n], dtype=torch.int32, device=dev)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mean_active = g['mean_active']
            while True:  # functions.py:258-266
                idx = torch.zeros(n * mean_active, dtype=torch.int32, device=dev)
                sl = torch.zeros((n, 2), dtype=torch.int32, device=dev)
                na = ref.ballquery_batch_p(xyz, bi, bo, idx, sl, n, mean_active, g['radius'])
                if na <= n * mean_active:
                    break
                mean_active = int(na // n + 1)
            idx = idx[:na]
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            ci, co = torch.IntTensor(), torch.IntTensor()
            ref.bfs_cluster(mean, idx.cpu(), sl.cpu(), ci, co, n, float(g['npoint_thr']), int(c))  # softgroup.py:458
            t2 = time.perf_counter()
            t_bq += t1 - t0
            t_bfs += t2 - t1
            nact += int(na)
            nprop += co.numel() - 1
        return t_bq * 1e3, t_bfs * 1e3, nact, nprop

    runs = sorted(grouping() for _ in range(reps))
    t_bq, t_bfs, nact, nprop = runs[len(runs) // 2]
    res['ballquery_batch_p'] = dict(ms=t_bq, nActive=nact, note='per-class calls incl. the overflow relaunches, wall clock around synchronised calls')
    res['bfs_cluster_cpu'] = dict(ms=t_bfs, proposals=nprop, note='includes the D2H of the neighbour lists (softgroup.py:458)')
    # ---- sec_min / sec_max / global_avg_pool on the proposals of this scan -----------------------------------------------
    pidx, poff = out['proposals_idx'], out['proposals_offset'].contiguous()
    if pidx.size(0) > 0:
        pc = cf[pidx[:, 1].long()].contiguous()
        nP = poff.numel() - 1

        def secs():
            a, b = torch.zeros((nP, 3), device=dev), torch.zeros((nP, 3), device=dev)
            ref.sec_min(pc, poff, a, nP, 3)
            ref.sec_max(pc, poff, b, nP, 3)

        _, (ms, wall) = timed(secs)
        res['sec_min+sec_max'] = dict(ms=ms, wall_ms=wall)
        f32 = torch.randn((pidx.size(0), 32), device=dev)

        def gap():
            o = torch.zeros((nP, 32), device=dev)
            ref.global_avg_pool_fp(f32, poff, o, nP, 32)

        _, (ms, wall) = timed(gap)
        res['global_avg_pool_fp'] = dict(ms=ms, wall_ms=wall, rows=int(pidx.size(0)))
    res['note'] = ('unmodified reference ops (oracle/_ref, sm_100a build) on this B200, same scan and injected predictions; '
                   'spconv (third party) is not part of the reference tree and has no entry here')
    return res


# ---------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))

    import torch
    from softgroup_b200 import synth
    from softgroup_b200.configs import model_cfg

    wl = WORKLOADS[args.workload]
    cfg = model_cfg(wl['cfg'])

    def make_workload_scan(seed):
        sc = synth.make_scan(wl['shape'], seed=seed, n_points=wl['n'])
        if wl.get('intensity_only'):
            sc['feats'] = sc['feats'][:, :1].copy()
        if wl.get('no_coords'):
            pass  # with_coords=False in the model config: feats stay rgb
        base = sc
        if wl.get('x4'):
            sc = synth.to_x4_split(sc)
        return sc, base  # base: the scan in point order = the order of the MERGED x4 outputs the predictions are injected in

    if args.impl == 'reference':
        assert args.workload == 'c2', 'the reference arm is defined on the metric configuration (c2)'

        if rank != 0:
            return 0
        from softgroup_b200.model import SoftGroup
        torch.manual_seed(0)
        model = SoftGroup(**cfg).eval()
        # identical synthetic checkpoint protocol, heads calibrated with the CPU fit below
        scan = synth.make_scan(WORKLOAD, seed=args.seed, n_points=N_POINTS)
        sd = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
        sd = calibrate_sd_cpu(sd, cfg, crop_scan(scan, args.cpu_sample_points))
        steps = max(1, min(args.steps, 3))
        warm = min(args.warmup, 1)
        cb, sec = cpu_leg(args, sd, cfg, scan, steps, warm)
        line = dict(metric=METRIC, value=cb['value'], unit='scans/sec', n_gpus=args.gpus, steps=steps, warmup=warm,
                    ms_per_step=sec * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
                    data='synthetic', impl='reference',
                    config=dict(workload='ScanNet-shape synthetic scan (~150k pts, 18 classes), SoftGroup inference',
                                note='reference arm steps are capped at 3 (each step is a bounded CPU sample)'),
                    cpu_baseline=cb,
                    e2e=dict(value=cb['value'], unit='scans/sec', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line))
        return 0

    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback)'
    torch.cuda.set_device(local_rank)
    # The host side of a scan is launch latency, not throughput: no intra-op pool and, with one rank per GPU, every rank on its
    # own share of the cores of ITS GPU's NUMA node (NVML's ideal CPU affinity; the GPUs of the 8-GPU box sit four per node).
    torch.set_num_threads(1)  # (1 / 8 / 128 threads measured the same on one GPU: GPU call 33; 1 keeps 8 ranks x 3 scan threads quiet)
    if world > 1:
        try:
            import pynvml
            pynvml.nvmlInit()
            allowed = set(os.sched_getaffinity(0))
            words = (max(allowed) // 64) + 1

            def cores_of(i):
                uuid = str(torch.cuda.get_device_properties(i).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(('GPU-' + uuid) if not uuid.startswith('GPU-') else uuid)
                mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
                return tuple(sorted(c for c in allowed if (mask[c // 64] >> (c % 64)) & 1))

            n_local = min(world, torch.cuda.device_count())
            sets = [cores_of(i) for i in range(n_local)]
            mine = sets[local_rank]
            group = [i for i in range(n_local) if sets[i] == mine]
            k = group.index(local_rank)
            os.sched_setaffinity(0, set(mine[k::len(group)]))  # strided: a core and its hyper-thread sibling stay with one rank
        except Exception:
            try:  # no NVML: an even split of the allowed cores in rank order
                cores = sorted(os.sched_getaffinity(0))
                per = max(1, len(cores) // world)
                os.sched_setaffinity(0, set(cores[local_rank * per:(local_rank + 1) * per]))
            except Exception:
                pass
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    from softgroup_b200 import harness
    from softgroup_b200.model import SoftGroup
    from softgroup_b200.ops import _lib
    from softgroup_b200 import profiler

    torch.manual_seed(0)
    model = SoftGroup(**cfg).cuda().eval()
    scan, scan_points = make_workload_scan(args.seed + rank)
    hb = harness.to_host_batch(scan, pin=True)
    inj = harness.pointwise_injection(scan_points, sigma=wl['sigma'], seed=args.seed + rank, fragments=wl.get('fragments', 1),
                                      confusion=wl.get('confusion', 0.0))
    dev = harness.device_batch(hb)
    dev_in = {k: v for k, v in dev.items() if k not in ('voxel_coords', 'v2p_map', 'p2v_map')}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')  # 2x the 126 MB L2

    def step_device():
        # inputs resident in HBM; the step includes the GPU hash (point->voxel) and the whole forward
        from softgroup_b200 import ops
        vc, v2p, p2v = ops.voxelization_idx(dev_in['coords'], dev_in['batch_size'])
        d = dict(dev_in)
        d.pop('coords')
        return model.forward_test(device_only=True, inject_pointwise=inj, voxel_coords=vc, v2p_map=v2p, p2v_map=p2v,
                                  **d)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, instrument=False):
        with torch.no_grad():
            out = None
            for _ in range(warmup):
                out = fn()  # (kept while the next call runs, like in the timed loop: the second set of pinned result buffers
                            #  is then allocated here and not by a 25 ms cudaHostAlloc inside the second timed step)
            # every object alive after the warm-up (model, plans, cached tensors) moves to the permanent generation: a full
            # collection of Python's cyclic GC in the middle of a timed step cost 10-20 ms once per leg (one 23-31 ms step
            # among 20 of 10.9 ms end to end, GPU call 40)
            gc.collect()
            gc.freeze()
            barrier()
            evs = []
            t_wall = time.perf_counter()
            for _ in range(steps):
                flush.zero_()  # L2 flush between iterations, outside the per-step events
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                if instrument:
                    profiler.enable()
                e0.record()
                out = fn()
                e1.record()
                if instrument:
                    profiler.disable()
                evs.append((e0, e1))
            barrier()
            wall = time.perf_counter() - t_wall
        per_step = [a.elapsed_time(b) for a, b in evs]
        timed.last_per_step = per_step
        ms = sum(per_step)
        return ms, wall, out

    pipe = harness.ScanPipeline(model, workers=args.inflight) if args.inflight > 1 else None

    def timed_inflight(fn, steps, warmup):
        """`steps` scans with args.inflight of them in flight (one host thread + CUDA stream each, harness.ScanPipeline): the
        timed region runs from an event every worker stream waits on to an event recorded after all of them; the L2 flush of
        every scan is INSIDE it (on the scan's own stream)."""
        with torch.no_grad():
            def call(_):  # results are dropped at once: a retained result dict pins its host buffers, and every later scan
                fn()      # would then pay a fresh cudaHostAlloc for its own
                return None
            pipe.map(call, range(warmup))
            gc.collect()
            gc.freeze()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t_wall = time.perf_counter()
            e0.record()
            res, evs = pipe.map(call, range(steps), start_event=e0, before=flush.zero_)
            for ev in evs:
                torch.cuda.current_stream().wait_event(ev)
            e1.record()
            barrier()
            wall = time.perf_counter() - t_wall
        return e0.elapsed_time(e1), wall

    sampler = ClockSampler(local_rank)
    with sampler:
        l0 = _lib.lib().sgb_launch_count()
        seq_dev_ms, dev_wall, out = timed(step_device, args.steps, max(args.warmup, 3))
        launches = (_lib.lib().sgb_launch_count() - l0)
        seq_dev_steps = sorted(timed.last_per_step)
        if args.dump_outputs and rank == 0:  # before the later legs run the model on this thread again
            dump_outputs(out, args.dump_outputs)
        seq_e2e_ms, e2e_wall, ret = timed(lambda: harness.run_scan(model, hb, inject_pointwise=inj), args.steps, 3)
        seq_e2e_steps = sorted(timed.last_per_step)
        if pipe is not None:
            dev_ms, dev_wall = timed_inflight(step_device, args.steps, max(args.warmup, 3))
            e2e_ms, e2e_wall = timed_inflight(lambda: harness.run_scan(model, hb, inject_pointwise=inj), args.steps, 3)
        else:
            dev_ms, e2e_ms = seq_dev_ms, seq_e2e_ms
        # instrumented pass (per-op CUDA events) -> dominant kernel and its roofline. It runs the module path (one ctypes call
        # per launch, same kernels and arguments as the compiled plan of the timed legs) so that every launch has its own event
        profiler.reset()
        model.use_plan = False
        timed(step_device, min(args.steps, 5), 1, instrument=True)
        model.use_plan = True
    from softgroup_b200 import spconv as _spconv
    _spconv.check_overflow()  # the device-resident legs keep the forward free of host waits: checked once here
    # launches counted over warmup+steps of the first leg -> per timed region
    launches_per_step = launches // (args.steps + max(args.warmup, 3))

    t = torch.tensor([dev_ms, e2e_ms, seq_dev_ms, seq_e2e_ms], dtype=torch.float64, device='cuda')
    per_rank = None
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)  # a few bytes over NCCL: per-rank timings, so that a slow rank is visible in the line
        per_rank = dict(device_ms_per_step=[round(float(x[0]) / args.steps, 3) for x in allt],
                        e2e_ms_per_step=[round(float(x[1]) / args.steps, 3) for x in allt])
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_ms_max = float(t[0]), float(t[1])
    seq_dev_ms_max, seq_e2e_ms_max = float(t[2]), float(t[3])
    value = world * args.steps / (dev_ms_max / 1e3)
    e2e_value = world * args.steps / (e2e_ms_max / 1e3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
        peak_src = 'measured (MEASURED_PEAKS.json)' if 'hbm_gbs' in peaks else 'fallback (B200_PROFILING.md)'
        prof = profiler.summary()
        dom = prof['dominant']
        traffic = None
        traffic_note = None
        try:  # dram__bytes_read+write of the conv launches from the committed OFFLINE ncu capture (per step, like achieved)
            tj = json.load(open(os.path.join(ROOT, 'profiles', 'r2_dominant_kernel_traffic.json')))
            if tj.get('kernel') == dom['name'] and args.workload == 'c2':
                traffic = tj['dram_bytes_per_step']
                traffic_note = tj.get('note')
        except Exception:
            pass
        for k, v in prof['by_kernel'].items():
            v['frac_of_hbm_peak'] = round(v['gbs'] / hbm_peak, 4)
        if args.workload == 'c2' and 'ballquery_batch_p' in prof['by_kernel']:
            # the ball query is bound by instruction issue, not bytes (DESIGN.md 6): its floor from the committed ncu capture
            # (8.2 M warp-level blocks of 32 exact distance tests per scan at >= 9 thread-instructions per test on 148 SMs x 128
            # lanes at 1.965 GHz ~ 63 us; 416 M warp instructions executed at 57 % issue-slot utilisation)
            bq = prof['by_kernel']['ballquery_batch_p']
            bq['issue_floor_us'] = 63.0
            bq['frac_of_issue_floor'] = round(63.0 / max(bq['ms_per_step'] * 1e3, 1e-9), 4)
            bq['issue_floor_source'] = 'offline: profiles/r2_ncu_grouping_per_launch.tsv + the instruction count of the test loop'
        roofline = dict(bound='hbm', kernel=dom['name'], achieved=dom['gbs'], peak=hbm_peak, unit='GB/s',
                        frac=dom['gbs'] / hbm_peak, traffic=traffic, traffic_source=traffic_note, peak_source=peak_src,
                        launches_per_step=dom['launches_per_step'], avg_launch_us=dom['avg_us'],
                        share_of_step=dom['share'], algorithmic_bytes_per_step=dom['bytes_per_step'],
                        by_kernel=prof['by_kernel'])
        d2h = 0
        if isinstance(ret, dict):
            d2h = int(sum(v.nbytes for v in ret.values() if isinstance(v, np.ndarray)))
            d2h += int(sum(len(p['pred_mask']['counts']) for p in ret.get('pred_instances', [])))
        line = dict(metric=wl['metric'], value=value, unit='scans/sec', n_gpus=world, steps=args.steps,
                    warmup=max(args.warmup, 3), ms_per_step=dev_ms_max / args.steps, higher_is_better=True,
                    scaling='weak', vs_baseline=None, dtype='f32', data='synthetic',
                    config=dict(workload=wl['what'], workload_key=args.workload, points=wl['n'],
                                path='%s hyper-parameters (%d channels x %d U-Net levels), random-init weights; point-wise head '
                                'outputs are computed, then overwritten by synthetic predictions (one-hot*8+N(0,1), centroid '
                                'offsets+N(0,sigma)) so grouping sees a trained-checkpoint load' %
                                (wl['cfg'], cfg['channels'], cfg['num_blocks']),
                                l2='flushed: 256 MiB memset (2x the L2) before every scan (between the per-step events of the sequential legs; inside the timed '
                                'region, on the scan\'s own stream, with scans in flight)',
                                parallelism='dp%d (independent scans, no data-path collective)' % world,
                                inflight='%d scans in flight per GPU (host thread + CUDA stream each); one at a time: see '
                                '`sequential`' % args.inflight,
                                proposals=int(out['proposals_offset'].numel() - 1),
                                proposal_points=int(out['proposals_idx'].size(0))),
                    e2e=dict(value=e2e_value, unit='scans/sec', h2d_bytes_per_step=harness.h2d_bytes(hb),
                             d2h_bytes_per_step=d2h, ms_per_step=e2e_ms_max / args.steps),
                    sequential=dict(note='one scan at a time (latency): device step with inputs resident / end to end from '
                                    'pinned host tensors', ms_per_step=seq_dev_ms_max / args.steps,
                                    e2e_ms_per_step=seq_e2e_ms_max / args.steps,
                                    this_rank_ms_min_median_max=[round(seq_dev_steps[0], 3), round(seq_dev_steps[len(seq_dev_steps) // 2], 3),
                                                                 round(seq_dev_steps[-1], 3)],
                                    this_rank_e2e_ms_min_median_max=[round(seq_e2e_steps[0], 3),
                                                                     round(seq_e2e_steps[len(seq_e2e_steps) // 2], 3),
                                                                     round(seq_e2e_steps[-1], 3)],
                                    value=world * args.steps / (seq_dev_ms_max / 1e3),
                                    e2e_value=world * args.steps / (seq_e2e_ms_max / 1e3)),
                    gpu_launches=int(launches_per_step * args.steps), gpu_launches_per_step=int(launches_per_step),
                    clocks=sampler.summary(), roofline=roofline, stage_ms=prof.get('stage_ms'))
        if per_rank is not None:
            line['per_rank'] = per_rank
        if not args.no_cpu_baseline and world == 1 and args.workload == 'c2':
            sd = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
            cb, _ = cpu_leg(args, sd, cfg, scan, 1, 0)
            line['cpu_baseline'] = cb
            try:
                with torch.no_grad():
                    rg = reference_gpu_ops_leg(scan, cfg, inj, out)
                if rg is not None:
                    line['reference_gpu_ops'] = rg
            except Exception as e:  # a baseline leg must never take the bench line down
                line['reference_gpu_ops'] = dict(unavailable=repr(e)[:200])
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def calibrate_sd_cpu(sd, cfg, scan):
    """CPU twin of harness.calibrate_heads for the reference arm (numpy, same ridge fit)."""
    import oracle
    from oracle import spconv_oracle as so
    vc, v2p, p2v = oracle.voxelization_idx(scan['coords'], 1, 4)
    feats = np.concatenate([scan['feats'], scan['coords_float']], 1).astype(np.float32)
    out = so.backbone(oracle.voxelization(feats, p2v, 4), vc.astype(np.int32), scan['spatial_shape'], sd,
                      cfg['channels'], cfg['num_blocks'])
    pf = out[v2p].astype(np.float64)

    def fit(p, target, ridge=1e-3):
        h = pf @ sd[p + '.0.weight'].T.astype(np.float64) + sd[p + '.0.bias']
        h = so._bn_relu(h.astype(np.float32), sd, p + '.1').astype(np.float64)
        A = np.concatenate([h, np.ones((h.shape[0], 1))], 1)
        G = A.T @ A + ridge * h.shape[0] * np.eye(A.shape[1])
        sol = np.linalg.solve(G, A.T @ target)
        sd[p + '.3.weight'] = sol[:-1].T.astype(np.float32)
        sd[p + '.3.bias'] = sol[-1].astype(np.float32)

    onehot = np.zeros((pf.shape[0], cfg['semantic_classes']))
    onehot[np.arange(pf.shape[0]), scan['semantic_labels']] = 6.0
    fit('semantic_linear', onehot)
    off = scan['pt_offset_labels'].astype(np.float64).copy()
    off[scan['instance_labels'] < 0] = 0
    fit('offset_linear', off)
    return sd


if __name__ == '__main__':
    sys.exit(main())
