"""Occupancy evaluation per frame: the fused path (NeuSHead.occupancy + the histogram metrics) against the fp32
reference composition (get_uniform_sdf lattice + F.grid_sample + argmax + LUT + borders + the reference's per-class
metric loops, oracle/occupancy.py) on the same GPU.

Workloads:
  occ3d   nuscenes_occ.py head (257 x 257 x 25, 3 colour + 21 semantic channels), scene_size 4 at 0.2 m, Occ3D points,
          semantics on, MeanIoU (masked) on the semantic labels;
  kitti   kitti_occ.py head (257 x 257 x 33, colour 3), the KITTI range at 0.4 m and at 0.2 m, IoU + SSCMetrics(2).
Scene: the analytic sdf of selfocc_b200.synth plus seeded random colour / semantic channels (a random-init decode is all
free space).  The decode (so_tpv_decode of random planes, embed dims 96) is common to both arms and timed on its own.

Timing: CUDA events around one frame, warm-up first, median of --reps (>= 20) frames; the L2 is flushed before every
frame by writing a 512 MB buffer (outside the timed window).  Peak memory = torch.cuda.max_memory_allocated growth over
the decoded volume during one frame.  Writes one JSON document (--out) with the card's name and power limit, read in
the same run, and how many labels differ between the two arms.

    python scripts/bench_occ.py --reps 25 --out /tmp/bench_occ.json
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import occupancy as oo                     # noqa: E402
from selfocc_b200 import metric, occupancy, ops, synth  # noqa: E402
from selfocc_b200.head import NeuSHead                 # noqa: E402
from selfocc_b200.mapping import GridMeterMapping      # noqa: E402

NUSC_OCC = dict(nonlinear_mode='linear', h_size=[128, 0], h_range=[40.0, 0], h_half=False, w_size=[128, 0], w_range=[40.0, 0],
                w_half=False, d_size=[24, 0], d_range=[-1.0, 5.4, 5.4])
KITTI_OCC = dict(nonlinear_mode='linear', h_size=[256, 0], h_range=[51.2, 0], h_half=True, w_size=[128, 0], w_range=[25.6, 0],
                 w_half=False, d_size=[32, 0], d_range=[-2.0, 4.4, 4.4])


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else ''
    name, _, power = line.partition(',')
    return {'name': name.strip() or torch.cuda.get_device_name(0), 'power_limit': power.strip() or 'unknown'}


def make_head(margs, aabb, color_dims, return_sem, ground_z, dev):
    head = NeuSHead(roi_aabb=aabb, mapping_args=margs, color_dims=color_dims, return_sem=return_sem, tpv=True, embed_dims=96,
                    sh_deg=0).to(dev)
    f = head.model.field
    m = GridMeterMapping(**margs)
    f.vol_sdf = synth.pack_sdf_volume(synth.analytic_sdf_volume(m, ground_z=ground_z), f.desc.zpitch).to(dev)
    gen = torch.Generator().manual_seed(0)
    feat = torch.randn(color_dims, m.size_h, m.size_w, m.size_d, generator=gen)
    f.vol_feat = synth.pack_feat_volume(feat, f.desc.feat_pitch).to(dev)
    return head, m


def timed(fn, reps, warmup, flush):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times, peaks = [], []
    for _ in range(reps):
        flush.fill_(1.0)                                      # evict the L2 (outside the timed window)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
        peaks.append(torch.cuda.max_memory_allocated() - base)
        del out
    return {'median_ms': float(np.median(times)), 'min_ms': float(np.min(times)), 'max_ms': float(np.max(times)),
            'reps': reps, 'peak_mem_growth_mb': float(max(peaks)) / 2 ** 20}


def decode_time(head, margs, reps, warmup, flush):
    f = head.model.field
    d = f.desc
    m = GridMeterMapping(**margs)
    planes = [p.to(f.vol_sdf.device) for p in synth.random_planes(m, 96, seed=1)]
    w1, b1, w2, b2 = (t.to(f.vol_sdf.device) for t in synth.random_mlp(96, 1 + d.n_feat, seed=1))
    return timed(lambda: ops.tpv_decode(*planes, w1, b1, w2, b2, d), reps, warmup, flush)


def occ3d(args, dev, flush):
    pcr, _ = occupancy.SCENE_SIZES[4]
    head, _ = make_head(NUSC_OCC, pcr, 24, True, 0.07, dev)
    a = math.radians(-90.0)
    e2l = np.array([[math.cos(a), -math.sin(a), 0, 0.0], [math.sin(a), math.cos(a), 0, 0.94], [0, 0, 1, -1.84], [0, 0, 0, 1.]])
    pts = occupancy.occ3d_points(e2l, 4, device=dev)
    z_keep, border = occupancy.OCC3D_BORDERS
    lut = occupancy.OPENSEED2NUSCENES
    lut_t = torch.tensor(lut, device=dev)
    gen = torch.Generator().manual_seed(3)
    gt = torch.randint(0, 18, (200, 200, 16), generator=gen).to(dev)
    gt[gt == 17] = 0
    mask = (torch.rand(200, 200, 16, generator=gen) < 0.6).to(dev)
    names = ['c%d' % i for i in range(16)]
    m = metric.MeanIoU(list(range(1, 17)), 0, names)
    m.reset()
    m_ref = oo.MeanIoURef(list(range(1, 17)), 0, names)

    def fused():
        out = head.occupancy(aabb=pcr, resolution=0.2, points=pts, sem_lut=lut, z_keep=z_keep, border=border)
        m._after_step(out['sem'], gt, mask)
        return out

    def composition():
        sdf, _, logits, _ = head.get_uniform_sdf(pcr, 0.2, dev)
        occ, sem = oo.labels_ref(sdf, 0., logits, pts, lut_t, z_keep, border)
        m_ref._after_step(sem, gt, mask)
        return {'occ': occ, 'sem': sem}

    f, c = fused(), composition()
    diff = {'occ': int((f['occ'].long() != c['occ'].long()).sum()), 'sem': int((f['sem'].long() != c['sem'].long()).sum()),
            'voxels': f['occ'].numel(), 'occupied': int(f['occ'].sum())}
    return {'workload': 'occ3d nuscenes_occ head 257x257x25 (25 ch), scene_size 4, 0.2 m, 200x200x16, semantics + masked MeanIoU',
            'decode': decode_time(head, NUSC_OCC, args.reps, args.warmup, flush),
            'fused': timed(fused, args.reps, args.warmup, flush),
            'composition': timed(composition, args.reps, args.warmup, flush), 'labels_differ': diff}


def kitti(args, dev, flush, res):
    aabb = occupancy.KITTI_RANGE
    head, _ = make_head(KITTI_OCC, aabb, 3, False, -0.87, dev)
    z_keep, border = occupancy.KITTI_BORDERS
    shape = tuple(int((aabb[3 + i] - aabb[i]) / res) for i in (1, 0, 2))
    gen = torch.Generator().manual_seed(4)
    gt = torch.randint(0, 20, shape, generator=gen)
    gt[torch.rand(shape, generator=gen) < 0.6] = 0
    gt[torch.rand(shape, generator=gen) < 0.1] = 255
    gt = gt.to(dev)
    g0 = gt.clone()
    g0[g0 == 255] = 0
    iou, ssc = metric.IoU(), metric.SSCMetrics(2)
    iou.reset()
    iou_ref, ssc_ref = oo.IoURef(), oo.SSCMetricsRef(2)

    def fused():
        out = head.occupancy(aabb=aabb, resolution=res, z_keep=z_keep, border=border)
        iou._after_step(out['occ'], gt)
        ssc.add_batch(out['occ'], gt)
        return out

    def composition():
        sdf, _ = head.get_uniform_sdf(aabb, res, dev)
        occ, _ = oo.labels_ref(sdf, 0., None, None, None, z_keep, border)
        iou_ref._after_step(occ, torch.nonzero(g0))
        ssc_ref.add_batch(occ, gt)
        return {'occ': occ}

    f, c = fused(), composition()
    diff = {'occ': int((f['occ'].long() != c['occ'].long()).sum()), 'voxels': f['occ'].numel(), 'occupied': int(f['occ'].sum())}
    return {'workload': 'kitti kitti_occ head 257x257x33 (4 ch), %.1f m, %dx%dx%d lattice, IoU + SSCMetrics(2)' % ((res,) + shape),
            'decode': decode_time(head, KITTI_OCC, args.reps, args.warmup, flush),
            'fused': timed(fused, args.reps, args.warmup, flush),
            'composition': timed(composition, args.reps, args.warmup, flush), 'labels_differ': diff}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=25)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if args.reps < 20:
        ap.error('--reps must be >= 20')
    if not torch.cuda.is_available():
        raise SystemExit('bench_occ.py needs a CUDA device')
    dev = torch.device('cuda:0')
    flush = torch.empty(512 * 2 ** 20 // 4, device=dev)
    res = {'card': card(), 'torch': torch.__version__, 'timing': 'CUDA events per frame, median of reps after warm-up, '
           'L2 flushed (512 MB write) before every frame', 'workloads': []}
    res['workloads'].append(occ3d(args, dev, flush))
    for r in (0.4, 0.2):
        res['workloads'].append(kitti(args, dev, flush, r))
    for w in res['workloads']:
        w['speedup_median'] = w['composition']['median_ms'] / w['fused']['median_ms']
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
