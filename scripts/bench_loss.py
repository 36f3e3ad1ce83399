"""Reprojection loss, forward + backward w.r.t. the weights: the kernels (so_reproj_forward / so_reproj_backward) against
the fp32 composition of the reference's ops (oracle/loss.py: grid_sample, the 4x4 projection, per-ray sums, SSIM, min;
autograd backward) on the same GPU.

Workloads (the shipped configs' loss settings, SSIM and automask on, no deltas):
  nuscenes  ReprojLossMonoMultiNewCombine, 6 cameras x 48 x 100 rays x 256 samples, 900 x 1600 images (7.4 M samples);
  kitti     ReprojLossMonoMultiNew, 1 camera x 44 x 152 rays x 256 samples, 370 x 1216 images (1.7 M samples).
Inputs: tests/test_gpu_loss.real_frame (seeded).  Timing: CUDA events around one forward + backward, warm-up first,
median of --reps; the L2 is flushed before every rep by writing a 512 MB buffer (outside the timed window).  Writes one
JSON document (--out) with the card's name and power limit read in the same run, and the two arms' loss difference.

    python scripts/bench_loss.py --reps 30 --out profiles/r4_bench_loss.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from oracle import loss as ol           # noqa: E402
from selfocc_b200 import ops            # noqa: E402
from test_gpu_loss import real_frame    # noqa: E402

WORKLOADS = {'nuscenes': dict(combine=True, n_cam=6, grid=(48, 100), S=256, img=(900, 1600), seed=0),
             'kitti': dict(combine=False, n_cam=1, grid=(44, 152), S=256, img=(370, 1216), seed=1)}


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else ''
    name, _, power = line.partition(',')
    return {'name': name.strip() or torch.cuda.get_device_name(0), 'power_limit': power.strip() or 'unknown'}


def timed(fn, reps, flush):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.add_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.percentile(ts, 10)), float(np.percentile(ts, 90))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=30)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_loss.py measures on the GPU'
    dev = torch.device('cuda:0')
    flush = torch.empty(128 * 1024 * 1024, device=dev)
    res = {'card': card(), 'reps': a.reps, 'workloads': {}}
    for name, wl in WORKLOADS.items():
        x, img, grid = real_frame(dev, wl['n_cam'], wl['grid'], wl['S'], wl['img'], wl['seed'])
        R = grid[0] * grid[1]
        desc = ops.make_reproj_desc(wl['combine'], wl['n_cam'], R, wl['S'], img, img, grid, True, True)
        imgs = tuple(x[k][0].contiguous() for k in ('curr', 'prev', 'next'))
        w = x['weights'].clone().requires_grad_(True)

        def kernel():
            loss = ops.ReprojLossFunction.apply(w, desc, *imgs, x['pix'], x['img2prev'], x['img2next'], x['ts'], None)
            loss.backward()
            return loss

        def composition():
            loss = ol.reproj_loss_ref(wl['combine'], x['curr'], x['prev'], x['next'], x['pix'], x['img2prev'], x['img2next'],
                                      w, x['ts'], None, img, grid)
            loss.backward()
            return loss

        lk, lc = float(kernel()), float(composition())
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        k = timed(kernel, a.reps, flush)
        mk = torch.cuda.max_memory_allocated() - base
        torch.cuda.reset_peak_memory_stats()
        c = timed(composition, a.reps, flush)
        mc = torch.cuda.max_memory_allocated() - base
        n = wl['n_cam'] * R * wl['S']
        res['workloads'][name] = {
            'samples': n, 'kernel_ms': {'median': k[0], 'p10': k[1], 'p90': k[2]},
            'composition_ms': {'median': c[0], 'p10': c[1], 'p90': c[2]}, 'speedup': c[0] / k[0],
            'kernel_peak_extra_mb': mk / 2 ** 20, 'composition_peak_extra_mb': mc / 2 ** 20,
            # weights + ts read in the forward and again in the backward, g_weights written: the per-sample HBM floor
            'per_sample_bytes_min': 4 * (2 + 2 + 1), 'loss_kernel': lk, 'loss_composition': lc,
            'loss_rel_diff': abs(lk - lc) / abs(lc)}
        print(name, json.dumps(res['workloads'][name]))
    doc = json.dumps(res, indent=1)
    print(doc)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, 'w').write(doc)


if __name__ == '__main__':
    main()
