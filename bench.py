#!/usr/bin/env python
"""bench.py -- rendered rays/second of the SelfOcc hot path on B200 (see DESIGN.md "Measurement").

A step = ONE pass of the hot path over one synthetic 6-camera frame:
    TPVQueryLifter -> TPVFormerEncoder (4 layers of self + image cross attention) -> NeuSHead.prepare
    (TPV -> decoded volume) -> NeuSHead.render (6 x 900 x 1600 rays x 256 samples -> depth, max-depth, acc, normal, rgb)
i.e. BASELINE.json configs[2] ("nuScenes novel-depth 900x1600 full-res render"), the configuration the
metric "rendered rays/sec (6-cam 900x1600)" is quoted on, with the head of config/nuscenes/nuscenes_novel_depth.py:
color_dims=3 (decode writes 4 channels, colour is composited), render_bkgd='random'.  `--color-dims 0` is the depth-only
head of config/nuscenes/nuscenes_depth.py on the same ray grid (a second workload, stated in config.color_dims).  The image backbone (third-party cuDNN ResNet/FPN) is
outside the hot path: the step starts from synthetic FPN features.

  python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
  python bench.py --impl reference --gpus N ...            # the CPU oracle port (the reference is not installable)
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

N > 1 (torchrun): data-parallel frames exactly like the reference's DDP evaluation -- rank r lifts and renders
its own frame -- plus the north-star's single all_gather of the rendered maps; per-GPU work is fixed (weak scaling).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (ray grid per camera, image size, FPN input (h, w) the level shapes derive from)
    'nuscenes_novel_depth_900x1600': dict(ray_number=(900, 1600), ray_img_size=(900, 1600), fpn_hw=(768, 1600)),
    'nuscenes_depth_450x800': dict(ray_number=(450, 800), ray_img_size=(900, 1600), fpn_hw=(896, 1600)),
    'tiny': dict(ray_number=(32, 32), ray_img_size=(900, 1600), fpn_hw=(128, 256)),
}
# rays kept by --dump-outputs: 11 floats per ray over all outputs (depth, max-depth, acc, normal, rgb, pixel) = 46 MB
DUMP_RAYS = 1 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='nuscenes_novel_depth_900x1600', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-e2e-pipeline', action='store_true', help='e2e with serial copies on the compute stream')
    ap.add_argument('--no-train-probe', action='store_true', help='skip the training-form render forward side figure')
    ap.add_argument('--color-dims', type=int, default=3, choices=[0, 3],
                    help='3: the configs[2] head (nuscenes_novel_depth.py:326); 0: depth-only head (nuscenes_depth.py)')
    ap.add_argument('--no-parity', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='strong mode: issue the sharded frame eagerly instead of replaying a CUDA graph')
    ap.add_argument('--graph', action='store_true', help='strong mode at N > 1: capture the NCCL collectives into the graph too (opt-in)')
    ap.add_argument('--no-strong', action='store_true', help='skip the strong-scaling (one frame sharded over the ranks) measurement')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'], help='which measurement is the headline `value`')
    ap.add_argument('--no-reference-gpu', action='store_true', help='skip the reference-style eager-PyTorch-on-GPU side figure')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the timed step returned in its last step to DIR/<name>.npy '
                         '(float32; a fixed, seeded sample of rays when the frame has more than %d)' % DUMP_RAYS)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be >= 1')
    if a.dump_outputs and a.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    return a


# ------------------------------------------------------------------------------------------ synthetic frame
def make_frame(workload, seed):
    """Synthetic inputs of one frame (SURVEY.md 8d): FPN features ~ N(0,1), the 6-camera nuScenes-like rig."""
    from selfocc_b200 import synth
    w = WORKLOADS[workload]
    g = torch.Generator().manual_seed(seed)
    shapes = synth.fpn_level_shapes(w['fpn_hw'][0] // 2 * 2, w['fpn_hw'][1])
    feats = [torch.randn(1, 6, 96, h, ww, generator=g) for h, ww in shapes]
    l2i, i2l = synth.camera_rig()
    metas = [dict(lidar2img=list(l2i), img2lidar=list(i2l), img_shape=(w['ray_img_size'][0], w['ray_img_size'][1]))]
    return feats, metas, shapes


def build_model(workload, device, color_dims=3):
    from selfocc_b200 import configs
    from selfocc_b200.registry import build_head
    import selfocc_b200.segmentor  # noqa: F401
    w = WORKLOADS[workload]
    torch.manual_seed(0)
    cfg = configs.hot_path_config(ray_number=w['ray_number'], ray_img_size=w['ray_img_size'], return_max_depth=True,
                                  color_dims=color_dims, render_bkgd='random' if color_dims else 'white')
    model = build_head(cfg)
    model.encoder.init_weights()
    with torch.no_grad():
        g = torch.Generator().manual_seed(1)
        for n, p in model.named_parameters():       # "stress" init of SURVEY 8d: non-trivial offsets / softmax
            if 'sampling_offsets.weight' in n or 'attention_weights.weight' in n:
                p.copy_(0.02 * torch.randn(p.shape, generator=g))
        for p in (model.lifter.tpv_hw, model.lifter.tpv_zh, model.lifter.tpv_wz):
            p.mul_(0.1)
        model.head.model.field.deviation_network.variance.fill_(0.3)
    return model.eval().to(device), cfg


def dump_outputs(out, path):
    """NeuSHead.render's return value as path/<key>.npy (float32): one row per (camera, ray) in the frame's flat order, and
    ms_rays, the pixel table every camera shares, as each row's pixel.  A frame of more than DUMP_RAYS rays keeps the same
    seeded sample of DUMP_RAYS rows in every array, so that the dumps of two runs with the same arguments line up.  With the
    random background, ms_colors also depends on how many draws torch's CUDA generator made before the last step, which
    --steps and --warmup change."""
    import numpy as np
    total = out['ms_depths'][0].numel()
    n_pix = out['ms_rays'].shape[0]
    idx = torch.arange(total)
    if total > DUMP_RAYS:
        idx = torch.randperm(total, generator=torch.Generator().manual_seed(0))[:DUMP_RAYS].sort().values
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        t, rows = (v, idx % n_pix) if k == 'ms_rays' else (v[0].reshape(total, *v[0].shape[3:]), idx)
        np.save(os.path.join(path, k + '.npy'), t[rows.to(t.device)].float().cpu().numpy())


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0, set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return None
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': mx, 'reasons': sorted(reasons), 'samples': len(sm)}


# ------------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch.distributed as dist
    from selfocc_b200 import _lib
    from selfocc_b200.dist import all_gather_rays
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    cpu_line = None
    if world == 1 and not args.no_cpu_baseline:
        # BEFORE CUDA is initialised: inside the GPU arm the same port once measured 27x slower than in the reference arm
        # on the same box (CUDA's spinning host threads vs the 128 OpenMP workers) -- see VERDICT r1 weak #11
        cpu_line = cpu_reference(args.workload, steps=5, warmup=1, color_dims=args.color_dims)
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl b200 needs a CUDA device: the hot path has no CPU fallback')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        import datetime
        dist.init_process_group('nccl', device_id=dev, timeout=datetime.timedelta(seconds=180))   # a lost rank must fail, not hang
    assert world == args.gpus or world == 1, 'launch with torchrun --nproc-per-node == --gpus'
    _lib.load()
    model, cfg = build_model(args.workload, dev, args.color_dims)
    has_rgb = args.color_dims >= 3
    feats_h, metas, shapes = make_frame(args.workload, seed=100 + rank)
    feats_h = [f.pin_memory() for f in feats_h]
    feats_d = [f.to(dev) for f in feats_h]
    import numpy as np
    to_dev = lambda k: torch.as_tensor(np.asarray(metas[0][k]), dtype=torch.float32, device=dev)
    metas_d = [dict(lidar2img=to_dev('lidar2img'), img2lidar=to_dev('img2lidar'), img_shape=metas[0]['img_shape'])]
    n_cam, n_ray = 6, model.head.ray_sampler.ray_number
    rays_per_frame = n_cam * n_ray
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    @torch.no_grad()
    def step(feats, m):
        r = model.lifter(ms_img_feats=feats)
        r = model.encoder(representation=r['representation'], ms_img_feats=feats, metas=m)
        model.head.prepare(representation=r['representation'], metas=m)
        return model.head.render(metas=m, batch=0)

    pending = []                                       # (work, buffers): the previous frame's gather, still in flight

    def gather_join():
        while pending:
            pending.pop()[0].wait()

    def gather(out):
        """The one collective of the weak mode (depth / max-depth / RGB of every rank's frame), issued ASYNCHRONOUSLY: NCCL runs
        it on its own stream while the compute stream already lifts the next frame; it is joined one step later (and by
        `gather_join` at the end of the timed region, so every gather is paid for inside the region)."""
        if world == 1:
            return out['ms_depths'][0]
        cols = [out['ms_depths'][0].reshape(-1), out['ms_max_depths'][0].reshape(-1)]
        if has_rgb:
            cols.append(out['ms_colors'][0].reshape(-1))
        local = torch.cat(cols)                                        # planar pack: contiguous copies (an interleaved [R, 5] pack
        full = local.new_empty(world * local.numel())                  # is a strided write of every column, ~1 ms per frame)
        gather_join()                                                  # frame k-1's gather must be done before frame k's starts
        pending.append((dist.all_gather_into_tensor(full, local, async_op=True), (full, local)))
        return full

    def timed(fn, K, W, sampler=None, sample_clocks=False, finalize=None):
        if sampler:
            sampler.start()                                        # nvidia-smi needs ~100s of ms to start: sample from warm-up on
        if sample_clocks:
            for _ in range(20):                                    # extra untimed steps (ALL ranks: fn may hold a collective)
                fn()                                               # so that the clocks are sampled under load
        for _ in range(W):
            flush.zero_()
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        evs = []
        l0 = _lib.launch_count()
        _lib.profile_reset()
        for _ in range(K):
            flush.zero_()                                          # evict L2 between timed steps (untimed)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            evs.append((a, b))
        if finalize is not None:                                   # e.g. join the download stream: still inside the timed region
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            finalize()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)               # max over ranks
        return float(t.item()), _lib.launch_count() - l0, clocks

    K, W = args.steps, max(args.warmup, 3)
    _lib.profile_enable(True)
    sampler = ClockSampler(local) if rank == 0 else None
    last = {}                                          # what the timed step returned last (--dump-outputs)

    def step_eager():
        last['out'] = step(feats_d, metas_d)
        return gather(last['out'])
    total_ms, launches, clocks = timed(step_eager, K, W, sampler, sample_clocks=True,
                                       finalize=gather_join if world > 1 else None)
    prof = _lib.profile_read()
    ms_per_step_eager = total_ms / K
    # The same step replayed from a CUDA graph (one capture per rank: ~95 launches of lift + decode + pack + render; the NCCL
    # gather stays OUTSIDE the graph and reads a fresh packed copy of the outputs).  The eager pass above supplies the per-kernel
    # breakdown (library events cannot be read back from a captured stream) and stays the fallback.
    issue = 'eager issue'
    have_graph = False
    if not args.no_graph:
        try:
            _lib.profile_enable(False)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    step(feats_d, metas_d)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                g_out = step(feats_d, metas_d)
            ok, why = 1, ''
        except Exception as e:
            ok, why = 0, repr(e)[:200]
        if world > 1:
            flag = torch.tensor([ok], device=dev, dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok = int(flag.item())
        have_graph = bool(ok)
        if ok:
            def step_graph():
                graph.replay()
                return gather(g_out)
            total_ms, _, _ = timed(step_graph, K, W, finalize=gather_join if world > 1 else None)
            last['out'] = g_out
            issue = 'CUDA graph replay of the step (collective outside the graph)'
        else:
            issue = 'eager issue (graph capture failed: %s)' % why
    ms_per_step = total_ms / K
    value = world * rays_per_frame / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:              # before anything below replays the graph into g_out again
        dump_outputs(last['out'], args.dump_outputs)

    # ---- strong scaling of ONE frame (SURVEY 8e): query-sharded lifting (one all_gather of the planes per layer), slab-sharded
    # decode, ray-sharded render, one final all_gather -- selfocc_b200/dist.py.  Total work is fixed as N grows.
    strong = None
    if not args.no_strong:
        from selfocc_b200.dist import ShardedLifter, frame_sharded
        _lib.profile_enable(False)
        sl = ShardedLifter(model.encoder)
        feats_0 = feats_d
        if world > 1:                                                  # every rank works on rank 0's frame
            feats_0 = [f.clone() for f in feats_d]
            for f in feats_0:
                dist.broadcast(f, 0)
        # the sharded frame is ~110 launches + 7 collectives for a few ms of GPU work per rank: captured once into a CUDA graph
        # per rank (NCCL included) and replayed; eager issue is the fallback (and is reported next to it)
        from selfocc_b200.dist import GraphedFrame
        s_eager_ms, _, _ = timed(lambda: frame_sharded(model, feats_0, metas_d, lifter=sl), K, W)
        step_strong, mode_s = None, 'eager issue'
        if (world == 1 and not args.no_graph) or args.graph:   # NCCL inside a captured graph is opt-in: see GraphedFrame's docstring
            try:
                gf = GraphedFrame(model, feats_0, metas_d, lifter=sl)
                ok, why = 1, ''
            except Exception as e:
                ok, why = 0, repr(e)[:200]
            if world > 1:
                flag = torch.tensor([ok], device=dev, dtype=torch.int32)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                ok = int(flag.item())
            if ok:
                step_strong, mode_s = gf.replay, 'CUDA graph replay (kernels + NCCL captured per rank)'
            else:
                mode_s = 'eager issue (graph capture failed: %s)' % why
        s_ms = s_eager_ms
        if step_strong is not None:
            s_ms, _, _ = timed(step_strong, K, W)
        strong = {'value': rays_per_frame / (s_ms / K * 1e-3), 'unit': 'rays/s', 'ms_per_step': s_ms / K, 'scaling': 'strong',
                  'frames_per_step': 1, 'issue': mode_s, 'ms_per_step_eager': s_eager_ms / K,
                  'parallelism': 'query-sharded lifting (1 all_gather/layer) + slab-sharded decode + '
                  'ray-sharded render + 1 all_gather over %d rank(s)' % world}
        _lib.profile_enable(True)

    # ---- e2e: same step through the public module API with HOST inputs / outputs inside the timed region
    e2e = None
    if not args.no_e2e:
        out_h = torch.empty(5 if has_rgb else 2, rays_per_frame, dtype=torch.float32).pin_memory()
        rgb_h = out_h[2:].view(rays_per_frame, 3) if has_rgb else None          # [R, 3] like ms_colors

        def fetch(o):
            return (o['ms_depths'][0].reshape(-1), o['ms_max_depths'][0].reshape(-1)) + \
                ((o['ms_colors'][0].reshape(-1, 3),) if has_rgb else ())
        hosts = [out_h[0], out_h[1]] + ([rgb_h] if has_rgb else [])

        # the camera matrices of the step travel from PINNED host memory (non-blocking) into the device tensors the step reads:
        # a pageable upload would synchronise the stream on every call and expose the host's launch time
        l2i_h = torch.as_tensor(np.asarray(metas[0]['lidar2img']), dtype=torch.float32).pin_memory()
        i2l_h = torch.as_tensor(np.asarray(metas[0]['img2lidar']), dtype=torch.float32).pin_memory()

        def metas_upload():
            metas_d[0]['lidar2img'].copy_(l2i_h, non_blocking=True)
            metas_d[0]['img2lidar'].copy_(i2l_h, non_blocking=True)
            return metas_d

        def compute_eager(fd):
            return step(fd, metas_upload())

        def compute_graph(fd):
            """the captured step (it reads feats_d / metas_d and writes g_out): stage this frame's uploaded inputs into the
            graph's input tensors, replay, and hand out copies of the outputs so that the download of frame k does not
            race with the replay of frame k+1 (two device-to-device copies, 58 + 173 MB: ~0.1 ms)"""
            for d_, s_ in zip(feats_d, fd):
                d_.copy_(s_, non_blocking=True)
            metas_upload()
            graph.replay()
            keys = ('ms_depths', 'ms_max_depths') + (('ms_colors',) if has_rgb else ())
            return {k: [g_out[k][0].clone()] for k in keys}
        compute = compute_graph if have_graph else compute_eager
        issue_e2e = 'CUDA graph replay' if have_graph else 'eager issue'

        def step_e2e():
            fd = [f.to(dev, non_blocking=True) for f in feats_h]     # H2D of this step's inputs (pinned)
            out = compute(fd)
            for h, t in zip(hosts, fetch(out)):
                h.copy_(t, non_blocking=True)
            return gather(out) if world > 1 else None
        _lib.profile_enable(False)
        # the same frames through selfocc_b200.pipeline.FramePipeline: upload of frame k+1 and download of frame k overlap
        # the compute of their neighbours (every step still uploads its inputs and downloads its result inside the region)
        step_fn, finalize, mode = step_e2e, (gather_join if world > 1 else None), 'serial copies on the compute stream, ' + issue_e2e
        if not args.no_e2e_pipeline:
            try:
                from selfocc_b200.pipeline import FramePipeline
                pipe = FramePipeline(compute, fetch, hosts, dev)

                def step_pipe():
                    out = pipe.submit(feats_h, next_host=feats_h)
                    return gather(out) if world > 1 else None
                probe = pipe.submit(feats_h, next_host=feats_h)      # one probe frame outside the timed region (no collective)
                pipe.drain()
                torch.cuda.synchronize()
                if not torch.equal(out_h[0], probe['ms_depths'][0].reshape(-1).cpu()):
                    raise RuntimeError('downloaded depth differs from the device result')
                ok, why = 1, ''
            except Exception as e:                                   # never lose the e2e figure to the overlap machinery
                ok, why = 0, ' (FramePipeline failed: %s)' % repr(e)[:200]
                compute, issue_e2e = compute_eager, 'eager issue'
            if world > 1:                                            # all ranks must take the same path: both hold a collective
                flag = torch.tensor([ok], device=dev, dtype=torch.int32)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                ok = int(flag.item())
            if ok:
                step_fn, finalize, mode = step_pipe, (lambda: (pipe.drain(), gather_join())), \
                    'FramePipeline: H2D of frame k+1 / D2H of frame k overlap compute; compute = ' + issue_e2e
            else:
                mode = 'serial copies on the compute stream, ' + issue_e2e + why
        e_ms, _, _ = timed(step_fn, K, W, finalize=finalize)
        h2d = sum(f.numel() * 4 for f in feats_h) + 2 * 6 * 16 * 4
        e2e = {'value': world * rays_per_frame / (e_ms / K * 1e-3), 'unit': 'rays/s', 'ms_per_step': e_ms / K,
               'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': out_h.numel() * 4, 'mode': mode}
        # what this host's PCIe path gives the same pinned buffers with the GPU otherwise idle (outside every timed region):
        # when d2h_bytes / d2h_GBps exceeds the device step, the e2e figure above is bound by the link, not by the kernels
        try:
            probe_d = torch.empty(out_h.shape, device=dev)
            feats_d0 = [torch.empty(f.shape, device=dev) for f in feats_h]
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            torch.cuda.synchronize()
            ev[0].record()
            out_h.copy_(probe_d, non_blocking=True)
            ev[1].record()
            for dd, hh in zip(feats_d0, feats_h):
                dd.copy_(hh, non_blocking=True)
            ev[2].record()
            torch.cuda.synchronize()
            e2e['pcie_probe'] = {'d2h_GBps': out_h.numel() * 4 / (ev[0].elapsed_time(ev[1]) * 1e-3) / 1e9,
                                 'h2d_GBps': sum(f.numel() * 4 for f in feats_h) / (ev[1].elapsed_time(ev[2]) * 1e-3) / 1e9,
                                 'd2h_ms_per_step_alone': ev[0].elapsed_time(ev[1]), 'h2d_ms_per_step_alone': ev[1].elapsed_time(ev[2])}
            del probe_d, feats_d0
        except Exception as e:
            e2e['pcie_probe'] = {'error': repr(e)[:120]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    r_ms, r_calls = prof.get('render_infer', (0.0, 0))
    d = model.head.model.field.desc
    # algorithmic bytes of one render launch (DESIGN.md section 4): per ray the outputs actually written (rays are generated
    # in-kernel: 0 B in) + ONE read of the packed volume the kernel gathers from
    vol_bytes = (d.H * d.W * d.Z * 16) if has_rgb else (d.H * d.W * d.zpitch * 8)
    bytes_per_ray = 4 + 4 + 4 + 12 + (12 + 12 if has_rgb else 0)   # depth, max_depth, acc, normal_vis (+ rgb out, random background in)
    alg_bytes = rays_per_frame * bytes_per_ray + vol_bytes
    dur = (r_ms / max(r_calls, 1)) * 1e-3
    achieved = alg_bytes / dur / 1e9 if dur > 0 else 0.0
    flop_per_ray = 256 * 150.0                # SURVEY 8d estimate: ~150 flop per sample
    roofline = {'kernel': 'render_packed_kernel<RGB=%d>' % int(has_rgb), 'bound': 'hbm', 'achieved': achieved, 'peak': hbm_peak,
                'unit': 'GB/s', 'frac': achieved / hbm_peak, 'peak_source': 'measured' if peaks else 'fallback',
                'launch_ms': dur * 1e3, 'algorithmic_bytes_per_launch': alg_bytes}
    roofline.update(static_ncu_facts(has_rgb, args.workload))
    roofline['note'] = ('inference render is issue-slot bound by construction (~600 flop/B, SURVEY 8d caveat), not HBM-bound: '
                        'fp32 throughput estimate %.1f TFLOP/s; the HBM-bound form of this kernel is `roofline_train_form`'
                        % (rays_per_frame * flop_per_ray / dur / 1e12 if dur > 0 else 0))
    breakdown = {k: round(v[0] / K, 4) for k, v in prof.items()}
    line = {'metric': 'rendered rays/sec (6-cam 900x1600)', 'value': value, 'unit': 'rays/s', 'n_gpus': world, 'steps': K,
            'warmup': W, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic', 'impl': 'b200',
            'config': {'workload': args.workload, 'rays_per_frame': rays_per_frame, 'samples_per_ray': 256,
                       'tpv': '257x257x31x96', 'fpn_levels': shapes, 'encoder_layers': 4,
                       'color_dims': args.color_dims, 'render_bkgd': 'random' if has_rgb else 'white',
                       'outputs': 'depth, max_depth, acc, normal' + (', rgb' if has_rgb else ''),
                       'frames_per_step': world, 'parallelism': 'dp%d frames + 1 all_gather (async, overlaps the next lift)' % world,
                       'l2_flush_between_steps': True, 'issue': issue, 'ms_per_step_eager': ms_per_step_eager},
            'e2e': e2e, 'gpu_launches': int(launches), 'clocks': clocks, 'roofline': roofline,
            'kernel_ms_per_step': breakdown}
    if strong is not None:
        line['strong_scaling'] = strong
        if args.scaling == 'strong':                                   # make the one-frame-sharded number the headline
            line['weak_scaling'] = {'value': value, 'ms_per_step': ms_per_step, 'scaling': 'weak'}
            line.update(value=strong['value'], ms_per_step=strong['ms_per_step'], scaling='strong')
            line['config'].update(frames_per_step=1, parallelism=strong['parallelism'])
    if world == 1 and not args.no_train_probe:
        try:
            line['roofline_train_form'] = train_form_probe(dev, hbm_peak)
        except Exception as e:                 # a side figure must never cost the bench line
            line['roofline_train_form'] = {'error': repr(e)[:300]}
    if world == 1 and not args.no_reference_gpu:
        try:                                   # the north-star's ">= 10x the reference GPU path" anchor, render only
            line['reference_style_gpu'] = reference_style_gpu(dev, args.color_dims, dur, rays_per_frame)
        except Exception as e:
            line['reference_style_gpu'] = {'error': repr(e)[:300]}
    if cpu_line is not None:
        line['cpu_baseline'] = cpu_line
    parity_ok = True
    if world == 1 and not args.no_parity:
        try:                                   # CPU leg: the oracle as checker on the bench workload ("AbsRel vs reference")
            line['parity'] = parity_probe(model, feats_d, metas_d, args.workload, dev, args.color_dims)
        except Exception as e:
            line['parity'] = {'ok': False, 'error': repr(e)[:300]}
        parity_ok = bool(line['parity'].get('ok', False))
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if not parity_ok:
        sys.stderr.write('bench.py: PARITY FAILED (see "parity" in the JSON line)\n')
        sys.exit(3)


def static_ncu_facts(has_rgb, workload):
    """DRAM traffic and pipe utilisation of the render kernel cannot be measured inside a timed run; they come from the committed
    `ncu --set full` capture of this same kernel and workload (profiles/, file named here).  `traffic` stays null until such a
    capture exists for the variant."""
    path = os.path.join(ROOT, 'profiles', 'r2_render_packed_ncu.json')
    out = {'traffic': None, 'traffic_source': None}
    try:
        facts = json.load(open(path))
        f = facts.get(workload, {}).get('rgb' if has_rgb else 'depth')
        if f:
            out = {'traffic': f['dram_bytes_read'] + f['dram_bytes_write'], 'traffic_source': 'static: profiles/r2_render_packed_ncu.json '
                   '(ncu --set full of this kernel at this workload), not a measurement of this run', 'ncu': f}
    except Exception:
        pass
    return out


def reference_style_gpu(dev, color_dims, our_launch_s, rays_per_frame):
    """BASELINE.md section 3 "reference-style GPU path": the oracle port in EAGER PyTorch on this B200 with the reference's own
    structure -- python chunk loop of 90 000 rays (`--batch 90000`), autograd `grid_sample` field query, `cumprod`
    compositing, max-depth on the CPU (neus_head.py:329-374, 430-438).  Stands in for "the reference GPU path" of the
    north-star's >= 10x target (the reference cannot be installed offline).  Render only; bounded sample: 1 camera x
    450 x 800 rays (4 chunks) of the frame's 6 x 900 x 1600, scaled linearly."""
    import numpy as np
    from oracle.mapping import GridMeterMappingRef
    from oracle import render as orender, rays as orays
    from selfocc_b200 import synth
    mref = GridMeterMappingRef(**synth.NUSC_MAPPING)
    H, W, Z = mref.size_h, mref.size_w, mref.size_d
    g = torch.Generator().manual_seed(0)
    vol = (0.55 + 0.11 * torch.randn(1 + color_dims, H, W, Z, generator=g)).to(dev)
    _, i2l = synth.camera_rig()
    i2l = torch.tensor(np.asarray(i2l), dtype=torch.float32, device=dev)[None, :1]
    ny, nx = 450, 800
    pix = orays.fixed_ray_grid([ny, nx], [900, 1600]).to(dev)
    origin, direction = orays.img2lidar_rays(i2l, pix)

    def run():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        orender.head_render_ref(vol, mref, origin, direction, synth.NUSC_RANGE, 20.0, batch=90000, S=256, max_depth_on_cpu=True,
                                color_dims=color_dims, bkgd='white')
        torch.cuda.synchronize()
        return time.perf_counter() - t0
    run()
    ts = sorted(run() for _ in range(3))
    t = ts[1]
    rps = ny * nx / t
    ours = rays_per_frame / our_launch_s if our_launch_s > 0 else 0.0
    return {'impl': 'oracle port, eager PyTorch on this GPU, chunked 90000 rays, CPU max-depth (stands in for the reference GPU path)',
            'sample': '1 cam x %d x %d rays x 256 samples, median of 3' % (ny, nx), 'seconds': t, 'spread_s': [ts[0], ts[-1]],
            'rays_per_s_render_only': rps, 'this_repo_render_rays_per_s': ours, 'render_speedup': ours / rps if rps > 0 else None}


# ------------------------------------------------------------------------------------------ CPU reference arm
def train_form_probe(dev, hbm_peak, iters=10, cf=25, frames=1):
    """North-star side figure (SURVEY 8d caveat): the TRAINING-form render forward -- the kernel that must emit ~6 KB of
    per-sample tensors per ray -- at BASELINE configs[4] sizes (6 cams x 48 x 100 rays x 256 samples, TPV 257x257x25) with the
    REAL head of config/nuscenes/nuscenes_occ.py:350 (color_dims = 24: Cf = 25 decoded channels, rgb + 21 semantic classes
    rendered), timed with the library's CUDA events (L2 flushed before every launch), against the measured HBM peak.
    Algorithmic bytes = SURVEY 8d's per-ray figure (28 + 16 + S * (weights 4 + ts 4 + deltas 4 + eik_grad 12) = 6 188 B/ray,
    178 MB per step); the volume (sdf + 24 feature channels, 165 MB) and jitter reads are reported separately.  Same set-up as
    scripts/bench_train_render.py; the Cf = 1 figure of round 1 is kept as `cf1`."""
    from selfocc_b200 import ops, synth, _lib
    from selfocc_b200.mapping import GridMeterMapping
    margs = dict(synth.NUSC_MAPPING, d_size=[24, 0], d_range=[-4.0, 4.0, 4.0])
    aabb = [-51.2, -51.2, -4.0, 51.2, 51.2, 4.0]
    m = GridMeterMapping(**margs)
    _, i2l = synth.camera_rig()
    i2l = torch.tensor(i2l, dtype=torch.float32, device=dev).repeat(frames, 1, 1)
    ncam = 6 * frames
    ny, nx, S = 48, 100, 256
    n = ncam * ny * nx
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run(cfv):
        n_feat = cfv - 1
        desc = m.volume_desc(n_feat)
        vs = synth.pack_sdf_volume(synth.analytic_sdf_volume(m, noise=0.02), desc.zpitch).to(dev)
        vf = (0.5 * torch.randn(desc.H, desc.W, desc.Z, desc.feat_pitch, device=dev)) if n_feat else None
        jit = torch.rand(n, S + 1, device=dev)
        bk = torch.rand(n, 3, device=dev) if n_feat else None
        invs = torch.tensor([20.0], device=dev)
        want = ['depth', 'acc', 'fars', 'weights', 'ts', 'deltas', 'eik_grad'] + (['rgb'] if n_feat >= 3 else []) + (['sem'] if n_feat > 3 else [])
        cfg = dict(desc=desc, cam_mats=i2l, rays=ops.make_ray_desc(ncam, grid=(ny, nx, 16.0, 3.0, 16.0, 5.0)),
                   params=ops.make_render_params(aabb, S, 20.0, training=True, bkgd='random' if n_feat else 'white'), jitter=jit,
                   bkgd_rand=bk, want=want)
        _lib.profile_enable(True)
        with torch.no_grad():
            for it in range(iters + 3):
                if it == 3:
                    torch.cuda.synchronize()
                    _lib.profile_reset()
                flush.zero_()
                ops.RenderTrainFunction.apply(vs, vf, invs, cfg)
        torch.cuda.synchronize()
        ms, calls = _lib.profile_read()['render_train_fwd']
        fwd_ms = ms / calls
        per_ray = 28 + 16 + S * (4 + 4 + 4 + 12)
        out_extra = n * ((12 if n_feat >= 3 else 0) + 4 * max(n_feat - 3, 0))
        vol_bytes = desc.H * desc.W * desc.zpitch * 4 + (desc.H * desc.W * desc.Z * desc.feat_pitch * 4 if n_feat else 0)
        jit_bytes = n * (S + 1) * 4
        alg = n * per_ray + out_extra
        gbs = alg / (fwd_ms * 1e-3) / 1e9
        return {'launch_ms': fwd_ms, 'algorithmic_bytes_per_launch': alg, 'achieved': gbs, 'frac': gbs / hbm_peak,
                'volume_bytes': vol_bytes, 'jitter_bytes': jit_bytes,
                'frac_incl_volume_and_jitter': (alg + vol_bytes + jit_bytes) / (fwd_ms * 1e-3) / 1e9 / hbm_peak,
                'rays_per_s': n / (fwd_ms * 1e-3)}
    main = run(cf)
    out = {'kernel': 'render_train_fwd_kernel<RGB, SEM=24> (one ray per warp, lane = sample)' if cf == 25 else 'render_train_fwd5_kernel',
           'workload': 'nuscenes_occ_train %dx48x100 rays x256, Cf=%d (config/nuscenes/nuscenes_occ.py:350)' % (ncam, cf),
           'bound': 'hbm', 'peak': hbm_peak, 'unit': 'GB/s', 'bytes_per_ray': 28 + 16 + S * 24}
    out.update(main)
    if cf != 1:
        c1 = run(1)
        out['cf1'] = {k: c1[k] for k in ('launch_ms', 'achieved', 'frac', 'frac_incl_volume_and_jitter', 'rays_per_s')}
        out['cf1']['kernel'] = 'render_train_fwd5_kernel (+ zpair_pack_kernel), depth-only head'
    return out


def parity_probe(model, feats, metas, workload, dev, color_dims, stride=50):
    """CPU leg, the oracle as the CHECKER (never the thing measured): BASELINE's "AbsRel vs reference" on the bench workload
    itself.  The bench model's own TPV planes and MLP go through the fp64 oracle (decode + render) on a strided sub-grid of the
    frame (every `stride`-th pixel of all 6 cameras); the same sub-grid is rendered by the CUDA kernels from the decoded
    volume the timed steps used.  oracle/parity.py explains the three comparisons (geometry / same cells / independent) and why
    the analytic-gradient discontinuity across cell faces makes the split necessary; `ok` is the gate bench.py exits on."""
    from oracle.mapping import GridMeterMappingRef
    from oracle import render as orender, rays as orays
    from oracle.parity import render_parity
    from selfocc_b200 import ops, synth
    import numpy as np
    w = WORKLOADS[workload]
    head = model.head
    f = head.model.field
    with torch.no_grad():
        r = model.lifter(ms_img_feats=feats)
        r = model.encoder(representation=r['representation'], ms_img_feats=feats, metas=metas)
        planes = r['representation']
        head.prepare(representation=planes, metas=metas)
        ny, nx = max(w['ray_number'][0] // stride, 1), max(w['ray_number'][1] // stride, 1)
        H_img, W_img = w['ray_img_size']
        M = head.img2lidar.matrices(metas, dev)[0].contiguous()
        rd = ops.make_ray_desc(M.shape[0], grid=(ny, nx, W_img / nx, 0.0, H_img / ny, 0.0))
        pr = ops.make_render_params(head.aabb, head.num_samples, head._inv_s(), bkgd='white')
        want = ['depth', 'max_idx', 'acc', 'normal_vis'] + (['rgb'] if color_dims else [])
        got = ops.render_infer(f.vol_sdf, f.vol_feat, f.desc, M, rd, pr, want=want, pack=f.render_pack(), probe_grid=True)
        got = {k: v.cpu() for k, v in got.items()}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    torch.set_num_threads(os.cpu_count())
    mref = GridMeterMappingRef(**synth.NUSC_MAPPING)
    l1, l2 = f.density_net[1], f.density_net[3]
    cpu64 = lambda t: t.detach().cpu().double()
    vol = orender.tpv_decode_ref(cpu64(planes[0][0]), cpu64(planes[1][0]), cpu64(planes[2][0]),
                                 (mref.size_h, mref.size_w, mref.size_d), cpu64(l1.weight), cpu64(l1.bias), cpu64(l2.weight), cpu64(l2.bias))
    pix = orays.fixed_ray_grid([ny, nx], [H_img, W_img])
    i2l = torch.tensor(np.asarray(metas[0]['img2lidar']), dtype=torch.float32) if not torch.is_tensor(metas[0]['img2lidar']) \
        else metas[0]['img2lidar'].detach().cpu().float()
    origin, direction = orays.img2lidar_rays(i2l[None], pix)
    rep = render_parity(got, vol, mref, origin, direction, list(head.aabb), head._inv_s(), head.num_samples, color_dims=color_dims,
                        bkgd='white')
    rep.update({'sub_grid': 'every %dth pixel of %d cameras' % (stride, M.shape[0]),
                'oracle': 'fp64 CPU restatement (decode + render) on the bench model\'s own planes and MLP; see oracle/parity.py',
                'oracle_seconds': time.perf_counter() - t0})
    return rep


def cpu_reference(workload, steps, warmup, color_dims=3):
    """The reference's CPU PyTorch path = the oracle port (the reference itself cannot be installed: mmcv / sdfstudio fork
    absent, DESIGN.md).  Bounded sample (~20-40 s of CPU work), linearly extrapolated to the frame:
      lift   : ONE encoder layer on a TPV lattice reduced to 65 x 65 x 9 (same FPN features, same points per pillar), scaled
               by the query-count ratio and x4 layers                    (measured once)
      decode : 32 of the 257 h-rows of the full-size TPV decode, scaled  (measured once)
      render : 1 camera x 45x80 rays of 6 x 900 x 1600, 256 samples, full 257x257x31 volume, reference-style chunk loop
               with the CPU max-depth step                               (every step; MEDIAN of the timed samples, spread reported)
    value = rays_per_frame / (t_lift + t_decode + t_render * scale)."""
    import numpy as np
    from oracle.mapping import GridMeterMappingRef
    from oracle import lifting as ol, render as orender, rays as orays
    from selfocc_b200 import synth
    # 32 OpenMP threads: on the shared 128-core hosts of this pool 128 threads spin against the other tenants and the same
    # sample took 0.28 s .. 11.3 s from run to run (BENCH_r01, profiles/r2_bench_v1_rgb.json); `cores` reports what is used
    torch.set_num_threads(min(32, os.cpu_count()))
    w = WORKLOADS[workload]
    feats, metas, shapes = make_frame(workload, seed=100)
    mref = GridMeterMappingRef(**synth.NUSC_MAPPING)
    H, W, Z = mref.size_h, mref.size_w, mref.size_d
    g = torch.Generator().manual_seed(0)
    rays_per_frame = 6 * w['ray_number'][0] * w['ray_number'][1]
    tiny = workload == 'tiny'
    C = 96
    # --- lifting sample on a reduced lattice
    small = dict(synth.NUSC_MAPPING, h_size=[32, 0], w_size=[32, 0], d_size=[8, 0])
    msm = GridMeterMappingRef(**small)
    q_small = msm.size_h * msm.size_w + 2 * msm.size_d * msm.size_h
    q_full = H * W + Z * H + W * Z
    planes_s = [0.1 * torch.randn(1, n, C, generator=g) for n in (msm.size_h * msm.size_w, msm.size_d * msm.size_h, msm.size_w * msm.size_d)]
    p = _random_encoder_params(C, g)
    l2i = torch.tensor(np.asarray(metas[0]['lidar2img']), dtype=torch.float32)
    cfg = dict(num_freqs=[12] * 3, tot_range=synth.NUSC_RANGE, num_points_cross=[48, 48, 8], num_points_self=12, num_layers=1,
               num_heads=6, num_cams=6)
    t0 = time.perf_counter()
    with torch.no_grad():
        ol.tpv_encoder_ref(p, msm, planes_s, feats, l2i[None], metas[0]['img_shape'], cfg)
    t_lift_s = time.perf_counter() - t0
    t_lift = t_lift_s * (q_full / q_small) * 4
    # --- decode sample
    planes = [0.1 * torch.randn(n, C, generator=g) for n in (H * W, Z * H, W * Z)]
    w1, b1, w2, b2 = synth.random_mlp(C, 1 + color_dims)
    hs = 32
    t0 = time.perf_counter()
    with torch.no_grad():
        orender.tpv_decode_ref(planes[0][:hs * W], planes[1].view(Z, H, C)[:, :hs].reshape(-1, C), planes[2], (hs, W, Z), w1, b1, w2, b2)
    t_dec_s = time.perf_counter() - t0
    t_decode = t_dec_s * H / hs
    vol = 0.55 + 0.11 * torch.randn(1 + color_dims, H, W, Z, generator=g)      # free-space-like scene, like the bench's decoded volume
    # --- per-step bounded render sample
    ny, nx = (8, 8) if tiny else (45, 80)
    pix = orays.fixed_ray_grid([ny, nx], list(w['ray_img_size']))
    i2l = torch.tensor(np.asarray(metas[0]['img2lidar']), dtype=torch.float32)[None, :1]
    origin, direction = orays.img2lidar_rays(i2l, pix)
    scale = rays_per_frame / (ny * nx)

    def render_sample():
        t0 = time.perf_counter()
        orender.head_render_ref(vol, mref, origin, direction, synth.NUSC_RANGE, 20.0, batch=90000, S=256, max_depth_on_cpu=True,
                                color_dims=color_dims, bkgd='white')
        return time.perf_counter() - t0
    for _ in range(warmup):
        render_sample()
    ts = sorted(render_sample() for _ in range(max(steps, 1)))
    t_r = ts[len(ts) // 2]
    frame_s = t_lift + t_decode + t_r * scale
    return {'value': rays_per_frame / frame_s, 'unit': 'rays/s', 'cores': torch.get_num_threads(), 'host_cores': os.cpu_count(), 'kind': 'port',
            'sample': 'oracle port (reference not installable), before CUDA init: 1 encoder layer on a 65x65x9 lattice (%.2fs) scaled x%.1f '
                      'queries x4 layers + decode of %d/%d h-rows (%.2fs) scaled + render of 1 cam x %dx%d rays x 256 samples '
                      '(median %.3fs of %d, min %.3f max %.3f) scaled x%.0f to %d rays, color_dims=%d'
                      % (t_lift_s, q_full / q_small, hs, H, t_dec_s, ny, nx, t_r, len(ts), ts[0], ts[-1], scale, rays_per_frame, color_dims),
            'render_sample_s': ts, 'ms_per_step_extrapolated': frame_s * 1e3, 'threads': torch.get_num_threads()}


def _random_encoder_params(C, g):
    """Parameter dict for one oracle encoder layer (state_dict key names of the reference modules)."""
    p = {}

    def lin(key, o, i, s=0.05):
        p[key + '.weight'] = s * torch.randn(o, i, generator=g)
        p[key + '.bias'] = s * torch.randn(o, generator=g)
    for n in ('hw', 'zh', 'wz'):
        lin('positional_encoding.position_layer_' + n, C, 48)
    p['cams_embeds'] = torch.randn(6, C, generator=g)
    p['level_embeds'] = torch.randn(4, C, generator=g)
    a = 'layers.0.attentions.0.'
    lin(a + 'sampling_offsets', 6 * 3 * 12 * 2, C); lin(a + 'attention_weights', 6 * 3 * 12, C)
    lin(a + 'value_proj', C, C); lin(a + 'output_proj', C, C)
    for n, D in (('attn_hw', 8), ('attn_zh', 48), ('attn_wz', 48)):
        b = 'layers.0.attentions.1.%s.' % n
        lin(b + 'deformable_attention.sampling_offsets', 6 * 4 * D * 2, C)
        lin(b + 'deformable_attention.attention_weights', 6 * 4 * D, C)
        lin(b + 'deformable_attention.value_proj', C, C)
        lin(b + 'output_proj', C, C)
    lin('layers.0.ffns.0.layers.0.0', 2 * C, C); lin('layers.0.ffns.0.layers.1', C, 2 * C)
    for i in range(3):
        p['layers.0.norms.%d.weight' % i] = torch.ones(C)
        p['layers.0.norms.%d.bias' % i] = torch.zeros(C)
    return p


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return                                     # rank 0 alone runs the CPU arm
    K, W = args.steps, args.warmup
    t0 = time.perf_counter()
    cb = cpu_reference(args.workload, steps=K, warmup=min(W, 1), color_dims=args.color_dims)
    w = WORKLOADS[args.workload]
    line = {'metric': 'rendered rays/sec (6-cam 900x1600)', 'value': cb['value'], 'unit': 'rays/s', 'n_gpus': args.gpus,
            'steps': K, 'warmup': W, 'ms_per_step': cb['ms_per_step_extrapolated'], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'impl': 'reference',
            'config': {'workload': args.workload, 'rays_per_frame': 6 * w['ray_number'][0] * w['ray_number'][1],
                       'samples_per_ray': 256, 'tpv': '257x257x31x96', 'color_dims': args.color_dims},
            'cpu_baseline': cb, 'e2e': {'value': cb['value'], 'unit': 'rays/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0, 'wall_s': time.perf_counter() - t0}
    print(json.dumps(line))


if __name__ == '__main__':
    a = parse()
    run_reference(a) if a.impl == 'reference' else run_b200(a)
