"""GPU: strong-scaling path (selfocc_b200/dist.py).  Single-GPU tests emulate the ranks one after the other (every kernel
is row-independent, so the sharded result must be BIT-IDENTICAL to the unsharded encoder / decode / render); the torchrun
test runs the real NCCL path when the machine has >= 2 GPUs."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

from test_gpu_pipeline import _setup

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize('world', [2, 3, 8])
def test_query_sharded_lifting_is_bit_identical(world):
    from selfocc_b200.dist import ShardedLifter
    model, cfg, margs, rng, metas, feats, l2i, i2l = _setup()
    dev = torch.device('cuda:0')
    model.to(dev)
    feats = [f.to(dev) for f in feats]
    with torch.no_grad():
        rep = model.lifter(ms_img_feats=feats)['representation']
        ref = model.encoder(representation=rep, ms_img_feats=feats, metas=metas)['representation']
        sl = ShardedLifter(model.encoder)
        st = sl.prepare(feats, metas)
        qfull = torch.cat([p[0] for p in rep], 0).contiguous()
        for li in range(len(model.encoder.layers)):
            bufs = [sl.pad_local(sl.layer_local(li, qfull, st, r, world), r, world) for r in range(world)]
            qfull = sl.assemble(torch.stack(bufs, 0), world)            # what all_gather_into_tensor delivers
        got = torch.split(qfull, sl.sizes, 0)
    for a, b in zip(got, ref):
        assert torch.equal(a, b[0])
    # the per-plane split balances the image cross-attention work: every rank owns ~1/world of EACH plane
    for r in range(world):
        for (b, c), n in zip(sl.slices(r, world), sl.sizes):
            assert c <= -(-n // world)


def test_slab_sharded_decode_is_bit_identical():
    from selfocc_b200 import ops
    from selfocc_b200.dist import ray_slice
    model, cfg, margs, rng, metas, feats, l2i, i2l = _setup(color_dims=3)
    dev = torch.device('cuda:0')
    model.to(dev)
    f = model.head.model.field
    planes = [0.5 * torch.randn_like(p).to(dev) for p in (model.lifter.tpv_hw, model.lifter.tpv_zh, model.lifter.tpv_wz)]
    l1, l2 = f.density_net[1], f.density_net[3]
    args = [p[0].contiguous() for p in planes] + [l1.weight, l1.bias, l2.weight, l2.bias, f.desc]
    with torch.no_grad():
        vs, vf = ops.tpv_decode(*args)
        bs, bf = torch.full_like(vs, float('nan')), torch.full_like(vf, float('nan'))
        for r in range(3):
            ops.tpv_decode(*args, rows=ray_slice(f.desc.H, 3, r), out=(bs, bf))
    assert torch.equal(bs, vs) and torch.equal(bf, vf)


WORKER = r'''
import os, sys, json
import numpy as np
import torch, torch.distributed as dist
sys.path.insert(0, %r); sys.path.insert(0, os.path.join(%r, 'tests'))
from test_gpu_pipeline import _setup
from selfocc_b200.dist import frame_sharded, uniform_sdf_sharded
rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
torch.cuda.set_device(int(os.environ['LOCAL_RANK']))
dev = torch.device('cuda', int(os.environ['LOCAL_RANK']))
dist.init_process_group('nccl', device_id=dev)
model, cfg, margs, rng, metas, feats, l2i, i2l = _setup(color_dims=3)
model.head.num_samples = 64
model.head.render_bkgd = 'white'
model.to(dev)
feats = [f.to(dev) for f in feats]
with torch.no_grad():
    res = model(ms_img_feats=feats, metas=metas, prepare=True)
    one = model.head.render(metas=metas)
    sdf1 = model.head.forward_occ(res['representation'], aabb=rng, resolution=0.5)['sdf']
    got = frame_sharded(model, feats, metas)
    sdfN, _ = uniform_sdf_sharded(model.head, rng, 0.5)
ok = True
ok = ok and torch.equal(got['depth'], one['ms_depths'][0].reshape(-1)) and torch.equal(got['max_depth'], one['ms_max_depths'][0].reshape(-1)) \
    and torch.equal(got['acc'], one['ms_accs'][0].reshape(-1)) and torch.equal(got['rgb'], one['ms_colors'][0].reshape(-1, 3)) \
    and torch.equal(sdfN, sdf1)
flag = torch.tensor([int(ok)], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    print('DIST_OK' if int(flag) == 1 else 'DIST_MISMATCH', world)
dist.destroy_process_group()
'''


def test_frame_sharded_and_lattice_sharded_over_nccl(tmp_path):
    """BASELINE configs[3] ("4 x B200 ray-sharded") / configs[4]: the real collectives.  Needs >= 2 GPUs."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs (torchrun over 2 or 4 ranks)')
    n = 4 if torch.cuda.device_count() >= 4 else 2
    script = tmp_path / 'worker.py'
    script.write_text(WORKER % (ROOT, ROOT))
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(n), '--master-addr',
                        '127.0.0.1', '--master-port', '29741', str(script)], capture_output=True, text=True, timeout=900)
    assert 'DIST_OK %d' % n in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_graphed_frame_single_gpu_equals_eager():
    """GraphedFrame at world size 1 (no collectives): replaying the captured frame reproduces the eager result bit for bit and
    follows the static input buffers."""
    from selfocc_b200.dist import GraphedFrame, frame_sharded
    import numpy as np
    model, cfg, margs, rng, metas, feats, l2i, i2l = _setup(color_dims=3)
    dev = torch.device('cuda:0')
    model.to(dev)
    model.head.num_samples = 64
    model.head.render_bkgd = 'white'
    feats = [f.to(dev) for f in feats]
    metas_d = [dict(lidar2img=torch.tensor(np.asarray(metas[0]['lidar2img']), dtype=torch.float32, device=dev),
                    img2lidar=torch.tensor(np.asarray(metas[0]['img2lidar']), dtype=torch.float32, device=dev), img_shape=metas[0]['img_shape'])]
    with torch.no_grad():
        eager = frame_sharded(model, feats, metas_d)
        gf = GraphedFrame(model, feats, metas_d)
        rep = gf.replay()
        torch.cuda.synchronize()
        for k in eager:
            assert torch.equal(rep[k], eager[k]), k
        for f in feats:                                  # new frame through the same static buffers
            f.mul_(0.5)
        eager2 = frame_sharded(model, feats, metas_d)
        rep2 = gf.replay()
        torch.cuda.synchronize()
        for k in eager2:
            assert torch.equal(rep2[k], eager2[k]), k
        assert not torch.equal(eager2['depth'], eager['depth'])
