"""Golden vectors for the reprojection losses, from the reference's own loss classes (see ``loss_golden``), and the loss
dicts of the shipped configs (see ``dump_loss_configs``).

Uses the same reference location and loader as ``make_golden.py``; inputs are seeded and stored beside the outputs.
Run once where the reference tree is present:  python tests/golden/make_golden_loss.py
"""
import glob
import json
import os
import sys
import types
import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from make_golden import HERE, REF  # noqa: E402
from oracle.loss import project_ref  # noqa: E402

N_CAM, GRID, S = 2, (4, 5), 16
IMG_SIZE, IMG_HW = (24, 40), (12, 20)     # img_size the pixels are normalised by != the image tensor size


def _reference_losses():
    """Imports loss/reproj_loss_mono_multi_new{,_combine}.py UNMODIFIED with two stand-ins: a ``loss`` package whose
    OPENOCC_LOSS.register_module() is a pass-through decorator (the real package __init__ needs mmengine), and a
    ``utils.tb_wrapper`` whose WrappedTBWriter has no instances (base_loss.py:2-6: no TensorBoard writer)."""
    import importlib

    class _Reg:
        def register_module(self, *a, **k):
            return lambda cls: cls
    pkg = types.ModuleType('loss')
    pkg.__path__ = [os.path.join(REF, 'loss')]
    pkg.OPENOCC_LOSS = _Reg()
    utils = types.ModuleType('utils')
    utils.__path__ = []
    tb = types.ModuleType('utils.tb_wrapper')
    tb.WrappedTBWriter = type('WrappedTBWriter', (), {'_instance_dict': {}})
    sys.modules.update({'loss': pkg, 'utils': utils, 'utils.tb_wrapper': tb})
    comb = importlib.import_module('loss.reproj_loss_mono_multi_new_combine')
    mono = importlib.import_module('loss.reproj_loss_mono_multi_new')
    return comb.ReprojLossMonoMultiNewCombine, mono.ReprojLossMonoMultiNew


def make_inputs(seed=7):
    """Seeded inputs shaped as the training head returns them.  Camera 1 sees both neighbour frames from 2.5 m behind the
    current one (samples with t < ~2.5 project behind the camera; rays 3 and 4 have only such samples, so they hit the
    1e3 rows); sideways shifts send samples outside the image; rays 0 and 1 look from outside img_size, so the current
    frame is sampled on the border.  Samples within 1e-4 (relative) of a mask bound are pushed away from it, so the
    fp64 oracle and the fp32 reference agree on every mask."""
    gen = torch.Generator().manual_seed(seed)
    R = GRID[0] * GRID[1]
    h, w = IMG_SIZE
    imgs = [torch.rand(1, N_CAM, 3, *IMG_HW, generator=gen) for _ in range(3)]
    pix = torch.rand(R, 2, generator=gen) * torch.tensor([w, h])
    pix[0], pix[1] = torch.tensor([-3.0, 5.0]), torch.tensor([w + 4.5, h + 2.0])
    f, cx, cy = 30.0, w / 2, h / 2
    K = torch.tensor([[f, 0, cx, 0], [0, f, cy, 0], [0, 0, 1, 0], [0, 0, 0, 1]], dtype=torch.float64)
    Ts = []
    for cam in range(N_CAM):
        for sgn in (-1.0, 1.0):
            a = 0.05 * sgn + 0.02 * cam
            rot = torch.tensor([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]], dtype=torch.float64)
            E = torch.eye(4, dtype=torch.float64)
            E[:3, :3] = rot
            E[:3, 3] = torch.tensor([0.4 * sgn, 0.1, -2.5 if cam == 1 else 0.3 * sgn], dtype=torch.float64)
            Ts.append((K @ E @ torch.linalg.inv(K)).float())
    T = torch.stack(Ts).reshape(N_CAM, 2, 4, 4)
    ts = 0.5 + 15 * torch.rand(N_CAM, R, S, generator=gen)
    ts[1, 3:5] = 0.1 + 1.5 * torch.rand(2, S, generator=gen)
    for _ in range(20):
        near = torch.zeros_like(ts, dtype=torch.bool)
        for cam in range(N_CAM):
            for j in range(2):
                _, _, _, mg = project_ref(T[cam, j].double(), pix.double(), ts[cam].double(), IMG_SIZE)
                near[cam] |= mg < 1e-4
        if not near.any():
            break
        ts[near] *= 1.013
    weights = torch.rand(N_CAM, R, S, generator=gen)
    deltas = 0.05 + 0.5 * torch.rand(N_CAM, R, S, generator=gen)
    deltas[torch.rand(N_CAM, R, S, generator=gen) < 0.1] = 0.0
    return dict(curr=imgs[0], prev=imgs[1], next=imgs[2], pix=pix, img2prev=T[:, 0].contiguous(), img2next=T[:, 1].contiguous(),
                weights=weights.reshape(N_CAM, -1), ts=ts.reshape(N_CAM, -1), deltas=deltas.reshape(N_CAM, -1))


CASES = [(cls, ssim, am, dl) for cls in ('combine', 'mono') for ssim in (1, 0) for am in (1, 0) for dl in (0, 1)]


def case_name(cls, ssim, am, dl):
    return '%s_ssim%d_am%d_dl%d' % (cls, ssim, am, dl)


def loss_golden():
    """Pins oracle/loss.py and the kernels to ReprojLossMonoMultiNewCombine / ReprojLossMonoMultiNew executed UNMODIFIED
    on the CPU (fp32) over no_ssim x no_automask x deltas, with ray_indices = arange(R).repeat_interleave(S) as the
    head builds them.  Writes tests/golden/reference_golden_loss.npz: the inputs, the loss and d loss / d weights per
    case."""
    Comb, Mono = _reference_losses()
    x = make_inputs()
    out = {k: v.numpy() for k, v in x.items()}
    R = GRID[0] * GRID[1]
    ray_idx = torch.arange(R).repeat_interleave(S)
    for cls, ssim, am, dl in CASES:
        kw = dict(weight=1.0, no_ssim=not ssim, img_size=list(IMG_SIZE), ray_resize=list(GRID), no_automask=not am,
                  input_dict={})
        mod = (Comb if cls == 'combine' else Mono)(**kw)
        weights = [x['weights'][c].clone().requires_grad_(True) for c in range(N_CAM)]
        metas = [{'img2prevImg': x['img2prev'].numpy(), 'img2nextImg': x['img2next'].numpy()}]
        loss = mod.reproj_loss(x['curr'], x['prev'], x['next'], [ray_idx] * N_CAM, weights, list(x['ts']), metas, x['pix'],
                               deltas=list(x['deltas']) if dl else None)
        loss.backward()
        name = case_name(cls, ssim, am, dl)
        out['loss_' + name] = np.array(float(loss))
        out['gw_' + name] = torch.stack([w.grad for w in weights]).numpy()
    np.savez_compressed(os.path.join(HERE, 'reference_golden_loss.npz'), **out)
    print('wrote loss golden:', len(CASES), 'cases')


def dump_loss_configs():
    """The `loss` dict and `loss_input_convertion` of every shipped config (plain `exec` of config/<set>/<name>.py, as in
    make_golden.dump_reference_model_configs).  Written to tests/golden/reference_loss_cfgs.json."""
    out = {}
    for f in sorted(glob.glob(os.path.join(REF, 'config', '*', '*.py'))):
        if '_base_' in f:
            continue
        ns = {}
        exec(compile(open(f).read(), f, 'exec'), ns)
        if 'loss' not in ns:
            continue
        out[os.path.relpath(f, os.path.join(REF, 'config'))] = {'loss': ns['loss'],
                                                                  'loss_input_convertion': ns.get('loss_input_convertion')}
    json.dump(out, open(os.path.join(HERE, 'reference_loss_cfgs.json'), 'w'), indent=1, sort_keys=True)
    print('wrote loss configs of', sorted(out))


if __name__ == '__main__':
    loss_golden()
    dump_loss_configs()
