"""CPU: the training losses -- the fp64 oracle of both reprojection losses against the reference's own classes
(tests/golden/reference_golden_loss.npz), the shipped configs' loss dicts built through MultiLoss / OPENOCC_LOSS, the
plain-torch losses against the oracle, the unsupported knobs, and the error paths of the so_reproj_* entry points."""
import ctypes as C
import json
import os
import numpy as np
import pytest
import torch

from oracle import loss as ol
from selfocc_b200 import loss as sl
from selfocc_b200.registry import Registry

HERE = os.path.dirname(os.path.abspath(__file__))
G = np.load(os.path.join(HERE, 'golden', 'reference_golden_loss.npz'))
CFGS = json.load(open(os.path.join(HERE, 'golden', 'reference_loss_cfgs.json')))
GRID, IMG_SIZE = (4, 5), (24, 40)
CASES = [(cls, ssim, am, dl) for cls in ('combine', 'mono') for ssim in (1, 0) for am in (1, 0) for dl in (0, 1)]
# The golden values are the reference's fp32 arithmetic, the oracle is fp64.  Measured on these inputs: loss within
# 1.7e-7 relative (fp32 rounding of a sum of a few hundred terms); gradient within 1.2e-5 of the largest entry (the
# fp32 reference's SSIM forms sigma = E[x^2] - mu^2 by cancellation, which loses ~1e-5 relative in its derivative).
LOSS_RTOL, GRAD_TOL = 1e-6, 3e-5


def golden_inputs(dtype=torch.float64, device='cpu'):
    return {k: torch.from_numpy(G[k]).to(device=device, dtype=dtype)
            for k in ('curr', 'prev', 'next', 'pix', 'img2prev', 'img2next', 'weights', 'ts', 'deltas')}


def case_name(cls, ssim, am, dl):
    return '%s_ssim%d_am%d_dl%d' % (cls, ssim, am, dl)


@pytest.mark.parametrize('case', CASES, ids=[case_name(*c) for c in CASES])
def test_reproj_oracle_matches_reference(case):
    cls, ssim, am, dl = case
    x = golden_inputs()
    w = x['weights'].clone().requires_grad_(True)
    loss = ol.reproj_loss_ref(cls == 'combine', x['curr'], x['prev'], x['next'], x['pix'], x['img2prev'], x['img2next'], w,
                              x['ts'], x['deltas'] if dl else None, IMG_SIZE, GRID, not ssim, not am)
    loss.backward()
    name = case_name(*case)
    np.testing.assert_allclose(loss.item(), float(G['loss_' + name]), rtol=LOSS_RTOL)
    gw = G['gw_' + name]
    assert np.abs(w.grad.numpy() - gw).max() <= GRAD_TOL * np.abs(gw).max()


def test_golden_covers_the_edge_cases():
    """Behind-camera, out-of-image and no-valid-sample rays are all present, for two cameras."""
    x = golden_inputs()
    R = x['pix'].shape[0]
    t = x['ts'].reshape(2, R, -1)
    behind = outside = 0
    for cam in range(2):
        for T in (x['img2prev'][cam], x['img2next'][cam]):
            c = torch.stack([x['pix'][:, :1] * t[cam], x['pix'][:, 1:] * t[cam], t[cam], torch.ones_like(t[cam])], -1)
            p = c @ T.T
            behind += int((p[..., 2] <= 0).sum())
            _, _, m, _ = ol.project_ref(T, x['pix'], t[cam], IMG_SIZE)
            outside += int(((p[..., 2] > 0) & ~m).sum())
    assert behind > 0 and outside > 0
    d = {}
    ol.reproj_loss_ref(False, x['curr'], x['prev'], x['next'], x['pix'], x['img2prev'], x['img2next'], x['weights'], x['ts'],
                       None, IMG_SIZE, GRID, diag=d)
    assert sum(int((c == 0).all(-1).sum()) for c in d['count']) > 0       # rays on the 1e3 rows
    assert (x['deltas'] == 0).any()                                        # deltas below eps


def test_shipped_configs_build_through_multiloss():
    for name, typ in (('nuscenes/nuscenes_depth.py', sl.ReprojLossMonoMultiNewCombine),
                      ('kitti_raw/kitti_raw_depth.py', sl.ReprojLossMonoMultiNew)):
        cfg = CFGS[name]['loss']
        m = sl.OPENOCC_LOSS.build(cfg)
        assert isinstance(m, sl.MultiLoss) and m.num_losses == len(cfg['loss_cfgs'])
        assert [type(x) for x in m.losses] == [typ, sl.EikonalLoss, sl.EdgeLoss3DMS]
        r = m.losses[0]
        c0 = cfg['loss_cfgs'][0]
        assert (r.weight, r.img_size, r.ray_resize, r.no_ssim) == (c0['weight'], c0['img_size'], c0['ray_resize'], False)
        assert r.input_dict == c0['input_dict'] and r.no_automask == c0.get('no_automask', False)
        assert m.losses[1].weight == 0.1 and m.losses[2].weight == 0.01
    # every shipped config's loss list names only classes this package or (out of scope here) the reference's own
    # registry provides, and every config leads with one of the two reprojection losses
    external = ('RGBLossMS', 'SemLossMS', 'SemCELossMS', 'SparsityLoss', 'HardSparsityLoss', 'SoftSparsityLoss',
                'AdaptiveSparsityLoss')
    for name, c in CFGS.items():
        assert c['loss']['loss_cfgs'][0]['type'] in ('ReprojLossMonoMultiNewCombine', 'ReprojLossMonoMultiNew'), name
        for lc in c['loss']['loss_cfgs']:
            assert lc['type'] in sl.OPENOCC_LOSS or lc['type'] in external, (name, lc['type'])


def test_plain_losses_match_oracle():
    torch.manual_seed(0)
    eik = torch.randn(40, 8, 3, dtype=torch.float64)
    sg = torch.randn(40, 8, 3, dtype=torch.float64)
    assert torch.allclose(sl.EikonalLoss(0.1)({'eik_grad': eik}), 0.1 * ol.eikonal_ref(eik))
    assert torch.allclose(sl.SecondGradLoss(0.01)({'second_grad': sg}), 0.01 * ol.second_grad_ref(sg))
    imgs = torch.rand(1, 2, 3, 12, 20, dtype=torch.float64)
    depth = torch.rand(1, 2, 20, dtype=torch.float64) * 10 + 1
    rays = torch.rand(20, 2, dtype=torch.float64) * torch.tensor([40., 24.], dtype=torch.float64)
    e = sl.EdgeLoss3DMS(0.01, img_size=list(IMG_SIZE), ray_resize=list(GRID))
    got = e({'curr_imgs': imgs, 'ms_depths': [depth], 'ms_rays': rays})
    assert torch.allclose(got, 0.01 * ol.edge_ref(imgs, [depth], rays, IMG_SIZE, GRID))


def test_multiloss_sums_and_reports():
    m = sl.MultiLoss([dict(type='EikonalLoss', weight=0.1), dict(type='SecondGradLoss', weight=0.01)])
    g = torch.randn(10, 4, 3, dtype=torch.float64)
    tot, d = m({'eik_grad': g, 'second_grad': g})
    assert set(d) == {'EikonalLoss', 'SecondGradLoss'}
    assert abs(float(tot) - (d['EikonalLoss'] + d['SecondGradLoss'])) < 1e-12


def test_unsupported_knobs_and_types_raise():
    with pytest.raises(NotImplementedError, match='dims'):
        sl.ReprojLossMonoMultiNewCombine(dims=2)
    with pytest.raises(NotImplementedError, match='sdf_loss'):
        sl.ReprojLossMonoMultiNew(sdf_loss=True)
    with pytest.raises(KeyError):
        sl.OPENOCC_LOSS.build(dict(type='NoSuchLoss'))
    with pytest.raises(KeyError):                   # not provided here: the reference's registry holds it (see below)
        sl.MultiLoss([dict(type='RGBLossMS')])
    assert sl.ReprojLossMonoMultiNewCombine(no_ssim=False, ray_resize=None).no_ssim     # ray_resize=None forces no_ssim
    r = sl.ReprojLossMonoMultiNew(img_size=[24, 40], ray_resize=[4, 5])
    x = golden_inputs(torch.float32)
    ts = [t.clone().requires_grad_(True) for t in x['ts']]
    inputs = dict(curr_imgs=x['curr'], prev_imgs=x['prev'], next_imgs=x['next'], ray_indices=[torch.arange(20).repeat_interleave(16)] * 2,
                  weights=list(x['weights']), ts=ts, metas=[{}], ms_rays=x['pix'])
    with pytest.raises(ValueError, match='ts must not require grad'):
        r(inputs)
    inputs['ts'] = list(x['ts'])
    inputs['weights'] = [x['weights'][0], x['weights'][1][:-1]]
    with pytest.raises(ValueError, match='R \\* S'):
        r(inputs)


def _stub(name):
    """A stand-in for a reference loss this package does not provide: records its constructor kwargs."""
    def __init__(self, weight=1.0, input_dict=None, **kwargs):
        torch.nn.Module.__init__(self)
        self.weight, self.kwargs = weight, kwargs
    return type(name, (torch.nn.Module,), {'__init__': __init__})


def test_register_into_keeps_other_entries():
    reg = Registry('openocc_loss')
    RGBLossMS = _stub('RGBLossMS')

    class MultiLoss:              # a stale entry of the same name is replaced
        pass
    reg.register_module(module=RGBLossMS)
    reg.register_module(module=MultiLoss)
    sl.register_into(reg)
    assert reg.get('RGBLossMS') is RGBLossMS
    assert issubclass(reg.get('MultiLoss'), sl.MultiLoss) and reg.get('MultiLoss').registry is reg
    for cls in sl.LOSSES[1:]:
        assert reg.get(cls.__name__) is cls
    assert sl.OPENOCC_LOSS.get('MultiLoss') is sl.MultiLoss         # the package's own entry is untouched


def test_every_shipped_loss_dict_builds_through_a_registry_it_was_registered_into():
    """train.py:116 builds cfg.loss from the reference's OPENOCC_LOSS: after register_into, the MultiLoss found there
    must build the reference-only entries (RGBLossMS, Sem*, SoftSparsityLoss) from that same registry."""
    reg = Registry('openocc_loss')
    stubs = {n: _stub(n) for n in ('RGBLossMS', 'SemLossMS', 'SemCELossMS', 'SparsityLoss', 'HardSparsityLoss',
                                   'SoftSparsityLoss', 'AdaptiveSparsityLoss')}
    for cls in stubs.values():
        reg.register_module(module=cls)
    sl.register_into(reg)
    assert len(CFGS) >= 6
    for name, c in CFGS.items():
        m = reg.build(c['loss'])
        assert [type(x).__name__ for x in m.losses] == [lc['type'] for lc in c['loss']['loss_cfgs']], name
        for x, lc in zip(m.losses, c['loss']['loss_cfgs']):
            assert type(x) is (stubs.get(lc['type']) or reg.get(lc['type'])), (name, lc['type'])
            assert x.weight == lc.get('weight', 1.0), (name, lc['type'])


def test_reproj_entry_points_reject_bad_arguments_without_a_gpu():
    from selfocc_b200 import _lib, build
    build.build()
    lib = _lib.load()
    N, one = None, C.c_void_p(16)

    def desc(**k):
        d = _lib.ReprojDesc()
        d.variant, d.n_cam, d.n_rays, d.n_samples, d.img_h, d.img_w = 0, 2, 20, 16, 12, 20
        d.size_h, d.size_w, d.grid_h, d.grid_w, d.ssim, d.automask = 24., 40., 4, 5, 1, 1
        for a, v in k.items():
            setattr(d, a, v)
        return d
    assert lib.so_reproj_workspace_floats(C.byref(desc())) == 2 * 20 * 53
    for bad in (dict(variant=2), dict(n_cam=0), dict(n_samples=0), dict(img_w=0), dict(size_h=0.), dict(grid_w=4),
                dict(grid_h=1, grid_w=20)):
        assert lib.so_reproj_workspace_floats(C.byref(desc(**bad))) == -1, bad
    assert lib.so_reproj_workspace_floats(C.byref(desc(grid_w=4, ssim=0))) > 0       # the grid is only read for SSIM
    fwd = lambda d, **k: lib.so_reproj_forward(C.byref(d), *[k.get(n, one) for n in ('curr', 'prev', 'next', 'pix', 'tp', 'tn', 'w', 'ts')],
                                               k.get('deltas', N), k.get('loss', one), k.get('ws', one), N)
    assert fwd(desc(), curr=N) == -1
    assert fwd(desc(), ts=N) == -1
    assert fwd(desc(), loss=N) == -1
    assert fwd(desc(), ws=N) == -1
    assert fwd(desc(grid_w=3)) == -1
    assert lib.so_reproj_forward(N, *[one] * 8, N, one, one, N) == -1
    bwd = lambda d, **k: lib.so_reproj_backward(C.byref(d), *[one] * 8, N, k.get('g', one), k.get('gw', one), one, N)
    assert bwd(desc(), g=N) == -1
    assert bwd(desc(), gw=N) == -1
    assert bwd(desc(n_rays=0)) == -1
    assert lib.so_reproj_check_layout(N, 10, 2, one, N) == -1
    assert lib.so_reproj_check_layout(one, 10, 0, one, N) == -1
    assert lib.so_reproj_check_layout(one, 10, 2, N, N) == -1
    assert lib.so_reproj_check_layout(one, 0, 2, one, N) == 0                        # n = 0: nothing to do
