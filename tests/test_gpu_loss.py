"""GPU: the reprojection-loss kernels (so_reproj_*) against the fp64 oracle and the fp32 composition (oracle/loss.py) on
the golden inputs and at the nuScenes / KITTI sizes, end to end through NeuSHead.forward, bit-reproducibility, the
ray-layout guard, and the absence of host syncs in a loss step."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import loss as ol
from selfocc_b200 import ops

GOLD_GRID, GOLD_SIZE = (4, 5), (24, 40)
OPTS = [(c, ssim, am, dl) for c in (True, False) for ssim in (1, 0) for am in (1, 0) for dl in (0, 1)]
OPT_IDS = ['%s_ssim%d_am%d_dl%d' % ('combine' if c else 'mono', s, a, d) for c, s, a, d in OPTS]
# Tolerances.  A mask is a comparison of an fp32 projection with a bound: the kernel's fp32 matmul order is not the
# composition's, so a mask may differ where the projected coordinate is within fp32 rounding of the bound -- accepted
# only where the oracle puts some sample of the ray within MARGIN of a bound (relative), and reported.
MARGIN = 1e-5
# Values are held to the reference's own fp32 arithmetic: the kernel's distance to the fp64 oracle may be at most
# SLACK times that of the fp32 composition (same inputs, same GPU), plus a floor.  The measured cause of that distance:
# the reference forms the sample position as ((2 u / 1600 - 1) + 1) / 2 * 1599 in fp32, ~2e-4 px off at 900 x 1600,
# which moves a bilinear sample of these seeded (unsmoothed) images by up to ~2e-4 -- 3e-4 relative in a per-ray loss.
# The chosen branch may differ only where the two smallest candidates are closer than TIE_SLACK times that per-ray
# distance.  On the golden inputs (24 x 40 pixels) the kernel is within 2e-5 of the oracle outright.
SLACK, TIE_SLACK, FLOOR = 2.0, 4.0, 1e-6
LOSS_RTOL, GRAD_TOL = 2e-5, 1e-4


def _dev():
    if not torch.cuda.is_available():
        pytest.skip('needs CUDA')
    return torch.device('cuda:0')


def golden_frame(dev, dtype=torch.float32):
    import os
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_golden_loss.npz'))
    x = {k: torch.from_numpy(G[k]).to(dev, dtype) for k in ('curr', 'prev', 'next', 'pix', 'img2prev', 'img2next', 'weights',
                                                            'ts', 'deltas')}
    return x, GOLD_SIZE, GOLD_GRID


def real_frame(dev, n_cam, grid, S, img_hw, seed=0):
    """A frame at a shipped size: pixels on the ray grid, depths 1..60 m, neighbour frames 0.6 m behind / ahead with a
    small yaw, pinhole cameras of focal 0.8 * width."""
    g = torch.Generator().manual_seed(seed)
    h, w = img_hw
    gh, gw = grid
    R = gh * gw
    ii, jj = torch.meshgrid(torch.arange(gh), torch.arange(gw), indexing='ij')
    pix = torch.stack([(jj.flatten() + torch.rand(R, generator=g)) * w / gw, (ii.flatten() + torch.rand(R, generator=g)) * h / gh], -1)
    f = 0.8 * w
    K = torch.tensor([[f, 0, w / 2, 0], [0, f, h / 2, 0], [0, 0, 1, 0], [0, 0, 0, 1]], dtype=torch.float64)
    Ts = []
    for cam in range(n_cam):
        for sgn in (-1.0, 1.0):
            a = 0.02 * sgn * (1 + cam % 3)
            E = torch.eye(4, dtype=torch.float64)
            E[0, 0], E[0, 2], E[2, 0], E[2, 2] = np.cos(a), np.sin(a), -np.sin(a), np.cos(a)
            E[:3, 3] = torch.tensor([0.1 * sgn, 0.02, -0.6 * sgn], dtype=torch.float64)
            Ts.append((K @ E @ torch.linalg.inv(K)).float())
    T = torch.stack(Ts).reshape(n_cam, 2, 4, 4)
    edges = torch.sort(1 + 59 * torch.rand(n_cam, R, S + 1, generator=g), -1).values
    ts = 0.5 * (edges[..., 1:] + edges[..., :-1])
    deltas = edges[..., 1:] - edges[..., :-1]
    wts = torch.rand(n_cam, R, S, generator=g) ** 4 / S * 4
    x = dict(curr=torch.rand(1, n_cam, 3, h, w, generator=g), prev=torch.rand(1, n_cam, 3, h, w, generator=g),
             next=torch.rand(1, n_cam, 3, h, w, generator=g), pix=pix, img2prev=T[:, 0].contiguous(), img2next=T[:, 1].contiguous(),
             weights=wts.reshape(n_cam, -1), ts=ts.reshape(n_cam, -1), deltas=deltas.reshape(n_cam, -1))
    return {k: v.to(dev) for k, v in x.items()}, img_hw, grid


def run_kernel(x, combine, ssim, am, dl, img_size, grid):
    N, R = x['curr'].shape[1], x['pix'].shape[0]
    S = x['weights'].shape[1] // R
    desc = ops.make_reproj_desc(combine, N, R, S, x['curr'].shape[-2:], img_size, grid if ssim else None, ssim, am)
    args = (x['curr'][0].contiguous(), x['prev'][0].contiguous(), x['next'][0].contiguous(), x['pix'], x['img2prev'],
            x['img2next'], x['weights'], x['ts'], x['deltas'] if dl else None)
    loss, ws = ops.reproj_forward(desc, *args)
    g = ops.reproj_backward(desc, *args, torch.ones(1, device=loss.device), ws)
    v = ops.reproj_workspace_views(desc, ws)
    return loss[0], g, {k: t.clone() for k, t in v.items()}


def run_ref(x, combine, ssim, am, dl, img_size, grid, dtype):
    y = {k: t.to(dtype) for k, t in x.items()}
    w = y['weights'].clone().requires_grad_(True)
    d = {}
    loss = ol.reproj_loss_ref(combine, y['curr'], y['prev'], y['next'], y['pix'], y['img2prev'], y['img2next'], w, y['ts'],
                              y['deltas'] if dl else None, img_size, grid, not ssim, not am, diag=d)
    loss.backward()
    return loss.detach(), w.grad, {k: torch.stack(v) for k, v in d.items()}


def _dilate(m, grid, k):
    """rays within a k x k window of a flagged ray on the ray grid"""
    N = m.shape[0]
    return torch.nn.functional.max_pool2d(m.reshape(N, 1, *grid).float(), k, 1, k // 2).reshape(N, -1) > 0.5


def compare(x, opts, img_size, grid, report, real=False):
    """Kernel vs the fp64 oracle; at the real sizes held to the fp32 composition's own distance from the oracle."""
    combine, ssim, am, dl = opts
    loss, g, kv = run_kernel(x, *opts, img_size, grid)
    rloss, rg, d = run_ref(x, *opts, img_size, grid, torch.float64)
    closs, cg, dc = run_ref(x, *opts, img_size, grid, torch.float32)
    N, R = kv['proj'].shape
    near = (d['margin'] < MARGIN).any(-1)
    mask_bad = (kv['counts'] != d['count'].to(torch.float32)).any(-1)            # [N, R]
    cmask_bad = (dc['count'] != d['count']).any(-1)
    assert not (mask_bad & ~near).any(), 'mask disagreement away from a bound on %d rays' % int((mask_bad & ~near).sum())
    # with SSIM a ray's candidates read its 3 x 3 neighbours' composed colours: a mask disagreement there moves them too
    dil = (lambda m: _dilate(m, grid, 3)) if ssim else (lambda m: m)
    cand = d['cand']
    pr = cand.gather(-1, d['choice'][..., None])[..., 0].double()
    pc = dc['cand'].gather(-1, dc['choice'][..., None])[..., 0].double()
    cok = ~(dil(cmask_bad) | (dc['choice'] != d['choice']))
    e_comp = float((pc - pr)[cok].abs().max()) if real else 0.
    top2 = cand.sort(-1).values[..., :2] if cand.shape[-1] > 1 else cand.repeat(1, 1, 2)
    gap = (top2[..., 1] - top2[..., 0]).abs()
    ch_bad = kv['choice'].long() != d['choice']
    odd = ch_bad & (gap > max(TIE_SLACK * e_comp, LOSS_RTOL * float(top2[..., 0].abs().max()))) & ~dil(mask_bad)
    assert not odd.any(), 'branch disagreement away from a tie on %d rays, gaps %s' % (int(odd.sum()), gap[odd].tolist())
    bad = dil(mask_bad) | ch_bad
    ok = ~bad
    e_kern = float((kv['proj'].double() - pr)[ok].abs().max())
    assert e_kern <= SLACK * e_comp + LOSS_RTOL * float(pr.abs().max()), (e_kern, e_comp)
    slack = float((kv['proj'][bad].double() - pr[bad]).abs().sum()) / (N * R)
    assert abs(float(loss) - float(rloss)) <= SLACK * abs(float(closs) - float(rloss)) + LOSS_RTOL * abs(float(rloss)) + slack
    # gradients on the rays whose whole SSIM neighbourhood (two grid cells) agrees in both fp32 arms
    cbad = dil(cmask_bad) | (dc['choice'] != d['choice'])
    keep = ~_dilate(bad | cbad, grid, 5) if ssim else ~(bad | cbad)
    S = g.shape[1] // R
    rk = rg.reshape(N, R, S)[keep]
    scale = max(float(rk.abs().max()), 1e-30)
    err = float((g.reshape(N, R, S)[keep].double() - rk).abs().max()) / scale
    cerr = float((cg.reshape(N, R, S)[keep].double() - rk).abs().max()) / scale if real else 0.
    report.append(dict(mask=int(mask_bad.sum()), branch=int(ch_bad.sum()), e_kern=e_kern, e_comp=e_comp, g_kern=err, g_comp=cerr))
    assert err <= SLACK * cerr + GRAD_TOL, (err, cerr)
    return loss, g


@pytest.mark.parametrize('opts', OPTS, ids=OPT_IDS)
def test_small_against_fp64_oracle_and_fp32_composition(opts):
    dev = _dev()
    x, size, grid = golden_frame(dev)
    rep = []
    compare(x, opts, size, grid, rep)
    print('small', opts, rep)
    assert rep[0]['mask'] == rep[0]['branch'] == 0       # the golden inputs keep every sample 1e-4 away from the bounds


@pytest.mark.parametrize('opts', OPTS, ids=OPT_IDS)
@pytest.mark.parametrize('size', ['nuscenes', 'kitti'])
def test_real_size_against_fp64_oracle_and_fp32_composition(opts, size):
    dev = _dev()
    if size == 'nuscenes':
        x, img, grid = real_frame(dev, 6, (48, 100), 256, (900, 1600))
    else:
        x, img, grid = real_frame(dev, 1, (44, 152), 256, (370, 1216), seed=1)
    rep = []
    compare(x, opts, img, grid, rep, real=True)
    print('real', size, opts, rep)


def test_two_runs_are_bit_identical():
    dev = _dev()
    x, img, grid = real_frame(dev, 6, (48, 100), 256, (900, 1600))
    for combine in (True, False):
        a = run_kernel(x, combine, 1, 1, 1, img, grid)
        b = run_kernel(x, combine, 1, 1, 1, img, grid)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def _loss_inputs(x, n_cam, R, S):
    return dict(curr_imgs=x['curr'], prev_imgs=x['prev'], next_imgs=x['next'],
                ray_indices=[torch.arange(R, device=x['pix'].device).repeat_interleave(S)] * n_cam,
                weights=list(x['weights']), ts=list(x['ts']), ms_rays=x['pix'],
                metas=[{'img2prevImg': x['img2prev'].cpu().numpy(), 'img2nextImg': x['img2next'].cpu().numpy()}])


def test_loss_classes_match_the_composition_and_step_does_not_sync():
    dev = _dev()
    from selfocc_b200 import loss as sl
    x, img, grid = real_frame(dev, 6, (48, 100), 64, (900, 1600))
    for cls, combine in ((sl.ReprojLossMonoMultiNewCombine, True), (sl.ReprojLossMonoMultiNew, False)):
        m = cls(weight=0.5, img_size=list(img), ray_resize=list(grid))
        inp = _loss_inputs(x, 6, 4800, 64)
        w = [t.clone().requires_grad_(True) for t in x['weights']]
        inp['weights'] = w
        loss = m(inp)
        loss.backward()
        ref = 0.5 * ol.reproj_loss_ref(combine, x['curr'], x['prev'], x['next'], x['pix'], x['img2prev'], x['img2next'],
                                       x['weights'], x['ts'], None, img, grid)
        assert abs(float(loss) - float(ref)) <= 1e-4 * abs(float(ref))
        assert all(t.grad is not None and torch.isfinite(t.grad).all() for t in w)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode('error')
        try:
            loss = m(inp)
            loss.backward()
        finally:
            torch.cuda.set_sync_debug_mode(0)
        m.check_layout()


def test_wrong_ray_layout_raises_at_the_multiloss_item():
    dev = _dev()
    from selfocc_b200 import loss as sl
    x, img, grid = golden_frame(dev)
    ml = sl.MultiLoss([dict(type='ReprojLossMonoMultiNewCombine', img_size=list(img), ray_resize=list(grid),
                            input_dict={k: k for k in sl._REPROJ_INPUTS})])
    inp = _loss_inputs(x, 2, 20, 16)
    tot, d = ml(inp)
    assert abs(d['ReprojLossMonoMultiNewCombine'] - float(tot)) < 1e-6
    inp['ray_indices'] = [torch.arange(20, device=dev).repeat(16)] * 2     # sample-major: not the head's layout
    with pytest.raises(ValueError, match='ray_indices'):
        ml(inp)


def test_head_forward_loss_backward_matches_the_composition():
    """NeuSHead.forward -> ReprojLossMonoMultiNewCombine -> backward gives the plane and MLP gradients of the same head
    outputs fed to the fp32 composition."""
    dev = _dev()
    from selfocc_b200 import synth, configs
    from selfocc_b200 import loss as sl
    from selfocc_b200.registry import build_head
    import selfocc_b200.segmentor  # noqa: F401
    torch.manual_seed(0)
    margs, rng = synth.small_mapping(8, 4, rng=20.0, z0=-2.0, z1=4.0)
    cfg = configs.hot_path_config(mapping_args=margs, pc_range=rng, num_cams=6, num_layers=1, num_points_cross=(6, 6, 4),
                                  num_points_self=4, num_samples=32, ray_number=(6, 8), ray_img_size=(90, 160))
    head = build_head(cfg['head']).to(dev).train()
    with torch.no_grad():
        head.model.field.deviation_network.variance.fill_(0.25)
    l2i, i2l = synth.camera_rig(f=126.6, cx=80., cy=45., height=0.5, radius=0.2)
    metas = [dict(lidar2img=list(l2i), img2lidar=list(i2l), img_shape=(90, 160))]
    x, _, _ = real_frame(dev, 6, (6, 8), 32, (90, 160))
    metas[0]['img2prevImg'], metas[0]['img2nextImg'] = x['img2prev'].cpu().numpy(), x['img2next'].cpu().numpy()
    planes = [(0.5 * torch.randn(1, n, 96, device=dev)).requires_grad_(True) for n in (17 * 17, 5 * 17, 17 * 5)]
    jitter = torch.rand(6 * 48, 33, device=dev)
    params = [planes[0], planes[1], planes[2]] + list(head.model.field.density_net.parameters())

    def grads(use_kernel):
        out = head(representation=planes, metas=metas, jitter=jitter)
        if use_kernel:
            m = sl.ReprojLossMonoMultiNewCombine(img_size=[90, 160], ray_resize=[6, 8])
            loss = m(dict(curr_imgs=x['curr'], prev_imgs=x['prev'], next_imgs=x['next'], ray_indices=out['ray_indices'],
                          weights=out['weights'], ts=out['ts'], metas=metas, ms_rays=out['ms_rays']))
        else:
            loss = ol.reproj_loss_ref(True, x['curr'], x['prev'], x['next'], out['ms_rays'], x['img2prev'], x['img2next'],
                                      out['weights'], out['ts'], None, (90, 160), (6, 8))
        return loss, torch.autograd.grad(loss, params)

    lk, gk = grads(True)
    lr, gr = grads(False)
    assert abs(float(lk) - float(lr)) <= 1e-5 * abs(float(lr))
    for a, b in zip(gk, gr):
        assert torch.isfinite(a).all() and b.abs().max() > 0
        assert float((a - b).abs().max()) <= 1e-3 * float(b.abs().max()), float((a - b).abs().max() / b.abs().max())


def test_nuscenes_depth_multiloss_drives_a_full_training_step():
    """The loss dict of config/nuscenes/nuscenes_depth.py, built through MultiLoss, on the outputs of the whole hot path
    (lifter -> encoder -> NeuSHead.forward) at the nuScenes geometry (TPV 257 x 257 x 31, 6 cameras x 48 x 100 rays x 256
    samples, 900 x 1600 images), its loss_input_convertion applied: backward() reaches every stage with finite gradients."""
    import json
    import os
    dev = _dev()
    from selfocc_b200 import configs, synth
    from selfocc_b200 import loss as sl
    from selfocc_b200.registry import build_head
    import selfocc_b200.segmentor  # noqa: F401
    c = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_loss_cfgs.json')))
    c = c['nuscenes/nuscenes_depth.py']
    torch.manual_seed(0)
    cfg = configs.hot_path_config(ray_number=(48, 100), ray_img_size=(900, 1600), color_dims=0, ray_sample_mode='cellular',
                                  return_max_depth=False)
    model = build_head(cfg)
    model.encoder.init_weights()
    with torch.no_grad():
        for p in (model.lifter.tpv_hw, model.lifter.tpv_zh, model.lifter.tpv_wz):
            p.mul_(0.1)
        model.head.model.field.deviation_network.variance.fill_(0.3)
    model.train().to(dev)
    l2i, i2l = synth.camera_rig()
    x, _, _ = real_frame(dev, 6, (48, 100), 1, (900, 1600))
    metas = [dict(lidar2img=list(l2i), img2lidar=list(i2l), img_shape=(900, 1600),
                  img2prevImg=x['img2prev'].cpu().numpy(), img2nextImg=x['img2next'].cpu().numpy())]
    g = torch.Generator().manual_seed(1)
    feats = [torch.randn(1, 6, 96, h, w, generator=g).to(dev) for h, w in synth.fpn_level_shapes(900, 1600)]
    multi = sl.OPENOCC_LOSS.build(c['loss'])
    r = model.lifter(ms_img_feats=feats)
    r = model.encoder(representation=r['representation'], ms_img_feats=feats, metas=metas)
    out = model.head(representation=r['representation'], metas=metas)
    inputs = {k: out[v] for k, v in c['loss_input_convertion'].items()}
    inputs.update(curr_imgs=x['curr'], prev_imgs=x['prev'], next_imgs=x['next'], metas=metas)
    tot, loss_dict = multi(inputs)
    assert set(loss_dict) == {'ReprojLossMonoMultiNewCombine', 'EikonalLoss', 'EdgeLoss3DMS'}
    assert all(np.isfinite(v) for v in loss_dict.values()) and abs(sum(loss_dict.values()) - float(tot)) < 1e-4
    tot.backward()
    grads = {n: p.grad for n, p in model.named_parameters() if p.grad is not None}
    assert all(torch.isfinite(t).all() for t in grads.values())
    for stage in ('lifter.', 'encoder.', 'head.'):
        assert any(n.startswith(stage) and t.abs().sum() > 0 for n, t in grads.items()), stage
