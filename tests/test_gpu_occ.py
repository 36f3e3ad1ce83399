"""GPU: occupancy evaluation.  NeuSHead.occupancy (so_occ_classify) against the fp32 reference composition
(get_uniform_sdf lattice + F.grid_sample + argmax + LUT + borders, oracle/occupancy.py on the same GPU) and the fp64
oracle, voxel for voxel; so_occ_hist against torch.bincount; the device MeanIoU / IoU / SSCMetrics against the oracle's
restatement of the reference's loops; and neither the labels nor the metric step synchronise with the host."""
import math
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import occupancy as oo
from oracle.mapping import GridMeterMappingRef
from selfocc_b200 import metric, occupancy, synth
from selfocc_b200.head import NeuSHead
from selfocc_b200.mapping import GridMeterMapping

TIE = 1e-6
# Against the fp64 oracle the fp32 labels carry the rounding of two chained 8-term trilinear sums (the field query of a
# lattice node, then the resample): a few ulp of |logit| ~ 4 on each of the two compared channels.  At 640 k voxels x 21
# channels, labels at top-two gaps of 1-3e-6 differ from fp64 (86 voxels, 0.013 %, on a B200), so the oracle comparison
# uses a 1e-5 band; the kernel itself equals the fp32 composition (same GPU) within TIE.
TIE64 = 1e-5


def _dev():
    if not torch.cuda.is_available():
        pytest.skip('needs CUDA')
    return torch.device('cuda:0')


def _head(margs, aabb, return_sem, ground_z, seed=0):
    """NeuSHead (color_dims 24: 3 colour + 21 semantic channels) holding an analytic scene plus seeded random channels."""
    dev = _dev()
    head = NeuSHead(roi_aabb=aabb, mapping_args=margs, color_dims=24, return_sem=return_sem, tpv=True, embed_dims=32,
                    sh_deg=0).to(dev)
    f = head.model.field
    m = GridMeterMapping(**margs)
    f.vol_sdf = synth.pack_sdf_volume(synth.analytic_sdf_volume(m, ground_z=ground_z), f.desc.zpitch).to(dev)
    gen = torch.Generator().manual_seed(seed)
    feat = torch.randn(24, m.size_h, m.size_w, m.size_d, generator=gen)
    f.vol_feat = synth.pack_feat_volume(feat, f.desc.feat_pitch).to(dev)
    return head


def _oracle_volume(head, dtype, device):
    f = head.model.field
    d = f.desc
    sdf = f.vol_sdf[..., :d.Z]
    feat = f.vol_feat[..., :d.n_feat].permute(3, 0, 1, 2)
    return torch.cat([sdf[None], feat], 0).to(device=device, dtype=dtype)


def _points(e2l, n, lo, hi, pcr, expansion, device):
    """Voxel centres of an n[0] x n[1] x n[2] ego grid moved into the lidar frame and normalised (eval_iou.py:211-218)."""
    axes = [torch.linspace(lo[i], hi[i], n[i]) for i in range(3)]
    xyz = torch.stack([axes[0][:, None, None].expand(*n), axes[1][None, :, None].expand(*n), axes[2][None, None, :].expand(*n),
                       torch.ones(*n)], -1).to(device)
    p = torch.matmul(xyz.new_tensor(e2l).unsqueeze(0), xyz.reshape(-1, 4, 1)).squeeze(-1)[:, :3]
    for i in range(3):
        p[:, i] = (p[:, i] - pcr[i]) / expansion[i]
    return p.reshape(*n, 3)


def _ego2lidar(yaw_deg, t):
    a = math.radians(yaw_deg)
    return np.array([[math.cos(a), -math.sin(a), 0, t[0]], [math.sin(a), math.cos(a), 0, t[1]], [0, 0, 1, t[2]], [0, 0, 0, 1.]])


def _check_labels(got, ref, thresh, lut, what, tie=TIE):
    """got = head.occupancy(...); ref = labels_ref(..., return_values=True).  Every voxel equal, except near-ties of the
    thresholded sdf or of the top-two logits; those must be <= 0.1 % and must pick one of the tied options."""
    occ_r, sem_r, s, lg = ref
    occ_g = got['occ'].to(occ_r.device).long()
    s = s.to(occ_r.device)
    tie_occ = (s - thresh).abs() <= tie * s.abs().clamp_min(1)
    bad_occ = occ_g != occ_r.long()
    assert not (bad_occ & ~tie_occ).any(), '%s: %d occupancy labels differ away from a tie' % (what, int((bad_occ & ~tie_occ).sum()))
    n_tie = int((bad_occ & tie_occ).sum())
    if sem_r is not None:
        top = lg.topk(2, -1)
        gap = (top.values[..., 0] - top.values[..., 1]).abs()
        tie_lg = gap <= tie * top.values[..., 0].abs().clamp_min(1)
        lut_t = torch.as_tensor(lut if lut is not None else list(range(lg.shape[-1])), device=lg.device)
        sem_g = got['sem'].to(occ_r.device).long()
        bad = sem_g != sem_r.long()
        options = (sem_g == occ_g * lut_t[top.indices[..., 0]]) | (sem_g == occ_g * lut_t[top.indices[..., 1]])
        assert not (bad & ~(tie_occ | tie_lg)).any(), '%s: %d semantic labels differ away from a tie' % (what, int((bad & ~(tie_occ | tie_lg)).sum()))
        assert bool(options[bad].all()), '%s: a tied semantic label picked neither option' % what
        assert bool(((sem_g == 0) | (occ_g == 1)).all())
        n_tie += int((bad & ~bad_occ).sum())
        if bool((bad & ~bad_occ).any()):
            print('%s: largest top-two logit gap among differing labels %.2e' % (what, float(gap[bad & ~bad_occ].max())))
    print('%s: %d voxels, %d near-tie differences' % (what, occ_g.numel(), n_tie))
    assert n_tie <= 1e-3 * occ_g.numel()


SMALL = synth.small_mapping(16, 8, rng=12.8, z0=-2.0, z1=3.0)
SETTINGS = {
    # name: (resample, lut, z_keep, border)
    'occ3d': (True, occupancy.OPENSEED2NUSCENES, (0, 8), (3, 3, 3, 3)),
    'openocc': (False, occupancy.OPENSEED2NUSCENES, (2, -2), (3, 3, 3, 3)),
    'kitti': (False, None, (0, 10), (0, 3, 3, 3)),
}


@pytest.mark.parametrize('setting', sorted(SETTINGS))
@pytest.mark.parametrize('sem', [False, True])
def test_occupancy_labels_match_composition_and_oracle(setting, sem):
    dev = _dev()
    margs, aabb = SMALL
    resample, lut, z_keep, border = SETTINGS[setting]
    head = _head(margs, aabb, sem, ground_z=-0.87)
    res, thresh = 0.4, 0.
    pts = None
    if resample:
        pts = _points(_ego2lidar(7.0, (0.3, -0.4, 0.25)), (40, 40, 10), (-10., -10., -1.5), (10., 10., 2.5), aabb,
                      [aabb[3] - aabb[0], aabb[4] - aabb[1], aabb[5] - aabb[2]], dev)
    got = head.occupancy(aabb=aabb, resolution=res, thresh=thresh, points=pts, sem_lut=lut if sem else None,
                         z_keep=z_keep, border=border)
    assert got['occ'].dtype == torch.uint8 and ('sem' in got) == sem
    # fp32 reference composition on the same GPU: forward_occ's lattice (get_uniform_sdf) + the eval_iou*.py ops
    lat = head.get_uniform_sdf(aabb, res, dev)
    logits = lat[2] if sem else None
    comp = oo.labels_ref(lat[0], thresh, logits, pts, lut if sem else None, z_keep, border, return_values=True)
    _check_labels(got, comp, thresh, lut, '%s sem=%d vs fp32 composition' % (setting, sem))
    # fp64 oracle on the CPU
    vol = _oracle_volume(head, torch.float64, 'cpu')
    sdf64, lg64 = oo.lattice_ref(vol, GridMeterMappingRef(**margs), aabb, res)
    ref = oo.labels_ref(sdf64, thresh, lg64 if sem else None, None if pts is None else pts.cpu().double(), lut if sem else None,
                        z_keep, border, return_values=True)
    _check_labels({k: v.cpu() for k, v in got.items()}, ref, thresh, lut, '%s sem=%d vs fp64 oracle' % (setting, sem), TIE64)
    assert int(got['occ'].sum()) > 0.02 * got['occ'].numel()           # the scene is not all free space


def test_occ3d_real_size_labels_and_memory():
    """nuscenes_occ.py head sizes (257 x 257 x 25, 25 decoded channels), scene_size 4 at 0.2 m, 200 x 200 x 16 output."""
    dev = _dev()
    margs = dict(nonlinear_mode='linear', h_size=[128, 0], h_range=[40.0, 0], h_half=False, w_size=[128, 0],
                 w_range=[40.0, 0], w_half=False, d_size=[24, 0], d_range=[-1.0, 5.4, 5.4])
    pcr, _ = occupancy.SCENE_SIZES[4]
    head = _head(margs, pcr, True, ground_z=0.07, seed=1)
    pts = occupancy.occ3d_points(_ego2lidar(-90.0, (0.0, 0.94, -1.84)), 4, device=dev)
    z_keep, border = occupancy.OCC3D_BORDERS
    lut = occupancy.OPENSEED2NUSCENES
    head.occupancy(aabb=pcr, resolution=0.2, points=pts, sem_lut=lut, z_keep=z_keep, border=border)     # caches the LUT
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    got = head.occupancy(aabb=pcr, resolution=0.2, points=pts, sem_lut=lut, z_keep=z_keep, border=border)
    torch.cuda.synchronize()
    growth = torch.cuda.max_memory_allocated() - base
    print('fused occupancy: peak growth over the decoded volume %.2f MB' % (growth / 2 ** 20))
    assert growth < 64 * 2 ** 20
    assert got['occ'].shape == (200, 200, 16) and int(got['occ'].sum()) > 1000
    lat = head.get_uniform_sdf(pcr, 0.2, dev)
    comp = oo.labels_ref(lat[0], 0., lat[2], pts, lut, z_keep, border, return_values=True)
    del lat
    _check_labels(got, comp, 0., lut, 'Occ3D real size vs fp32 composition')
    del comp
    vol = _oracle_volume(head, torch.float64, dev)            # the fp64 oracle, run on the GPU at this size
    sdf64, lg64 = _lattice64(vol, margs, pcr, dev)
    ref = oo.labels_ref(sdf64, 0., lg64, pts.double(), lut, z_keep, border, return_values=True)
    _check_labels(got, ref, 0., lut, 'Occ3D real size vs fp64 oracle', TIE64)


def _lattice64(vol, margs, aabb, dev):
    """oracle.render.uniform_sdf_ref on the device, in chunks of lattice rows (the whole fp64 query is several GB)."""
    from oracle.render import field_query_ref, uniform_lattice
    xyz = uniform_lattice(aabb, 0.2).to(dev).double()
    mref = GridMeterMappingRef(**margs)
    H, W, D = xyz.shape[:3]
    out = torch.cat([field_query_ref(vol, mref, xyz[h:h + 50].reshape(-1, 3), with_grad=False)[0] for h in range(0, H, 50)])
    return out[:, 0].reshape(H, W, D), out[:, 4:].reshape(H, W, D, -1)


@pytest.mark.parametrize('P', [2, 17, 32])
def test_hist_equals_bincount(P):
    dev = _dev()
    gen = torch.Generator(device=dev).manual_seed(P)
    hist = torch.zeros(256, P, dtype=torch.int64, device=dev)
    ref = torch.zeros(256 * P, dtype=torch.int64, device=dev)
    from selfocc_b200 import ops
    for n, masked in ((1_000_003, False), (777_777, True), (255, True), (96_001, False)):
        pred = torch.randint(0, 40, (n,), generator=gen, device=dev, dtype=torch.int32).to(torch.uint8)
        pred[torch.rand(n, generator=gen, device=dev) < 0.6] = 0               # realistic skew: most voxels empty
        gt = torch.randint(0, 256, (n,), generator=gen, device=dev, dtype=torch.int32).to(torch.uint8)
        gt[torch.rand(n, generator=gen, device=dev) < 0.7] = 0
        mask = (torch.rand(n, generator=gen, device=dev) < 0.5).to(torch.uint8) if masked else None
        ops.occ_hist(pred, gt, hist, mask)
        key = gt.long() * P + pred.long().clamp(max=P - 1)
        if masked:
            key = key[mask.bool()]
        ref += torch.bincount(key, minlength=256 * P)
        assert torch.equal(hist.reshape(-1), ref)


def test_metrics_match_oracle_over_frames():
    dev = _dev()
    gen = torch.Generator().manual_seed(5)
    names = ['c%d' % i for i in range(16)]
    m, m_ref = metric.MeanIoU(list(range(1, 17)), 0, names), oo.MeanIoURef(list(range(1, 17)), 0, names)
    mm, mm_ref = metric.MeanIoU(list(range(1, 17)), 0, names), oo.MeanIoURef(list(range(1, 17)), 0, names)
    iou, iou_ref = metric.IoU(), oo.IoURef()
    ssc, ssc_ref = metric.SSCMetrics(2), oo.SSCMetricsRef(2)
    for x in (m, mm, iou):
        x.reset()
    shape = (64, 48, 16)
    for _ in range(4):
        pred = (torch.rand(shape, generator=gen) < 0.4).long() * torch.tensor(occupancy.OPENSEED2NUSCENES)[torch.randint(0, 21, shape, generator=gen)]
        gt = torch.randint(0, 18, shape, generator=gen)
        gt[torch.rand(shape, generator=gen) < 0.05] = 255
        mask = torch.rand(shape, generator=gen) < 0.6
        m._after_step(pred.to(dev), gt.to(dev))
        m_ref._after_step(pred, gt)
        mm._after_step(pred.to(dev), gt.to(dev), mask.to(dev))
        mm_ref._after_step(pred, gt, mask)
        occ = (torch.rand(shape, generator=gen) < 0.3).long()
        kgt = torch.randint(0, 20, shape, generator=gen)
        kgt[torch.rand(shape, generator=gen) < 0.1] = 255
        g0 = kgt.clone()
        g0[g0 == 255] = 0
        iou._after_step(occ.to(dev), kgt.to(dev))                    # the label volume: no nonzero()/tolist() sync
        iou_ref._after_step(occ, torch.nonzero(g0))
        ssc.add_batch(occ.to(dev), kgt.to(dev))
        ssc_ref.add_batch(occ, kgt)
    for d, r in ((m, m_ref), (mm, mm_ref)):
        assert [list(c) for c in d.counts()] == [r.total_seen, r.total_correct, r.total_positive]
        np.testing.assert_allclose(d._after_epoch(), r._after_epoch(), rtol=1e-6)
    assert list(iou.counts()) == [iou_ref.total_seen, iou_ref.total_correct, iou_ref.total_positive]
    np.testing.assert_allclose(iou._after_epoch(), iou_ref._after_epoch(), rtol=1e-6)
    tp, fp, fn, tps, fps, fns = ssc.counts()
    assert [tp, fp, fn, tps, fps, fns] == [ssc_ref.completion_tp, ssc_ref.completion_fp, ssc_ref.completion_fn,
                                           ssc_ref.tps, ssc_ref.fps, ssc_ref.fns]
    a, b = ssc.get_stats(), ssc_ref.get_stats()
    for k in ('precision', 'recall', 'iou', 'iou_ssc_mean'):
        np.testing.assert_allclose(a[k], b[k], rtol=1e-6)
    # the coordinate-list form of IoU._after_step counts the same
    iou2 = metric.IoU()
    iou2.reset()
    iou2._after_step(occ.to(dev), torch.nonzero(g0).to(dev))
    iou3 = metric.IoU()
    iou3.reset()
    iou3._after_step(occ.to(dev), kgt.to(dev))
    assert iou2.counts() == iou3.counts()


def test_occupancy_and_metric_step_do_not_sync():
    dev = _dev()
    margs, aabb = SMALL
    head = _head(margs, aabb, True, ground_z=-0.87)
    lut = occupancy.OPENSEED2NUSCENES
    pts = _points(_ego2lidar(3.0, (0.1, 0.2, 0.0)), (20, 20, 8), (-8., -8., -1.), (8., 8., 2.), aabb,
                  [aabb[3] - aabb[0], aabb[4] - aabb[1], aabb[5] - aabb[2]], dev)
    gt = torch.randint(0, 18, (20, 20, 8), device=dev)
    mask = torch.rand(20, 20, 8, device=dev) < 0.5
    m = metric.MeanIoU(list(range(1, 17)), 0, ['c%d' % i for i in range(16)])
    m.reset()
    iou = metric.IoU()
    iou.reset()
    head.occupancy(aabb=aabb, resolution=0.4, points=pts, sem_lut=lut, z_keep=(0, 6), border=(2, 2, 2, 2))   # caches the LUT
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        out = head.occupancy(aabb=aabb, resolution=0.4, points=pts, sem_lut=lut, z_keep=(0, 6), border=(2, 2, 2, 2))
        out2 = head.occupancy(aabb=aabb, resolution=0.4, z_keep=(1, -1), border=(2, 2, 2, 2))
        m._after_step(out['sem'], gt, mask)
        iou._after_step(out2['occ'], out2['occ'])
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert m.counts()[0][-1] == int(((gt != 0) & mask).sum())
