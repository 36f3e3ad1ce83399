"""CPU: occupancy evaluation -- the oracle's label pipeline and metric loops against the reference's own metric classes
(tests/golden/reference_golden_occ.npz), the histogram formulas of selfocc_b200.metric, the Occ3D point builder, and the
error paths of so_occ_classify / so_occ_hist."""
import ctypes as C
import os
import numpy as np
import pytest
import torch

from oracle import occupancy as oo
from selfocc_b200 import metric, occupancy

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_golden_occ.npz'))
FRAMES = 3
NAMES = ['c%d' % i for i in range(16)]


def _t(a):
    return torch.from_numpy(a.astype(np.int64))


def _bincount_hist(pairs, P):
    """int64 [256, P] joint histogram of (gt, min(pred, P - 1)) pairs via torch.bincount (the kernel's definition)."""
    h = torch.zeros(256 * P, dtype=torch.int64)
    for pred, gt, mask in pairs:
        p, g = pred.reshape(-1).clamp(max=P - 1), gt.reshape(-1)
        if mask is not None:
            p, g = p[mask.reshape(-1)], g[mask.reshape(-1)]
        h += torch.bincount(g * P + p, minlength=256 * P)
    return h.reshape(256, P)


def test_luts_match_reference():
    assert tuple(G['lut_openseed2nuscenes']) == occupancy.OPENSEED2NUSCENES
    assert tuple(G['lut_cityscapes2semantickitti']) == occupancy.CITYSCAPES2SEMANTICKITTI


@pytest.mark.parametrize('masked', [False, True])
def test_miou_oracle_and_histogram_match_reference(masked):
    tag = 'mask' if masked else 'plain'
    ref = oo.MeanIoURef(list(range(1, 17)), 0, NAMES)
    pairs = []
    for f in range(FRAMES):
        pred, gt = _t(G['miou_pred%d' % f]), _t(G['miou_gt%d' % f])
        mask = torch.from_numpy(G['miou_mask%d' % f]) if masked else None
        ref._after_step(pred, gt, mask)
        pairs.append((pred, gt, mask))
    counts = G['miou_%s_counts' % tag]
    assert [ref.total_seen, ref.total_correct, ref.total_positive] == counts.astype(np.int64).tolist()
    miou, occ_iou = ref._after_epoch()
    assert (miou, occ_iou) == tuple(G['miou_%s_result' % tag])          # the reference's float32 arithmetic, exactly
    # the device class's epoch step on the same counts, fed as a hand-filled histogram
    m = metric.MeanIoU(list(range(1, 17)), 0, NAMES)
    m.reset()
    m.hist = _bincount_hist(pairs, m.P)
    assert [list(c) for c in m.counts()] == counts.astype(np.int64).tolist()
    np.testing.assert_allclose(m._after_epoch(), G['miou_%s_result' % tag], rtol=1e-6)


def test_iou_and_ssc_oracle_and_histogram_match_reference():
    iou, ssc = oo.IoURef(), oo.SSCMetricsRef(2)
    pairs = []
    for f in range(FRAMES):
        pred, gt_raw = _t(G['kitti_pred%d' % f]), _t(G['kitti_gt%d' % f])
        gt = gt_raw.clone()
        gt[gt == 255] = 0
        iou._after_step(pred, torch.nonzero(gt))
        ssc.add_batch(pred, gt_raw)
        pairs.append((pred, gt_raw, None))
    assert [iou.total_seen, iou.total_correct, iou.total_positive] == G['iou_counts'].astype(np.int64).tolist()
    assert iou._after_epoch() == G['iou_result'][0]
    assert [ssc.completion_tp, ssc.completion_fp, ssc.completion_fn] == G['ssc_completion'].astype(np.int64).tolist()
    assert [ssc.tps, ssc.fps, ssc.fns] == G['ssc_class_counts'].astype(np.int64).tolist()
    st = ssc.get_stats()
    assert [st['precision'], st['recall'], st['iou'], st['iou_ssc_mean']] == G['ssc_result'].tolist()
    assert torch.equal(st['iou_ssc'], torch.from_numpy(G['ssc_iou_ssc']))

    d_iou, d_ssc = metric.IoU(), metric.SSCMetrics(2)
    d_iou.reset()
    d_iou.hist = _bincount_hist(pairs, d_iou.P)
    d_ssc.hist = _bincount_hist(pairs, d_ssc.P)
    assert list(d_iou.counts()) == G['iou_counts'].astype(np.int64).tolist()
    np.testing.assert_allclose(d_iou._after_epoch(), G['iou_result'][0], rtol=1e-6)
    tp, fp, fn, tps, fps, fns = d_ssc.counts()
    assert [tp, fp, fn] == G['ssc_completion'].astype(np.int64).tolist()
    assert [tps, fps, fns] == G['ssc_class_counts'].astype(np.int64).tolist()
    st = d_ssc.get_stats()
    np.testing.assert_allclose([st['precision'], st['recall'], st['iou'], st['iou_ssc_mean']], G['ssc_result'], rtol=1e-6)
    np.testing.assert_allclose(st['iou_ssc'].numpy(), G['ssc_iou_ssc'], rtol=1e-6)


def test_histogram_clamps_out_of_range_predictions():
    """MeanIoU's last histogram column collects every other non-empty prediction: a label above the classes (or a
    negative one, which wraps to 255 in uint8) is non-empty but matches no class, as in the reference."""
    m = metric.MeanIoU([1, 2], 0, ['a', 'b'])
    ref = oo.MeanIoURef([1, 2], 0, ['a', 'b'])
    pred = torch.tensor([0, 1, 2, 7, 200, 1, 0, 2])
    gt = torch.tensor([0, 1, 1, 7, 0, 2, 2, 2])
    ref._after_step(pred, gt)
    m.reset()
    m.hist = _bincount_hist([(pred, gt, None)], m.P)
    assert [list(c) for c in m.counts()] == [ref.total_seen, ref.total_correct, ref.total_positive]


def test_labels_ref_borders_follow_slice_semantics():
    sdf = -torch.ones(10, 9, 8, dtype=torch.float64)
    occ, _ = oo.labels_ref(sdf, z_keep=(2, -3), border=(1, 2, 0, 4))
    want = torch.ones(10, 9, 8, dtype=torch.int)
    want[..., -3:] = 0
    want[..., :2] = 0
    want[:1] = 0
    want[-2:] = 0
    want[:, -4:] = 0
    assert torch.equal(occ, want)


def test_occ3d_points_equal_oracle_bitwise():
    rng = np.random.default_rng(3)
    a = np.deg2rad(rng.uniform(-10, 10))
    e2l = np.array([[np.cos(a), -np.sin(a), 0, 0.3], [np.sin(a), np.cos(a), 0, -0.2], [0, 0, 1, -1.8], [0, 0, 0, 1]])
    for s in (1, 4, 6):
        pcr, exp = occupancy.SCENE_SIZES[s]
        assert torch.equal(occupancy.occ3d_points(e2l, s), oo.occ3d_points_ref(e2l, pcr, exp))


def test_occ_entry_points_reject_bad_arguments_without_a_gpu():
    from selfocc_b200 import _lib, build
    build.build()
    lib = _lib.load()
    N, one = None, C.c_void_p(16)
    d = _lib.VolumeDesc()
    d.H, d.W, d.Z, d.zpitch, d.n_feat, d.feat_pitch = 9, 9, 5, 8, 24, 24
    for i in range(3):
        d.axis[i].range0, d.axis[i].size0 = 1.0, 4.0
    g = _lib.OccGrid()
    g.n0, g.n1, g.n2, g.z_lo, g.z_hi = 4, 3, 2, 0, 2
    args = lambda **k: [k.get('sdf', one), k.get('feat', one), C.byref(k.get('desc', d)), one, one, one, 3, 4, 2,
                        k.get('pts', N), C.byref(k.get('grid', g)), k.get('lut', N), k.get('lut_len', 0), k.get('occ', one),
                        k.get('sem', N), N]
    assert lib.so_occ_classify(*args(sdf=N)) == -1                         # NULL volume
    assert lib.so_occ_classify(*args(occ=N)) == -1                         # NULL output
    assert lib.so_occ_classify(*args(pts=one, sem=one, lut=one, lut_len=20)) == -1   # LUT shorter than the 21 classes
    assert lib.so_occ_classify(*args(pts=one, sem=one, feat=N)) == -1      # semantics without a feature volume
    bad = _lib.VolumeDesc()
    bad.H, bad.W, bad.Z, bad.zpitch = 4, 4, 4, 2                           # zpitch < Z
    assert lib.so_occ_classify(*args(desc=bad)) == -1
    g2 = _lib.OccGrid()
    g2.n0, g2.n1, g2.n2 = 5, 3, 2
    assert lib.so_occ_classify(*args(grid=g2)) == -1                       # lattice mode: the output must be the lattice
    g2.border[1] = -1
    assert lib.so_occ_classify(*args(grid=g2, pts=one)) == -1              # negative border
    wide = _lib.VolumeDesc()
    wide.H, wide.W, wide.Z, wide.zpitch, wide.n_feat, wide.feat_pitch = 9, 9, 5, 8, 40, 40
    for i in range(3):
        wide.axis[i].range0, wide.axis[i].size0 = 1.0, 4.0
    assert lib.so_occ_classify(*args(desc=wide, pts=one, sem=one)) == -2   # more than 32 semantic channels
    g0 = _lib.OccGrid()
    g0.n0, g0.n1, g0.n2 = 0, 3, 2
    assert lib.so_occ_classify(*args(grid=g0, pts=one)) == 0               # n = 0: nothing to do
    assert lib.so_occ_hist(N, one, N, 10, 2, one, N) == -1
    assert lib.so_occ_hist(one, one, N, 10, 2, N, N) == -1
    assert lib.so_occ_hist(one, one, N, 10, 0, one, N) == -1
    assert lib.so_occ_hist(one, one, N, 10, 33, one, N) == -2              # P > 32
    assert lib.so_occ_hist(one, one, N, 0, 17, one, N) == 0                # n = 0: nothing to do
