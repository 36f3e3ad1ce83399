"""Golden vectors for the occupancy metrics, from the reference's own metric classes (see ``occ_golden``).

Uses the same reference location and loader as ``make_golden.py``; inputs are seeded and stored beside the outputs.
"""
import os
import sys
import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from make_golden import HERE, load  # noqa: E402


def occ_golden():
    """Pins the occupancy metrics (oracle/occupancy.py, selfocc_b200.metric.MeanIoU / IoU / SSCMetrics) to the reference's
    own classes, executed UNMODIFIED on seeded random label volumes: MeanIoU, IoU, openseed2nuscenes and
    cityscapes2semantickitti from utils/metric_util.py, SSCMetrics from utils/scenerf_metric.py.  Two stand-ins, as for
    the BEVNeRF vectors: (a) ``mmengine.MMLogger`` (metric_util.py:4-5 builds a module-level logger) is a plain
    ``logging`` logger, and (b) ``Tensor.cuda()`` -- the classes allocate their counters with it -- is the identity, so
    they run on the CPU.  IoU._after_epoch / SSCMetrics.get_stats all-reduce unconditionally, so a one-process gloo group
    is initialised.  Writes tests/golden/reference_golden_occ.npz.

    Run once where the reference tree is present:  python tests/golden/make_golden_occ.py"""
    import logging
    import tempfile
    import types
    import torch.distributed as dist

    class MMLogger:
        @staticmethod
        def get_instance(name):
            return logging.getLogger(name)
    mm = types.ModuleType('mmengine')
    mm.MMLogger = MMLogger
    sys.modules.setdefault('mmengine', mm)
    torch.Tensor.cuda = lambda self, *a, **k: self
    if not dist.is_initialized():
        dist.init_process_group('gloo', init_method='file://' + tempfile.mktemp(), rank=0, world_size=1)
    mu = load('utils/metric_util.py', 'ref_metric_util')
    sm = load('utils/scenerf_metric.py', 'ref_scenerf_metric')

    gen = torch.Generator().manual_seed(2024)
    out = {}
    out['lut_openseed2nuscenes'] = mu.openseed2nuscenes(torch.arange(21)).numpy()
    out['lut_cityscapes2semantickitti'] = mu.cityscapes2semantickitti(torch.arange(19)).numpy()
    shape, frames = (12, 10, 6), 3
    names = ['barrier', 'bicycle', 'bus', 'car', 'construction_vehicle', 'motorcycle', 'pedestrian', 'traffic_cone',
             'trailer', 'truck', 'driveable_surface', 'other_flat', 'sidewalk', 'terrain', 'manmade', 'vegetation']
    # nuScenes mIoU (eval_iou.py:140-149, :283-294): pred = occ * openseed2nuscenes(argmax); gt 0..17 with 255 sprinkled in
    m_plain, m_mask = mu.MeanIoU(list(range(1, 17)), 0, names, True, 0), mu.MeanIoU(list(range(1, 17)), 0, names, True, 0)
    m_plain.reset(); m_mask.reset()
    for f in range(frames):
        occ = (torch.rand(shape, generator=gen) < 0.4).to(torch.int)
        arg = torch.randint(0, 21, shape, generator=gen)
        pred = occ * mu.openseed2nuscenes(arg)
        gt = torch.randint(0, 18, shape, generator=gen)
        gt[torch.rand(shape, generator=gen) < 0.05] = 255
        gt[torch.rand(shape, generator=gen) < 0.3] = 0
        mask = torch.rand(shape, generator=gen) < 0.7
        m_plain._after_step(pred, gt)
        m_mask._after_step(pred, gt, mask)
        out['miou_pred%d' % f], out['miou_gt%d' % f] = pred.numpy().astype(np.uint8), gt.numpy().astype(np.uint8)
        out['miou_mask%d' % f] = mask.numpy()
    for tag, m in (('plain', m_plain), ('mask', m_mask)):
        out['miou_%s_counts' % tag] = torch.stack([m.total_seen, m.total_correct, m.total_positive]).numpy()
        miou, occ_iou = m._after_epoch()
        out['miou_%s_result' % tag] = np.array([miou, float(occ_iou)])
    # KITTI IoU + SSCMetrics(2) (eval_iou_kitti.py:167-190): pred 0/1 occupancy, gt raw SemanticKITTI labels incl. 255
    iou, ssc = mu.IoU(), sm.SSCMetrics(2)
    iou.reset()
    for f in range(frames):
        pred = (torch.rand(shape, generator=gen) < 0.35).to(torch.int)
        gt_raw = torch.randint(0, 20, shape, generator=gen)
        gt_raw[torch.rand(shape, generator=gen) < 0.5] = 0
        gt_raw[torch.rand(shape, generator=gen) < 0.1] = 255
        gt = gt_raw.clone()
        gt[gt == 255] = 0
        iou._after_step(pred, torch.nonzero(gt))
        ssc.add_batch(pred, gt_raw.clone())
        out['kitti_pred%d' % f], out['kitti_gt%d' % f] = pred.numpy().astype(np.uint8), gt_raw.numpy().astype(np.uint8)
    out['iou_counts'] = torch.cat([iou.total_seen, iou.total_correct, iou.total_positive]).numpy()
    out['iou_result'] = np.array([iou._after_epoch()])
    out['ssc_completion'] = torch.cat([ssc.completion_tp, ssc.completion_fp, ssc.completion_fn]).numpy()
    out['ssc_class_counts'] = torch.stack([ssc.tps, ssc.fps, ssc.fns]).numpy()
    st = ssc.get_stats()
    out['ssc_result'] = np.array([float(st['precision']), float(st['recall']), float(st['iou']), float(st['iou_ssc_mean'])])
    out['ssc_iou_ssc'] = st['iou_ssc'].numpy()
    dist.destroy_process_group()
    np.savez_compressed(os.path.join(HERE, 'reference_golden_occ.npz'), **out)
    print('wrote occupancy golden:', len(out), 'arrays')


if __name__ == '__main__':
    occ_golden()
