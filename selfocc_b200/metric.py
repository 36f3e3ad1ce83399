"""8f-3: DepthMetric on the device (reference utils/metric_util.py:282-397) -- same buffers, same
``_reset / _after_step / _after_epoch`` surface and the same numbers, but the per-camera boolean-mask indexing
(``depth_gt_i[depth_mask_i]``: a device->host sync per camera per frame) is replaced by two small kernels
(``so_depth_metric_sample`` + ``so_depth_metric_sums``) and a sort-based masked median, so a frame's metric step
enqueues without synchronising."""
import ctypes as C
import logging
import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .ops import _chk, _p, _stream

KEYS = ('abs_rel', 'sq_rel', 'rmse', 'rmse_log', 'a1', 'a2', 'a3')


def depth_sample(depth_pred, depth_loc):
    """depth_pred [N,h,w], depth_loc [N,n,2] in [0,1] -> [N,n] (grid_sample bilinear / border / align_corners=True)."""
    lib = _lib.load()
    _chk(depth_pred, name='depth_pred'); _chk(depth_loc, name='depth_loc')
    N, h, w = depth_pred.shape
    n = depth_loc.shape[1]
    out = torch.empty(N, n, device=depth_pred.device)
    _lib.check(lib.so_depth_metric_sample(_p(depth_pred), _p(depth_loc), N, n, h, w, _p(out), _stream()), 'so_depth_metric_sample')
    return out


def depth_metric_sums(sampled, depth_gt, mask_u8, scale=None):
    lib = _lib.load()
    _chk(sampled, name='sampled'); _chk(depth_gt, name='depth_gt'); _chk(mask_u8, torch.uint8, 'depth_mask'); _chk(scale, name='scale')
    N, n = sampled.shape
    sums = torch.empty(N, 8, device=sampled.device)
    _lib.check(lib.so_depth_metric_sums(_p(sampled), _p(depth_gt), _p(mask_u8), _p(scale), N, n, _p(sums), _stream()),
               'so_depth_metric_sums')
    return sums


def masked_median(x, mask):
    """torch.median(x_i[mask_i]) per row (the LOWER median, like torch.median) without boolean indexing."""
    filled = torch.where(mask, x, torch.full_like(x, float('inf')))
    srt = filled.sort(dim=1).values
    cnt = mask.sum(1)
    idx = ((cnt - 1).clamp_min(0) // 2).unsqueeze(1)
    return srt.gather(1, idx).squeeze(1)


def metrics_from_sums(sums):
    """[N,8] error sums -> dict of [N] metrics (cal_depth_metric, metric_util.py:247-279)."""
    c = sums[:, 7].clamp_min(1.0)
    return {'abs_rel': sums[:, 0] / c, 'sq_rel': sums[:, 1] / c, 'rmse': (sums[:, 2] / c).sqrt(), 'rmse_log': (sums[:, 3] / c).sqrt(),
            'a1': sums[:, 4] / c, 'a2': sums[:, 5] / c, 'a3': sums[:, 6] / c}


class DepthMetric(nn.Module):
    def __init__(self, camera_names=['front'], eval_types=['raw', 'median']):
        super().__init__()
        self.num_cams, self.camera_names = len(camera_names), camera_names
        self.num_types, self.eval_types = len(eval_types), eval_types
        for k in KEYS + ('scaling',):
            self.register_buffer(k, torch.zeros(self.num_types, self.num_cams))
        self.register_buffer('count', torch.zeros(1))

    def _reset(self):
        for k in KEYS + ('scaling', 'count'):
            getattr(self, k).zero_()

    @torch.no_grad()
    def _after_step(self, depth_loc, depth_gt, depth_mask, depth_pred):
        """depth_loc [N,n,2], depth_gt [N,n], depth_mask bool [N,n], depth_pred [N,h,w] (metric_util.py:311-349)."""
        depth_loc, depth_gt, depth_pred = depth_loc.float().contiguous(), depth_gt.float().contiguous(), depth_pred.float().contiguous()
        mask = depth_mask.bool()
        mask_u8 = mask.to(torch.uint8).contiguous()
        sampled = depth_sample(depth_pred, depth_loc)
        for ti, typ in enumerate(self.eval_types):
            if typ == 'raw':
                scale = torch.ones(self.num_cams, device=sampled.device)
            elif typ == 'median':
                scale = masked_median(depth_gt, mask) / masked_median(sampled, mask)
            else:
                raise NotImplementedError(typ)
            m = metrics_from_sums(depth_metric_sums(sampled, depth_gt, mask_u8, scale.contiguous()))
            self.scaling[ti] += scale
            for k in KEYS:
                getattr(self, k)[ti] += m[k]
        self.count += 1

    def _after_epoch(self, logger=None):
        """metric_util.py:351-397: all-reduce over ranks when torch.distributed is initialised, then average."""
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.barrier()
            for k in ('count',) + KEYS + ('scaling',):
                dist.all_reduce(getattr(self, k))
            dist.barrier()
        res = {k: getattr(self, k) / self.count for k in KEYS + ('scaling',)}
        if logger is not None and (not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0):
            logger.info('Averaging over %s samples.' % self.count.item())
            for ti, typ in enumerate(self.eval_types):
                logger.info('%s evaluation:' % typ)
                for cam, name in enumerate(self.camera_names):
                    logger.info('%12s | ' % name + ' '.join('%s %.3f' % (k, res[k][ti, cam]) for k in KEYS + ('scaling',)))
                logger.info('%12s | ' % 'All' + ' '.join('%s %.3f' % (k, res[k][ti].mean()) for k in KEYS + ('scaling',)))
        return res


# --------------------------------------------------------------------------------------- occupancy metrics
# utils/metric_util.py:66-244 and utils/scenerf_metric.py.  The reference accumulates per-class float32 counters with a
# host sync per class per frame (.item() / .tolist()); every one of its numbers is a function of the joint (gt, pred)
# label histogram, which so_occ_hist accumulates on the device as exact int64 counts without synchronising.  The float32
# totals of the reference stop counting exactly once a total passes 2^24 voxels (a few dozen Occ3D frames for the
# empty class); these counts do not, and the ratios are formed in float64.
def _occ_labels(t):
    return t.to(torch.uint8).contiguous().reshape(-1)


class _OccHistogram:
    """int64 hist[g, min(p, P - 1)] over uint8 labels; column P - 1 collects every prediction >= P - 1."""

    P = 2

    def reset(self):
        self.hist = torch.zeros(256, self.P, dtype=torch.int64, device='cuda' if torch.cuda.is_available() else 'cpu')

    def _accumulate(self, outputs, targets, mask=None):
        from .ops import occ_hist
        pred, gt = _occ_labels(outputs), _occ_labels(targets)
        occ_hist(pred, gt, self.hist, None if mask is None else _occ_labels(mask))

    def _reduced(self):
        """The histogram summed over ranks (when torch.distributed is initialised), as a host int64 tensor."""
        import torch.distributed as dist
        h = self.hist
        if dist.is_available() and dist.is_initialized():
            h = h.clone()
            dist.all_reduce(h)
        return h.cpu()


def _ratio(a, b):
    return a / b if b else float('nan')


class MeanIoU(_OccHistogram):
    """Per-class IoU + non-empty IoU (utils/metric_util.py:66-165): same constructor, ``reset / _after_step /
    _after_epoch``.  Labels are integers in [0, 255]; outputs outside [0, max(class_indices, empty_label)] count as
    "some other non-empty class", as in the reference.  The dict-target branch (metric_util.py:93-105) is not
    provided: no reference script uses it."""

    def __init__(self, class_indices, empty_label, label_str, use_mask=False, dataset_empty_label=17, name='none'):
        self.class_indices = list(class_indices)
        self.num_classes = len(self.class_indices)
        self.empty_label, self.dataset_empty_label = empty_label, dataset_empty_label
        self.label_str, self.use_mask, self.name = label_str, use_mask, name
        self.P = max(self.class_indices + [empty_label]) + 2
        if min(self.class_indices + [empty_label]) < 0 or self.P > 32:
            raise ValueError('MeanIoU: class indices and the empty label must lie in [0, 30]')

    @torch.no_grad()
    def _after_step(self, outputs, targets, mask=None):
        """outputs, targets: integer label volumes of one shape; mask: bool / 0-1 voxels to count (None = all)."""
        if not torch.is_tensor(targets):
            raise NotImplementedError('MeanIoU: the dict-target branch of the reference is not provided')
        self._accumulate(outputs, targets, mask)

    def counts(self):
        """(total_seen, total_correct, total_positive) int lists of the reference, the last entry the non-empty row."""
        h = self._reduced()
        e = self.empty_label
        seen = [int(h[c].sum()) for c in self.class_indices]
        correct = [int(h[c, c]) for c in self.class_indices]
        positive = [int(h[:, c].sum()) for c in self.class_indices]
        total = int(h.sum())
        ne = torch.ones(256, dtype=torch.bool)
        ne[e] = False
        ne_p = torch.ones(self.P, dtype=torch.bool)
        ne_p[e] = False
        seen.append(total - int(h[e].sum()))
        correct.append(int(h[ne][:, ne_p].sum()))
        positive.append(total - int(h[:, e].sum()))
        return seen, correct, positive

    def _after_epoch(self):
        """(mIoU * 100, non-empty IoU * 100); a class never seen in the ground truth counts as IoU 1."""
        seen, correct, positive = self.counts()
        ious = [1.0 if seen[i] == 0 else _ratio(correct[i], seen[i] + positive[i] - correct[i]) for i in range(self.num_classes)]
        miou = float(np.mean(ious))
        log = logging.getLogger('selfocc_b200')
        log.info('Validation per class iou %s:', self.name)
        for i, s in enumerate(self.label_str):
            prec = _ratio(correct[i], positive[i]) if positive[i] else 0.
            rec = _ratio(correct[i], seen[i]) if seen[i] else 1.
            log.info('%s : %.2f%%, %.2f, %.2f', s, ious[i] * 100, prec, rec)
        occ_iou = _ratio(correct[-1], seen[-1] + positive[-1] - correct[-1])
        return miou * 100, occ_iou * 100


class IoU(_OccHistogram):
    """Occupied-voxel IoU of eval_iou_kitti.py (utils/metric_util.py:168-244).  ``_after_step(outputs, targets)``:
    outputs a 0/1 occupancy volume; targets either the raw label volume of the same shape (occupied = label not in
    {0, 255}, no host sync) or, as in the reference, the [K, 3] coordinates of the occupied voxels."""

    P = 2

    def __init__(self, use_mask=False):
        self.class_indices, self.num_classes, self.label_str, self.use_mask = [0], 1, ['occupied'], use_mask

    @torch.no_grad()
    def _after_step(self, outputs, targets, occ3d=False):
        if occ3d:
            raise NotImplementedError('IoU._after_step_occ3d is not provided: no reference script uses it')
        if targets.shape != outputs.shape:
            idx = targets.long()
            occ = torch.zeros(outputs.shape, dtype=torch.uint8, device=outputs.device)
            occ[tuple(idx.t())] = 1
            targets = occ
        self._accumulate(outputs, targets)

    def counts(self):
        h = self._reduced()
        occ_rows = h[1:255]
        return int(occ_rows.sum()), int(occ_rows[:, 1].sum()), int(h[:, 1].sum())

    def _after_epoch(self):
        """IoU * 100 of the occupied class (1 if no voxel is occupied in the ground truth)."""
        seen, correct, positive = self.counts()
        iou = 1.0 if seen == 0 else _ratio(correct, seen + positive - correct)
        logging.getLogger('selfocc_b200').info('Final iou: %s', iou * 100)
        return iou * 100


class SSCMetrics(_OccHistogram):
    """Scene-completion metrics of eval_iou_kitti.py (utils/scenerf_metric.py:39-215): ``reset / add_batch /
    get_stats``.  Completion counts voxels with gt != 255 (occupied: label > 0); the per-class counts compare RAW labels
    0 .. n_classes - 1, so SSCMetrics(2) fed SemanticKITTI labels scores "class 1" as gt == 1, as the reference does."""

    def __init__(self, n_classes):
        self.n_classes = n_classes
        self.P = n_classes + 1
        if not 1 <= n_classes <= 31:
            raise ValueError('SSCMetrics: n_classes must lie in [1, 31]')
        self.reset()

    @torch.no_grad()
    def add_batch(self, y_pred, y_true, nonempty=None, nonsurface=None):
        if nonsurface is not None:
            raise NotImplementedError('SSCMetrics: nonsurface is not provided (no reference script passes it)')
        self._accumulate(y_pred, y_true, nonempty)

    def counts(self):
        """(completion tp, fp, fn, per-class tps, fps, fns) as ints."""
        h = self._reduced()
        h = torch.cat([h[:255], torch.zeros(1, self.P, dtype=h.dtype)])      # gt == 255 is ignored
        occ_g = h[1:]
        tp, fp, fn = int(occ_g[:, 1:].sum()), int(h[0, 1:].sum()), int(occ_g[:, 0].sum())
        C = self.n_classes
        tps = [int(h[j, j]) for j in range(C)]
        fps = [int(h[:, j].sum()) - tps[j] for j in range(C)]
        fns = [int(h[j].sum()) - tps[j] for j in range(C)]
        return tp, fp, fn, tps, fps, fns

    def get_stats(self):
        tp, fp, fn, tps, fps, fns = self.counts()
        if tp != 0:
            precision, recall, iou = tp / (tp + fp), tp / (tp + fn), tp / (tp + fp + fn)
        else:
            precision, recall, iou = 0., 0., 0.
        iou_ssc = torch.tensor([a / (a + b + c + 1e-5) for a, b, c in zip(tps, fps, fns)], dtype=torch.float64)
        return {'precision': precision, 'recall': recall, 'iou': iou, 'iou_ssc': iou_ssc,
                'iou_ssc_mean': float(iou_ssc[1:].mean())}
