"""Oracle: occupancy evaluation (test infrastructure, see oracle/__init__.py).

Restates, with the reference's own torch ops:
* the label pipeline of eval_iou.py:206-258 (Occ3D: F.grid_sample of the get_uniform_sdf lattice at the Occ3D points;
  OpenOccupancy: the lattice itself) and eval_iou_kitti.py:167-196 -- threshold, border rows, argmax of the semantic
  logits h[..., 4:], lookup table, ``pred_occ * sem``;
* the per-class counting loops of MeanIoU / IoU (utils/metric_util.py:66-244) and SSCMetrics (utils/scenerf_metric.py),
  with the reference's float32 formation of the returned numbers (exact while every count is below 2^24).

Device-agnostic and dtype-preserving: fp64 on the CPU it is the oracle; fp32 on CUDA, fed the lattice of
``NeuSHead.get_uniform_sdf``, it is the reference composition the fused path is compared with and benchmarked against.
"""
import numpy as np
import torch
import torch.nn.functional as F

from .render import uniform_sdf_ref


def lattice_ref(vol, mapping, aabb, resolution):
    """get_uniform_sdf (neus_head.py:265-293) of a decoded volume [Cf, H, W, Z]: (sdf [H, W, D], logits [H, W, D, C] or
    None)."""
    sdf, sem, _ = uniform_sdf_ref(vol, mapping, aabb, resolution)
    return sdf, sem


def occ3d_points_ref(ego2lidar, pcr, expansion, device=None):
    """eval_iou.py:151-164 and :211-218."""
    xx = torch.linspace(-40.0, 40.0, 200)
    yy = torch.linspace(-40.0, 40.0, 200)
    zz = torch.linspace(-1.0, 5.4, 16)
    xyz = torch.stack([xx[:, None, None].expand(-1, 200, 16), yy[None, :, None].expand(200, -1, 16),
                       zz[None, None, :].expand(200, 200, -1), torch.ones(200, 200, 16)], dim=-1)
    if device is not None:
        xyz = xyz.to(device)
    ego2lidar = xyz.new_tensor(ego2lidar)
    lidar_points = torch.matmul(ego2lidar.unsqueeze(0), xyz.reshape(-1, 4, 1))
    lidar_points = lidar_points.squeeze(-1)[:, :3]
    lidar_points[:, 0] = (lidar_points[:, 0] - pcr[0]) / expansion[0]
    lidar_points[:, 1] = (lidar_points[:, 1] - pcr[1]) / expansion[1]
    lidar_points[:, 2] = (lidar_points[:, 2] - pcr[2]) / expansion[2]
    return lidar_points.reshape(200, 200, 16, 3)


def labels_ref(sdf, thresh=0., logits=None, points=None, lut=None, z_keep=None, border=None, return_values=False):
    """Lattice sdf [H, W, D] (+ logits [H, W, D, C]) -> (occ int [n0, n1, n2], sem int or None).  points [n0, n1, n2, 3]
    normalised: resample as eval_iou.py:219-223 / 243-248.  z_keep / border as NeuSHead.occupancy.  return_values also
    returns the thresholded sdf values and the per-voxel logits (for near-tie accounting)."""
    grid = None
    if points is not None:
        grid = (points[..., [2, 0, 1]] * 2 - 1)[None].to(sdf.dtype)
        s = F.grid_sample(sdf[None, None], grid, mode='bilinear', align_corners=True)[0, 0]
    else:
        s = sdf
    occ = (s <= thresh).to(torch.int)
    n2 = occ.shape[2]
    lo, hi = (0, n2) if z_keep is None else z_keep
    hi = n2 + hi if hi < 0 else hi
    occ[..., hi:] = 0
    occ[..., :lo] = 0
    b = (0, 0, 0, 0) if border is None else border
    occ[:b[0]] = 0
    if b[1]:
        occ[-b[1]:] = 0
    occ[:, :b[2]] = 0
    if b[3]:
        occ[:, -b[3]:] = 0
    sem, lg = None, None
    if logits is not None:
        if grid is not None:
            lg = F.grid_sample(logits.permute(3, 0, 1, 2)[None], grid, mode='bilinear', align_corners=True)[0].permute(1, 2, 3, 0)
        else:
            lg = logits
        arg = torch.argmax(lg, dim=-1)
        if lut is not None:
            arg = torch.as_tensor(lut, device=arg.device)[arg.flatten()].reshape(arg.shape)
        sem = occ * arg
    return (occ, sem, s, lg) if return_values else (occ, sem)


class MeanIoURef:
    """utils/metric_util.py:66-165 (tensor-target branch)."""

    def __init__(self, class_indices, empty_label, label_str, use_mask=False, dataset_empty_label=17, name='none'):
        self.class_indices, self.num_classes, self.empty_label = list(class_indices), len(class_indices), empty_label
        self.reset()

    def reset(self):
        n = self.num_classes + 1
        self.total_seen, self.total_correct, self.total_positive = [0] * n, [0] * n, [0] * n

    def _after_step(self, outputs, targets, mask=None):
        if mask is not None:
            outputs, targets = outputs[mask], targets[mask]
        for i, c in enumerate(self.class_indices):
            self.total_seen[i] += torch.sum(targets == c).item()
            self.total_correct[i] += torch.sum((targets == c) & (outputs == c)).item()
            self.total_positive[i] += torch.sum(outputs == c).item()
        self.total_seen[-1] += torch.sum(targets != self.empty_label).item()
        self.total_correct[-1] += torch.sum((targets != self.empty_label) & (outputs != self.empty_label)).item()
        self.total_positive[-1] += torch.sum(outputs != self.empty_label).item()

    def _after_epoch(self):
        seen, correct, positive = (torch.tensor(v, dtype=torch.float32) for v in
                                   (self.total_seen, self.total_correct, self.total_positive))
        ious = []
        for i in range(self.num_classes):
            if seen[i] == 0:
                ious.append(1)
            else:
                ious.append((correct[i] / (seen[i] + positive[i] - correct[i])).item())
        occ_iou = correct[-1] / (seen[-1] + positive[-1] - correct[-1])
        return np.mean(ious) * 100, float(occ_iou * 100)


class IoURef:
    """utils/metric_util.py:168-244 (``_after_step`` with the [K, 3] coordinates of the occupied ground-truth voxels)."""

    def __init__(self, use_mask=False):
        self.reset()

    def reset(self):
        self.total_seen, self.total_correct, self.total_positive = 0, 0, 0

    def _after_step(self, outputs, targets):
        self.total_seen += targets.shape[0]
        self.total_correct += int(outputs[tuple(targets.transpose(0, 1))].sum())
        self.total_positive += int(outputs.sum())

    def _after_epoch(self):
        seen, correct, positive = (torch.tensor([v], dtype=torch.float32) for v in
                                   (self.total_seen, self.total_correct, self.total_positive))
        if seen[0] == 0:
            return np.mean([1]) * 100
        return np.mean([(correct[0] / (seen[0] + positive[0] - correct[0])).item()]) * 100


class SSCMetricsRef:
    """utils/scenerf_metric.py:39-215 (batch axis = the first axis of the label volume, as eval_iou_kitti.py feeds it)."""

    def __init__(self, n_classes):
        self.n_classes = n_classes
        self.reset()

    def reset(self):
        self.completion_tp = self.completion_fp = self.completion_fn = 0
        self.tps, self.fps, self.fns = [0] * self.n_classes, [0] * self.n_classes, [0] * self.n_classes

    def add_batch(self, y_pred, y_true, nonempty=None):
        mask = y_true != 255
        if nonempty is not None:
            mask = mask & nonempty
        pred, true = y_pred.clone(), y_true.clone()
        pred[true == 255] = 0
        true[true == 255] = 0
        for idx in range(pred.shape[0]):
            m = mask[idx].reshape(-1)
            yt, yp = (true[idx].reshape(-1) > 0)[m], (pred[idx].reshape(-1) > 0)[m]
            self.completion_tp += int((yt & yp).sum())
            self.completion_fp += int((~yt & yp).sum())
            self.completion_fn += int((yt & ~yp).sum())
            yt, yp = true[idx].reshape(-1)[m], pred[idx].reshape(-1)[m]
            for j in range(self.n_classes):
                self.tps[j] += int(((yt == j) & (yp == j)).sum())
                self.fps[j] += int(((yt != j) & (yp == j)).sum())
                self.fns[j] += int(((yt == j) & (yp != j)).sum())

    def get_stats(self):
        tp, fp, fn = (torch.tensor([v], dtype=torch.float32) for v in (self.completion_tp, self.completion_fp, self.completion_fn))
        if tp != 0:
            precision, recall, iou = tp / (tp + fp), tp / (tp + fn), tp / (tp + fp + fn)
        else:
            precision, recall, iou = 0, 0, 0
        tps, fps, fns = (torch.tensor(v, dtype=torch.float32) for v in (self.tps, self.fps, self.fns))
        iou_ssc = tps / (tps + fps + fns + 1e-5)
        return {'precision': float(precision), 'recall': float(recall), 'iou': float(iou), 'iou_ssc': iou_ssc,
                'iou_ssc_mean': float(torch.mean(iou_ssc[1:]))}
