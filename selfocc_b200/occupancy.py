"""Occupancy-evaluation data of the reference scripts (eval_iou.py, eval_iou_kitti.py, utils/metric_util.py) and the
Occ3D sample points.  The labels themselves come from ``NeuSHead.occupancy`` (so_occ_classify), the scores from
``selfocc_b200.metric.MeanIoU / IoU / SSCMetrics`` (so_occ_hist)."""
import torch

# utils/metric_util.py:37-64: OpenSeeD class -> nuScenes occupancy class (index = argmax of the 21 semantic channels)
OPENSEED2NUSCENES = (1, 2, 3, 4, 5, 5, 6, 7, 8, 9, 9, 10, 11, 12, 13, 14, 14, 15, 15, 16, 0)
# utils/metric_util.py:10-35: Cityscapes class -> SemanticKITTI class
CITYSCAPES2SEMANTICKITTI = (9, 11, 13, 13, 14, 18, 19, 19, 15, 17, 0, 6, 7, 1, 4, 5, 5, 3, 2)

# eval_iou.py:174-196: --scene-size -> (point_cloud_range, expansion) of the Occ3D evaluation
SCENE_SIZES = {
    0: ([-51.2, -51.2, -4, 51.2, 51.2, 4], [102.4, 102.4, 8]),
    1: ([-40.0, -40.0, -2.8, 40.0, 40.0, 3.6], [80.0, 80.0, 6.4]),
    2: ([-40.0, -40.0, -3.1, 40.0, 40.0, 3.9], [80.0, 80.0, 7.0]),
    3: ([-40.0, -40.0, -3.2, 40.0, 40.0, 4.0], [80.0, 80.0, 7.2]),
    4: ([-40.0, -40.0, -1.0, 40.0, 40.0, 5.4], [80.0, 80.0, 6.4]),
    5: ([-51.2, -51.2, -5, 51.2, 51.2, 3], [102.4, 102.4, 8]),
    6: ([-51.2, -51.2, -4, 51.2, 51.2, 5], [102.4, 102.4, 9]),
}
# eval_iou.py:175: the OpenOccupancy evaluation range (no resampling)
OPENOCC_RANGE = [-51.2, -51.2, -5, 51.2, 51.2, 3]
# eval_iou_kitti.py:163
KITTI_RANGE = [-25.6, 0, -2.0, 25.6, 51.2, 4.4]

# border rules: (z_keep, border) arguments of NeuSHead.occupancy; None in z_keep = the lattice depth D
OCC3D_BORDERS = ((0, 12), (6, 6, 6, 6))                 # eval_iou.py:228-232
OPENOCC_BORDERS = ((5, -4), (6, 6, 6, 6))               # eval_iou.py:252-257: [..., :5] and [..., -4:] zeroed
KITTI_BORDERS = ((0, 28), (0, 6, 6, 6))                 # eval_iou_kitti.py:182-186: the first rows are kept


def lut_tensor(table, device):
    return torch.tensor(table, dtype=torch.uint8, device=device)


def occ3d_grid(device=None):
    """eval_iou.py:151-164: the homogeneous 200 x 200 x 16 Occ3D voxel centres in ego metres, [200, 200, 16, 4]."""
    xx = torch.linspace(-40.0, 40.0, 200)
    yy = torch.linspace(-40.0, 40.0, 200)
    zz = torch.linspace(-1.0, 5.4, 16)
    xyz = torch.stack([xx[:, None, None].expand(-1, 200, 16), yy[None, :, None].expand(200, -1, 16),
                       zz[None, None, :].expand(200, 200, -1), torch.ones(200, 200, 16)], dim=-1)
    return xyz if device is None else xyz.to(device)


def occ3d_points(ego2lidar, scene_size=4, xyz=None, device=None):
    """eval_iou.py:211-218: the Occ3D voxel centres moved into the lidar frame and normalised by the scene range ->
    [200, 200, 16, 3] (x, y, z) in [0, 1], the ``points`` argument of ``NeuSHead.occupancy``.  Same torch ops in the
    same order as the reference, so the points are bit-identical to its ``lidar_points``.  ``xyz``: occ3d_grid() of the
    target device, computed once per evaluation like the reference does."""
    pcr, expansion = SCENE_SIZES[scene_size]
    if xyz is None:
        xyz = occ3d_grid(device)
    e2l = xyz.new_tensor(ego2lidar)
    pts = torch.matmul(e2l.unsqueeze(0), xyz.reshape(-1, 4, 1))
    pts = pts.squeeze(-1)[:, :3]
    pts[:, 0] = (pts[:, 0] - pcr[0]) / expansion[0]
    pts[:, 1] = (pts[:, 1] - pcr[1]) / expansion[1]
    pts[:, 2] = (pts[:, 2] - pcr[2]) / expansion[2]
    return pts.reshape(200, 200, 16, 3)
