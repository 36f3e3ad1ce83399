"""Training losses of the shipped configs (reference loss/*.py) under the reference's class names and constructors.

* ReprojLossMonoMultiNewCombine / ReprojLossMonoMultiNew: the self-supervised reprojection loss every shipped config
  puts first in its MultiLoss, as CUDA kernels (csrc/reproj.cu) with a backward to the head's per-sample weights.
* EikonalLoss, EdgeLoss3DMS, SecondGradLoss: plain torch (element-wise or ray-grid sized).
* MultiLoss with the reference's ``(tot, loss_dict)`` return.
* OPENOCC_LOSS: mmengine's ``Registry('openocc_loss')`` when mmengine is importable, else the package's Registry;
  ``register_into(registry)`` puts these classes into the reference's own OPENOCC_LOSS (train.py builds the loss from it),
  next to its RGBLossMS / Sem* / *SparsityLoss.

No TensorBoard scalars are written: the reference's ``masked/{cam}`` count and ``loss/*`` scalars need a host sync each.
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from .registry import Registry

try:  # pragma: no cover - mmengine is absent in the build container
    from mmengine.registry import Registry as _MMRegistry
    OPENOCC_LOSS = _MMRegistry('openocc_loss')
except Exception:
    OPENOCC_LOSS = Registry('openocc_loss')


class BaseLoss(nn.Module):
    """loss/base_loss.py: ``forward(inputs)`` picks ``input_dict``'s entries out of ``inputs`` and returns
    ``weight * loss_func(**picked)``."""

    def __init__(self, weight=1.0, input_dict=None, **kwargs):
        super().__init__()
        self.weight = weight
        self.input_dict = input_dict if input_dict is not None else {'input': 'input'}
        self.loss_func = lambda: 0

    def forward(self, inputs):
        return self.weight * self.loss_func(**{k: inputs[v] for k, v in self.input_dict.items()})


_REPROJ_INPUTS = ('curr_imgs', 'prev_imgs', 'next_imgs', 'ray_indices', 'weights', 'ts', 'metas', 'ms_rays')


def _pinned_upload(trans, n_cam, dev):
    """list2tensor (reproj_loss_mono_multi_new.py:101-110) of metas[i]['img2prevImg' / 'img2nextImg'] (numpy, lists or
    tensors) -> [N, 4, 4] fp32 on `dev`, staged through pinned memory so the copy does not synchronise."""
    if isinstance(trans[0], torch.Tensor):
        t = torch.stack(list(trans)).to(torch.float32)
        if t.device == dev:
            return t.reshape(n_cam, 4, 4).contiguous()
        t = t.cpu()
    else:
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(trans, dtype=np.float32)))
    return t.reshape(n_cam, 4, 4).contiguous().pin_memory().to(dev, non_blocking=True)


def _stack(ts):
    if isinstance(ts, torch.Tensor):
        return ts.reshape(ts.shape[0], -1).contiguous()
    return torch.stack([t.reshape(-1) for t in ts]).contiguous()


class _ReprojLoss(BaseLoss):
    COMBINE = True

    def __init__(self, weight=1.0, input_dict=None, **kwargs):
        super().__init__(weight, input_dict if input_dict is not None else {k: k for k in _REPROJ_INPUTS})
        self.no_ssim = kwargs.get('no_ssim', False)
        self.img_size = kwargs.get('img_size', [768, 1600])
        self.ray_resize = kwargs.get('ray_resize', None)
        self.no_automask = kwargs.get('no_automask', False)
        self.dims = kwargs.get('dims', 3)
        self.no_ssim = self.no_ssim or (self.ray_resize is None)
        if self.dims != 3:
            raise NotImplementedError('%s: dims=%r, the kernels implement 3 colour channels' % (type(self).__name__, self.dims))
        self.loss_func = self.reproj_loss
        self.iter_counter = 0
        self._pending = []          # (event, pinned flag) of layout checks not yet read

    def check_layout(self):
        """Raises if a completed step was handed a ray_indices other than arange(R).repeat_interleave(S).  Reads only
        checks whose copy has finished (an event query, no synchronisation); MultiLoss calls it after its .item()."""
        keep = []
        for ev, flag in self._pending:
            if not ev.query():
                keep.append((ev, flag))
            elif int(flag[0]):
                self._pending = []
                raise ValueError('%s: ray_indices must be arange(R).repeat_interleave(S) per camera (S contiguous samples '
                                 'per ray, rays in order), as NeuSHead.forward returns them' % type(self).__name__)
        self._pending = keep

    def _enqueue_layout_check(self, ray_indices, n_samples, dev):
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        seen = set()
        for idx in ray_indices:
            if idx.data_ptr() in seen:
                continue
            seen.add(idx.data_ptr())
            ops.reproj_check_layout(idx.reshape(-1).contiguous(), n_samples, bad)
        flag = torch.empty(1, dtype=torch.int32, pin_memory=True)
        flag.copy_(bad, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._pending.append((ev, flag))

    def reproj_loss(self, curr_imgs, prev_imgs, next_imgs, ray_indices, weights, ts, metas, ms_rays, deltas=None,
                    sample_sdfs=None):
        self.check_layout()
        bs, num_cams = curr_imgs.shape[:2]
        assert bs == 1
        R = ms_rays.shape[0]
        if len(weights) != num_cams or len(ts) != num_cams or len(ray_indices) != num_cams:
            raise ValueError('%s: one weights / ts / ray_indices entry per camera expected' % type(self).__name__)
        if any(isinstance(t, torch.Tensor) and t.requires_grad for t in ts):
            raise ValueError('%s: ts must not require grad (no gradient w.r.t. ts is computed)' % type(self).__name__)
        n = weights[0].numel()
        if n % R or any(w.numel() != n for w in weights) or any(i.numel() != n for i in ray_indices):
            raise ValueError('%s: every camera needs R * S weights, ts and ray_indices (R = %d rays)' % (type(self).__name__, R))
        S = n // R
        dev = curr_imgs.device
        W = _stack(weights)
        T = _stack(ts).detach()
        D = _stack(deltas).detach() if deltas is not None else None
        tp = _pinned_upload([m['img2prevImg'] for m in metas], num_cams, dev)
        tn = _pinned_upload([m['img2nextImg'] for m in metas], num_cams, dev)
        self._enqueue_layout_check(ray_indices, S, dev)
        desc = ops.make_reproj_desc(self.COMBINE, num_cams, R, S, curr_imgs.shape[-2:], self.img_size,
                                    None if self.no_ssim else self.ray_resize, not self.no_ssim, not self.no_automask)
        img = lambda x: x[0].to(torch.float32).contiguous()
        loss = ops.ReprojLossFunction.apply(W, desc, img(curr_imgs), img(prev_imgs), img(next_imgs),
                                            ms_rays.to(torch.float32).contiguous(), tp, tn, T, D)
        self.iter_counter += 1
        return loss


class ReprojLossMonoMultiNewCombine(_ReprojLoss):
    """loss/reproj_loss_mono_multi_new_combine.py: one l1 (+ SSIM) term of the colour composed from both neighbour frames
    per ray, automasked against the static-frame losses; border padding.  Kwargs as the reference: weight, input_dict,
    no_ssim, img_size, ray_resize (None forces no_ssim), no_automask, dims (3 only)."""
    COMBINE = True


class ReprojLossMonoMultiNew(_ReprojLoss):
    """loss/reproj_loss_mono_multi_new.py with sdf_loss=False: separate prev / next terms, min over them (and the
    automask terms); zeros padding.  Kwargs as ReprojLossMonoMultiNewCombine plus sdf_loss (False only)."""
    COMBINE = False

    def __init__(self, weight=1.0, input_dict=None, **kwargs):
        if kwargs.get('sdf_loss', False):
            raise NotImplementedError('ReprojLossMonoMultiNew: sdf_loss=True is not provided (no shipped config enables it)')
        super().__init__(weight, input_dict, **kwargs)


class EikonalLoss(BaseLoss):
    """loss/eikonal_loss.py: mean (|grad| - 1)^2."""

    def __init__(self, weight=1.0, input_dict=None, **kwargs):
        super().__init__(weight, input_dict if input_dict is not None else {'eik_grad': 'eik_grad'})
        self.loss_func = self.eikonal_loss

    def eikonal_loss(self, eik_grad):
        return ((eik_grad.norm(2, dim=-1) - 1) ** 2).mean()


class SecondGradLoss(BaseLoss):
    """loss/second_grad_loss.py: mean |second_grad|."""

    def __init__(self, weight=1.0, input_dict=None, **kwargs):
        super().__init__(weight, input_dict if input_dict is not None else {'second_grad': 'second_grad'})
        self.loss_func = self.second_grad_loss

    def second_grad_loss(self, second_grad):
        return second_grad.abs().mean()


class EdgeLoss3DMS(BaseLoss):
    """loss/edge_loss_3d_ms.py: edge-aware smoothness of the mean-normalised depth on the ray_resize grid."""

    def __init__(self, weight=1.0, input_dict=None, **kwargs):
        super().__init__(weight, input_dict if input_dict is not None else
                         {'curr_imgs': 'curr_imgs', 'ms_depths': 'ms_depths', 'ms_rays': 'ms_rays'})
        self.img_size = kwargs.get('img_size', [768, 1600])
        self.ray_resize = kwargs.get('ray_resize', None)
        self.use_inf_mask = kwargs.get('use_inf_mask', False)
        if self.ray_resize is None:
            raise ValueError('EdgeLoss3DMS needs ray_resize')
        self.loss_func = self.edge_loss

    def edge_loss(self, curr_imgs, ms_depths, ms_rays, ms_accs=None, max_depths=None):
        if self.use_inf_mask and (ms_accs is None or max_depths is None):
            raise ValueError('EdgeLoss3DMS(use_inf_mask=True) needs ms_accs and max_depths')
        if not isinstance(ms_rays, (list, tuple)):
            ms_rays = [ms_rays] * len(ms_depths)
        bs, num_cams, num_rays = ms_depths[0].shape
        tot = 0.
        for scale, (depth, rays) in enumerate(zip(ms_depths, ms_rays)):
            g = rays.reshape(1, 1, num_rays, 2).repeat(bs * num_cams, 1, 1, 1) \
                / rays.new_tensor([self.img_size[1], self.img_size[0]]) * 2 - 1
            rgb = F.grid_sample(curr_imgs.flatten(0, 1), g, mode='bilinear', padding_mode='border', align_corners=True)
            rgb = rgb.reshape(bs * num_cams, -1, *self.ray_resize)
            if self.use_inf_mask:
                depth = depth * ms_accs[scale] + max_depths[scale] * (1 - ms_accs[scale])
            d = depth.reshape(bs * num_cams, 1, *self.ray_resize)
            d = d / (d.mean(2, True).mean(3, True) + 1e-6)
            gdx = (d[..., :-1] - d[..., 1:]).abs() * torch.exp(-(rgb[..., :-1] - rgb[..., 1:]).abs().mean(1, True))
            gdy = (d[..., :-1, :] - d[..., 1:, :]).abs() * torch.exp(-(rgb[..., :-1, :] - rgb[..., 1:, :]).abs().mean(1, True))
            tot = tot + gdx.mean() + gdy.mean()
        return tot / len(ms_depths)


class MultiLoss(nn.Module):
    """loss/multi_loss.py: the sum of the configured losses and {class name: value} (one .item() per loss, as the
    reference).  The reprojection losses' ray-layout checks are read right after those .item() calls.  The sub-losses are
    built from ``registry``: this package's OPENOCC_LOSS here, the target registry in the class register_into installs."""

    registry = None        # None: this module's OPENOCC_LOSS (bound late: it is created after the class)

    def __init__(self, loss_cfgs):
        super().__init__()
        assert isinstance(loss_cfgs, list)
        self.num_losses = len(loss_cfgs)
        reg = type(self).registry if type(self).registry is not None else OPENOCC_LOSS
        self.losses = nn.ModuleList([reg.build(c) for c in loss_cfgs])
        self.iter_counter = 0

    def forward(self, inputs):
        loss_dict = {}
        tot_loss = 0.
        for loss_func in self.losses:
            loss = loss_func(inputs)
            tot_loss += loss
            loss_dict[loss_func.__class__.__name__] = loss.detach().item()
            check = getattr(loss_func, 'check_layout', None)
            if check is not None:
                check()
        self.iter_counter += 1
        return tot_loss, loss_dict


LOSSES = (MultiLoss, ReprojLossMonoMultiNewCombine, ReprojLossMonoMultiNew, EikonalLoss, EdgeLoss3DMS, SecondGradLoss)


def register_into(registry):
    """Register this module's losses into `registry` (e.g. the reference's loss.OPENOCC_LOSS) under their class names,
    replacing entries of the same name; returns the registry.  The MultiLoss installed there is a subclass that builds
    its sub-losses from `registry` itself, so the entries this module does not provide (the reference's RGBLossMS,
    SemLossMS, SemCELossMS, *SparsityLoss) keep resolving to the registry's own classes."""
    for cls in LOSSES:
        if cls is MultiLoss and registry is not OPENOCC_LOSS:
            cls = type('MultiLoss', (MultiLoss,), {'registry': registry, '__module__': __name__,
                                                    '__qualname__': 'MultiLoss', '__doc__': MultiLoss.__doc__})
        registry.register_module(name=cls.__name__, module=cls, force=True)
    return registry


register_into(OPENOCC_LOSS)
