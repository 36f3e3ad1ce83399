"""B1-B13: NeuSHead behind the reference's head API (model/head/neus_head/neus_head.py:21-721).

The reference head is an adapter over the un-vendored sdfstudio fork; here the same public surface
(``prepare`` / ``render`` / ``forward_occ`` / ``forward``, constructor kwargs, output dict keys) drives
the fused sm_100a kernels.  Fork-only knobs whose semantics cannot be recovered from the reference
(SURVEY.md 8c) are rejected when set to a non-default value instead of being silently ignored.
"""
import math
import os
import numpy as np
import torch
import torch.nn as nn

from . import ops
from .encoder import _metas_matrix
from .mapping import GridMeterMapping
from .registry import HEADS


class RaySampler(nn.Module):
    """B1.  model/head/nerfacc_head/ray_sampler.py:5-68.  ``forward()`` returns the [R, 2] (x, y) pixel
    table like the reference; ``grid()`` exposes the same rays as strided-grid parameters so the render
    kernel can generate them in registers (bit-identical: one fp32 multiply and one add per coordinate)."""

    def __init__(self, ray_sample_mode='fixed', ray_number=[192, 400], ray_img_size=[768, 1600], ray_upper_crop=0,
                 ray_x_dsr_max=None, ray_y_dsr_max=None):
        super().__init__()
        assert ray_sample_mode in ['fixed', 'cellular', 'random']
        self.ray_sample_mode = ray_sample_mode
        self.ray_number = ray_number[0] * ray_number[1]
        self.ray_resize = list(ray_number)
        self.ray_img_size = list(ray_img_size)
        self.ray_upper_crop = ray_upper_crop
        ny, nx = ray_number
        xs, ys = torch.arange(nx, dtype=torch.float), torch.arange(ny, dtype=torch.float)
        if ray_sample_mode == 'fixed':
            self._grid = (ny, nx, 1.0 * ray_img_size[1] / nx, 0.0, 1.0 * ray_img_size[0] / ny, 0.0)
            xs, ys = xs * self._grid[2], ys * self._grid[4]
        elif ray_sample_mode == 'cellular':
            self.ray_x_dsr_max = 1.0 * ray_img_size[1] / nx if ray_x_dsr_max is None else ray_x_dsr_max
            self.ray_y_dsr_max = 1.0 * (ray_img_size[0] - ray_upper_crop) / ny if ray_y_dsr_max is None else ray_y_dsr_max
            assert self.ray_x_dsr_max > 1 and self.ray_y_dsr_max > 1
            self._grid = None
        table = torch.stack([xs[None, :].expand(ny, -1), ys[:, None].expand(-1, nx)], -1)
        self.register_buffer('rays', table.flatten(0, 1) if ray_sample_mode == 'fixed' else table, False)

    def draw(self):
        """Advance the sampler (host RNG exactly like ray_sampler.py:58-63) and return the grid tuple
        (ny, nx, sx, ox, sy, oy), or None for the 'random' mode."""
        ny, nx = self.ray_resize
        if self.ray_sample_mode == 'fixed':
            return self._grid
        if self.ray_sample_mode == 'cellular':
            x_dsr = np.random.uniform() * (self.ray_x_dsr_max - 1) + 1
            y_dsr = np.random.uniform() * (self.ray_y_dsr_max - 1) + 1
            x_emp = np.random.uniform() * (self.ray_img_size[1] - nx * x_dsr)
            y_emp = np.random.uniform() * (self.ray_img_size[0] - self.ray_upper_crop - ny * y_dsr)
            return (ny, nx, x_dsr, x_emp, y_dsr, y_emp + self.ray_upper_crop)
        return None

    def table(self, grid):
        if self.ray_sample_mode == 'fixed':
            return self.rays
        if self.ray_sample_mode == 'random':
            rays = torch.rand(self.ray_number, 2, device=self.rays.device)
            rays[:, 0] *= self.ray_img_size[1]
            rays[:, 1] *= self.ray_img_size[0]
            return rays
        ny, nx, sx, ox, sy, oy = grid
        rays = self.rays.clone()
        rays[..., 0] = rays[..., 0] * sx + ox
        # ray_sampler.py:67 adds y_emp and the crop separately; oy carries their fp64 sum
        rays[..., 1] = rays[..., 1] * sy + oy
        return rays.flatten(0, 1)

    def forward(self):
        return self.table(self.draw())


class Img2LiDAR(nn.Module):
    """B2.  model/head/nerfacc_head/img2lidar.py:6-70: selects the per-camera 4x4 pixel->lidar matrices
    (the kernel derives origin = M[:3,3] and direction = M[:3,:3](x,y,1) itself)."""

    def __init__(self, trans_kw, trans_kw_eval=None, novel_view=None):
        super().__init__()
        if not isinstance(trans_kw, list):
            trans_kw, self.two_split = [trans_kw], False
        else:
            assert trans_kw == ['img2lidar', 'temImg2lidar']
            self.two_split = True
        self.trans_kw = trans_kw
        self.trans_kw_eval = trans_kw if trans_kw_eval is None else trans_kw_eval
        self.novel_view = novel_view

    def matrices(self, metas, device):
        kws = self.trans_kw_eval if os.environ.get('eval', 'false') == 'true' else self.trans_kw
        if not isinstance(kws, list):
            kws = [kws]
        M = torch.cat([_metas_matrix(metas, k, device) for k in kws], 1).clone()   # B, N, 4, 4
        return self.apply_novel_view(M) if self.novel_view is not None else M

    def apply_novel_view(self, M):
        """img2lidar.py:51-61: z-rotation (degrees) of the 3x3 block, then an xyz translation of the origin.  M [B, N, 4, 4]."""
        a = math.radians(self.novel_view[3])
        R = torch.tensor([[math.cos(a), -math.sin(a), 0.], [math.sin(a), math.cos(a), 0.], [0., 0., 1.]], device=M.device)
        M = M.clone()
        M[..., :3, :3] = R[None, None] @ M[..., :3, :3]
        for i in range(3):
            M[..., i, 3] = M[..., i, 3] + self.novel_view[i]
        return M

    def forward(self, metas, rays):
        M = self.matrices(metas, rays.device)
        pad = torch.cat([rays.float().reshape(1, 1, -1, 2), torch.ones(1, 1, rays.shape[0], 1, device=rays.device)], -1)
        return M[..., :3, 3], torch.matmul(M[..., :3, :3].unsqueeze(2), pad.unsqueeze(-1)).squeeze(-1)


class _Deviation(nn.Module):
    """upstream SingleVarianceNetwork: inv_s = exp(10 * variance) clipped to [1e-6, 1e6]."""

    def __init__(self, init_val):
        super().__init__()
        self.variance = nn.Parameter(init_val * torch.ones(1))

    def get_variance(self):
        return torch.exp(self.variance * 10.0).clip(1e-6, 1e6)


class _SDFField(nn.Module):
    """TPV SDF field: per-frame decoded volume + trilinear queries (SURVEY.md rows B5, B7, B8, B12).
    Parameter layout follows the in-repo analogue bev_nerf.py:62-71 (``density_net.{1,3}``)."""

    def __init__(self, mapping_args, embed_dims, color_dims, density_layers, sh_deg, sh_act, beta_init, tpv):
        super().__init__()
        if not tpv:
            raise NotImplementedError('tpv=False (single BEV plane decode) is not used by the target configs')
        if density_layers != 2:
            raise NotImplementedError('density_layers=%d: the fused decode kernel implements the 2-layer MLP' % density_layers)
        if sh_deg != 0:
            raise NotImplementedError('sh_deg=%d: all shipped configs use degree 0' % sh_deg)
        if color_dims not in (0,) and color_dims < 3:
            raise ValueError('color_dims must be 0 or >= 3')
        self.mapping = GridMeterMapping(**mapping_args)
        self.embed_dims, self.color_dims, self.sh_act = embed_dims, color_dims, sh_act
        self.density_net = nn.Sequential(nn.Softplus(), nn.Linear(embed_dims, embed_dims), nn.Softplus(),
                                         nn.Linear(embed_dims, 1 + color_dims))
        self.deviation_network = _Deviation(beta_init)
        self.desc = self.mapping.volume_desc(color_dims)
        self.vol_sdf = self.vol_feat = None
        self._pack = None

    def pre_compute_density_color(self, representation):
        hw, zh, wz = representation
        assert hw.shape[0] == 1, 'only support bs = 1 currently'
        l1, l2 = self.density_net[1], self.density_net[3]
        self.vol_sdf, self.vol_feat = ops.tpv_decode(hw[0].contiguous(), zh[0].contiguous(), wz[0].contiguous(),
                                                     l1.weight, l1.bias, l2.weight, l2.bias, self.desc)
        self._pack = None

    def render_pack(self):
        """The frame's packed render volume (ops.render_pack), built on the first render after a decode and reused by
        every further render of the frame (eval_novel_depth.py:143-172: one prepare, several poses).  Keyed on the
        volume tensors' identity and version, so a volume swapped in from outside (training forward, tests) is repacked."""
        vf = self.vol_feat
        key = (self.vol_sdf.data_ptr(), self.vol_sdf._version, None if vf is None else (vf.data_ptr(), vf._version))
        if self._pack is None or self._pack[0] != key:
            self._pack = (key, ops.render_pack(self.vol_sdf, vf, self.desc))    # None: no packed form for this channel count
        return self._pack[1]

    def forward_geonetwork(self, xyz):
        s, _, f = ops.field_query(self.vol_sdf, self.vol_feat, self.desc, xyz.reshape(-1, 3).contiguous(), want_feat=True)
        return torch.cat([s[:, None], f], -1).reshape(*xyz.shape[:-1], -1)

    def forward_sdfnetwork(self, xyz):
        return ops.field_query(self.vol_sdf, self.vol_feat, self.desc, xyz.reshape(-1, 3).contiguous())[0].reshape(xyz.shape[:-1])


class _Model(nn.Module):
    def __init__(self, field):
        super().__init__()
        self.field = field


# Options whose semantics live only in the un-vendored sdfstudio fork: rejected at construction when non-default.
# `return_second_grad` / `use_compact_2nd_grad` are NOT in this list: four of the six shipped TPV configs set them, they
# only add the `second_grad` training output (SecondGradLoss), so construction, prepare(), render() and forward_occ()
# work with those configs and only the training-form forward() refuses (see forward()).
_UNSUPPORTED_DEFAULTS = dict(use_numerical_gradients=False, use_uniform_gradient=False, calculate_online=False,
                             beta_hand_tune=False, estimate_flow=False, disp_sampler=False,
                             anneal_aabb=False, using_2d_img_feats=False,
                             num_samples_importance=0, num_up_sample_steps=0)


@HEADS.register_module()
class NeuSHead(nn.Module):
    def __init__(self, roi_aabb, resolution=0.4, near_plane=0.0, far_plane=1e10, num_samples=64, num_samples_importance=0,
                 num_up_sample_steps=0, base_variance=64, beta_init=0.1, beta_max=0.195, total_iters=3516 * 11,
                 use_numerical_gradients=False, numerical_gradients_delta=0.01, use_uniform_gradient=False,
                 nbr_gradient_points=128 * 128 * 16, calculate_online=False, sample_gradient=True, use_compact_2nd_grad=False,
                 beta_hand_tune=False, return_uniform_sdf=False, estimate_flow=False, return_max_depth=False,
                 return_surface_sdf=False, return_second_grad=False, return_sample_sdf=False, return_sem=False,
                 disp_sampler=False, anneal_aabb=False, aabb_every_iters=3516, aabb_min_near=10., aabb_min_far_frac=0.25,
                 ray_sample_mode='fixed', ray_number=[192, 400], ray_img_size=[768, 1600], ray_upper_crop=0,
                 ray_x_dsr_max=None, ray_y_dsr_max=None, trans_kw='img2lidar', trans_kw_eval=None, novel_view=None,
                 render_bkgd='white', mapping_args=None, embed_dims=128, color_dims=0, density_layers=2, sh_deg=2,
                 sh_act='relu', init_cfg=None, print_freq=50, two_split=True, tpv=False, using_2d_img_feats=False,
                 sample_anchor='mid', second_grad_assumption=None, **kwargs):
        super().__init__()
        given = dict(use_numerical_gradients=use_numerical_gradients, use_uniform_gradient=use_uniform_gradient,
                     calculate_online=calculate_online, beta_hand_tune=beta_hand_tune, estimate_flow=estimate_flow,
                     disp_sampler=disp_sampler, anneal_aabb=anneal_aabb, using_2d_img_feats=using_2d_img_feats,
                     num_samples_importance=num_samples_importance, num_up_sample_steps=num_up_sample_steps)
        bad = {k: v for k, v in given.items() if v != _UNSUPPORTED_DEFAULTS[k]}
        if bad:
            raise NotImplementedError('NeuSHead options outside the restated semantics (sdfstudio-fork only): %r' % bad)
        if render_bkgd not in ('white', 'black', 'random'):
            raise NotImplementedError('render_bkgd=%r' % render_bkgd)
        if mapping_args is None:
            raise ValueError('mapping_args is required')
        rs = dict(ray_number=ray_number, ray_img_size=ray_img_size, ray_upper_crop=ray_upper_crop)
        self.ray_sampler = RaySampler(ray_sample_mode=ray_sample_mode, ray_x_dsr_max=ray_x_dsr_max, ray_y_dsr_max=ray_y_dsr_max, **rs)
        self.ray_sampler_eval = RaySampler(ray_sample_mode='fixed', **rs)
        self.img2lidar = Img2LiDAR(trans_kw=trans_kw, trans_kw_eval=trans_kw_eval, novel_view=novel_view)
        self.model = _Model(_SDFField(mapping_args, embed_dims, color_dims, density_layers, sh_deg, sh_act, beta_init, tpv))
        self.near_plane, self.far_plane, self.num_samples = near_plane, far_plane, num_samples
        self.render_bkgd, self.sample_anchor = render_bkgd, sample_anchor
        self.print_freq, self.resolution, self.aabb = print_freq, resolution, list(roi_aabb)
        self.return_uniform_sdf, self.return_max_depth = return_uniform_sdf, return_max_depth
        self.return_surface_sdf, self.return_sample_sdf, self.return_sem = return_surface_sdf, return_sample_sdf, return_sem
        self.return_second_grad = return_second_grad
        self.second_grad_assumption = (os.environ.get('SELFOCC_B200_SECOND_GRAD', '0') == '1') if second_grad_assumption is None \
            else bool(second_grad_assumption)
        if return_sem and color_dims <= 3:
            raise ValueError('return_sem needs color_dims > 3 (3 rgb + semantic logits)')
        self.z_size = self.model.field.mapping.size_d
        self.bev_size = [self.model.field.mapping.size_h, self.model.field.mapping.size_w]
        self.two_split = two_split
        self.cos_anneal_ratio = 1.0

    # ------------------------------------------------------------------ checkpoints
    # The field's parameters follow the in-repo analogue's names (bev_nerf.py:62-71: ``density_net.{1,3}``) under
    # ``model.field``; a checkpoint written by the un-vendored fork may keep them under another module path.  On load, a
    # key of this head that is missing is looked up (i) through ``checkpoint_key_map`` ({regex: replacement}, applied to the
    # key relative to the head) and (ii) by its unambiguous suffix anywhere under the head's prefix.
    FIELD_SUFFIXES = ('density_net.1.weight', 'density_net.1.bias', 'density_net.3.weight', 'density_net.3.bias',
                      'deviation_network.variance')
    checkpoint_key_map = {}

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        import re
        for k in [k for k in state_dict if k.startswith(prefix)]:
            rel = k[len(prefix):]
            for pat, rep in self.checkpoint_key_map.items():
                new = re.sub(pat, rep, rel)
                if new != rel and prefix + new not in state_dict:
                    state_dict[prefix + new] = state_dict.pop(k)
                    break
        for suf in self.FIELD_SUFFIXES:
            tgt = prefix + 'model.field.' + suf
            if tgt in state_dict:
                continue
            cands = [k for k in state_dict if k.startswith(prefix) and k.endswith('.' + suf) and k != tgt]
            if len(cands) == 1:
                state_dict[tgt] = state_dict.pop(cands[0])
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)

    # ------------------------------------------------------------------ helpers
    def _sampler(self):
        return self.ray_sampler_eval if os.environ.get('eval', 'false') == 'true' else self.ray_sampler

    def _inv_s(self):
        """exp(10 * variance) as a host float, cached on the parameter's version so eval does not sync per frame."""
        v = self.model.field.deviation_network.variance
        key = (v._version, v.data_ptr())
        if getattr(self, '_inv_s_key', None) != key:
            self._inv_s_key, self._inv_s_val = key, float(self.model.field.deviation_network.get_variance())
        return self._inv_s_val

    def _params(self, training):
        f = self.model.field
        return ops.make_render_params(self.aabb, self.num_samples, self._inv_s(),
                                      near_plane=self.near_plane, training=training, cos_anneal=self.cos_anneal_ratio,
                                      anchor_mid=self.sample_anchor == 'mid', sh_act=f.sh_act, bkgd=self.render_bkgd)

    # ------------------------------------------------------------------ reference API
    def prepare(self, representation, metas=None, **kwargs):
        """neus_head.py:295-306."""
        self.model.field.pre_compute_density_color(representation)
        return {}

    @torch.no_grad()
    def render(self, metas=None, batch=0, ray_range=None, **kwargs):
        """neus_head.py:308-471: all cameras, all rays, one fused launch.  ``batch`` keeps the reference's
        chunking SEMANTICS (the per-chunk clip of the expected depth) without a python loop.
        ``ray_range=(begin, count)`` renders a contiguous slice of the flat (cam, ray) order (ray sharding)."""
        f = self.model.field
        if f.vol_sdf is None:
            raise RuntimeError('render() called before prepare()/forward(): no decoded volume')
        sampler = self._sampler()
        dev = f.vol_sdf.device
        grid = sampler.draw()
        rays = sampler.table(grid)
        M = self.img2lidar.matrices(metas, dev)
        bs, num_cams = M.shape[:2]
        assert bs == 1, 'only support bs = 1 currently'
        num_rays = rays.shape[0]
        total = num_cams * num_rays
        chunk_len = 0
        if batch > 0:
            chunks = int(math.ceil(total * 1.0 / batch))
            chunk_len = int(math.ceil(total / chunks))                 # torch.chunk sizes (neus_head.py:341-345)
        begin, count = (0, total) if ray_range is None else ray_range
        rd = ops.make_ray_desc(num_cams, grid=grid, n_pix=num_rays, ray_begin=begin, ray_count=count, chunk_len=chunk_len)
        has_rgb = f.color_dims >= 3
        want = ['depth', 'acc', 'normal_vis'] + (['max_depth'] if self.return_max_depth else []) \
            + (['rgb'] if has_rgb else []) + (['sem'] if self.return_sem else [])
        bk = torch.rand(count, 3, device=dev) if (self.render_bkgd == 'random' and has_rgb) else None
        out = ops.render_infer(f.vol_sdf, f.vol_feat, f.desc, M[0].contiguous(), rd, self._params(False),
                               pix=None if grid is not None else rays.contiguous(), bkgd_rand=bk, want=want,
                               pack=f.render_pack())
        full = ray_range is None
        shp = (lambda t, *tail: t.reshape(bs, num_cams, num_rays, *tail)) if full else (lambda t, *tail: t)
        outputs = {'ms_depths': [shp(out['depth'])],
                   'ms_colors': [shp(out['rgb'], 3) if has_rgb else out['depth'].new_empty(bs, num_cams, num_rays, 0)],
                   'vis_normal': [shp(out['normal_vis'], 3)], 'ms_accs': [shp(out['acc'])], 'ms_rays': rays}
        if self.return_max_depth:
            outputs['ms_max_depths'] = [shp(out['max_depth'])]
        if self.return_sem:
            outputs['sem'] = [shp(out['sem'], out['sem'].shape[-1])]
        return outputs

    @torch.no_grad()
    def render_poses(self, metas=None, poses=None, batch=0, want=None, **kwargs):
        """8f-3: K renders of the prepared frame in ONE launch.  The reference's novel-depth evaluation issues one
        ``head.render`` per source pose after a single ``prepare`` (eval_novel_depth.py:159-172,
        ``metas['render_img2lidar'] = temImg2lidars[source_id]``); here ``poses`` = those K matrix sets ([K, N, 4, 4] array /
        tensor or a list of K [N, 4, 4]; default: ``metas[0]['temImg2lidars']``) are rendered as K * N cameras of one ray
        set.  Every pose keeps its own expected-depth clip (the renderer clips per ``self.model(ray_bundle)`` call), so the
        result equals K separate ``render`` calls; returns the ``render`` dict with a leading pose axis: ms_depths[0] is
        [K, N, R].  ``batch > 0`` (the reference's chunking) falls back to K launches when a chunk would straddle poses."""
        f = self.model.field
        if f.vol_sdf is None:
            raise RuntimeError('render_poses() called before prepare()/forward(): no decoded volume')
        dev = f.vol_sdf.device
        if poses is None:
            poses = metas[0]['temImg2lidars']
        P = torch.as_tensor(np.asarray([np.asarray(p) for p in poses]) if not torch.is_tensor(poses) else poses,
                            dtype=torch.float32, device=dev)
        assert P.dim() == 4 and P.shape[-2:] == (4, 4), 'poses must be [K, N, 4, 4]'
        K, N = P.shape[:2]
        sampler = self._sampler()
        grid = sampler.draw()
        rays = sampler.table(grid)
        R = rays.shape[0]
        per_pose = N * R
        chunk_len = per_pose
        if batch > 0:
            chunks = int(math.ceil(per_pose * 1.0 / batch))
            chunk_len = int(math.ceil(per_pose / chunks))
            if per_pose % chunk_len:              # a chunk would straddle two poses: keep the reference's exact clip groups
                outs = []
                for k in range(K):
                    m2 = [dict(metas[0], render_img2lidar=P[k])]
                    saved = self.img2lidar.trans_kw, self.img2lidar.trans_kw_eval
                    self.img2lidar.trans_kw = self.img2lidar.trans_kw_eval = ['render_img2lidar']
                    try:
                        outs.append(self.render(metas=m2, batch=batch))
                    finally:
                        self.img2lidar.trans_kw, self.img2lidar.trans_kw_eval = saved
                keys = [k for k in outs[0] if isinstance(outs[0][k], list)]
                merged = {k: [torch.cat([o[k][0] for o in outs], 0)] for k in keys}
                merged['ms_rays'] = rays
                return merged
        M = P.reshape(K * N, 4, 4).clone()
        if self.img2lidar.novel_view is not None:
            M = self.img2lidar.apply_novel_view(M[None])[0]
        has_rgb = f.color_dims >= 3
        if want is None:
            want = ['depth', 'acc', 'normal_vis'] + (['max_depth'] if self.return_max_depth else []) + (['rgb'] if has_rgb else [])
        rd = ops.make_ray_desc(K * N, grid=grid, n_pix=R, chunk_len=chunk_len)
        bk = torch.rand(K * per_pose, 3, device=dev) if (self.render_bkgd == 'random' and 'rgb' in want) else None
        out = ops.render_infer(f.vol_sdf, f.vol_feat, f.desc, M.contiguous(), rd, self._params(False),
                               pix=None if grid is not None else rays.contiguous(), bkgd_rand=bk, want=want, pack=f.render_pack())
        shp = lambda t, *tail: t.reshape(K, N, R, *tail)
        res = {'ms_rays': rays}
        names = dict(depth='ms_depths', acc='ms_accs', max_depth='ms_max_depths')
        for k, v in out.items():
            if k in names:
                res[names[k]] = [shp(v)]
            elif k == 'rgb':
                res['ms_colors'] = [shp(v, 3)]
            elif k == 'normal_vis':
                res['vis_normal'] = [shp(v, 3)]
        return res

    def get_uniform_sdf(self, aabb, resolution, device, shift=False):
        """neus_head.py:265-293."""
        xs = torch.linspace(aabb[0], aabb[3], int((aabb[3] - aabb[0]) / resolution), device=device)
        ys = torch.linspace(aabb[1], aabb[4], int((aabb[4] - aabb[1]) / resolution), device=device)
        zs = torch.linspace(aabb[2], aabb[5], int((aabb[5] - aabb[2]) / resolution), device=device)
        W, H, D = len(xs), len(ys), len(zs)
        xyzs = torch.stack([xs[None, :, None].expand(H, W, D), ys[:, None, None].expand(H, W, D),
                            zs[None, None, :].expand(H, W, D)], dim=-1).flatten(0, 2)
        if shift:
            xyzs = xyzs + torch.rand_like(xyzs) * resolution
        if self.return_sem:
            h = self.model.field.forward_geonetwork(xyzs)
            sem = h[..., 4:]
            return h[..., 0].reshape(H, W, D), torch.argmax(sem, dim=-1).reshape(H, W, D), sem.reshape(H, W, D, -1), \
                xyzs.reshape(H, W, D, -1)
        return self.model.field.forward_sdfnetwork(xyzs).reshape(H, W, D), xyzs.reshape(H, W, D, -1)

    @torch.no_grad()
    def forward_occ(self, representation, metas=None, **kwargs):
        """neus_head.py:237-263."""
        device = representation[0].device if isinstance(representation, (tuple, list)) else representation.device
        self.model.field.pre_compute_density_color(representation)
        aabb = kwargs['aabb'] if 'aabb' in kwargs else self.aabb
        reso = kwargs['resolution'] if 'resolution' in kwargs else self.resolution
        if self.return_sem:
            sdf, sem, sem_logits, xyz = self.get_uniform_sdf(aabb, reso, device=device)
            return {'sdf': sdf, 'rep': representation, 'sem': sem, 'logits': sem_logits, 'xyz': xyz}
        sdf, xyz = self.get_uniform_sdf(aabb, reso, device=device)
        return {'sdf': sdf, 'rep': representation, 'xyz': xyz}

    @torch.no_grad()
    def occupancy(self, aabb=None, resolution=None, thresh=0., points=None, sem_lut=None, z_keep=None, border=None):
        """Occupancy / semantic labels of the prepared frame (eval_iou.py:206-258, eval_iou_kitti.py:167-196) in one
        launch, without the get_uniform_sdf lattice of ``forward_occ``.  Returns {'occ': uint8} plus 'sem' (uint8) when
        the head was built with ``return_sem``, shaped like the [H(y), W(x), D(z)] lattice of ``get_uniform_sdf(aabb,
        resolution)`` or, when ``points`` ([n0, n1, n2, 3] normalised (x, y, z), e.g. occupancy.occ3d_points) is given,
        like ``points[..., 0]``: the lattice trilinearly resampled there as F.grid_sample(align_corners=True) does.
        occ = sdf <= thresh, zeroed outside third-axis ``z_keep = (lo, hi)`` (hi < 0 counts from the end, like a slice)
        and in the ``border = (first lo, first hi, second lo, second hi)`` rows; sem = occ * sem_lut[argmax of the
        semantic logits] (sem_lut None: the raw argmax).  Enqueues without synchronising once a list ``sem_lut`` has
        been seen (its device copy is cached)."""
        f = self.model.field
        if f.vol_sdf is None:
            raise RuntimeError('occupancy() called before prepare(): no decoded volume')
        if sem_lut is not None and not self.return_sem:
            raise ValueError('sem_lut needs a head built with return_sem=True')
        dev = f.vol_sdf.device
        aabb = self.aabb if aabb is None else aabb
        resolution = self.resolution if resolution is None else resolution
        # the node coordinates of get_uniform_sdf, computed the same way (neus_head.py:266-268)
        xs = torch.linspace(aabb[0], aabb[3], int((aabb[3] - aabb[0]) / resolution), device=dev)
        ys = torch.linspace(aabb[1], aabb[4], int((aabb[4] - aabb[1]) / resolution), device=dev)
        zs = torch.linspace(aabb[2], aabb[5], int((aabb[5] - aabb[2]) / resolution), device=dev)
        n2 = zs.numel() if points is None else points.shape[-2]
        if z_keep is not None:
            lo, hi = z_keep
            z_keep = (lo, n2 + hi if hi < 0 else hi)
        lut = None
        if sem_lut is not None:
            if torch.is_tensor(sem_lut):
                lut = sem_lut.to(device=dev, dtype=torch.uint8).contiguous()
            else:
                key = (tuple(int(v) for v in sem_lut), dev)
                if getattr(self, '_lut_cache', (None,))[0] != key:
                    self._lut_cache = (key, torch.tensor(key[0], dtype=torch.uint8, device=dev))
                lut = self._lut_cache[1]
        pts = None if points is None else points.to(device=dev, dtype=torch.float32).contiguous()
        occ, sem = ops.occ_classify(f.vol_sdf, f.vol_feat, f.desc, xs, ys, zs, points=pts, thresh=thresh, z_keep=z_keep,
                                    border=border, lut=lut, want_sem=self.return_sem)
        return {'occ': occ, 'sem': sem} if self.return_sem else {'occ': occ}

    def forward(self, representation, metas=None, **kwargs):
        """neus_head.py:473-713 (training form: per-sample weights / ts / deltas / eik_grad)."""
        if self.return_second_grad and not self.second_grad_assumption:
            raise NotImplementedError(
                "return_second_grad=True: the `second_grad` training output is computed inside the un-vendored sdfstudio fork "
                "(cuda_gridsample_grad2, `use_compact_2nd_grad`) and its definition cannot be recovered from the reference.  "
                "Construct the head with second_grad_assumption=True (or set SELFOCC_B200_SECOND_GRAD=1) to opt into the declared "
                "restatement -- row sums of the Hessian of the trilinear field, see so_field_second_grad in include/selfocc_b200.h "
                "-- or set return_second_grad=False and drop SecondGradLoss; prepare()/render()/forward_occ() are unaffected")
        from .head_train import forward_train
        return forward_train(self, representation, metas, **kwargs)
