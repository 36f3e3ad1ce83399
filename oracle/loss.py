"""Oracle: the self-supervised training losses (test infrastructure, see oracle/__init__.py).

Restates, with plain torch ops:
* ReprojLossMonoMultiNewCombine.reproj_loss (loss/reproj_loss_mono_multi_new_combine.py:108-245) and
  ReprojLossMonoMultiNew.reproj_loss with sdf_loss=False (loss/reproj_loss_mono_multi_new.py:117-288), for the training
  head's ray layout (S contiguous samples per ray, rays in order), where every ``index_add_`` over ``ray_indices`` is a
  sum over the sample axis;
* the SSIM module both files define (:7-37);
* EikonalLoss (loss/eikonal_loss.py:19-22), EdgeLoss3DMS (loss/edge_loss_3d_ms.py:7-20, :44-76) and SecondGradLoss
  (loss/second_grad_loss.py:19-20).

Device-agnostic and dtype-preserving: fp64 on the CPU it is the oracle; fp32 on CUDA it is the reference composition the
kernels are compared with and benchmarked against.  Gradients come from autograd.
"""
import torch
import torch.nn.functional as F

EPS32 = float(torch.finfo(torch.float32).eps)   # the reference takes finfo of the (float32) weight dtype


def ssim_ref(x, y):
    """SSIM module (:7-37): reflection pad 1, 3x3 mean, C1 = 0.01^2, C2 = 0.03^2, clamp((1 - n / d) / 2, 0, 1)."""
    x, y = F.pad(x, (1, 1, 1, 1), mode='reflect'), F.pad(y, (1, 1, 1, 1), mode='reflect')
    mean = lambda a: F.avg_pool2d(a, 3, 1)
    mx, my = mean(x), mean(y)
    sx, sy, sxy = mean(x * x) - mx ** 2, mean(y * y) - my ** 2, mean(x * y) - mx * my
    n = (2 * mx * my + 0.01 ** 2) * (2 * sxy + 0.03 ** 2)
    d = (mx ** 2 + my ** 2 + 0.01 ** 2) * (sx + sy + 0.03 ** 2)
    return torch.clamp((1 - n / d) / 2, 0, 1)


def sample_ref(img, u, v, img_size, border):
    """sample_pixel (:151-170 / :151-163): img [3, H, W], pixel (u, v) [...] -> [..., 3]."""
    g = torch.stack([u / img_size[1], v / img_size[0]], -1) * 2 - 1
    out = F.grid_sample(img[None], g.reshape(1, 1, -1, 2), mode='bilinear', padding_mode='border' if border else 'zeros',
                        align_corners=True)
    return out[0, :, 0].transpose(0, 1).reshape(*u.shape, 3)


def project_ref(T, pix, t, img_size):
    """cal_pixel (:133-144): T [4, 4], pix [R, 2], t [R, S] -> u, v, mask [R, S] and the distance of the sample to the
    nearest mask bound relative to its scale (for telling fp32 rounding from a real disagreement)."""
    c = torch.stack([pix[:, :1] * t, pix[:, 1:] * t, t, torch.ones_like(t)], -1)
    p = (T[None, None] * c[..., None, :]).sum(-1)
    z = p[..., 2]
    den = torch.clamp_min(z, 1e-5)
    u, v = p[..., 0] / den, p[..., 1] / den
    m = (z > 0) & (u > 0) & (u < img_size[1]) & (v > 0) & (v < img_size[0])
    zs = (T[2].abs()[None, None] * c.abs()).sum(-1).clamp_min(1e-30)
    margin = torch.stack([z.abs() / zs, u.abs() / img_size[1], (u - img_size[1]).abs() / img_size[1],
                          v.abs() / img_size[0], (v - img_size[0]).abs() / img_size[0]], -1).amin(-1)
    return u, v, m, margin


def _trans(t, n_cam, like):
    if isinstance(t, torch.Tensor):
        return t.to(like).reshape(n_cam, 4, 4)
    return torch.stack([torch.as_tensor(x).to(like) for x in t]).reshape(n_cam, 4, 4)


def reproj_loss_ref(combine, curr, prev, nxt, pix, img2prev, img2next, weights, ts, deltas=None, img_size=(768, 1600),
                    ray_resize=None, no_ssim=False, no_automask=False, diag=None):
    """Reprojection loss of one frame.  combine: True = ReprojLossMonoMultiNewCombine, False = ReprojLossMonoMultiNew.
    curr / prev / nxt [1, N, 3, H, W]; pix [R, 2]; img2prev / img2next [N, 4, 4] (or lists); weights, ts, deltas: per camera
    [R * S] (lists or [N, R * S]).  Returns the loss (before the loss weight).  diag: optional dict filled with per-camera
    lists 'count' [R, k] (valid samples per ray and branch), 'margin' [R, S] (min over both projections), 'cand' [R, k]
    (the min's candidates) and 'choice' [R]."""
    no_ssim = no_ssim or ray_resize is None
    N, R = curr.shape[1], pix.shape[0]
    like = weights[0]
    Tp, Tn = _trans(img2prev, N, like), _trans(img2next, N, like)
    tot = 0.
    for cam in range(N):
        w = weights[cam].reshape(R, -1)
        t = ts[cam].reshape(R, -1).detach()
        if deltas is not None:                                              # :120-125
            d = deltas[cam].reshape(R, -1).detach()
            w = torch.where(d < EPS32, torch.zeros_like(w), w / d.clamp_min(EPS32))
        up, vp, mp, mgp = project_ref(Tp[cam], pix, t, img_size)
        un, vn, mn, mgn = project_ref(Tn[cam], pix, t, img_size)
        rp = sample_ref(prev[0, cam], up, vp, img_size, combine)            # [R, S, 3]
        rn = sample_ref(nxt[0, cam], un, vn, img_size, combine)
        tc = sample_ref(curr[0, cam], pix[:, 0], pix[:, 1], img_size, combine)     # [R, 3]
        grid = lambda a: a.transpose(0, 1).reshape(1, 3, *ray_resize)
        ssim = lambda a, b: ssim_ref(grid(a), grid(b)).mean(1).flatten()

        def plain(target):                                                   # automask terms, weight-free
            l1 = (tc - target).abs().mean(-1)
            return l1 if no_ssim else 0.85 * ssim(target, tc) + 0.15 * l1

        if combine:                                                          # :172-213
            rp, rn = rp * mp[..., None], rn * mn[..., None]
            dp = (tc[:, None] - rp).abs().mean(-1) * mp
            dn = (tc[:, None] - rn).abs().mean(-1) * mn
            cnt = mp.to(w) + mn.to(w)
            g = cnt > 0
            cnt = cnt.clamp_min(1.0)
            w = torch.where(g, w, torch.zeros_like(w))
            wn = w / w.sum(1, keepdim=True).clamp_min(EPS32)
            pn = (wn * (dp + dn) / cnt).sum(1)
            if not no_ssim:
                x = (wn[..., None] * (rp + rn) / cnt[..., None]).sum(1)
                pn = 0.15 * pn + 0.85 * ssim(x, tc)
            cands, counts = [pn], [g.sum(1)]
            if not no_automask:                                              # :228-246
                cands[0] = torch.where(g.any(1), pn, torch.full_like(pn, 1e3))
        else:                                                                # :165-246
            cands, counts = [], []
            for r_b, m_b in ((rp, mp), (rn, mn)):
                wb = torch.where(m_b, w, torch.zeros_like(w))
                wb = wb / wb.sum(1, keepdim=True).clamp_min(EPS32)
                l1 = (wb * (tc[:, None] - r_b).abs().mean(-1)).sum(1)
                if not no_ssim:
                    l1 = 0.85 * ssim((wb[..., None] * r_b).sum(1), tc) + 0.15 * l1
                cands.append(torch.where(m_b.any(1), l1, torch.full_like(l1, 1e3)))
                counts.append(m_b.sum(1))
        if not no_automask:
            for img in (prev, nxt):
                cands.append(plain(sample_ref(img[0, cam], pix[:, 0], pix[:, 1], img_size, combine)))
        cand = torch.stack(cands, -1)
        proj, choice = cand.min(-1)
        tot = tot + proj.mean()
        if diag is not None:
            for k, v in (('count', torch.stack(counts, -1)), ('margin', torch.minimum(mgp, mgn)), ('cand', cand.detach()),
                         ('choice', choice)):
                diag.setdefault(k, []).append(v)
    return tot / N


def eikonal_ref(eik_grad):
    """EikonalLoss (eikonal_loss.py:19-22)."""
    return ((eik_grad.norm(2, dim=-1) - 1) ** 2).mean()


def second_grad_ref(second_grad):
    """SecondGradLoss (second_grad_loss.py:19-20)."""
    return second_grad.abs().mean()


def edge_ref(curr_imgs, ms_depths, ms_rays, img_size, ray_resize):
    """EdgeLoss3DMS without use_inf_mask (edge_loss_3d_ms.py:7-20, :44-76): edge-aware smoothness of the mean-normalised
    depth on the ray grid, weighted by the border-padded image colour at the ray pixels."""
    if not isinstance(ms_rays, (list, tuple)):
        ms_rays = [ms_rays] * len(ms_depths)
    tot = 0.
    for depth, rays in zip(ms_depths, ms_rays):
        bs, n, r = depth.shape
        g = rays.reshape(1, 1, r, 2).repeat(bs * n, 1, 1, 1) / rays.new_tensor([img_size[1], img_size[0]]) * 2 - 1
        rgb = F.grid_sample(curr_imgs.flatten(0, 1), g, mode='bilinear', padding_mode='border', align_corners=True)
        rgb = rgb.reshape(bs * n, -1, *ray_resize)
        d = depth.reshape(bs * n, 1, *ray_resize)
        d = d / (d.mean(2, True).mean(3, True) + 1e-6)
        gdx, gdy = (d[..., :-1] - d[..., 1:]).abs(), (d[..., :-1, :] - d[..., 1:, :]).abs()
        gix = (rgb[..., :-1] - rgb[..., 1:]).abs().mean(1, True)
        giy = (rgb[..., :-1, :] - rgb[..., 1:, :]).abs().mean(1, True)
        tot = tot + (gdx * torch.exp(-gix)).mean() + (gdy * torch.exp(-giy)).mean()
    return tot / len(ms_depths)
