"""Torch-tensor front end of the C ABI: pointer/stream plumbing only, no arithmetic.

Every function validates device/dtype/contiguity, passes raw device pointers plus the current CUDA
stream to ``libselfocc_b200.so`` and returns the output tensors.  There is no CPU path: a non-CUDA
tensor raises ``RuntimeError``.
"""
import ctypes as C
import torch
from . import _lib


def _chk(t, dtype=torch.float32, name='tensor'):
    if t is None:
        return None
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError('%s must be a CUDA tensor: selfocc_b200 has no CPU fallback' % name)
    if t.dtype != dtype:
        raise TypeError('%s must be %s, got %s' % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError('%s must be contiguous' % name)
    return t


def _p(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# --------------------------------------------------------------------------------------- B5
def tpv_decode(tpv_hw, tpv_zh, tpv_wz, w1, b1, w2, b2, desc, rows=None, out=None):
    """planes [H*W,C], [Z*H,C], [W*Z,C] + MLP -> (vol_sdf [H,W,zpitch], vol_feat [H,W,Z,feat_pitch] | None).
    rows=(h_begin, h_count): decode that slab of h rows only (voxel-sharded decode); out=(vol_sdf, vol_feat): write into
    existing full-size buffers (rows outside the slab are left untouched)."""
    lib = _lib.load()
    for n, t in (('tpv_hw', tpv_hw), ('tpv_zh', tpv_zh), ('tpv_wz', tpv_wz), ('w1', w1), ('b1', b1), ('w2', w2), ('b2', b2)):
        _chk(t, name=n)
    Cc = tpv_hw.shape[-1]
    assert tpv_hw.numel() == desc.H * desc.W * Cc and tpv_zh.numel() == desc.Z * desc.H * Cc \
        and tpv_wz.numel() == desc.W * desc.Z * Cc, 'plane shapes do not match the mapping'
    assert w1.shape == (Cc, Cc) and w2.shape == (1 + desc.n_feat, Cc)
    dev = tpv_hw.device
    if out is not None:
        vol_sdf, vol_feat = out
        _chk(vol_sdf, name='vol_sdf'); _chk(vol_feat, name='vol_feat')
        assert vol_sdf.shape == (desc.H, desc.W, desc.zpitch)
    else:
        vol_sdf = torch.empty(desc.H, desc.W, desc.zpitch, device=dev, dtype=torch.float32)
        vol_feat = torch.empty(desc.H, desc.W, desc.Z, desc.feat_pitch, device=dev, dtype=torch.float32) if desc.n_feat else None
    h0, hc = (0, desc.H) if rows is None else rows
    if vol_feat is not None and desc.feat_pitch > desc.n_feat:
        vol_feat[h0:h0 + hc].zero_()
    _lib.check(lib.so_tpv_decode_rows(_p(tpv_hw), _p(tpv_zh), _p(tpv_wz), Cc, _p(w1), _p(b1), _p(w2), _p(b2), C.byref(desc),
                                      int(h0), int(hc), _p(vol_sdf), _p(vol_feat), _stream()), 'so_tpv_decode_rows')
    return vol_sdf, vol_feat


# --------------------------------------------------------------------------------------- B1-B11
def make_ray_desc(n_cam, grid=None, n_pix=None, ray_begin=0, ray_count=None, chunk_len=0):
    """grid = (ny, nx, sx, ox, sy, oy) for the in-kernel strided pixel grid, or n_pix with a pixel table."""
    r = _lib.RayDesc()
    r.n_cam = n_cam
    if grid is not None:
        ny, nx, sx, ox, sy, oy = grid
        r.nx, r.ny, r.sx, r.ox, r.sy, r.oy = int(nx), int(ny), float(sx), float(ox), float(sy), float(oy)
        r.rays_per_cam = int(nx) * int(ny)
    else:
        r.rays_per_cam = int(n_pix)
    total = r.n_cam * r.rays_per_cam
    r.ray_begin = int(ray_begin)
    r.ray_count = int(total - ray_begin if ray_count is None else ray_count)
    r.chunk_len = int(chunk_len)
    return r


def make_render_params(aabb, num_samples, inv_s, near_plane=0.0, training=False, cos_anneal=1.0, anchor_mid=True,
                       sh_act='relu', bkgd='white'):
    p = _lib.RenderParams()
    for i in range(6):
        p.aabb[i] = float(aabb[i])
    p.near_plane = float(near_plane)
    p.training = int(bool(training))
    p.num_samples = int(num_samples)
    p.inv_s = float(inv_s)
    p.cos_anneal = float(cos_anneal)
    p.anchor_mid = int(bool(anchor_mid))
    p.sh_act = {'relu': 0, 'sigmoid': 1}[sh_act]
    p.bkgd_mode = {'black': 0, 'white': 1, 'random': 2}[bkgd]
    return p


def render_pack(vol_sdf, vol_feat, desc):
    """Once-per-frame repack of the decoded volume for the packed render kernels (so_render_pack): float2 z-pairs when no
    colour is decoded, float4 (r, g, b, sdf) for color_dims == 3.  Returns None when this channel count has no packed form."""
    lib = _lib.load()
    _chk(vol_sdf, name='vol_sdf'); _chk(vol_feat, name='vol_feat')
    n = lib.so_render_pack_floats(C.byref(desc))
    if n <= 0:
        return None
    pack = torch.empty(n, device=vol_sdf.device, dtype=torch.float32)
    _lib.check(lib.so_render_pack(_p(vol_sdf), _p(vol_feat), C.byref(desc), _p(pack), _stream()), 'so_render_pack')
    return pack


def render_infer(vol_sdf, vol_feat, desc, cam_mats, rays, params, pix=None, bkgd_rand=None, want=('depth',),
                 out=None, pack=None, probe_grid=False):
    """Fused inference render.  ``want`` subset of depth,max_depth,max_idx,acc,normal_vis,rgb,sem.
    Returns a dict of flat per-ray tensors for rays [ray_begin, ray_begin+ray_count).
    ``pack`` = render_pack(...) selects the packed-volume kernels; ``probe_grid`` (tests) adds 'grid' [n, S, 3], the fp32
    grid coordinates of every sample as the packed kernel computed them."""
    lib = _lib.load()
    _chk(pack, name='pack')
    _chk(vol_sdf, name='vol_sdf'); _chk(vol_feat, name='vol_feat'); _chk(cam_mats, name='cam_mats')
    _chk(pix, name='pix'); _chk(bkgd_rand, name='bkgd_rand')
    assert cam_mats.shape == (rays.n_cam, 4, 4)
    n = rays.ray_count
    dev = vol_sdf.device
    total = rays.n_cam * rays.rays_per_cam
    n_chunks = (total + rays.chunk_len - 1) // rays.chunk_len if rays.chunk_len > 0 else 1
    ws = torch.empty(lib.so_render_workspace_floats(n_chunks), device=dev, dtype=torch.float32)
    shapes = dict(depth=((n,), torch.float32), max_depth=((n,), torch.float32), max_idx=((n,), torch.int64),
                  acc=((n,), torch.float32), normal_vis=((n, 3), torch.float32), rgb=((n, 3), torch.float32),
                  sem=((n, max(desc.n_feat - 3, 0)), torch.float32))
    res = {}
    for k in want:
        if out is not None and k in out:
            res[k] = _chk(out[k], shapes[k][1], k)
        else:
            res[k] = torch.empty(shapes[k][0], device=dev, dtype=shapes[k][1])
    g = lambda k: _p(res.get(k))
    if pack is None and not probe_grid:
        _lib.check(lib.so_render_infer(_p(vol_sdf), _p(vol_feat), C.byref(desc), _p(cam_mats), _p(pix), C.byref(rays),
                                       C.byref(params), _p(bkgd_rand), g('depth'), g('max_depth'), g('max_idx'), g('acc'),
                                       g('normal_vis'), g('rgb'), g('sem'), _p(ws), _stream()), 'so_render_infer')
        return res
    if probe_grid:
        res['grid'] = torch.empty(n, params.num_samples, 3, device=dev, dtype=torch.float32)
    _lib.check(lib.so_render_infer_packed(_p(vol_sdf), _p(vol_feat), C.byref(desc), _p(pack), _p(cam_mats), _p(pix), C.byref(rays),
                                          C.byref(params), _p(bkgd_rand), g('depth'), g('max_depth'), g('max_idx'), g('acc'),
                                          g('normal_vis'), g('rgb'), g('sem'), _p(ws), g('grid'), _stream()),
               'so_render_infer_packed')
    return res


def field_query(vol_sdf, vol_feat, desc, points, want_grad=False, want_feat=False):
    lib = _lib.load()
    _chk(vol_sdf, name='vol_sdf'); _chk(vol_feat, name='vol_feat'); _chk(points, name='points')
    n = points.shape[0]
    dev = points.device
    sdf = torch.empty(n, device=dev)
    grad = torch.empty(n, 3, device=dev) if want_grad else None
    feat = torch.empty(n, desc.n_feat, device=dev) if want_feat else None
    _lib.check(lib.so_field_query(_p(vol_sdf), _p(vol_feat), C.byref(desc), _p(points), n, _p(sdf), _p(grad), _p(feat),
                                  _stream()), 'so_field_query')
    return sdf, grad, feat


# --------------------------------------------------------------------------------------- occupancy evaluation
def occ_classify(vol_sdf, vol_feat, desc, xs, ys, zs, points=None, thresh=0., z_keep=None, border=None, lut=None, want_sem=False):
    """Decoded volume -> (occ u8, sem u8 | None) shaped like the [len(ys), len(xs), len(zs)] lattice (points None) or like
    points[..., 0] (points [n0, n1, n2, 3] normalised (x, y, z), trilinear resample of the lattice).  z_keep = (lo, hi)
    kept third-axis range (default all), border = (first lo, first hi, second lo, second hi) zeroed rows (default 0);
    lut: uint8 table applied to the semantic argmax (None = raw argmax)."""
    lib = _lib.load()
    _chk(vol_sdf, name='vol_sdf'); _chk(vol_feat, name='vol_feat')
    _chk(xs, name='xs'); _chk(ys, name='ys'); _chk(zs, name='zs'); _chk(points, name='points'); _chk(lut, torch.uint8, 'lut')
    shape = (ys.numel(), xs.numel(), zs.numel()) if points is None else tuple(points.shape[:-1])
    if len(shape) != 3 or (points is not None and points.shape[-1] != 3):
        raise ValueError('points must be [n0, n1, n2, 3], got %s' % (tuple(points.shape),))
    g = _lib.OccGrid()
    g.n0, g.n1, g.n2 = shape
    g.z_lo, g.z_hi = (0, shape[2]) if z_keep is None else (int(z_keep[0]), int(z_keep[1]))
    for i, b in enumerate((0, 0, 0, 0) if border is None else border):
        g.border[i] = int(b)
    g.thresh = float(thresh)
    occ = torch.empty(shape, device=vol_sdf.device, dtype=torch.uint8)
    sem = torch.empty(shape, device=vol_sdf.device, dtype=torch.uint8) if want_sem else None
    _lib.check(lib.so_occ_classify(_p(vol_sdf), _p(vol_feat), C.byref(desc), _p(xs), _p(ys), _p(zs), xs.numel(), ys.numel(),
                                   zs.numel(), _p(points), C.byref(g), _p(lut), 0 if lut is None else lut.numel(), _p(occ), _p(sem),
                                   _stream()), 'so_occ_classify')
    return occ, sem


def occ_hist(pred, gt, hist, mask=None):
    """hist int64 [256, P] += joint (gt, min(pred, P - 1)) counts over the voxels where mask != 0; pred, gt, mask uint8."""
    lib = _lib.load()
    _chk(pred, torch.uint8, 'pred'); _chk(gt, torch.uint8, 'gt'); _chk(mask, torch.uint8, 'mask'); _chk(hist, torch.int64, 'hist')
    n = pred.numel()
    if gt.numel() != n or (mask is not None and mask.numel() != n) or hist.dim() != 2 or hist.shape[0] != 256:
        raise ValueError('occ_hist: pred %s, gt %s, mask %s, hist %s' % (tuple(pred.shape), tuple(gt.shape),
                                                                        None if mask is None else tuple(mask.shape), tuple(hist.shape)))
    _lib.check(lib.so_occ_hist(_p(pred), _p(gt), _p(mask), n, hist.shape[1], _p(hist), _stream()), 'so_occ_hist')
    return hist


# --------------------------------------------------------------------------------------- A4-A8
def msda_forward(value, spatial_shapes, level_start_index, loc, weights):
    lib = _lib.load()
    _chk(value, name='value'); _chk(loc, name='sampling_locations'); _chk(weights, name='attention_weights')
    _chk(spatial_shapes, torch.int64, 'spatial_shapes'); _chk(level_start_index, torch.int64, 'level_start_index')
    B, Nv, Hd, Dh = value.shape
    _, Nq, _, L, P, _ = loc.shape
    out = torch.empty(B, Nq, Hd * Dh, device=value.device, dtype=torch.float32)
    _lib.check(lib.so_msda_forward(_p(value), _p(spatial_shapes), _p(level_start_index), _p(loc), _p(weights), _p(out),
                                   B, Nv, Hd, Dh, Nq, L, P, _stream()), 'so_msda_forward')
    return out


def msda_backward(value, spatial_shapes, level_start_index, loc, weights, grad_out):
    lib = _lib.load()
    _chk(grad_out, name='grad_out')
    B, Nv, Hd, Dh = value.shape
    _, Nq, _, L, P, _ = loc.shape
    gv = torch.zeros_like(value)
    gl = torch.empty_like(loc)
    gw = torch.empty_like(weights)
    _lib.check(lib.so_msda_backward(_p(value), _p(spatial_shapes), _p(level_start_index), _p(loc), _p(weights),
                                    _p(grad_out), _p(gv), _p(gl), _p(gw), B, Nv, Hd, Dh, Nq, L, P, _stream()),
               'so_msda_backward')
    return gv, gl, gw


class MultiScaleDeformableAttnFunction(torch.autograd.Function):
    """Same call contract as mmcv.ops.multi_scale_deform_attn.MultiScaleDeformableAttnFunction
    (reference call sites image_cross_attention.py:340-342, cross_view_hybrid_attention.py:111-113)."""

    @staticmethod
    def forward(ctx, value, value_spatial_shapes, value_level_start_index, sampling_locations, attention_weights,
                im2col_step=64):
        value, sampling_locations, attention_weights = (t.contiguous() for t in (value, sampling_locations, attention_weights))
        ctx.save_for_backward(value, value_spatial_shapes, value_level_start_index, sampling_locations, attention_weights)
        return msda_forward(value, value_spatial_shapes, value_level_start_index, sampling_locations, attention_weights)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_output):
        value, shapes, lsi, loc, w = ctx.saved_tensors
        gv, gl, gw = msda_backward(value, shapes, lsi, loc, w, grad_output.contiguous())
        return gv, None, None, gl, gw, None


def point_sampling(ref_3d, lidar2img, img_shape):
    """ref_3d [D,Q,3], lidar2img [N,4,4] -> uv [N,Q,D,2], mask uint8 [N,Q,D], vis uint8 [N,Q]."""
    lib = _lib.load()
    _chk(ref_3d, name='ref_3d'); _chk(lidar2img, name='lidar2img')
    D, Q, _ = ref_3d.shape
    N = lidar2img.shape[0]
    dev = ref_3d.device
    uv = torch.empty(N, Q, D, 2, device=dev)
    mask = torch.empty(N, Q, D, device=dev, dtype=torch.uint8)
    vis = torch.empty(N, Q, device=dev, dtype=torch.uint8)
    _lib.check(lib.so_point_sampling(_p(ref_3d), _p(lidar2img), D, Q, N, float(img_shape[0]), float(img_shape[1]),
                                     _p(uv), _p(mask), _p(vis), _stream()), 'so_point_sampling')
    return uv, mask, vis


def visible_index_lists(mask):
    """mask uint8 [N,Q,D] -> (lists int64 [N,Q], lens int32 [N]) -- device-side ``nonzero``."""
    lib = _lib.load()
    _chk(mask, torch.uint8, 'mask')
    N, Q, D = mask.shape
    lists = torch.empty(N, Q, device=mask.device, dtype=torch.int64)
    lens = torch.empty(N, device=mask.device, dtype=torch.int32)
    _lib.check(lib.so_visible_index_lists(_p(mask), N, Q, D, _p(lists), _p(lens), _stream()), 'so_visible_index_lists')
    return lists, lens


def tpv_cross_attn_forward(value, spatial_shapes, level_start_index, offsets, logits, uv, vis, want_count=False):
    """value [N,Nv,Hd,Dh], offsets [Q,Hd,L,D,2], logits [Q,Hd,L,D], uv [N,Q,D,2], vis [N,Q] -> slots [Q,Hd*Dh]."""
    lib = _lib.load()
    for n, t in (('value', value), ('offsets', offsets), ('logits', logits), ('uv', uv)):
        _chk(t, name=n)
    _chk(vis, torch.uint8, 'vis')
    _chk(spatial_shapes, torch.int64, 'spatial_shapes'); _chk(level_start_index, torch.int64, 'level_start_index')
    N, Nv, Hd, Dh = value.shape
    Q, _, L, D, _ = offsets.shape
    slots = torch.empty(Q, Hd * Dh, device=value.device)
    count = torch.empty(Q, device=value.device, dtype=torch.int32) if want_count else None
    _lib.check(lib.so_tpv_cross_attn_forward(_p(value), _p(spatial_shapes), _p(level_start_index), _p(offsets), _p(logits),
                                             _p(uv), _p(vis), _p(slots), _p(count), N, Nv, Hd, Dh, Q, L, D, _stream()),
               'so_tpv_cross_attn_forward')
    return (slots, count) if want_count else slots


def tpv_self_attn_forward(value, spatial_shapes, level_start_index, offsets, logits, ref):
    """value [Nv,Hd,Dh], offsets [Q,Hd,L,P,2], logits [Q,Hd,L,P], ref [Q,L,P,2] -> out [Q,Hd*Dh]."""
    lib = _lib.load()
    for n, t in (('value', value), ('offsets', offsets), ('logits', logits), ('ref', ref)):
        _chk(t, name=n)
    _chk(spatial_shapes, torch.int64, 'spatial_shapes'); _chk(level_start_index, torch.int64, 'level_start_index')
    Nv, Hd, Dh = value.shape
    Q, _, L, P, _ = offsets.shape
    out = torch.empty(Q, Hd * Dh, device=value.device)
    _lib.check(lib.so_tpv_self_attn_forward(_p(value), _p(spatial_shapes), _p(level_start_index), _p(offsets), _p(logits),
                                            _p(ref), _p(out), Nv, Hd, Dh, Q, L, P, _stream()), 'so_tpv_self_attn_forward')
    return out


# --------------------------------------------------------------------------------------- training form (B6-B10, B13)
def _render_ws(lib, rays, dev):
    total = rays.n_cam * rays.rays_per_cam
    n_chunks = (total + rays.chunk_len - 1) // rays.chunk_len if rays.chunk_len > 0 else 1
    return torch.empty(lib.so_render_workspace_floats(n_chunks), device=dev, dtype=torch.float32)


class RenderTrainFunction(torch.autograd.Function):
    """Differentiable (w.r.t. the decoded volume and inv_s) training-form render.
    forward(vol_sdf, vol_feat_or_None, inv_s[1], cfg) -> (depth, acc, fars, max_depth, rgb, sem, weights, ts, deltas,
    eik_grad, sample_sdf); entries not requested in cfg['want'] are returned as empty tensors."""

    ORDER = ('depth', 'acc', 'fars', 'max_depth', 'rgb', 'sem', 'weights', 'ts', 'deltas', 'eik_grad', 'sample_sdf')

    @staticmethod
    def forward(ctx, vol_sdf, vol_feat, inv_s, cfg):
        lib = _lib.load()
        desc, cam_mats, rays, params = cfg['desc'], cfg['cam_mats'], cfg['rays'], cfg['params']
        pix, jitter, bkgd = cfg.get('pix'), cfg.get('jitter'), cfg.get('bkgd_rand')
        _chk(vol_sdf, name='vol_sdf'); _chk(vol_feat, name='vol_feat'); _chk(cam_mats, name='cam_mats')
        _chk(pix, name='pix'); _chk(jitter, name='jitter'); _chk(bkgd, name='bkgd_rand')
        n, S, dev = rays.ray_count, params.num_samples, vol_sdf.device
        if jitter is not None:
            assert jitter.shape == (rays.n_cam * rays.rays_per_cam, S + 1)
        n_sem = max(desc.n_feat - 3, 0)
        shapes = dict(depth=(n,), acc=(n,), fars=(n,), max_depth=(n,), rgb=(n, 3), sem=(n, n_sem), weights=(n, S), ts=(n, S),
                      deltas=(n, S), eik_grad=(n, S, 3), sample_sdf=(n, S))
        want = set(cfg['want'])
        out = {k: (torch.empty(shapes[k], device=dev) if k in want else None) for k in RenderTrainFunction.ORDER}
        ws = _render_ws(lib, rays, dev)
        # scratch for the z-pair copy of the sdf volume (cfg['zpair']=False: gather from the volume itself)
        pair = torch.empty(lib.so_render_train_pair_floats(C.byref(desc)), device=dev) if cfg.get('zpair', True) else None
        g = lambda k: _p(out[k])
        _lib.check(lib.so_render_train_forward(
            _p(vol_sdf), _p(vol_feat), C.byref(desc), _p(cam_mats), _p(pix), C.byref(rays), C.byref(params), _p(jitter), _p(bkgd),
            g('depth'), g('acc'), g('fars'), g('rgb'), g('sem'), g('max_depth'), g('weights'), g('ts'), g('deltas'),
            g('eik_grad'), g('sample_sdf'), _p(ws), _p(pair), _stream()), 'so_render_train_forward')
        ctx.cfg = cfg
        ctx.save_for_backward(vol_sdf, vol_feat if vol_feat is not None else vol_sdf.new_empty(0))
        ctx.has_feat = vol_feat is not None
        res = tuple(out[k] if out[k] is not None else vol_sdf.new_empty(0) for k in RenderTrainFunction.ORDER)
        ctx.mark_non_differentiable(res[2], res[3], res[7], res[8])       # fars, max_depth, ts, deltas: geometry only
        return res

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_depth, g_acc, g_fars, g_maxd, g_rgb, g_sem, g_weights, g_ts, g_deltas, g_eik, g_sdf):
        lib = _lib.load()
        cfg = ctx.cfg
        vol_sdf, vol_feat = ctx.saved_tensors
        vol_feat = vol_feat if ctx.has_feat else None
        desc, rays, params = cfg['desc'], cfg['rays'], cfg['params']
        want = set(cfg['want'])

        def gr(name, t):
            return t.contiguous() if (name in want and t is not None and t.numel()) else None
        gd, ga, grgb, gsem = gr('depth', g_depth), gr('acc', g_acc), gr('rgb', g_rgb), gr('sem', g_sem)
        gw, ge, gs = gr('weights', g_weights), gr('eik_grad', g_eik), gr('sample_sdf', g_sdf)
        gvs = torch.zeros_like(vol_sdf)
        gvf = torch.zeros_like(vol_feat) if vol_feat is not None else None
        ginv = torch.zeros(1, device=vol_sdf.device)
        ws = _render_ws(lib, rays, vol_sdf.device)
        _lib.check(lib.so_render_train_backward(
            _p(vol_sdf), _p(vol_feat), C.byref(desc), _p(cfg['cam_mats']), _p(cfg.get('pix')), C.byref(rays), C.byref(params),
            _p(cfg.get('jitter')), _p(cfg.get('bkgd_rand')), _p(gd), _p(ga), _p(grgb), _p(gsem), _p(gw), _p(ge), _p(gs),
            _p(gvs), _p(gvf), _p(ginv), _p(ws), _stream()), 'so_render_train_backward')
        return gvs, gvf, ginv, None


class FieldQueryFunction(torch.autograd.Function):
    """Differentiable (w.r.t. the volume) point query: (vol_sdf, vol_feat, desc, points[n,3]) -> (sdf[n], grad[n,3], feat[n,nf])."""

    @staticmethod
    def forward(ctx, vol_sdf, vol_feat, desc, points, want_grad, want_feat):
        s, g, f = field_query(vol_sdf, vol_feat, desc, points, want_grad=want_grad, want_feat=want_feat)
        ctx.desc, ctx.has_feat = desc, vol_feat is not None
        ctx.save_for_backward(points, vol_sdf, vol_feat if vol_feat is not None else vol_sdf.new_empty(0))
        e = vol_sdf.new_empty(0)
        return s, (g if g is not None else e), (f if f is not None else e)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_s, g_g, g_f):
        lib = _lib.load()
        points, vol_sdf, vol_feat = ctx.saved_tensors
        gvs = torch.zeros_like(vol_sdf)
        gvf = torch.zeros_like(vol_feat) if ctx.has_feat else None
        opt = lambda t: t.contiguous() if (t is not None and t.numel()) else None
        gf = opt(g_f) if ctx.has_feat else None
        _lib.check(lib.so_field_query_backward(C.byref(ctx.desc), _p(points), points.shape[0], _p(opt(g_s)), _p(opt(g_g)),
                                               _p(gf), _p(gvs), _p(gvf), _stream()), 'so_field_query_backward')
        return gvs, gvf, None, None, None, None


class FieldSecondGradFunction(torch.autograd.Function):
    """`second_grad` at sample points (declared assumption, see so_field_second_grad): (vol_sdf, desc, points[n,3]) -> [n,3],
    differentiable w.r.t. the volume (it is linear in it)."""

    @staticmethod
    def forward(ctx, vol_sdf, desc, points):
        lib = _lib.load()
        _chk(vol_sdf, name='vol_sdf'); _chk(points, name='points')
        out = torch.empty(points.shape[0], 3, device=points.device)
        _lib.check(lib.so_field_second_grad(_p(vol_sdf), C.byref(desc), _p(points), points.shape[0], _p(out), _stream()),
                   'so_field_second_grad')
        ctx.desc = desc
        ctx.save_for_backward(points, vol_sdf)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        lib = _lib.load()
        points, vol_sdf = ctx.saved_tensors
        gvs = torch.zeros_like(vol_sdf)
        _lib.check(lib.so_field_second_grad_backward(C.byref(ctx.desc), _p(points), points.shape[0], _p(g.contiguous()), _p(gvs),
                                                     _stream()), 'so_field_second_grad_backward')
        return gvs, None, None


class TPVDecodeFunction(torch.autograd.Function):
    """Decode with the fused sm_100a forward.  Backward (training only) recomputes the MLP slab by slab -- bounded memory,
    never the reference's 750 MB intermediate.  Default: the native slab backward (_backward_native: tcgen05 3xTF32 GEMMs
    + the fused element-wise kernels so_tpv_decode_bwd_*); SELFOCC_B200_DECODE_BWD=torch or an unsupported channel count
    takes the torch/cuBLAS autograd restatement of the same slab (_backward_torch), which is also what the tests compare
    the native path with."""

    SLAB_ROWS = 32

    @staticmethod
    def forward(ctx, hw, zh, wz, w1, b1, w2, b2, desc):
        ctx.desc = desc
        ctx.save_for_backward(hw, zh, wz, w1, b1, w2, b2)
        vs, vf = tpv_decode(hw.contiguous(), zh.contiguous(), wz.contiguous(), w1.contiguous(), b1.contiguous(),
                            w2.contiguous(), b2.contiguous(), desc)
        return vs, (vf if vf is not None else vs.new_empty(0))

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_vs, g_vf):
        import os
        saved, d = ctx.saved_tensors, ctx.desc
        Cc = saved[0].shape[-1]
        native = os.environ.get('SELFOCC_B200_DECODE_BWD', 'native') != 'torch' and linear_supported(Cc, Cc) \
            and tuple(saved[3].shape) == (Cc, Cc) and 1 + d.n_feat <= 32
        fn = TPVDecodeFunction._backward_native if native else TPVDecodeFunction._backward_torch
        return (*fn(saved, d, g_vs, g_vf), None)

    @staticmethod
    def _backward_native(saved, d, g_vs, g_vf):
        lib = _lib.load()
        hw, zh, wz, w1, b1, w2, b2 = [t.contiguous() for t in saved]
        H, W, Z, Cc, n_out = d.H, d.W, d.Z, hw.shape[-1], 1 + d.n_feat
        dev = hw.device
        g_vs = g_vs.contiguous() if g_vs is not None else None
        g_vf = g_vf.contiguous() if (g_vf is not None and d.n_feat) else None
        w1_hi, w1_lo = split_tf32(w1)
        w1t_hi, w1t_lo = split_tf32(w1.t().contiguous())
        g_hw, g_zh, g_wz = torch.empty_like(hw), torch.empty_like(zh), torch.zeros_like(wz)
        g_w1, g_b1, g_w2, g_b2 = (torch.zeros_like(t) for t in (w1, b1, w2, b2))
        step = min(H, TPVDecodeFunction.SLAB_ROWS)
        rows_max = step * W * Z
        a0b, z1b, g1b = (torch.empty(rows_max, Cc, device=dev) for _ in range(3))
        gob = torch.empty(rows_max, n_out, device=dev)
        st = _stream()
        for h0 in range(0, H, step):
            nh = min(H, h0 + step) - h0
            rows = nh * W * Z
            a0, z1, g1, go = a0b[:rows], z1b[:rows], g1b[:rows], gob[:rows]
            _lib.check(lib.so_tpv_decode_bwd_features(_p(hw), _p(zh), _p(wz), Cc, C.byref(d), h0, nh, _p(a0), st),
                       'so_tpv_decode_bwd_features')
            linear_3xtf32(a0, w1_hi, w1_lo, b1, out=z1)
            _lib.check(lib.so_tpv_decode_bwd_hidden(_p(z1), _p(g_vs), _p(g_vf), _p(w2), Cc, C.byref(d), h0, nh, _p(g1), _p(go), st),
                       'so_tpv_decode_bwd_hidden')
            # weight gradients: reductions over the slab's rows (cuBLAS; z1 now holds a1)
            g_w2.addmm_(go.t(), z1)
            g_b2.add_(go.sum(0))
            g_w1.addmm_(g1.t(), a0)
            g_b1.add_(g1.sum(0))
            g0 = linear_3xtf32(g1, w1t_hi, w1t_lo, None, out=z1)          # a1 no longer needed
            _lib.check(lib.so_tpv_decode_bwd_input(_p(g0), _p(a0), g0.numel(), st), 'so_tpv_decode_bwd_input')
            g4 = g0.view(nh, W, Z, Cc)
            g_hw.view(H, W, Cc)[h0:h0 + nh] = g4.sum(2)
            g_zh.view(Z, H, Cc)[:, h0:h0 + nh] = g4.sum(1).permute(1, 0, 2)
            g_wz.view(W, Z, Cc).add_(g4.sum(0))
        return g_hw, g_zh, g_wz, g_w1, g_b1, g_w2, g_b2

    @staticmethod
    def _backward_torch(saved, d, g_vs, g_vf):
        import torch.nn.functional as F
        hw, zh, wz, w1, b1, w2, b2 = saved
        H, W, Z, Cc = d.H, d.W, d.Z, hw.shape[-1]
        g_out = g_vs[..., :Z, None]
        if d.n_feat:
            g_out = torch.cat([g_out, g_vf[..., :d.n_feat]], -1)
        grads = [torch.zeros_like(t) for t in (hw, zh, wz, w1, b1, w2, b2)]
        zh3, wz3 = zh.view(Z, H, Cc), wz.view(W, Z, Cc)
        step = 8
        for h0 in range(0, H, step):
            h1 = min(H, h0 + step)
            with torch.enable_grad():
                a = hw.view(H, W, Cc)[h0:h1].detach().requires_grad_(True)
                b = zh3[:, h0:h1].detach().requires_grad_(True)
                c = wz3.detach().requires_grad_(True)
                ws = [t.detach().requires_grad_(True) for t in (w1, b1, w2, b2)]
                f = a[:, :, None, :] + b.permute(1, 0, 2)[:, None, :, :] + c[None]
                out = F.linear(F.softplus(F.linear(F.softplus(f), ws[0], ws[1])), ws[2], ws[3])
                gs = torch.autograd.grad(out, [a, b, c] + ws, g_out[h0:h1])
            grads[0].view(H, W, Cc)[h0:h1] += gs[0]
            grads[1].view(Z, H, Cc)[:, h0:h1] += gs[1]
            grads[2].view(W, Z, Cc).add_(gs[2])
            for i in range(4):
                grads[3 + i] += gs[3 + i]
        return tuple(grads)


# --------------------------------------------------------------------------------------- A6/A9 tensor-core projections
def split_tf32(w):
    """w fp32 -> (w_hi, w_lo) for the 3xTF32 GEMM (once per weight)."""
    lib = _lib.load()
    _chk(w, name='weight')
    hi, lo = torch.empty_like(w), torch.empty_like(w)
    _lib.check(lib.so_split_tf32(_p(w), _p(hi), _p(lo), w.numel(), _stream()), 'so_split_tf32')
    return hi, lo


def linear_ln_supported(N, K):
    """so_linear_3xtf32_ln: the whole output row must sit in one n-tile."""
    return K in (96, 192) and N % 32 == 0 and N <= 128


def linear_3xtf32(x, w_hi, w_lo, bias=None, relu=False, residual=None, out=None, ln=None):
    """y = act(x @ w^T + bias) (+ residual) on tcgen05 tensor cores with fp32-level accuracy.  x [..., K] contiguous.
    ``out``: optional pre-allocated contiguous [..., N] destination (e.g. a row range of a larger token buffer).
    ``ln`` = (gamma, beta, eps): LayerNorm over the N outputs folded into the epilogue (so_linear_3xtf32_ln)."""
    lib = _lib.load()
    _chk(x, name='x'); _chk(w_hi, name='w_hi'); _chk(w_lo, name='w_lo'); _chk(bias, name='bias'); _chk(residual, name='residual')
    N, K = w_hi.shape
    assert x.shape[-1] == K
    M = x.numel() // K
    if out is None:
        y = torch.empty(*x.shape[:-1], N, device=x.device, dtype=torch.float32)
    else:
        y = _chk(out, name='out')
        assert y.numel() == M * N and y.shape[-1] == N
    if residual is not None:
        assert residual.numel() == y.numel()
    if ln is not None:
        gamma, beta, eps = ln
        _chk(gamma, name='ln weight'); _chk(beta, name='ln bias')
        _lib.check(lib.so_linear_3xtf32_ln(_p(x), _p(w_hi), _p(w_lo), _p(bias), _p(residual), _p(gamma), _p(beta), float(eps), _p(y),
                                           M, N, K, int(bool(relu)), _stream()), 'so_linear_3xtf32_ln')
        return y
    _lib.check(lib.so_linear_3xtf32(_p(x), _p(w_hi), _p(w_lo), _p(bias), _p(residual), _p(y), M, N, K, int(bool(relu)), _stream()),
               'so_linear_3xtf32')
    return y


def linear_supported(K, N=None):
    """Shapes so_linear_3xtf32 accepts (gemm.cu): K = 96 or 192, N a multiple of 4 (16-byte TMA store rows).  Anything
    else takes cuBLAS in the callers instead of raising SO_ERR_UNSUPPORTED."""
    return K in (96, 192) and (N is None or N % 4 == 0)


class TCLinearFunction(torch.autograd.Function):
    """nn.Linear for the TRAINING path of the lifting encoder: y = x w^T + b and dL/dx = dL/dy w on the tcgen05 3xTF32 GEMM
    (fp32-level accuracy, so the step stays an fp32 step: mmcv's Linear layers run cuBLAS fp32 SIMT kernels there); the
    weight gradient is a reduction over the 10^5 token rows (dL/dy^T x, K = rows), which so_linear_3xtf32's tiling does not
    cover, and stays on cuBLAS.  When the contraction of dL/dx (the layer's out_features) is not 96 / 192 it takes cuBLAS too."""

    @staticmethod
    def forward(ctx, x, w, b):
        x2 = x.reshape(-1, x.shape[-1]).contiguous()
        hi, lo = split_tf32(w.detach().contiguous())
        y = linear_3xtf32(x2, hi, lo, None if b is None else b.detach().contiguous())
        ctx.save_for_backward(x2, w)
        ctx.has_bias, ctx.xshape = b is not None, x.shape
        return y.view(*x.shape[:-1], w.shape[0])

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        x2, w = ctx.saved_tensors
        N, K = w.shape
        g2 = gy.reshape(-1, N).contiguous()
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            if linear_supported(N, K):
                hi, lo = split_tf32(w.detach().t().contiguous())
                gx = linear_3xtf32(g2, hi, lo, None)
            else:
                gx = g2 @ w.detach()
            gx = gx.view(ctx.xshape)
        if ctx.needs_input_grad[1]:
            gw = g2.t() @ x2
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = g2.sum(0)
        return gx, gw, gb


def flatten_levels(img_feats, cams_embeds, level_embeds):
    """A3: [1, N, C, h, w] x L -> [N, sum(hw), 1, C] with camera + level embeddings, one transposing pass per level."""
    lib = _lib.load()
    N, Cc = img_feats[0].shape[1], img_feats[0].shape[2]
    hws = [f.shape[3] * f.shape[4] for f in img_feats]
    total = sum(hws)
    out = torch.empty(N, total, 1, Cc, device=img_feats[0].device, dtype=torch.float32)
    _chk(cams_embeds, name='cams_embeds'); _chk(level_embeds, name='level_embeds')
    start = 0
    for l, f in enumerate(img_feats):
        assert f.shape[0] == 1 and f.shape[1] == N and f.shape[2] == Cc
        _chk(f, name='img_feats[%d]' % l)
        _lib.check(lib.so_flatten_level(_p(f), _p(cams_embeds), _p(level_embeds[l]), _p(out), N, Cc, hws[l], start, total, _stream()),
                   'so_flatten_level')
        start += hws[l]
    return out


def layer_norm(x, gamma, beta, eps=1e-5, add=None):
    """y = LayerNorm(x [+ add]) over the last dim (fp32), one warp per row."""
    lib = _lib.load()
    _chk(x, name='x'); _chk(add, name='add'); _chk(gamma, name='weight'); _chk(beta, name='bias')
    Cn = x.shape[-1]
    y = torch.empty_like(x)
    _lib.check(lib.so_layer_norm(_p(x), _p(add), _p(gamma), _p(beta), _p(y), x.numel() // Cn, Cn, float(eps), _stream()),
               'so_layer_norm')
    return y


def _rows(t, name):
    """2-D row-major view whose rows may be a column slice of a wider matrix: returns (tensor, row stride in floats)."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != torch.float32:
        raise RuntimeError('%s must be a CUDA fp32 tensor: selfocc_b200 has no CPU fallback' % name)
    assert t.dim() == 2 and t.stride(1) == 1, '%s must be a [rows, cols] view with unit column stride' % name
    return t, t.stride(0)


def tpv_cross_attn_forward_rows(value_rows, n_cam, Hd, Dh, spatial_shapes, level_start_index, offsets_rows, logits_rows, uv, vis, L, D):
    """Strided form: value_rows [n_cam*Nv, >= Hd*Dh] view, offsets_rows [Q, Hd*L*D*2] view, logits_rows [Q, Hd*L*D] view."""
    lib = _lib.load()
    v, vld = _rows(value_rows, 'value'); o, old = _rows(offsets_rows, 'offsets'); lg, lld = _rows(logits_rows, 'logits')
    _chk(uv, name='uv'); _chk(vis, torch.uint8, 'vis')
    Q = o.shape[0]
    Nv = v.shape[0] // n_cam
    slots = torch.empty(Q, Hd * Dh, device=v.device)
    _lib.check(lib.so_tpv_cross_attn_forward_strided(_p(v), _p(spatial_shapes), _p(level_start_index), _p(o), _p(lg), _p(uv), _p(vis),
                                                     _p(slots), _p(None), n_cam, Nv, Hd, Dh, Q, L, D, vld, old, lld, _stream()),
               'so_tpv_cross_attn_forward_strided')
    return slots


def tpv_self_attn_forward_rows(value_rows, Hd, Dh, spatial_shapes, level_start_index, offsets_rows, logits_rows, ref, L, P):
    lib = _lib.load()
    v, vld = _rows(value_rows, 'value'); o, old = _rows(offsets_rows, 'offsets'); lg, lld = _rows(logits_rows, 'logits')
    _chk(ref, name='ref')
    Q = o.shape[0]
    out = torch.empty(Q, Hd * Dh, device=v.device)
    _lib.check(lib.so_tpv_self_attn_forward_strided(_p(v), _p(spatial_shapes), _p(level_start_index), _p(o), _p(lg), _p(ref), _p(out),
                                                    v.shape[0], Hd, Dh, Q, L, P, vld, old, lld, _stream()),
               'so_tpv_self_attn_forward_strided')
    return out


# --------------------------------------------------------------------------------------- reprojection loss
def make_reproj_desc(combine, n_cam, n_rays, n_samples, img_hw, img_size, ray_resize=None, ssim=True, automask=True):
    """so_reproj_desc of one loss call; img_hw = the image tensor's (H, W), img_size = the (h, w) pixels are normalised by."""
    d = _lib.ReprojDesc()
    d.variant = _lib.REPROJ_COMBINE if combine else _lib.REPROJ_MONO_MULTI_NEW
    d.n_cam, d.n_rays, d.n_samples = int(n_cam), int(n_rays), int(n_samples)
    d.img_h, d.img_w = int(img_hw[0]), int(img_hw[1])
    d.size_h, d.size_w = float(img_size[0]), float(img_size[1])
    d.grid_h, d.grid_w = (int(ray_resize[0]), int(ray_resize[1])) if ray_resize is not None else (0, 0)
    d.ssim, d.automask = int(bool(ssim)), int(bool(automask))
    return d


def _reproj_args(desc, curr, prev, nxt, pix, img2prev, img2next, weights, ts, deltas):
    N, R, S = desc.n_cam, desc.n_rays, desc.n_samples
    for n, t in (('curr', curr), ('prev', prev), ('next', nxt)):
        if _chk(t, name=n).shape != (N, 3, desc.img_h, desc.img_w):
            raise ValueError('%s must be [%d, 3, %d, %d], got %s' % (n, N, desc.img_h, desc.img_w, tuple(t.shape)))
    for n, t, shp in (('pix', pix, (R, 2)), ('img2prev', img2prev, (N, 4, 4)), ('img2next', img2next, (N, 4, 4)),
                      ('weights', weights, (N, R * S)), ('ts', ts, (N, R * S)), ('deltas', deltas, (N, R * S))):
        if t is not None and tuple(_chk(t, name=n).shape) != shp:
            raise ValueError('%s must be %s, got %s' % (n, shp, tuple(t.shape)))
    return [_p(t) for t in (curr, prev, nxt, pix, img2prev, img2next, weights, ts, deltas)]


def reproj_forward(desc, curr, prev, nxt, pix, img2prev, img2next, weights, ts, deltas=None):
    """-> (loss [1] before the loss weight, workspace for reproj_backward).  Shapes as in so_reproj_forward."""
    lib = _lib.load()
    args = _reproj_args(desc, curr, prev, nxt, pix, img2prev, img2next, weights, ts, deltas)
    nws = lib.so_reproj_workspace_floats(C.byref(desc))
    if nws < 0:
        raise ValueError('invalid reprojection loss configuration (ray_resize must tile the %d rays)' % desc.n_rays)
    ws = torch.empty(nws, device=curr.device, dtype=torch.float32)
    loss = torch.empty(1, device=curr.device, dtype=torch.float32)
    _lib.check(lib.so_reproj_forward(C.byref(desc), *args, _p(loss), _p(ws), _stream()), 'so_reproj_forward')
    return loss, ws


def reproj_backward(desc, curr, prev, nxt, pix, img2prev, img2next, weights, ts, deltas, g_loss, ws):
    """g_loss [1] (device) -> g_weights [N, R * S]; ws from the reproj_forward of the same inputs."""
    lib = _lib.load()
    args = _reproj_args(desc, curr, prev, nxt, pix, img2prev, img2next, weights, ts, deltas)
    _chk(g_loss, name='g_loss'); _chk(ws, name='workspace')
    g_w = torch.empty_like(weights)
    _lib.check(lib.so_reproj_backward(C.byref(desc), *args, _p(g_loss), _p(g_w), _p(ws), _stream()), 'so_reproj_backward')
    return g_w


def reproj_workspace_views(desc, ws):
    """Named views of a forward's workspace (test hook): counts [N, R, 2] of valid samples per ray (Combine: [.., 0] =
    samples with either projection valid), proj [N, R] per-ray loss, choice [N, R] index of the min."""
    N, R = desc.n_cam, desc.n_rays
    nr = N * R
    sums = ws[9 * nr:21 * nr].reshape(N, R, 12)
    counts = sums[..., 5:6] if desc.variant == _lib.REPROJ_COMBINE else sums[..., 10:12]
    return dict(counts=counts, proj=ws[21 * nr:22 * nr].reshape(N, R), choice=ws[22 * nr:23 * nr].reshape(N, R))


def reproj_check_layout(ray_idx, n_samples, bad):
    """bad int32 [1] |= 1 unless ray_idx == arange(n / n_samples).repeat_interleave(n_samples); no synchronisation."""
    lib = _lib.load()
    _chk(ray_idx, torch.int64, 'ray_indices'); _chk(bad, torch.int32, 'bad')
    _lib.check(lib.so_reproj_check_layout(_p(ray_idx), ray_idx.numel(), int(n_samples), _p(bad), _stream()),
               'so_reproj_check_layout')


class ReprojLossFunction(torch.autograd.Function):
    """Reprojection loss, differentiable w.r.t. the stacked per-camera weights [N, R * S] only (ts, deltas, images and
    transforms carry no gradient).  forward(weights, desc, curr, prev, next, pix, img2prev, img2next, ts, deltas) -> loss."""

    @staticmethod
    def forward(ctx, weights, desc, curr, prev, nxt, pix, img2prev, img2next, ts, deltas):
        loss, ws = reproj_forward(desc, curr, prev, nxt, pix, img2prev, img2next, weights, ts, deltas)
        ctx.desc = desc
        ctx.save_for_backward(weights, curr, prev, nxt, pix, img2prev, img2next, ts,
                              deltas if deltas is not None else weights.new_empty(0), ws)
        ctx.has_deltas = deltas is not None
        return loss.reshape(())

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        weights, curr, prev, nxt, pix, img2prev, img2next, ts, deltas, ws = ctx.saved_tensors
        g_w = reproj_backward(ctx.desc, curr, prev, nxt, pix, img2prev, img2next, weights, ts,
                              deltas if ctx.has_deltas else None, g.reshape(1).contiguous(), ws)
        return (g_w,) + (None,) * 9
