/*
 * selfocc_b200 -- C ABI of the sm_100a hot-path library (libselfocc_b200.so).
 *
 * The reference (huang-yh/SelfOcc) has no FFI of its own: its boundary for this path is the
 * mmengine registry + nn.Module contracts (SURVEY.md section 8b).  This C ABI sits UNDER
 * those Python modules; each entry point names the reference call site it replaces.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - tensors are dense, row-major, fp32 unless stated; index tensors are int64/int32 as stated;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - no internal allocation, no implicit synchronisation: work is enqueued on `stream`;
 *   - return value: SO_OK (0) or a negative SO_ERR_* code; never throws, never prints;
 *   - thread-safe for concurrent callers that use distinct streams and distinct outputs.
 */
#ifndef SELFOCC_B200_H
#define SELFOCC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SO_OK 0
#define SO_ERR_INVALID_ARG (-1)   /* null pointer / non-positive size / unsupported shape */
#define SO_ERR_UNSUPPORTED (-2)   /* valid request outside what the kernels implement */
#define SO_ERR_CUDA (-3)          /* a CUDA runtime call or launch failed; see so_last_cuda_error */
#define SO_ERR_NO_DEVICE (-4)

#define SO_ABI_VERSION 5   /* 2: so_render_train_forward gained pair_workspace; 3: packed render volume entry points;
                              4: occupancy evaluation entry points; 5: reprojection loss entry points */

/* ABI version of the loaded library (compare with SO_ABI_VERSION). */
int so_abi_version(void);
/* cudaError_t (as int) of the most recent failing CUDA call on this host thread, 0 if none. */
int so_last_cuda_error(void);
/* Static string for an SO_* code. */
const char* so_error_string(int code);
/* Number of kernel launches enqueued by this library since process start (bench.py's
 * gpu_launches claim is read from here). */
int64_t so_launch_count(void);

/* Optional per-kernel device timing (used by bench.py for the roofline line).  When enabled, the entry
 * points bracket their dominant kernel with cudaEventRecord on the launch stream.  Tags:
 * 0 render_infer, 1 tpv_decode, 2 tpv_cross_attn, 3 tpv_self_attn, 4 msda_forward, 5 msda_backward,
 * 6 render_train_fwd, 7 render_train_bwd, 8 linear_3xtf32.  so_profile_elapsed_ms returns the SUM over the calls since
 * the last so_profile_reset (the caller must have synchronised the stream) and the call count. */
#define SO_PROF_NUM_TAGS 10
int so_profile_enable(int on);
int so_profile_reset(void);
int so_profile_elapsed_ms(int tag, float* total_ms_host, int32_t* calls_host);

/* ---------------------------------------------------------------------------------------
 * Grid <-> metre mapping, one axis.  Restates LinearMapping.meter2grid
 * (reference model/encoder/bevformer/mappings.py:97-150):
 *     c = m - start;  a = |c|
 *     g = sign(c) * (a <= range0 || size1 == 0 ? a / range0 * size0
 *                                             : size0 + (a - range0) / range1 * size1) + offset
 * offset = size0 + size1 for a mirrored (non-half) h/w axis, else 0; start = d_range[0] for d.
 * Axis order everywhere: [0] = h (from metre y), [1] = w (from metre x), [2] = d (from metre z).
 */
typedef struct so_axis_map {
  float start, range0, range1, size0, size1, offset;
} so_axis_map;

typedef struct so_volume_desc {
  int32_t H, W, Z;      /* grid sizes (size_h, size_w, size_d) */
  int32_t zpitch;       /* floats between consecutive (h, w) columns of the sdf plane, >= Z */
  int32_t n_feat;       /* decoded channels besides sdf (colour + semantics), 0 if none */
  int32_t feat_pitch;   /* floats per voxel in the channel-last feature volume (>= n_feat, %4==0) */
  so_axis_map axis[3];
} so_volume_desc;

/* ---------------------------------------------------------------------------------------
 * B5  TPV planes -> decoded volume.  Replaces field.pre_compute_density_color(representation)
 * (call sites model/head/neus_head/neus_head.py:249,302,483; semantics from the in-repo analogue
 * model/head/nerfacc_head/bev_nerf.py:62-95, tpv=True, density_layers=2):
 *     f[h,w,z,:] = hw[h,w,:] + zh[z,h,:] + wz[w,z,:]
 *     out        = W2 * softplus(W1 * softplus(f) + b1) + b2          (C -> C -> 1 + n_feat)
 * tpv_hw [H*W, C], tpv_zh [Z*H, C], tpv_wz [W*Z, C]; w1 [C, C], b1 [C], w2 [1+n_feat, C], b2.
 * Outputs: vol_sdf [H, W, zpitch] (channel 0; pad entries zeroed), vol_feat [H, W, Z, feat_pitch]
 * (channels 1.., may be NULL when n_feat == 0).  C must be a multiple of 32, C <= 128.
 */
int so_tpv_decode(const float* tpv_hw, const float* tpv_zh, const float* tpv_wz, int32_t C,
                  const float* w1, const float* b1, const float* w2, const float* b2,
                  const so_volume_desc* vol_host, float* vol_sdf, float* vol_feat, void* stream);
/* Same, for the row range [h_begin, h_begin + h_count) of the volume only (voxel-sharded decode: every rank decodes its
 * slab of h rows into the full-size buffers and one all_gather assembles the volume; SURVEY 8e).  Other rows untouched. */
int so_tpv_decode_rows(const float* tpv_hw, const float* tpv_zh, const float* tpv_wz, int32_t C, const float* w1,
                       const float* b1, const float* w2, const float* b2, const so_volume_desc* vol_host, int32_t h_begin,
                       int32_t h_count, float* vol_sdf, float* vol_feat, void* stream);

/* Backward of the decode MLP over one slab of h rows (training).  The two [rows x C x C] products of the slab run through
 * so_linear_3xtf32; these are the element-wise pieces around them (reference: autograd through the decoder MLP,
 * model/head/neus_head/bev_nerf.py:150-190).  rows = h_count * W * Z, voxel order (h, w, z) inside the slab.
 *   features: a0[rows][C] = softplus(hw + zh + wz)
 *   hidden:   z1_a1[rows][C] holds z1 = a0 W1^T + b1 on entry and a1 = softplus(z1) on return;
 *             g1 = (W2^T g_out) * sigmoid(z1); g_out[rows][1 + n_feat] = the slab's output gradient gathered from
 *             g_vol_sdf [H][W][zpitch] (may be NULL = zero) and g_vol_feat [H][W][Z][feat_pitch] (may be NULL = zero)
 *   input:    g0[n] *= 1 - exp(-a0[n])   (= sigmoid of the pre-activation), n % 4 == 0                                   */
int so_tpv_decode_bwd_features(const float* tpv_hw, const float* tpv_zh, const float* tpv_wz, int32_t C,
                               const so_volume_desc* vol_host, int32_t h_begin, int32_t h_count, float* a0, void* stream);
int so_tpv_decode_bwd_hidden(float* z1_a1, const float* g_vol_sdf, const float* g_vol_feat, const float* w2, int32_t C,
                             const so_volume_desc* vol_host, int32_t h_begin, int32_t h_count, float* g1, float* g_out,
                             void* stream);
int so_tpv_decode_bwd_input(float* g0, const float* a0, int64_t n, void* stream);

/* Test hook: force the fp32 SIMT decode kernel (default: the tcgen05 3xTF32 kernel whenever C % 32 == 0). */
int so_tpv_decode_force_simt(int on);

/* ---------------------------------------------------------------------------------------
 * Ray set of one frame: n_cam cameras x rays_per_cam pixel rays, flattened (cam, ray)-major
 * exactly like neus_head.py:324-325.  Pixel coordinates come either from `pix` ([rays_per_cam, 2]
 * (x, y), RaySampler.forward(), ray_sampler.py:48-68) or, when pix == NULL, from the strided grid
 *     x = j * sx + ox,  y = i * sy + oy,  ray = i * nx + j          (ray_sampler.py:23-31,58-68)
 * cam_mats [n_cam, 4, 4] = metas[trans_kw] (img2lidar.py:25-70): origin = M[:3,3],
 * direction = M[:3,:3] * (x, y, 1), un-normalised; its norm converts ray length <-> camera depth.
 */
typedef struct so_ray_desc {
  int32_t n_cam, rays_per_cam;
  int32_t nx, ny;            /* grid shape, used when pix == NULL (nx * ny == rays_per_cam) */
  float sx, ox, sy, oy;
  int64_t ray_begin;         /* first flat ray index this call renders (ray sharding across GPUs) */
  int64_t ray_count;         /* number of flat rays this call renders */
  int64_t chunk_len;         /* rays per reference chunk (neus_head.py:341-345 `--batch`); the
                                expected-depth clip is taken per chunk.  <= 0: one chunk */
} so_ray_desc;

typedef struct so_render_params {
  float aabb[6];             /* roi_aabb x0 y0 z0 x1 y1 z1 (neus_head.py:189-195) */
  float near_plane;          /* near clamp, applied when `training` (collider) */
  int32_t training;          /* 0: eval (near clamp 0, rgb clamped), 1: train */
  int32_t num_samples;       /* S, uniform bins per ray (neus_head.py:136) */
  float inv_s;               /* exp(10 * variance) of the deviation network, clipped 1e-6..1e6 */
  float cos_anneal;          /* NeuS cos anneal ratio, 1.0 after warm-up */
  int32_t anchor_mid;        /* 1: field queried at bin midpoints, 0: at bin starts */
  int32_t sh_act;            /* 0: relu(C0*f + 0.5), 1: sigmoid(C0*f)  (sh_render.py:84-94, deg 0) */
  int32_t bkgd_mode;         /* 0 black, 1 white, 2 per-ray colours given in bkgd_rand */
} so_render_params;

/* Workspace floats needed by so_render_infer for `n_chunks` depth-clip chunks. */
int64_t so_render_workspace_floats(int64_t n_chunks);

/* B1-B4, B6-B11  fused inference render: ray generation -> AABB -> S samples -> trilinear gather
 * (+ analytic sdf gradient) -> NeuS alpha -> compositing -> depth / max-depth / acc / normal / rgb.
 * Replaces the chunk loop `self.model(ray_bundle)` + post-processing of NeuSHead.render
 * (model/head/neus_head/neus_head.py:319-438).  Outputs are indexed by (flat ray - ray_begin);
 * any output pointer may be NULL.  depth/max_depth are camera-z depths (divided by |direction|).
 *   depth [n], max_depth [n], max_idx int64 [n] (first-max argmax of w/delta, :430-438),
 *   acc [n], normal_vis [n,3], rgb [n,3] (needs n_feat >= 3), sem [n, n_feat-3] (needs n_feat > 3).
 * workspace: so_render_workspace_floats(n_chunks) floats, n_chunks = ceil(total rays / chunk_len).
 */
int so_render_infer(const float* vol_sdf, const float* vol_feat, const so_volume_desc* vol_host,
                    const float* cam_mats, const float* pix, const so_ray_desc* rays_host,
                    const so_render_params* params_host, const float* bkgd_rand,
                    float* depth, float* max_depth, int64_t* max_idx, float* acc,
                    float* normal_vis, float* rgb, float* sem, float* workspace, void* stream);

/* Packed render volume: a once-per-frame repack of the decoded volume into the layout the gather of the inference
 * render wants (built by NeuSHead.prepare, reused by every render of the frame -- eval_novel_depth.py:143-172 renders
 * several poses per prepare):
 *   n_feat == 0 : float2 [H][W][zpitch] {sdf[z], sdf[z+1]}  -- the 8 trilinear taps become 4 aligned 64-bit loads
 *   n_feat == 3 : float4 [H][W][Z]      {r, g, b, sdf}       -- 8 aligned 128-bit loads fetch sdf and colour together
 * so_render_pack_floats: floats needed (0: this channel count has no packed form).  pack must be 16-byte aligned. */
int64_t so_render_pack_floats(const so_volume_desc* vol_host);
int so_render_pack(const float* vol_sdf, const float* vol_feat, const so_volume_desc* vol_host, float* pack, void* stream);

/* so_render_infer on the packed volume (same outputs, same semantics; `pack` from so_render_pack, NULL = plain
 * so_render_infer).  Used when the metre->grid map is affine, num_samples is a power of two, the cos-anneal is finished,
 * samples are taken at bin midpoints and no semantics are rendered; any other configuration is routed to so_render_infer.
 * Rays that leave the volume take the zero-padding loop inside the same launch.  A warp stops marching when every
 * ray's transmittance is below 1e-9 (changes the outputs by < 1e-9 relative, never the max-depth index).
 * dbg_grid: optional probe [n, S, 3]: the fp32 (h, w, d) grid coordinates of every sample exactly as the kernel computed
 * them (test hook: lets a fp64 oracle be evaluated in the kernel's own cells, the analytic sdf gradient being
 * discontinuous across cell faces); NULL in production. */
int so_render_infer_packed(const float* vol_sdf, const float* vol_feat, const so_volume_desc* vol_host, const float* pack,
                           const float* cam_mats, const float* pix, const so_ray_desc* rays_host,
                           const so_render_params* params_host, const float* bkgd_rand,
                           float* depth, float* max_depth, int64_t* max_idx, float* acc,
                           float* normal_vis, float* rgb, float* sem, float* workspace, float* dbg_grid, void* stream);

/* B6-B10, B13  training-form render (NeuSHead.forward, neus_head.py:513-587): same sampling / field / alpha /
 * compositing as so_render_infer but it EMITS the per-sample tensors the losses consume (:667-682) and has a
 * backward.  `jitter` [total rays, S+1] uniforms in [0,1) for the stratified sampler (`perturb=True`), NULL =
 * no jitter.  Per-ray outputs [n]: depth, acc, fars (far / |dir|), max_depth, rgb [n,3], sem [n,n_feat-3];
 * per-sample outputs [n,S]: weights, ts = mid / |dir|, deltas = (end-start) / |dir|, sample_sdf; eik_grad [n,S,3]
 * = d sdf / d metre at the samples.  Any output may be NULL.  S <= 256.
 * pair_workspace: optional scratch of so_render_train_pair_floats(vol) floats (8-byte aligned), NULL = none.  When
 * given, the sdf volume is first repacked as {v[z], v[z+1]} pairs so that the 8 trilinear taps become 4 aligned
 * 64-bit loads (half the L1 requests of the gather-bound forward); results are bit-identical either way. */
int64_t so_render_train_pair_floats(const so_volume_desc* vol_host);
int so_render_train_forward(const float* vol_sdf, const float* vol_feat, const so_volume_desc* vol_host,
                            const float* cam_mats, const float* pix, const so_ray_desc* rays_host,
                            const so_render_params* params_host, const float* jitter, const float* bkgd_rand,
                            float* depth, float* acc, float* fars, float* rgb, float* sem, float* max_depth,
                            float* weights, float* ts, float* deltas, float* eik_grad, float* sample_sdf,
                            float* workspace, float* pair_workspace, void* stream);

/* Test hook: force the one-ray-per-warp forward kernel (default: the batched-ray kernel whenever the mapping is affine,
 * num_samples is a power of two >= 64, the cos-anneal is finished and no semantics are rendered). */
int so_render_train_force_fwd32(int on);
/* Test hook: render 24-channel feature volumes through the generic (any channel count) semantic path instead of the
 * vectorised 3 rgb + 21 class specialisation (config/nuscenes/nuscenes_occ.py:350). */
int so_render_train_force_sem_generic(int on);

/* Backward of so_render_train_forward w.r.t. the decoded volume and inv_s.  Incoming gradients (NULL = zero):
 * g_depth, g_acc [n], g_rgb [n,3], g_sem [n,n_feat-3], g_weights, g_sdf [n,S], g_eik [n,S,3].  Results are
 * ACCUMULATED (atomically) into g_vol_sdf [H,W,zpitch], g_vol_feat [H,W,Z,feat_pitch] (needed iff g_rgb/g_sem)
 * and the scalar g_inv_s; the caller zero-fills them.  Recomputes the forward (nothing is saved). */
int so_render_train_backward(const float* vol_sdf, const float* vol_feat, const so_volume_desc* vol_host,
                             const float* cam_mats, const float* pix, const so_ray_desc* rays_host,
                             const so_render_params* params_host, const float* jitter, const float* bkgd_rand,
                             const float* g_depth, const float* g_acc, const float* g_rgb, const float* g_sem,
                             const float* g_weights, const float* g_eik, const float* g_sdf,
                             float* g_vol_sdf, float* g_vol_feat, float* g_inv_s, float* workspace, void* stream);

/* Backward of so_field_query: g_sdf [n], g_grad [n,3], g_feat [n,n_feat] (NULL = zero) accumulated into
 * g_vol_sdf / g_vol_feat (caller zero-fills). */
int so_field_query_backward(const so_volume_desc* vol_host, const float* points, int64_t n, const float* g_sdf,
                            const float* g_grad, const float* g_feat, float* g_vol_sdf, float* g_vol_feat, void* stream);

/* B8  `second_grad` (neus_head.py:177,703-706 -> loss/second_grad_loss.py:19-20), DECLARED ASSUMPTION: the quantity lives in
 * the un-vendored fork; restated as the double-backward idiom d(sum_j d sdf/d x_j)/d x of the trilinear field = the row
 * sums of its Hessian in metres (pure second derivatives vanish inside a cell, the mixed ones do not).  points [n,3]
 * metres -> second_grad [n,3].  Backward: g_second_grad [n,3] accumulated atomically into g_vol_sdf (caller zero-fills). */
int so_field_second_grad(const float* vol_sdf, const so_volume_desc* vol_host, const float* points, int64_t n,
                         float* second_grad, void* stream);
int so_field_second_grad_backward(const so_volume_desc* vol_host, const float* points, int64_t n, const float* g_second_grad,
                                  float* g_vol_sdf, void* stream);

/* 8f-3  device-side DepthMetric step (utils/metric_util.py:247-279,311-349; eval_novel_depth.py:174-200).
 * so_depth_metric_sample: depth_pred [N,h,w], loc [N,n,2] in [0,1] (x,y) -> sampled [N,n] with the arithmetic of
 *   F.grid_sample(pred, loc*2-1, bilinear, padding_mode='border', align_corners=True).
 * so_depth_metric_sums: per camera, over points with mask != 0 and pred' = clamp(scale[cam] * sampled, 1e-3, 80)
 *   (scale NULL = 1): sums [N,8] = (sum |gt-pred'|/gt, sum (gt-pred')^2/gt, sum (gt-pred')^2, sum (log gt - log pred')^2,
 *   #(thresh < 1.25), #(< 1.25^2), #(< 1.25^3), #points); the metrics are sums / #points (rmse: sqrt).  One CTA per
 *   camera, deterministic. */
int so_depth_metric_sample(const float* depth_pred, const float* loc, int32_t N, int32_t n, int32_t h, int32_t w,
                           float* sampled, void* stream);
int so_depth_metric_sums(const float* sampled, const float* depth_gt, const uint8_t* mask, const float* scale, int32_t N,
                         int32_t n, float* sums, void* stream);

/* B12  field query at arbitrary points.  Replaces field.forward_sdfnetwork / forward_geonetwork
 * as used by NeuSHead.get_uniform_sdf (neus_head.py:265-293).  points [n,3] metres ->
 * sdf [n], grad [n,3] (NULL ok), feat [n, n_feat] raw decoded channels 1.. (NULL ok). */
int so_field_query(const float* vol_sdf, const float* vol_feat, const so_volume_desc* vol_host,
                   const float* points, int64_t n, float* sdf, float* grad, float* feat, void* stream);

/* ---------------------------------------------------------------------------------------
 * Occupancy evaluation (eval_iou.py:206-258, eval_iou_kitti.py:167-196).
 *
 * so_occ_classify: decoded volume -> uint8 labels per output voxel, without storing the get_uniform_sdf lattice
 * (neus_head.py:265-293).  The lattice is [H = ny, W = nx, D = nz] with node (h, w, d) at metres (xs[w], ys[h], zs[d]);
 * xs / ys / zs are the caller's torch.linspace vectors, and a node's value is exactly what so_field_query returns there.
 *   points == NULL  lattice mode: the output grid IS the lattice (grid->n0 = ny, n1 = nx, n2 = nz).
 *   points [n, 3]   resample mode (Occ3D): normalised (x, y, z) in [0, 1] (eval_iou.py:211-218); each output voxel is
 *                   F.grid_sample(lattice, points[..., [2, 0, 1]] * 2 - 1, bilinear, align_corners=True, zeros padding).
 * occ [n] = sdf <= thresh, then zeroed outside third-axis [z_lo, z_hi) and in the border rows (first axis: the first
 * border[0] and last border[1] indices, second axis: border[2] / border[3]).
 * sem [n] (NULL = not computed) = occ * lut[argmax_c logit_c], logits = vol_feat channels 3.. (h[..., 4:] of the
 * lattice), first maximum; lut [lut_len >= n_feat - 3] uint8 (NULL = identity).  Logits are only gathered where occ is
 * 1.  n_feat - 3 <= 32.  n = n0 * n1 * n2 voxels, row-major.
 *
 * so_occ_hist: hist[g * P + min(pred, P - 1)] += 1 for every i < n with mask[i] != 0 (mask NULL = all), g = gt[i];
 * hist int64 [256, P], zero-filled by the caller and ACCUMULATED (across frames).  1 <= P <= SO_OCC_HIST_MAX_P.
 * Integer counts: deterministic.  Every reference occupancy metric (MeanIoU, IoU, SSCMetrics) is a function of it.
 */
#define SO_OCC_HIST_MAX_P 32

typedef struct so_occ_grid {
  int32_t n0, n1, n2;     /* output grid shape */
  int32_t z_lo, z_hi;     /* kept third-axis index range [z_lo, z_hi) */
  int32_t border[4];      /* zeroed rows: first axis low, high; second axis low, high (>= 0) */
  float thresh;           /* occupied: sdf <= thresh */
} so_occ_grid;

int so_occ_classify(const float* vol_sdf, const float* vol_feat, const so_volume_desc* vol_host, const float* xs,
                    const float* ys, const float* zs, int32_t nx, int32_t ny, int32_t nz, const float* points,
                    const so_occ_grid* grid_host, const uint8_t* lut, int32_t lut_len, uint8_t* occ, uint8_t* sem,
                    void* stream);
int so_occ_hist(const uint8_t* pred, const uint8_t* gt, const uint8_t* mask, int64_t n, int32_t P, int64_t* hist,
                void* stream);

/* ---------------------------------------------------------------------------------------
 * Self-supervised reprojection loss (loss/reproj_loss_mono_multi_new_combine.py:108-245, variant SO_REPROJ_COMBINE;
 * loss/reproj_loss_mono_multi_new.py:117-288, variant SO_REPROJ_MONO_MULTI_NEW, sdf_loss=False).
 *
 * Inputs are the training head's per-sample outputs in its ray layout: N cameras x R rays x S CONTIGUOUS samples,
 * rays in order (ray_indices[cam] = arange(R).repeat_interleave(S); so_reproj_check_layout verifies that).
 *   curr, prev, next [N, 3, img_h, img_w]   pix [R, 2] pixel (x, y) = ms_rays   img2prev, img2next [N, 4, 4]
 *   weights, ts [N, R * S]   deltas [N, R * S] or NULL (w <- delta < eps ? 0 : w / max(delta, eps))
 * so_reproj_forward writes loss[0] = the reference's return value (mean over rays, then over cameras; the caller applies
 * the loss weight) and keeps in `workspace` what the backward needs; so_reproj_backward takes the device scalar
 * g_loss[0] = d total / d loss and the SAME inputs and workspace, and writes g_weights [N, R * S] (no gradient w.r.t. ts,
 * deltas, images or transforms).  Combine samples the images with padding_mode='border', MonoMultiNew with zeros.
 * ssim != 0 needs grid_h * grid_w == R (ray_resize), grid_h, grid_w >= 2.  Deterministic: no atomics.
 * so_reproj_workspace_floats: floats of workspace for `desc` (-1: invalid desc). */
#define SO_REPROJ_COMBINE 0
#define SO_REPROJ_MONO_MULTI_NEW 1

typedef struct so_reproj_desc {
  int32_t variant;                     /* SO_REPROJ_* */
  int32_t n_cam, n_rays, n_samples;    /* N, R, S */
  int32_t img_h, img_w;                /* image tensor size */
  float size_h, size_w;                /* img_size the pixel coordinates are normalised by */
  int32_t grid_h, grid_w;              /* ray_resize, read iff ssim */
  int32_t ssim, automask;              /* !no_ssim, !no_automask */
} so_reproj_desc;

int64_t so_reproj_workspace_floats(const so_reproj_desc* desc_host);
int so_reproj_forward(const so_reproj_desc* desc_host, const float* curr, const float* prev, const float* next,
                      const float* pix, const float* img2prev, const float* img2next, const float* weights, const float* ts,
                      const float* deltas, float* loss, float* workspace, void* stream);
int so_reproj_backward(const so_reproj_desc* desc_host, const float* curr, const float* prev, const float* next,
                       const float* pix, const float* img2prev, const float* img2next, const float* weights, const float* ts,
                       const float* deltas, const float* g_loss, float* g_weights, float* workspace, void* stream);
/* bad[0] |= 1 if ray_idx[i] != i / n_samples for some i < n (bad zero-filled by the caller; no synchronisation). */
int so_reproj_check_layout(const int64_t* ray_idx, int64_t n, int32_t n_samples, int32_t* bad, void* stream);

/* ---------------------------------------------------------------------------------------
 * A7/A8  multi-scale deformable attention forward.  Drop-in for
 * MultiScaleDeformableAttnFunction.apply(value, spatial_shapes, level_start_index,
 * sampling_locations, attention_weights, im2col_step) of mmcv==2.0.1 (reference call sites
 * model/encoder/bevformer/attention/image_cross_attention.py:340-342 and
 * model/encoder/tpvformer/attention/cross_view_hybrid_attention.py:111-113).
 *   value [B, Nv, Hd, Dh]   spatial_shapes int64 [L,2] (h,w)   level_start_index int64 [L]
 *   loc [B, Nq, Hd, L, P, 2] normalised (x,y)   weights [B, Nq, Hd, L, P]   out [B, Nq, Hd*Dh]
 * Dh must be 16 or 32.
 */
int so_msda_forward(const float* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                    const float* loc, const float* weights, float* out,
                    int32_t B, int32_t Nv, int32_t Hd, int32_t Dh, int32_t Nq, int32_t L, int32_t P,
                    void* stream);

/* Backward of so_msda_forward (the mmcv op's autograd contract): grad_out [B,Nq,Hd*Dh] ->
 * grad_value [B,Nv,Hd,Dh] (must be zero-filled by the caller; accumulated atomically),
 * grad_loc [B,Nq,Hd,L,P,2], grad_weights [B,Nq,Hd,L,P]. */
int so_msda_backward(const float* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                     const float* loc, const float* weights, const float* grad_out,
                     float* grad_value, float* grad_loc, float* grad_weights,
                     int32_t B, int32_t Nv, int32_t Hd, int32_t Dh, int32_t Nq, int32_t L, int32_t P,
                     void* stream);

/* A6/A9  dense projection on the tcgen05 tensor cores with fp32-level accuracy ("3xTF32" operand splitting):
 *     y[M,N] = act(x[M,K] * w[N,K]^T + bias[N]) (+ residual[M,N])
 * Replaces the nn.Linear calls of the attention modules and the FFN (image_cross_attention.py:36,218-223,309-317,
 * cross_view_hybrid_attention.py:79-86,118, tpvformer_encoder_layer.py:198-206).  w_hi / w_lo = so_split_tf32(w)
 * (w_hi = w with the low 13 mantissa bits cleared, w_lo = w - w_hi), computed once per weight.  K % 96 == 0;
 * x, w_hi, w_lo 16-byte aligned; relu: 0/1; bias / residual may be NULL. */
/* Test hook: 1 = so_linear_3xtf32 with both MMA operands in shared memory (SS, the round-1 pipeline); 0 (default) = the X
 * operand split into tensor memory (TS).  Both are parity-tested. */
int so_linear_force_ss(int on);
int so_split_tf32(const float* w, float* w_hi, float* w_lo, int64_t n, void* stream);
int so_linear_3xtf32(const float* x, const float* w_hi, const float* w_lo, const float* bias, const float* residual,
                     float* y, int64_t M, int32_t N, int32_t K, int32_t relu, void* stream);

/* A9  projection + LayerNorm in ONE launch: y = LayerNorm(act(x w^T + bias) + residual) * gamma + beta over the N output
 * columns, computed in the GEMM epilogue (an epilogue thread owns a whole output row, so the statistics are register-local).
 * Replaces `output_proj -> (+ identity) -> norm` and `ffn.layers[1] -> (+ identity) -> norm` of TPVFormerLayer
 * (tpvformer_encoder_layer.py:185-218).  N % 32 == 0, N <= 128; otherwise as so_linear_3xtf32. */
int so_linear_3xtf32_ln(const float* x, const float* w_hi, const float* w_lo, const float* bias, const float* residual,
                        const float* gamma, const float* beta, float eps, float* y, int64_t M, int32_t N, int32_t K,
                        int32_t relu, void* stream);

/* A9  y = LayerNorm(x [+ add]) over the last dimension C (nn.LayerNorm(C), biased variance, eps inside the sqrt),
 * replaces the norm steps of TPVFormerLayer (tpvformer_encoder_layer.py:185-196).  x, add, y [rows, C]; C <= 256. */
int so_layer_norm(const float* x, const float* add, const float* gamma, const float* beta, float* y, int64_t rows,
                  int32_t C, float eps, void* stream);

/* A3  one FPN level into the flattened token tensor (tpvformer_encoder.py:261-277): feat [N, C, hw] ->
 * out[n, level_start + p, :] = (feat[n, :, p] + cams_embeds[n, :]) + level_embed[:], out being [N, total, C].  Replaces
 * flatten(3).permute(...) + the two embedding adds + torch.cat over levels + .contiguous() (five passes over 59 MB). */
int so_flatten_level(const float* feat, const float* cams_embeds, const float* level_embed, float* out, int32_t N, int32_t C,
                     int32_t hw, int64_t level_start, int64_t total, void* stream);

/* A4  projection of pillar reference points into the cameras.  Replaces point_sampling
 * (model/encoder/bevformer/utils.py:116-206, no post_rots / focal_ratios branch).
 *   ref_3d [D, Q, 3] metres, lidar2img [N, 4, 4], img_h/img_w = metas[0]['img_shape']
 *   -> uv [N, Q, D, 2] normalised (x, y), mask uint8 [N, Q, D] (1 = in frustum),
 *      vis uint8 [N, Q] = any_d mask (the per-camera query visibility of
 *      image_cross_attention.py:92; NULL ok).
 * Arithmetic order is fixed (plain fp32 mul/add, no FMA contraction) so that `mask`, an index-
 * generating quantity, is reproducible bit for bit. */
int so_point_sampling(const float* ref_3d, const float* lidar2img, int32_t D, int32_t Q, int32_t N,
                      float img_h, float img_w, float* uv, uint8_t* mask, uint8_t* vis, void* stream);

/* A5+A6+A7  rebatch-free image cross-attention core for one TPV plane.  Replaces the
 * nonzero()/rebatch/scatter-add/count machinery of BEVCrossAttention.forward together with the
 * location arithmetic, softmax and op call of BEVDeformableAttention.forward
 * (model/encoder/bevformer/attention/image_cross_attention.py:84-136, 313-345):
 *   for every query q:  slots[q] = (1 / max(1, #visible cams)) *
 *        sum_{cam visible(q)} MSDA(value[cam], uv[cam,q,:] + offsets[q] / (w_l, h_l), softmax(logits[q]))
 * where visible(q, cam) = vis[cam, q] = any_d mask[cam, q, d] (from so_point_sampling).  offsets/logits depend on the query only, so they
 * are computed once per query instead of once per (camera, padded slot).
 *   value [N, Nv, Hd, Dh] (after value_proj), offsets [Q, Hd, L, D, 2], logits [Q, Hd, L, D],
 *   uv [N, Q, D, 2], vis uint8 [N, Q], spatial_shapes int64 [L,2], level_start_index int64 [L]
 *   -> slots [Q, Hd*Dh] (input of output_proj), count int32 [Q] (NULL ok). */
int so_tpv_cross_attn_forward(const float* value, const int64_t* spatial_shapes,
                              const int64_t* level_start_index, const float* offsets, const float* logits,
                              const float* uv, const uint8_t* vis, float* slots, int32_t* count,
                              int32_t N, int32_t Nv, int32_t Hd, int32_t Dh, int32_t Q, int32_t L, int32_t D,
                              void* stream);

/* Strided variants: the value / offsets / logits operands may be column slices of wider row-major matrices (row strides
 * value_ld / offsets_ld / logits_ld in floats), so ONE projection GEMM can produce the offsets and logits of a query (and
 * the value tensors of all three planes) side by side without a repacking copy. */
int so_tpv_cross_attn_forward_strided(const float* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                                      const float* offsets, const float* logits, const float* uv, const uint8_t* vis,
                                      float* slots, int32_t* count, int32_t N, int32_t Nv, int32_t Hd, int32_t Dh, int32_t Q,
                                      int32_t L, int32_t D, int32_t value_ld, int32_t offsets_ld, int32_t logits_ld, void* stream);

/* Test hook: 1 = run so_tpv_cross_attn_forward* / so_tpv_self_attn_forward* on the first-generation kernels (every lane of
 * a (query, head) redoes the sample set-up) instead of the shared-set-up kernels.  Both are parity-tested. */
int so_attn_force_v1(int on);

/* A5  visible-query index lists, as the reference builds them with nonzero()
 * (image_cross_attention.py:90-94), without a host sync: for each camera, ascending int64 query
 * indices with any in-frustum point.  index_lists [N, Q] (first lens[cam] entries valid),
 * lens int32 [N].  Single-CTA-per-camera ordered compaction. */
int so_visible_index_lists(const uint8_t* mask, int32_t N, int32_t Q, int32_t D,
                           int64_t* index_lists, int32_t* lens, void* stream);

/* A8 fused  cross-view hybrid (self) attention core: softmax + location arithmetic + sampling.
 * Replaces cross_view_hybrid_attention.py:83-116.
 *   value [Nv, Hd, Dh] (after value_proj; levels = the three planes), offsets [Q, Hd, L, P, 2],
 *   logits [Q, Hd, L, P], ref [Q, L, P, 2] -> out [Q, Hd*Dh] (input of output_proj). */
int so_tpv_self_attn_forward(const float* value, const int64_t* spatial_shapes,
                             const int64_t* level_start_index, const float* offsets, const float* logits,
                             const float* ref, float* out,
                             int32_t Nv, int32_t Hd, int32_t Dh, int32_t Q, int32_t L, int32_t P,
                             void* stream);

int so_tpv_self_attn_forward_strided(const float* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                                     const float* offsets, const float* logits, const float* ref, float* out, int32_t Nv,
                                     int32_t Hd, int32_t Dh, int32_t Q, int32_t L, int32_t P, int32_t value_ld,
                                     int32_t offsets_ld, int32_t logits_ld, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SELFOCC_B200_H */
