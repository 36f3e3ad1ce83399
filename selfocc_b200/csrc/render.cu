// SDF volume-render head kernels (SURVEY.md section 8a rows B1-B4, B6-B12).
//
// so_render_infer: ONE fused launch per frame (plus a tiny depth-clip-bounds pre-pass) replacing the
// reference's python chunk loop of `self.model(ray_bundle)` (neus_head.py:346-374) and its CPU
// max-depth step (:430-438).  Mapping: one thread per ray, a warp = 32 horizontally adjacent pixels of
// one camera, so the 8-corner gathers of a warp hit a handful of (h, w) columns of the L2-resident
// decoded volume and the per-ray outputs are written fully coalesced.  The 256-sample compositing
// recurrence is kept in registers in the reference's order (exclusive cumprod, first-max argmax).
#include "render_common.cuh"
#ifndef SO_RENDER_UNROLL
#define SO_RENDER_UNROLL 1     // measured 10.20 / 10.56 / 10.44 ms for unroll 1 / 2 / 4 at 8.64 M rays
#endif
#ifndef SO_RENDER_BLOCK
#define SO_RENDER_BLOCK 128
#endif
#ifndef SO_RENDER_MIN_CTAS
#define SO_RENDER_MIN_CTAS 8    // 64 registers, no spills (10 -> 48 registers spills inside the sample loop and is slower)
#endif

namespace so {

// ---- pre-pass: per-chunk [min first-mid, max last-mid] for the expected-depth clip ------------------
__global__ void bounds_init_kernel(float* ws, long long n_chunks) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n_chunks) {
    ws[2 * i] = INFINITY;
    ws[2 * i + 1] = 0.f;
  }
}

__global__ void __launch_bounds__(256) bounds_kernel(RayDev R, RenderDev P, float* ws) {
  long long gid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  bool ok = gid < R.total;
  float mn = INFINITY, mx = 0.f;
  long long chunk = 0;
  if (ok) {
    float o[3], d[3], nrm, tn, tf;
    make_ray(R, gid, o, d, nrm);
    slab(P, o, d, tn, tf);
    float step = 1.0f / (float)P.S;
    const float* u = P.jitter ? P.jitter + gid * (long long)(P.S + 1) : nullptr;
    float e0 = edge_t(bin_edge01_jit(0, P.S, step, u), tn, tf), e1 = edge_t(bin_edge01_jit(1, P.S, step, u), tn, tf);
    float eL = edge_t(bin_edge01_jit(P.S - 1, P.S, step, u), tn, tf), eE = edge_t(bin_edge01_jit(P.S, P.S, step, u), tn, tf);
    mn = __fmul_rn(__fadd_rn(e0, e1), 0.5f);
    mx = __fmul_rn(__fadd_rn(eL, eE), 0.5f);
    chunk = R.chunk_len > 0 ? gid / R.chunk_len : 0;
  }
  // aggregate per warp, then per CTA, when everybody sits in one chunk (the common case): ONE atomic pair per CTA.
  // (One pair per warp -- 270 k same-address atomics for 8.64 M rays -- made this pre-pass 165 us, ncu r2_launches.)
  unsigned full = __activemask();
  long long c0 = __shfl_sync(full, chunk, 0);
  bool uniform = __all_sync(full, (!ok) || chunk == c0);
  __shared__ float s_mn[8], s_mx[8];
  __shared__ long long s_chunk[8];
  __shared__ int s_uniform;
  if (threadIdx.x == 0) s_uniform = 1;
  __syncthreads();
  if (uniform) {
    for (int s = 16; s > 0; s >>= 1) {
      mn = fminf(mn, __shfl_xor_sync(full, mn, s));
      mx = fmaxf(mx, __shfl_xor_sync(full, mx, s));
    }
  }
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { s_mn[w] = mn; s_mx[w] = mx; s_chunk[w] = c0; }
  if (!uniform) atomicAnd(&s_uniform, 0);
  __syncthreads();
  bool cta_uniform = s_uniform != 0;
  if (cta_uniform) {
    for (int i = 1; i < 8; ++i) cta_uniform = cta_uniform && (s_chunk[i] == s_chunk[0] || s_mn[i] == INFINITY);
  }
  if (cta_uniform) {
    if (threadIdx.x == 0) {
      float bmn = s_mn[0], bmx = s_mx[0];
      long long bc = s_chunk[0];
      for (int i = 1; i < 8; ++i) { if (s_mn[i] != INFINITY) bc = s_chunk[i]; bmn = fminf(bmn, s_mn[i]); bmx = fmaxf(bmx, s_mx[i]); }
      if (bmn != INFINITY) {
        // all values are >= 0, so the int ordering equals the float ordering
        atomicMin((int*)(ws + 2 * bc), __float_as_int(bmn));
        atomicMax((int*)(ws + 2 * bc + 1), __float_as_int(bmx));
      }
    }
  } else if (uniform) {
    if ((threadIdx.x & 31) == 0 && mn != INFINITY) {
      atomicMin((int*)(ws + 2 * c0), __float_as_int(mn));
      atomicMax((int*)(ws + 2 * c0 + 1), __float_as_int(mx));
    }
  } else if (ok) {
    atomicMin((int*)(ws + 2 * chunk), __float_as_int(mn));
    atomicMax((int*)(ws + 2 * chunk + 1), __float_as_int(mx));
  }
}

// enqueue the two pre-pass kernels; ws receives [min first-mid, max last-mid] per reference chunk
int launch_depth_bounds(const RayDev& R, const RenderDev& P, float* ws, cudaStream_t st) {
  long long n_chunks = R.chunk_len > 0 ? ceil_div64(R.total, R.chunk_len) : 1;
  bounds_init_kernel<<<(unsigned)ceil_div64(n_chunks, 256), 256, 0, st>>>(ws, n_chunks);
  bounds_kernel<<<(unsigned)ceil_div64(R.total, 256), 256, 0, st>>>(R, P, ws);
  note_launch(2);
  return check_launch();
}


// FAST = affine metre->grid map, power-of-two S, cos-anneal finished, mid-point anchor (every shipped eval config):
// the uniform branches for the general cases are compiled out.
template <bool HAS_RGB, bool HAS_SEM, bool FAST>
__global__ void __launch_bounds__(SO_RENDER_BLOCK, SO_RENDER_MIN_CTAS) render_infer_kernel(VolumeDev V, RayDev R, RenderDev P, const float* __restrict__ ws,
                                                           const float* __restrict__ bkgd_rand, float* __restrict__ depth,
                                                           float* __restrict__ max_depth, long long* __restrict__ max_idx,
                                                           float* __restrict__ acc_out, float* __restrict__ normal_vis,
                                                           float* __restrict__ rgb_out, float* __restrict__ sem_out) {
  long long lid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const bool valid = lid < R.ray_count;            // lanes past the end stay alive for the warp votes below
  if (!valid) lid = R.ray_count - 1;
  long long gid = R.ray_begin + lid;
  float o[3], d[3], nrm, tn, tf;
  make_ray(R, gid, o, d, nrm);
  slab(P, o, d, tn, tf);

  const int S = P.S;
  const float step = 1.0f / (float)S;
  const bool pow2 = FAST || (S & (S - 1)) == 0;    // then i * (1/S) is exact and equals torch.linspace bit for bit
  const float eps = 1.1920928955078125e-07f;       // torch.finfo(float32).eps (neus_head.py:431)
  const float eps_len = eps * nrm;                 // delta / nrm < eps  <=>  delta < eps * nrm
  // metre -> grid is affine per axis when the mapping has no outer ring (every shipped config):
  // g(t) = g0 + gd * t along the ray, one FMA per axis per sample
  const bool affine = FAST || (V.ax[0].k1 == 0.f && V.ax[1].k1 == 0.f && V.ax[2].k1 == 0.f);
  const float kh0 = V.ax[0].k0, kw0 = V.ax[1].k0, kd0 = V.ax[2].k0;
  const float gh0 = fmaf(o[1] - V.ax[0].start, kh0, V.ax[0].offset), gdh = d[1] * kh0;
  const float gw0 = fmaf(o[0] - V.ax[1].start, kw0, V.ax[1].offset), gdw = d[0] * kw0;
  const float gd0 = fmaf(o[2] - V.ax[2].start, kd0, V.ax[2].offset), gdd = d[2] * kd0;
  const int Hm1 = V.H - 1, Wm1 = V.W - 1, Zm1 = V.Z - 1;
  const bool anneal_done = FAST || P.cos_anneal == 1.0f;   // -(relu(-tc)) == min(tc, 0)
  const float k_log2 = P.inv_s * 1.4426950408889634f;       // inv_s * log2(e)

  float T = 1.0f, acc = 0.f, dsum = 0.f, n0 = 0.f, n1 = 0.f, n2 = 0.f;
  float best = -INFINITY, best_mid = 0.f;
  int best_i = 0;
  float c_r = 0.f, c_g = 0.f, c_b = 0.f;
  float sem[HAS_SEM ? kMaxSem : 1];
  const int n_sem = HAS_SEM ? V.n_feat - 3 : 0;
  if (HAS_SEM)
    for (int i = 0; i < kMaxSem; ++i) sem[i] = 0.f;

  float e0 = edge_t(bin_edge01(0, S, step), tn, tf);
  // FAST path: uniform bins, so mid_s = tn + (s + 1/2) * span / S and delta = span / S is constant along the ray
  // (within 1-2 ulp of the reference's edge arithmetic, far inside the 1e-5 tolerance of depth / max-depth)
  const float span = tf - tn;
  const float delta_c = span * step;
  const float h_const = delta_c * (0.5f * k_log2);
  float bm = 0.5f * step;
  constexpr int kUnroll = SO_RENDER_UNROLL;
#pragma unroll kUnroll
  for (int s = 0; s < S; ++s) {
    float mid, delta, tq;
    if (FAST) {
      mid = fmaf(bm, span, tn);
      bm += step;
      delta = delta_c;
      tq = mid;
    } else {
      float b1 = pow2 ? (float)(s + 1) * step : bin_edge01(s + 1, S, step);
      float e1 = edge_t(b1, tn, tf);
      mid = __fmul_rn(__fadd_rn(e0, e1), 0.5f);
      delta = __fsub_rn(e1, e0);
      tq = P.anchor_mid ? mid : e0;
      e0 = e1;
    }
    float gh, gw, gd, kh = kh0, kw = kw0, kd = kd0;
    if (affine) {
      gh = fmaf(gdh, tq, gh0); gw = fmaf(gdw, tq, gw0); gd = fmaf(gdd, tq, gd0);
    } else {
      float x = fmaf(d[0], tq, o[0]), y = fmaf(d[1], tq, o[1]), z = fmaf(d[2], tq, o[2]);
      gh = axis_m2g(V.ax[0], y, kh); gw = axis_m2g(V.ax[1], x, kw); gd = axis_m2g(V.ax[2], z, kd);
    }
    float sdf, dgh, dgw, dgd;
    float flh = floorf(gh), flw = floorf(gw), flz = floorf(gd);
    int h0 = (int)flh, w0 = (int)flw, z0 = (int)flz;
    bool interior = (unsigned)h0 < (unsigned)Hm1 && (unsigned)w0 < (unsigned)Wm1 && (unsigned)z0 < (unsigned)Zm1;
    Taps t;
    if (__all_sync(0xffffffffu, interior)) {
      gather_sdf_interior(V, h0, w0, z0, gh - flh, gw - flw, gd - flz, sdf, dgh, dgw, dgd);
      if (HAS_RGB) t = make_taps(V, gh, gw, gd);
    } else {
      t = make_taps(V, gh, gw, gd);
      gather_sdf(V, t, sdf, dgh, dgw, dgd);
    }
    float gx = dgw * kw, gy = dgh * kh, gz = dgd * kd;  // d sdf / d metre (x, y, z)
    // NeuS alpha (upstream SDFField.get_alpha)
    float tc = d[0] * gx + d[1] * gy + d[2] * gz;
    float ic = anneal_done ? fminf(tc, 0.f)
                           : -(fmaxf(fmaf(-tc, 0.5f, 0.5f), 0.f) * (1.0f - P.cos_anneal) + fmaxf(-tc, 0.f) * P.cos_anneal);
    float alpha = neus_alpha_log2(sdf * k_log2, ic * (FAST ? h_const : delta * (0.5f * k_log2)));
    float w = alpha * T;
    T *= (1.0f - alpha + 1e-7f);
    acc += w;
    dsum = fmaf(w, mid, dsum);
    float wn = w * rsqrtf(fmaxf(gx * gx + gy * gy + gz * gz, 1e-24f));  // F.normalize(eps=1e-12)
    n0 = fmaf(wn, gx, n0); n1 = fmaf(wn, gy, n1); n2 = fmaf(wn, gz, n2);
    // max-depth candidate (neus_head.py:430-438): first maximum of w / clamp(delta', eps) with w := 0 where delta' < eps;
    // delta' = delta / |dir| and |dir| is constant along the ray, so the argmax is taken over w / delta
    float cand = FAST ? w : (delta < eps_len ? 0.f : __fdividef(w, delta));   // FAST: delta is a positive per-ray constant
    if (cand > best) { best = cand; best_i = s; best_mid = mid; }
    if (HAS_RGB) {
      float f[3];
      gather_feat<3>(V, t, 0, f);
      float r0 = f[0] * kC0, r1 = f[1] * kC0, r2 = f[2] * kC0;
      if (P.sh_act == 0) { r0 = fmaxf(r0 + 0.5f, 0.f); r1 = fmaxf(r1 + 0.5f, 0.f); r2 = fmaxf(r2 + 0.5f, 0.f); }
      else { r0 = sigmoidf_acc(r0); r1 = sigmoidf_acc(r1); r2 = sigmoidf_acc(r2); }
      c_r = fmaf(w, r0, c_r); c_g = fmaf(w, r1, c_g); c_b = fmaf(w, r2, c_b);
    }
    if (HAS_SEM) {
      // rendered semantics = sum_s w * softmax(logits) (bev_nerf.py:147-148 + SemanticRenderer)
      float lg[kMaxSem];
      float mx = -INFINITY;
      for (int c = 0; c < n_sem; ++c) { float f1[1]; gather_feat<1>(V, t, 3 + c, f1); lg[c] = f1[0]; mx = fmaxf(mx, f1[0]); }
      float den = 0.f;
      for (int c = 0; c < n_sem; ++c) { lg[c] = expf(lg[c] - mx); den += lg[c]; }
      float sc = w / den;
      for (int c = 0; c < n_sem; ++c) sem[c] = fmaf(sc, lg[c], sem[c]);
    }
  }
  if (!valid) return;
  if (FAST && delta_c < eps_len) { best_i = 0; best_mid = fmaf(0.5f * step, span, tn); }   // all candidates are 0: first index

  long long chunk = R.chunk_len > 0 ? gid / R.chunk_len : 0;
  float lo = __ldg(ws + 2 * chunk), hi = __ldg(ws + 2 * chunk + 1);
  if (depth) {
    float dd = dsum / (acc + 1e-10f);
    dd = fminf(fmaxf(dd, lo), hi);
    depth[lid] = dd / nrm;
  }
  if (max_depth) max_depth[lid] = best_mid / nrm;
  if (max_idx) max_idx[lid] = best_i;
  if (acc_out) acc_out[lid] = acc;
  if (normal_vis) {
    normal_vis[3 * lid + 0] = (n0 + 1.0f) * 0.5f;
    normal_vis[3 * lid + 1] = (n1 + 1.0f) * 0.5f;
    normal_vis[3 * lid + 2] = (n2 + 1.0f) * 0.5f;
  }
  if (HAS_RGB && rgb_out) {
    float b0, b1, b2;
    if (P.bkgd_mode == 2) { b0 = bkgd_rand[3 * lid]; b1 = bkgd_rand[3 * lid + 1]; b2 = bkgd_rand[3 * lid + 2]; }
    else { b0 = b1 = b2 = (P.bkgd_mode == 1) ? 1.f : 0.f; }
    float rem = 1.0f - acc;
    float r = fmaf(b0, rem, c_r), g = fmaf(b1, rem, c_g), b = fmaf(b2, rem, c_b);
    if (P.eval_clamp) { r = fminf(fmaxf(r, 0.f), 1.f); g = fminf(fmaxf(g, 0.f), 1.f); b = fminf(fmaxf(b, 0.f), 1.f); }
    rgb_out[3 * lid] = r; rgb_out[3 * lid + 1] = g; rgb_out[3 * lid + 2] = b;
  }
  if (HAS_SEM && sem_out)
    for (int c = 0; c < n_sem; ++c) sem_out[lid * n_sem + c] = sem[c];
}

__global__ void __launch_bounds__(256) field_query_kernel(VolumeDev V, const float* __restrict__ pts, long long n,
                                                          float* __restrict__ sdf_out, float* __restrict__ grad_out,
                                                          float* __restrict__ feat_out) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  float x = pts[3 * i], y = pts[3 * i + 1], z = pts[3 * i + 2];
  float kh, kw, kd;
  Taps t = field_taps(V, x, y, z, kh, kw, kd);
  float sdf, dgh, dgw, dgd;
  gather_sdf(V, t, sdf, dgh, dgw, dgd);
  if (sdf_out) sdf_out[i] = sdf;
  if (grad_out) { grad_out[3 * i] = dgw * kw; grad_out[3 * i + 1] = dgh * kh; grad_out[3 * i + 2] = dgd * kd; }
  if (feat_out)
    for (int c = 0; c < V.n_feat; ++c) { float f1[1]; gather_feat<1>(V, t, c, f1); feat_out[i * V.n_feat + c] = f1[0]; }
}

}  // namespace so

using namespace so;

extern "C" int64_t so_render_workspace_floats(int64_t n_chunks) { return 2 * (n_chunks > 0 ? n_chunks : 1); }

extern "C" int so_render_infer(const float* vol_sdf, const float* vol_feat, const so_volume_desc* vol_host,
                               const float* cam_mats, const float* pix, const so_ray_desc* rd,
                               const so_render_params* pr, const float* bkgd_rand, float* depth, float* max_depth,
                               int64_t* max_idx, float* acc, float* normal_vis, float* rgb, float* sem,
                               float* workspace, void* stream) {
  if (!vol_sdf || !cam_mats || !rd || !pr || !workspace) return SO_ERR_INVALID_ARG;
  int rc = validate_volume(vol_host);
  if (rc) return rc;
  if (rd->n_cam < 1 || rd->rays_per_cam < 1 || pr->num_samples < 1) return SO_ERR_INVALID_ARG;
  if (!pix && (rd->nx < 1 || rd->ny < 1 || (int64_t)rd->nx * rd->ny != rd->rays_per_cam)) return SO_ERR_INVALID_ARG;
  int64_t total = (int64_t)rd->n_cam * rd->rays_per_cam;
  if (rd->ray_begin < 0 || rd->ray_count < 0 || rd->ray_begin + rd->ray_count > total) return SO_ERR_INVALID_ARG;
  bool want_rgb = rgb != nullptr, want_sem = sem != nullptr;
  if (want_rgb && (vol_host->n_feat < 3 || !vol_feat)) return SO_ERR_INVALID_ARG;
  if (want_sem && (vol_host->n_feat <= 3 || !vol_feat || !want_rgb)) return SO_ERR_INVALID_ARG;
  if (want_sem && vol_host->n_feat - 3 > kMaxSem) return SO_ERR_UNSUPPORTED;
  if (pr->bkgd_mode == 2 && want_rgb && !bkgd_rand) return SO_ERR_INVALID_ARG;
  if (pr->bkgd_mode < 0 || pr->bkgd_mode > 2 || pr->sh_act < 0 || pr->sh_act > 1) return SO_ERR_INVALID_ARG;
  if (rd->ray_count == 0) return SO_OK;
  cudaStream_t st = (cudaStream_t)stream;

  VolumeDev V = make_volume(*vol_host, vol_sdf, vol_feat);
  RayDev R;
  if ((rc = make_ray_dev(rd, cam_mats, pix, &R))) return rc;
  RenderDev P = make_render_dev(*pr, nullptr);

  if ((rc = launch_depth_bounds(R, P, workspace, st))) return rc;

  unsigned grid = (unsigned)ceil_div64(rd->ray_count, SO_RENDER_BLOCK);
  ProfScope prof(0, st);
  long long* midx = reinterpret_cast<long long*>(max_idx);
  const bool fast = V.ax[0].k1 == 0.f && V.ax[1].k1 == 0.f && V.ax[2].k1 == 0.f && (P.S & (P.S - 1)) == 0 &&
                    P.cos_anneal == 1.0f && P.anchor_mid;
#define SO_RENDER(RGB, SEM, F) render_infer_kernel<RGB, SEM, F><<<grid, SO_RENDER_BLOCK, 0, st>>>(V, R, P, workspace, bkgd_rand, depth, max_depth, midx, acc, normal_vis, rgb, sem)
  if (want_sem) { if (fast) SO_RENDER(true, true, true); else SO_RENDER(true, true, false); }
  else if (want_rgb) { if (fast) SO_RENDER(true, false, true); else SO_RENDER(true, false, false); }
  else { if (fast) SO_RENDER(false, false, true); else SO_RENDER(false, false, false); }
#undef SO_RENDER
  note_launch(1);
  return check_launch();
}

extern "C" int so_field_query(const float* vol_sdf, const float* vol_feat, const so_volume_desc* vol_host,
                              const float* points, int64_t n, float* sdf, float* grad, float* feat, void* stream) {
  if (!vol_sdf || !points || n < 0) return SO_ERR_INVALID_ARG;
  int rc = validate_volume(vol_host);
  if (rc) return rc;
  if (feat && (vol_host->n_feat < 1 || !vol_feat)) return SO_ERR_INVALID_ARG;
  if (n == 0) return SO_OK;
  VolumeDev V = make_volume(*vol_host, vol_sdf, vol_feat);
  field_query_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, (cudaStream_t)stream>>>(V, points, n, sdf, grad, feat);
  note_launch(1);
  return check_launch();
}
