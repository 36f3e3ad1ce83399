// Device functions shared by the inference and training render kernels (render.cu, render_train.cu).
#pragma once
#include "common.cuh"
#include <math.h>

namespace so {

struct RayDev {
  const float* cam;  // [n_cam][16]
  const float* pix;  // [rays_per_cam][2] or nullptr
  int n_cam, rays_per_cam, nx;
  float sx, ox, sy, oy;
  long long ray_begin, ray_count, total, chunk_len;
};

struct RenderDev {
  float lo[3], hi[3];
  float near_clamp;
  int S;
  float inv_s, cos_anneal;
  int anchor_mid, sh_act, bkgd_mode, eval_clamp;
  const float* jitter;  // [total rays][S + 1] stratified-sampling uniforms (training) or nullptr
};

inline RenderDev make_render_dev(const so_render_params& pr, const float* jitter) {
  RenderDev P;
  for (int a = 0; a < 3; ++a) { P.lo[a] = pr.aabb[a]; P.hi[a] = pr.aabb[3 + a]; }
  P.near_clamp = pr.training ? pr.near_plane : 0.f;
  P.S = pr.num_samples; P.inv_s = pr.inv_s; P.cos_anneal = pr.cos_anneal;
  P.anchor_mid = pr.anchor_mid; P.sh_act = pr.sh_act; P.bkgd_mode = pr.bkgd_mode; P.eval_clamp = pr.training ? 0 : 1;
  P.jitter = jitter;
  return P;
}

inline int make_ray_dev(const so_ray_desc* rd, const float* cam_mats, const float* pix, RayDev* out) {
  if (rd->n_cam < 1 || rd->rays_per_cam < 1) return SO_ERR_INVALID_ARG;
  if (!pix && (rd->nx < 1 || rd->ny < 1 || (int64_t)rd->nx * rd->ny != rd->rays_per_cam)) return SO_ERR_INVALID_ARG;
  int64_t total = (int64_t)rd->n_cam * rd->rays_per_cam;
  if (rd->ray_begin < 0 || rd->ray_count < 0 || rd->ray_begin + rd->ray_count > total) return SO_ERR_INVALID_ARG;
  RayDev R;
  R.cam = cam_mats; R.pix = pix; R.n_cam = rd->n_cam; R.rays_per_cam = rd->rays_per_cam; R.nx = rd->nx > 0 ? rd->nx : 1;
  R.sx = rd->sx; R.ox = rd->ox; R.sy = rd->sy; R.oy = rd->oy;
  R.ray_begin = rd->ray_begin; R.ray_count = rd->ray_count; R.total = total;
  R.chunk_len = rd->chunk_len > 0 ? rd->chunk_len : 0;
  *out = R;
  return SO_OK;
}

__device__ __forceinline__ void make_ray(const RayDev& R, long long gid, float o[3], float d[3], float& nrm) {
  int cam = (int)(gid / R.rays_per_cam);
  int r = (int)(gid - (long long)cam * R.rays_per_cam);
  float px, py;
  if (R.pix) {
    px = __ldg(R.pix + 2 * r);
    py = __ldg(R.pix + 2 * r + 1);
  } else {
    int i = r / R.nx, j = r - i * R.nx;
    px = __fadd_rn(__fmul_rn((float)j, R.sx), R.ox);  // ray_sampler.py:24-25,65-66 (mul then add)
    py = __fadd_rn(__fmul_rn((float)i, R.sy), R.oy);
  }
  const float* M = R.cam + cam * 16;
  float dx = __ldg(M + 0) * px + __ldg(M + 1) * py + __ldg(M + 2);
  float dy = __ldg(M + 4) * px + __ldg(M + 5) * py + __ldg(M + 6);
  float dz = __ldg(M + 8) * px + __ldg(M + 9) * py + __ldg(M + 10);
  o[0] = __ldg(M + 3); o[1] = __ldg(M + 7); o[2] = __ldg(M + 11);
  nrm = sqrtf(dx * dx + dy * dy + dz * dz);
  d[0] = dx / nrm; d[1] = dy / nrm; d[2] = dz / nrm;
}

// upstream AABBBoxCollider: slab test with 1/(d + 1e-6)
__device__ __forceinline__ void slab(const RenderDev& P, const float o[3], const float d[3], float& tn, float& tf) {
  float nmax = -INFINITY, fmin = INFINITY;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float inv = 1.0f / (d[a] + 1e-6f);
    float t1 = (P.lo[a] - o[a]) * inv, t2 = (P.hi[a] - o[a]) * inv;
    nmax = fmaxf(nmax, fminf(t1, t2));
    fmin = fminf(fmin, fmaxf(t1, t2));
  }
  tn = fmaxf(nmax, P.near_clamp);
  tf = fmaxf(fmin, tn + 1e-6f);
}

// torch.linspace(0, 1, S + 1)[i] in fp32 (two-sided evaluation like ATen's CPU kernel)
__device__ __forceinline__ float bin_edge01(int i, int S, float step) {
  return (i < (S + 1) / 2) ? __fmul_rn(step, (float)i) : __fsub_rn(1.0f, __fmul_rn(step, (float)(S - i)));
}
__device__ __forceinline__ float edge_t(float b, float tn, float tf) {
  return __fadd_rn(__fmul_rn(b, tf), __fmul_rn(__fsub_rn(1.0f, b), tn));
}
// upstream UniformSampler with train_stratified: edge i is re-drawn inside its half-cell,
// bins = lower + (upper - lower) * u_i with lower/upper the neighbouring bin centres (u = NULL: no jitter)
__device__ __forceinline__ float bin_edge01_jit(int i, int S, float step, const float* __restrict__ u) {
  float bi = bin_edge01(i, S, step);
  if (!u) return bi;
  float lower = bi, upper = bi;
  if (i > 0) lower = __fmul_rn(__fadd_rn(bi, bin_edge01(i - 1, S, step)), 0.5f);
  if (i < S) upper = __fmul_rn(__fadd_rn(bin_edge01(i + 1, S, step), bi), 0.5f);
  return __fadd_rn(lower, __fmul_rn(__fsub_rn(upper, lower), __ldg(u + i)));
}


// ---- trilinear sdf + analytic gradient (w.r.t. grid coords) ------------------------------------------
__device__ __forceinline__ void gather_sdf(const VolumeDev& v, const Taps& t, float& s, float& dgh, float& dgw,
                                           float& dgd) {
  int h0 = min(max(t.h0, 0), v.H - 1), h1 = min(max(t.h0 + 1, 0), v.H - 1);
  int w0 = min(max(t.w0, 0), v.W - 1), w1 = min(max(t.w0 + 1, 0), v.W - 1);
  int z0 = min(max(t.z0, 0), v.Z - 1), z1 = min(max(t.z0 + 1, 0), v.Z - 1);
  const float* p00 = v.sdf + ((size_t)h0 * v.W + w0) * v.zpitch;
  const float* p01 = v.sdf + ((size_t)h0 * v.W + w1) * v.zpitch;
  const float* p10 = v.sdf + ((size_t)h1 * v.W + w0) * v.zpitch;
  const float* p11 = v.sdf + ((size_t)h1 * v.W + w1) * v.zpitch;
  float a000 = __ldg(p00 + z0), a001 = __ldg(p00 + z1);
  float a010 = __ldg(p01 + z0), a011 = __ldg(p01 + z1);
  float a100 = __ldg(p10 + z0), a101 = __ldg(p10 + z1);
  float a110 = __ldg(p11 + z0), a111 = __ldg(p11 + z1);
  float m00 = t.mh0 * t.mw0, m01 = t.mh0 * t.mw1, m10 = t.mh1 * t.mw0, m11 = t.mh1 * t.mw1;
  a000 *= m00 * t.mz0; a001 *= m00 * t.mz1;
  a010 *= m01 * t.mz0; a011 *= m01 * t.mz1;
  a100 *= m10 * t.mz0; a101 *= m10 * t.mz1;
  a110 *= m11 * t.mz0; a111 *= m11 * t.mz1;
  float dz00 = a001 - a000, dz01 = a011 - a010, dz10 = a101 - a100, dz11 = a111 - a110;
  float c00 = fmaf(t.fz, dz00, a000), c01 = fmaf(t.fz, dz01, a010);
  float c10 = fmaf(t.fz, dz10, a100), c11 = fmaf(t.fz, dz11, a110);
  float dw0 = c01 - c00, dw1 = c11 - c10;
  float c0 = fmaf(t.fw, dw0, c00), c1 = fmaf(t.fw, dw1, c10);
  float dz0 = fmaf(t.fw, dz01 - dz00, dz00), dz1 = fmaf(t.fw, dz11 - dz10, dz10);
  dgh = c1 - c0;
  s = fmaf(t.fh, dgh, c0);
  dgw = fmaf(t.fh, dw1 - dw0, dw0);
  dgd = fmaf(t.fh, dz1 - dz0, dz0);
}

// tap set of the field query at one point in metres (so_field_query; the occupancy lattice nodes of occupancy.cu)
__device__ __forceinline__ Taps field_taps(const VolumeDev& V, float x, float y, float z, float& kh, float& kw, float& kd) {
  float gh = axis_m2g(V.ax[0], y, kh), gw = axis_m2g(V.ax[1], x, kw), gd = axis_m2g(V.ax[2], z, kd);
  return make_taps(V, gh, gw, gd);
}

// interior fast path: all 8 corners inside the volume (true for every sample strictly inside the AABB)
__device__ __forceinline__ void gather_sdf_interior(const VolumeDev& v, int h0, int w0, int z0, float fh, float fw,
                                                    float fz, float& s, float& dgh, float& dgw, float& dgd) {
  const int zp = v.zpitch;
  const float* p00 = v.sdf + ((h0 * v.W + w0) * zp + z0);
  const float* p01 = p00 + zp;
  const float* p10 = p00 + v.W * zp;
  const float* p11 = p10 + zp;
  float a000 = __ldg(p00), a001 = __ldg(p00 + 1);
  float a010 = __ldg(p01), a011 = __ldg(p01 + 1);
  float a100 = __ldg(p10), a101 = __ldg(p10 + 1);
  float a110 = __ldg(p11), a111 = __ldg(p11 + 1);
  float dz00 = a001 - a000, dz01 = a011 - a010, dz10 = a101 - a100, dz11 = a111 - a110;
  float c00 = fmaf(fz, dz00, a000), c01 = fmaf(fz, dz01, a010);
  float c10 = fmaf(fz, dz10, a100), c11 = fmaf(fz, dz11, a110);
  float dw0 = c01 - c00, dw1 = c11 - c10;
  float c0 = fmaf(fw, dw0, c00), c1 = fmaf(fw, dw1, c10);
  float dz0 = fmaf(fw, dz01 - dz00, dz00), dz1 = fmaf(fw, dz11 - dz10, dz10);
  dgh = c1 - c0;
  s = fmaf(fh, dgh, c0);
  dgw = fmaf(fh, dw1 - dw0, dw0);
  dgd = fmaf(fh, dz1 - dz0, dz0);
}

// trilinear gather of `n` consecutive feature channels starting at `c0` (channel-last volume)
template <int N>
__device__ __forceinline__ void gather_feat(const VolumeDev& v, const Taps& t, int c0, float out[N]) {
#pragma unroll
  for (int i = 0; i < N; ++i) out[i] = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    int dh = k >> 2, dw = (k >> 1) & 1, dz = k & 1;
    float wgt = (dh ? t.fh * t.mh1 : (1.f - t.fh) * t.mh0) * (dw ? t.fw * t.mw1 : (1.f - t.fw) * t.mw0) *
                (dz ? t.fz * t.mz1 : (1.f - t.fz) * t.mz0);
    int h = min(max(t.h0 + dh, 0), v.H - 1), w = min(max(t.w0 + dw, 0), v.W - 1), z = min(max(t.z0 + dz, 0), v.Z - 1);
    const float* p = v.feat + (((size_t)h * v.W + w) * v.Z + z) * v.feat_pitch + c0;
#pragma unroll
    for (int i = 0; i < N; ++i) out[i] = fmaf(wgt, __ldg(p + i), out[i]);
  }
}

// sigmoid via one ex2.approx + one rcp.approx (abs error ~1e-7): exp(-|x|) never overflows
__device__ __forceinline__ float sigmoid_fast(float x) {
  // exp(-x) may overflow to +inf for very negative x; rcp.approx(inf) = 0 is the correct limit
  return __fdividef(1.0f, 1.0f + __expf(-x));
}
__device__ __forceinline__ float sigmoidf_acc(float x) {
  float e = expf(-fabsf(x));
  float s = 1.0f / (1.0f + e);
  return x >= 0.f ? s : e * s;
}

// 1 - exp(-x) for x >= 0 with ~1e-6 relative accuracy: 5-term series below 1/8, ex2.approx above
__device__ __forceinline__ float one_minus_exp_neg(float x) {
  float ser = x * (1.0f - x * 0.5f * (1.0f - x * (1.0f / 3.0f) * (1.0f - x * 0.25f * (1.0f - x * 0.2f))));
  float big = 1.0f - __expf(-x);
  return x < 0.125f ? ser : big;
}

// NeuS alpha = clip((Phi(prev) - Phi(next) + 1e-5) / (Phi(prev) + 1e-5), 0, 1) with Phi = sigmoid(inv_s * .),
// prev = sdf - half, next = sdf + half (half <= 0).  The difference of the two CDFs is evaluated without
// cancellation:  Phi(a) - Phi(b) = Phi(a) * Phi(-b) * (1 - exp(-(a - b))),  a - b = -2 * half * inv_s >= 0,
// which keeps fp32 within rounding of the fp64 evaluation of the reference formula (the reference's own fp32
// evaluation loses ~3 digits to cancellation here).  Every exponential is taken in base 2:
// s2 = sdf * inv_s * log2(e), h2 = half * inv_s * log2(e) (<= 0), so each logistic is one ex2.approx + one rcp.approx.
__device__ __forceinline__ float neus_alpha_log2(float s2, float h2) {
  float pa = __fdividef(1.0f, 1.0f + exp2f(h2 - s2));           // Phi(prev) = 1 / (1 + 2^-(s2 - h2))
  float qb = __fdividef(1.0f, 1.0f + exp2f(s2 + h2));           // Phi(-next)
  float x = h2 * (-2.0f * 0.6931471805599453f);                 // a - b in natural units (>= 0)
#ifdef SO_ALPHA_HORNER
  float ser = x * fmaf(x, fmaf(x, fmaf(x, fmaf(x, 1.0f / 120.0f, -1.0f / 24.0f), 1.0f / 6.0f), -0.5f), 1.0f);   // same polynomial, 5 ops
#else
  float ser = x * (1.0f - x * 0.5f * (1.0f - x * (1.0f / 3.0f) * (1.0f - x * 0.25f * (1.0f - x * 0.2f))));
#endif
  float omen = x < 0.125f ? ser : 1.0f - exp2f(2.0f * h2);
  return __saturatef(__fdividef(fmaf(pa * qb, omen, 1e-5f), pa + 1e-5f));
}

constexpr float kC0 = 0.28209479177387814f;  // sh_render.py:4

constexpr int kMaxSem = 32;  // rendered semantic classes (n_feat - 3) supported per ray

int launch_depth_bounds(const RayDev& R, const RenderDev& P, float* ws, cudaStream_t st);

}  // namespace so
