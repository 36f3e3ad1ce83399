// Self-supervised reprojection loss on the device, forward and backward w.r.t. the per-sample weights
// (loss/reproj_loss_mono_multi_new_combine.py:108-245 and loss/reproj_loss_mono_multi_new.py:117-288).
//
// The reference runs, camera by camera: a batched 4x4 matmul of [R*S, 4, 1] pixel coordinates into the previous and the
// next frame, three to five F.grid_sample calls, five to eight index_add_ segment sums, two or three SSIMs over the
// ray_resize grid and a torch.min.  Here the same loss takes four launches, and the backward three:
//   1. ray stage      thread per (camera, ray): the current image (and, for the automask, the previous and next images)
//                     sampled at the ray pixel;
//   2. sample stage   warp per ray, lanes striding its S contiguous samples: deltas scaling, projection, masks, bilinear
//                     samples of prev / next, per-sample colour terms, and the variant's per-ray weighted sums reduced
//                     in a fixed order (no atomics: bit-reproducible);
//   3. grid stage     thread per (camera, ray) on the ray_resize grid: normalisation by the clamped weight sum, SSIM,
//                     automask terms, the 1e3 rows and the min (first index on ties, as torch.min);
//   4. mean           one CTA: fixed-order mean over rays, then over cameras.
// Backward: SSIM backward on the grid (per-ray partials, then a gather over the 3x3 windows with the reflection pad),
// per-ray coefficients of the weight-sum normalisation, then the sample stage recomputed per sample to write g_weights
// (storing the per-sample projections would cost ~200 MB at the nuScenes size).
//
// Pixel arithmetic follows the reference's op order in fp32: p = T [x t, y t, t, 1], z > 0, division by max(1e-5, z),
// 0 < u < img_size[1], 0 < v < img_size[0]; sampling normalises by img_size, applies 2p - 1 and unnormalises with ATen's
// align_corners=True formula to the image tensor's size.  Combine samples with padding_mode='border', MonoMultiNew with
// the default zeros padding.
#include "common.cuh"
#include <float.h>

namespace so {

constexpr int kSums = 12;    // per-ray sums of the sample stage
constexpr int kGrad = 20;    // per-ray SSIM partials [branch][channel][3] + g_l1 [branch]
constexpr int kCoef = 10;    // per-ray backward coefficients [branch][cl, cx0, cx1, cx2, K]
constexpr float kEps = FLT_EPSILON;   // torch.finfo(torch.float32).eps
constexpr float kC1 = 1e-4f, kC2 = 9e-4f;

struct ReprojDev {
  const float *curr, *prev, *next;   // [N][3][H][W]
  const float* pix;                  // [R][2] (x, y)
  const float *Tp, *Tn;              // [N][4][4]
  const float *w, *ts, *deltas;      // [N][R * S]
  int N, R, S, H, W, gh, gw;
  float sh, sw;                      // img_size (h, w)
  int ssim, automask;
  float *rc, *tp, *tn;               // [N][R][3]
  float* sums;                       // [N][R][kSums]
  float *proj, *choice;              // [N][R]
  float* grad;                       // [N][R][kGrad]
  float* coef;                       // [N][R][kCoef]
};

// Corners and weights of F.grid_sample(img, 2 * (u, v) / img_size - 1, bilinear, align_corners=True) in ATen's arithmetic
struct Bilin {
  long long o;                    // offset of the north-west corner
  bool nw, ne, sw, se;            // corner inside the image
  float wnw, wne, wsw, wse;
};

template <bool BORDER>
__device__ __forceinline__ Bilin bilin(int H, int W, float u, float v, float sw, float sh) {
  const float gx = __fsub_rn(__fmul_rn(2.f, __fdiv_rn(u, sw)), 1.f);
  const float gy = __fsub_rn(__fmul_rn(2.f, __fdiv_rn(v, sh)), 1.f);
  float ix = __fmul_rn(__fdiv_rn(__fadd_rn(gx, 1.f), 2.f), (float)(W - 1));
  float iy = __fmul_rn(__fdiv_rn(__fadd_rn(gy, 1.f), 2.f), (float)(H - 1));
  if (BORDER) {
    ix = fminf((float)(W - 1), fmaxf(ix, 0.f));
    iy = fminf((float)(H - 1), fmaxf(iy, 0.f));
  }
  const float x0f = floorf(ix), y0f = floorf(iy);
  // clamp before the int conversion so far-out samples cannot overflow (every corner is then out of range anyway)
  const int x0 = (int)fminf(fmaxf(x0f, -2.f), (float)W), y0 = (int)fminf(fmaxf(y0f, -2.f), (float)H);
  const float tx = __fsub_rn(ix, x0f), ty = __fsub_rn(iy, y0f);
  const float ux = __fsub_rn(__fadd_rn(x0f, 1.f), ix), uy = __fsub_rn(__fadd_rn(y0f, 1.f), iy);
  const bool bx0 = (unsigned)x0 < (unsigned)W, bx1 = (unsigned)(x0 + 1) < (unsigned)W;
  const bool by0 = (unsigned)y0 < (unsigned)H, by1 = (unsigned)(y0 + 1) < (unsigned)H;
  Bilin b;
  b.o = (long long)y0 * W + x0;
  b.nw = by0 && bx0; b.ne = by0 && bx1; b.sw = by1 && bx0; b.se = by1 && bx1;
  b.wnw = __fmul_rn(ux, uy); b.wne = __fmul_rn(tx, uy); b.wsw = __fmul_rn(ux, ty); b.wse = __fmul_rn(tx, ty);
  return b;
}

// bilinear sample of a planar [3, H, W] image: 12 scattered loads.  A channel-last float4 copy of prev / next (one
// 16-byte load per corner) was measured against it on a B200: 0.54 vs 0.49 ms forward + backward at the nuScenes size
// (the repack of 2 x 6 images of 900 x 1600 costs more than the gathers save, and takes 264 MB), 0.18 vs 0.20 ms at
// the KITTI size; the planar gather is kept.
template <bool BORDER>
__device__ __forceinline__ void sample3(const float* __restrict__ img, int H, int W, float u, float v, float sw, float sh,
                                        float out[3]) {
  const Bilin b = bilin<BORDER>(H, W, u, v, sw, sh);
  const long long plane = (long long)H * W;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float* p = img + c * plane;
    float r = 0.f;
    if (b.nw) r = fmaf(__ldg(p + b.o), b.wnw, r);
    if (b.ne) r = fmaf(__ldg(p + b.o + 1), b.wne, r);
    if (b.sw) r = fmaf(__ldg(p + b.o + W), b.wsw, r);
    if (b.se) r = fmaf(__ldg(p + b.o + W + 1), b.wse, r);
    out[c] = r;
  }
}


// cal_pixel: p = T [x t, y t, t, 1]; mask z > 0 and the pixel strictly inside img_size
__device__ __forceinline__ bool project(const float T[16], float x, float y, float t, float sw, float sh, float& u, float& v) {
  const float c0 = __fmul_rn(x, t), c1 = __fmul_rn(y, t);
  const float p0 = fmaf(T[2], t, fmaf(T[1], c1, __fmul_rn(T[0], c0))) + T[3];
  const float p1 = fmaf(T[6], t, fmaf(T[5], c1, __fmul_rn(T[4], c0))) + T[7];
  const float p2 = fmaf(T[10], t, fmaf(T[9], c1, __fmul_rn(T[8], c0))) + T[11];
  const float z = fmaxf(1e-5f, p2);
  u = __fdiv_rn(p0, z);
  v = __fdiv_rn(p1, z);
  return p2 > 0.f && u > 0.f && u < sw && v > 0.f && v < sh;
}

__device__ __forceinline__ float mean_abs3(const float a[3], const float b[3]) {
  return __fdiv_rn(__fadd_rn(__fadd_rn(fabsf(a[0] - b[0]), fabsf(a[1] - b[1])), fabsf(a[2] - b[2])), 3.f);
}

// w <- (delta < eps ? 0 : w / max(delta, eps)); the factor d w_eff / d w
__device__ __forceinline__ float delta_scale(const float* deltas, long long i) {
  if (!deltas) return 1.f;
  const float d = __ldg(deltas + i);
  return d < kEps ? 0.f : __frcp_rn(fmaxf(d, kEps));
}
__device__ __forceinline__ float eff_weight(const float* deltas, long long i, float w) {
  if (!deltas) return w;
  const float d = __ldg(deltas + i);
  return d < kEps ? 0.f : __fdiv_rn(w, fmaxf(d, kEps));
}

__device__ __forceinline__ void load_T(const float* T, int cam, float out[16]) {
#pragma unroll
  for (int k = 0; k < 16; ++k) out[k] = __ldg(T + cam * 16 + k);
}

// ---- 1. ray stage
template <bool COMBINE>
__global__ void __launch_bounds__(256) reproj_ray_kernel(ReprojDev D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= D.N * D.R) return;
  const int cam = i / D.R, ray = i - cam * D.R;
  const float x = __ldg(D.pix + 2 * ray), y = __ldg(D.pix + 2 * ray + 1);
  const long long img = (long long)cam * 3 * D.H * D.W;
  float c[3];
  sample3<COMBINE>(D.curr + img, D.H, D.W, x, y, D.sw, D.sh, c);
  for (int k = 0; k < 3; ++k) D.rc[3 * i + k] = c[k];
  if (D.automask) {
    sample3<COMBINE>(D.prev + img, D.H, D.W, x, y, D.sw, D.sh, c);
    for (int k = 0; k < 3; ++k) D.tp[3 * i + k] = c[k];
    sample3<COMBINE>(D.next + img, D.H, D.W, x, y, D.sw, D.sh, c);
    for (int k = 0; k < 3; ++k) D.tn[3 * i + k] = c[k];
  }
}

// Per-sample terms of one sample.  Combine: general mask g, diff, composed colour rgbc.  MonoMultiNew: the prev / next
// masks, mean |target - rgb| per branch and the branch colours.
struct SampleTerms {
  bool vp, vn;
  float rp[3], rn[3];
};

template <bool COMBINE>
__device__ __forceinline__ SampleTerms sample_terms(const ReprojDev& D, const float Tp[16], const float Tn[16], int cam, float x,
                                                    float y, float t) {
  SampleTerms s;
  float up, vp, un, vn;
  s.vp = project(Tp, x, y, t, D.sw, D.sh, up, vp);
  s.vn = project(Tn, x, y, t, D.sw, D.sh, un, vn);
  const long long img = (long long)cam * 3 * D.H * D.W;
  // a masked sample contributes nothing in either variant: skip its gathers
  if (s.vp) sample3<COMBINE>(D.prev + img, D.H, D.W, up, vp, D.sw, D.sh, s.rp);
  else s.rp[0] = s.rp[1] = s.rp[2] = 0.f;
  if (s.vn) sample3<COMBINE>(D.next + img, D.H, D.W, un, vn, D.sw, D.sh, s.rn);
  else s.rn[0] = s.rn[1] = s.rn[2] = 0.f;
  return s;
}

// Combine: diff = (dp + dn) / max(cnt, 1), rgbc = (rp + rn) / max(cnt, 1) over the valid branches
__device__ __forceinline__ void combine_terms(const SampleTerms& s, const float rc[3], float& diff, float rgbc[3]) {
  const float cnt = fmaxf((s.vp ? 1.f : 0.f) + (s.vn ? 1.f : 0.f), 1.f);
  const float dp = s.vp ? mean_abs3(rc, s.rp) : 0.f, dn = s.vn ? mean_abs3(rc, s.rn) : 0.f;
  diff = __fdiv_rn(__fadd_rn(dp, dn), cnt);
#pragma unroll
  for (int c = 0; c < 3; ++c) rgbc[c] = __fdiv_rn(__fadd_rn(s.rp[c], s.rn[c]), cnt);
}

// ---- 2. sample stage (forward): warp per ray
// sums, Combine:      [0] sum w', [1] sum w' diff, [2..4] sum w' rgbc, [5] #samples with g
// sums, MonoMultiNew: [0] sum wp, [1] sum wn, [2] sum wp |tc - rp|, [3] sum wn |tc - rn|, [4..6] sum wp rp,
//                     [7..9] sum wn rn, [10] #vp, [11] #vn
template <bool COMBINE>
__global__ void __launch_bounds__(256) reproj_sample_fwd_kernel(ReprojDev D) {
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= (long long)D.N * D.R) return;
  const int cam = (int)(warp / D.R), ray = (int)(warp - (long long)cam * D.R);
  float Tp[16], Tn[16];
  load_T(D.Tp, cam, Tp);
  load_T(D.Tn, cam, Tn);
  const float x = __ldg(D.pix + 2 * ray), y = __ldg(D.pix + 2 * ray + 1);
  float rc[3];
  for (int c = 0; c < 3; ++c) rc[c] = D.rc[3 * warp + c];
  float acc[kSums];
#pragma unroll
  for (int k = 0; k < kSums; ++k) acc[k] = 0.f;
  const long long base = ((long long)cam * D.R + ray) * D.S;
  for (int s = lane; s < D.S; s += 32) {
    const long long i = base + s;
    const float w = eff_weight(D.deltas, i, __ldg(D.w + i));
    const SampleTerms st = sample_terms<COMBINE>(D, Tp, Tn, cam, x, y, __ldg(D.ts + i));
    if (COMBINE) {
      if (!(st.vp || st.vn)) continue;
      float diff, rgbc[3];
      combine_terms(st, rc, diff, rgbc);
      acc[0] += w;
      acc[1] = fmaf(w, diff, acc[1]);
#pragma unroll
      for (int c = 0; c < 3; ++c) acc[2 + c] = fmaf(w, rgbc[c], acc[2 + c]);
      acc[5] += 1.f;
    } else {
      if (st.vp) {
        acc[0] += w;
        acc[2] = fmaf(w, mean_abs3(rc, st.rp), acc[2]);
#pragma unroll
        for (int c = 0; c < 3; ++c) acc[4 + c] = fmaf(w, st.rp[c], acc[4 + c]);
        acc[10] += 1.f;
      }
      if (st.vn) {
        acc[1] += w;
        acc[3] = fmaf(w, mean_abs3(rc, st.rn), acc[3]);
#pragma unroll
        for (int c = 0; c < 3; ++c) acc[7 + c] = fmaf(w, st.rn[c], acc[7 + c]);
        acc[11] += 1.f;
      }
    }
  }
  // fixed-order butterfly: every lane ends with the same, launch-independent sum
#pragma unroll
  for (int k = 0; k < kSums; ++k) {
    float v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    acc[k] = v;
  }
  if (lane < kSums) {
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < kSums; ++k) v = lane == k ? acc[k] : v;
    D.sums[warp * kSums + lane] = v;
  }
}

// ---- SSIM on the ray grid (SSIM module of both reference files, :7-37 / :7-37): reflection pad 1, 3x3 mean,
// clamp((1 - n / d) / 2, 0, 1)
__device__ __forceinline__ int reflect(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

struct SsimStats {
  float mx, my, sx, sy, sxy, n, d, val;
};

// window statistics of one channel at grid pixel (gi, gj); X(r), Y(r) give the channel value at ray r
template <typename FX, typename FY>
__device__ __forceinline__ SsimStats ssim_stats(const ReprojDev& D, int gi, int gj, FX X, FY Y) {
  float ax = 0.f, ay = 0.f, axx = 0.f, ayy = 0.f, axy = 0.f;
  for (int di = -1; di <= 1; ++di) {
    const int ii = reflect(gi + di, D.gh);
    for (int dj = -1; dj <= 1; ++dj) {
      const int r = ii * D.gw + reflect(gj + dj, D.gw);
      const float x = X(r), y = Y(r);
      ax += x; ay += y;
      axx += __fmul_rn(x, x); ayy += __fmul_rn(y, y); axy += __fmul_rn(x, y);
    }
  }
  SsimStats s;
  s.mx = __fdiv_rn(ax, 9.f); s.my = __fdiv_rn(ay, 9.f);
  s.sx = __fsub_rn(__fdiv_rn(axx, 9.f), __fmul_rn(s.mx, s.mx));
  s.sy = __fsub_rn(__fdiv_rn(ayy, 9.f), __fmul_rn(s.my, s.my));
  s.sxy = __fsub_rn(__fdiv_rn(axy, 9.f), __fmul_rn(s.mx, s.my));
  s.n = __fmul_rn(__fadd_rn(__fmul_rn(__fmul_rn(2.f, s.mx), s.my), kC1), __fadd_rn(__fmul_rn(2.f, s.sxy), kC2));
  s.d = __fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(s.mx, s.mx), __fmul_rn(s.my, s.my)), kC1),
                  __fadd_rn(__fadd_rn(s.sx, s.sy), kC2));
  s.val = __fdiv_rn(__fsub_rn(1.f, __fdiv_rn(s.n, s.d)), 2.f);
  return s;
}

// mean over the three channels of SSIM(pred, target) at ray r; P(c, r), T(c, r) give the channel values
template <typename FP, typename FT>
__device__ __forceinline__ float ssim_mean(const ReprojDev& D, int r, FP P, FT T) {
  const int gi = r / D.gw, gj = r - gi * D.gw;
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const SsimStats st = ssim_stats(D, gi, gj, [&](int q) { return P(c, q); }, [&](int q) { return T(c, q); });
    s += fminf(fmaxf(st.val, 0.f), 1.f);
  }
  return __fdiv_rn(s, 3.f);
}

// composed colour of branch b at ray r of camera cam: C_b / max(A_b, eps)
template <bool COMBINE>
__device__ __forceinline__ float composed(const ReprojDev& D, int cam, int b, int c, int r) {
  const float* s = D.sums + ((long long)cam * D.R + r) * kSums;
  if (COMBINE) return __fdiv_rn(s[2 + c], fmaxf(s[0], kEps));
  return __fdiv_rn(s[4 + 3 * b + c], fmaxf(s[b], kEps));
}

// mask_{prev,next}_proj_loss: 0.85 ssim(target, rc) + 0.15 mean |rc - target| (or the l1 term alone)
__device__ __forceinline__ float automask_loss(const ReprojDev& D, int cam, const float* tgt, int r) {
  const float* rc = D.rc + (long long)cam * D.R * 3;
  const float* t = tgt + (long long)cam * D.R * 3;
  const float l1 = mean_abs3(rc + 3 * r, t + 3 * r);
  if (!D.ssim) return l1;
  const float s = ssim_mean(D, r, [&](int c, int q) { return t[3 * q + c]; }, [&](int c, int q) { return rc[3 * q + c]; });
  return __fadd_rn(__fmul_rn(0.85f, s), __fmul_rn(0.15f, l1));
}

// ---- 3. grid stage: per-ray loss and the chosen branch
// choice, Combine:      0 prev_next, 1 automask prev, 2 automask next
// choice, MonoMultiNew: 0 prev, 1 next, 2 automask prev, 3 automask next
template <bool COMBINE>
__global__ void __launch_bounds__(256) reproj_grid_fwd_kernel(ReprojDev D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= D.N * D.R) return;
  const int cam = i / D.R, r = i - cam * D.R;
  const float* s = D.sums + (long long)i * kSums;
  const float* rc = D.rc + (long long)cam * D.R * 3;
  float cand[4];
  int nb;
  if (COMBINE) {
    const float l1 = __fdiv_rn(s[1], fmaxf(s[0], kEps));
    float pn = l1;
    if (D.ssim) {
      const float ss = ssim_mean(D, r, [&](int c, int q) { return composed<true>(D, cam, 0, c, q); },
                                 [&](int c, int q) { return rc[3 * q + c]; });
      pn = __fadd_rn(__fmul_rn(0.15f, l1), __fmul_rn(0.85f, ss));
    }
    cand[0] = pn;
    nb = 1;
    if (D.automask && s[5] == 0.f) cand[0] = 1e3f;
  } else {
    for (int b = 0; b < 2; ++b) {
      const float l1 = __fdiv_rn(s[2 + b], fmaxf(s[b], kEps));
      float v = l1;
      if (D.ssim) {
        const float ss = ssim_mean(D, r, [&](int c, int q) { return composed<false>(D, cam, b, c, q); },
                                   [&](int c, int q) { return rc[3 * q + c]; });
        v = __fadd_rn(__fmul_rn(0.85f, ss), __fmul_rn(0.15f, l1));
      }
      cand[b] = s[10 + b] == 0.f ? 1e3f : v;
    }
    nb = 2;
  }
  if (D.automask) {
    cand[nb] = automask_loss(D, cam, D.tp, r);
    cand[nb + 1] = automask_loss(D, cam, D.tn, r);
    nb += 2;
  }
  int k = 0;
  for (int j = 1; j < nb; ++j)
    if (cand[j] < cand[k]) k = j;     // strict: the first index wins ties, as torch.min
  D.proj[i] = cand[k];
  D.choice[i] = (float)k;
}

// ---- 4. mean over rays, then over cameras; one CTA, fixed order
constexpr int kMeanThreads = 1024;
__global__ void __launch_bounds__(kMeanThreads) reproj_mean_kernel(const float* __restrict__ proj, int N, int R, float* loss) {
  __shared__ float sm[kMeanThreads / 32];
  float tot = 0.f;
  for (int cam = 0; cam < N; ++cam) {
    float v = 0.f;
    for (int r = threadIdx.x; r < R; r += kMeanThreads) v += proj[(long long)cam * R + r];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      float c = 0.f;
      for (int k = 0; k < kMeanThreads / 32; ++k) c += sm[k];
      tot += __fdiv_rn(c, (float)R);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) loss[0] = __fdiv_rn(tot, (float)N);
}

// ---- backward
// SSIM partials at grid pixel r for one branch: d S_c / d (mu_x, E[x^2], E[xy]) times the upstream gS / 3, zero where
// the clamp is active (torch.clamp passes the gradient on [0, 1] inclusive)
template <typename FX, typename FY>
__device__ __forceinline__ void ssim_partials(const ReprojDev& D, int r, float gS, FX X, FY Y, float* out /*[9]*/) {
  const int gi = r / D.gw, gj = r - gi * D.gw;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const SsimStats st = ssim_stats(D, gi, gj, [&](int q) { return X(c, q); }, [&](int q) { return Y(c, q); });
    float a = 0.f, bxx = 0.f, bxy = 0.f;
    if (gS != 0.f && st.val >= 0.f && st.val <= 1.f) {
      const float A1 = 2.f * st.mx * st.my + kC1, A2 = 2.f * st.sxy + kC2;
      const float B1 = st.mx * st.mx + st.my * st.my + kC1, B2 = st.sx + st.sy + kC2;
      // n = A1 A2, d = B1 B2 with A2 = 2 (E[xy] - mx my) + C2, B2 = E[x^2] - mx^2 + E[y^2] - my^2 + C2
      const float dn_dmx = 2.f * st.my * A2 - 2.f * st.my * A1, dd_dmx = 2.f * st.mx * B2 - 2.f * st.mx * B1;
      const float inv_d = 1.f / st.d, q = st.n * inv_d;
      const float g = -0.5f * gS / 3.f;                  // S = (1 - n / d) / 2, mean over 3 channels
      a = g * (dn_dmx - q * dd_dmx) * inv_d;             // d(n/d)/d mx
      bxx = g * (-q * B1) * inv_d;                       // d(n/d)/d E[x^2]
      bxy = g * (2.f * A1) * inv_d;                      // d(n/d)/d E[xy]
    }
    out[3 * c] = a; out[3 * c + 1] = bxx; out[3 * c + 2] = bxy;
  }
}

// grid backward, part 1 (per output pixel): upstream gradient of the chosen branch, SSIM partials, g_l1
template <bool COMBINE>
__global__ void __launch_bounds__(256) reproj_grid_bwd1_kernel(ReprojDev D, const float* __restrict__ g_loss) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= D.N * D.R) return;
  const int cam = i / D.R, r = i - cam * D.R;
  const float* s = D.sums + (long long)i * kSums;
  const float* rc = D.rc + (long long)cam * D.R * 3;
  const float gp = __fdiv_rn(__fdiv_rn(__ldg(g_loss), (float)D.N), (float)D.R);
  const int k = (int)D.choice[i];
  float* out = D.grad + (long long)i * kGrad;
  for (int b = 0; b < 2; ++b) {
    // the branch carries gradient iff it was chosen and is not a constant 1e3 row
    bool live;
    if (COMBINE) live = b == 0 && k == 0 && !(D.automask && s[5] == 0.f);
    else live = k == b && s[10 + b] != 0.f;
    const float g = live ? gp : 0.f;
    out[18 + b] = D.ssim ? 0.15f * g : g;
    if (D.ssim && (COMBINE ? b == 0 : true))
      ssim_partials(D, r, 0.85f * g, [&](int c, int q) { return composed<COMBINE>(D, cam, b, c, q); },
                    [&](int c, int q) { return rc[3 * q + c]; }, out + 9 * b);
    else
      for (int j = 0; j < 9; ++j) out[9 * b + j] = 0.f;
  }
}

// grid backward, part 2 (per source ray): gather the SSIM partials of every window that covers the ray (the reflection
// pad can cover it twice), then the coefficients of g_w' = cl diff + sum_c cx_c rgb_c - K per branch, from
// l1 = sum w' diff / ws, x_c = sum w' rgb_c / ws, ws = max(sum w', eps)
template <bool COMBINE>
__global__ void __launch_bounds__(256) reproj_grid_bwd2_kernel(ReprojDev D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= D.N * D.R) return;
  const int cam = i / D.R, r = i - cam * D.R;
  const float* s = D.sums + (long long)i * kSums;
  const float* rc = D.rc + 3LL * i;
  const int nbr = COMBINE ? 1 : 2;
  for (int b = 0; b < 2; ++b) {
    float* co = D.coef + (long long)i * kCoef + 5 * b;
    if (b >= nbr) { for (int j = 0; j < 5; ++j) co[j] = 0.f; continue; }
    float gx[3] = {0.f, 0.f, 0.f};
    float x[3];
    for (int c = 0; c < 3; ++c) x[c] = composed<COMBINE>(D, cam, b, c, r);
    if (D.ssim) {
      const int gi = r / D.gw, gj = r - gi * D.gw;
      float pa[3] = {0.f, 0.f, 0.f}, pxx[3] = {0.f, 0.f, 0.f}, pxy[3] = {0.f, 0.f, 0.f};
      for (int oi = max(gi - 2, 0); oi <= min(gi + 2, D.gh - 1); ++oi)
        for (int di = -1; di <= 1; ++di) {
          if (reflect(oi + di, D.gh) != gi) continue;
          for (int oj = max(gj - 2, 0); oj <= min(gj + 2, D.gw - 1); ++oj)
            for (int dj = -1; dj <= 1; ++dj) {
              if (reflect(oj + dj, D.gw) != gj) continue;
              const float* G = D.grad + ((long long)cam * D.R + oi * D.gw + oj) * kGrad + 9 * b;
              for (int c = 0; c < 3; ++c) { pa[c] += G[3 * c]; pxx[c] += G[3 * c + 1]; pxy[c] += G[3 * c + 2]; }
            }
        }
      for (int c = 0; c < 3; ++c) gx[c] = (pa[c] + 2.f * x[c] * pxx[c] + rc[c] * pxy[c]) / 9.f;
    }
    const float gl1 = D.grad[(long long)i * kGrad + 18 + b];
    const float A = COMBINE ? s[0] : s[b];
    const float L = COMBINE ? s[1] : s[2 + b];
    const float inv_ws = 1.f / fmaxf(A, kEps);
    const float l1 = __fdiv_rn(L, fmaxf(A, kEps));
    float K = gl1 * l1 + gx[0] * x[0] + gx[1] * x[1] + gx[2] * x[2];
    K = A >= kEps ? K * inv_ws : 0.f;                    // clamp_min passes the gradient where sum >= eps
    co[0] = gl1 * inv_ws;
    for (int c = 0; c < 3; ++c) co[1 + c] = gx[c] * inv_ws;
    co[4] = K;
  }
}

// sample backward: thread per sample, recomputes the sample stage and writes g_weights
template <bool COMBINE>
__global__ void __launch_bounds__(256) reproj_sample_bwd_kernel(ReprojDev D, float* __restrict__ g_w) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long n = (long long)D.N * D.R * D.S;
  if (i >= n) return;
  const long long rr = i / D.S;
  const int cam = (int)(rr / D.R), ray = (int)(rr - (long long)cam * D.R);
  float co[kCoef];
  bool any = false;
#pragma unroll
  for (int k = 0; k < kCoef; ++k) { co[k] = D.coef[rr * kCoef + k]; any |= co[k] != 0.f; }
  const float ds = delta_scale(D.deltas, i);
  if (!any || ds == 0.f) { g_w[i] = 0.f; return; }
  float Tp[16], Tn[16];
  load_T(D.Tp, cam, Tp);
  load_T(D.Tn, cam, Tn);
  const float x = __ldg(D.pix + 2 * ray), y = __ldg(D.pix + 2 * ray + 1);
  float rc[3];
  for (int c = 0; c < 3; ++c) rc[c] = D.rc[3 * rr + c];
  const SampleTerms st = sample_terms<COMBINE>(D, Tp, Tn, cam, x, y, __ldg(D.ts + i));
  float g = 0.f;
  if (COMBINE) {
    if (st.vp || st.vn) {
      float diff, rgbc[3];
      combine_terms(st, rc, diff, rgbc);
      g = co[0] * diff + co[1] * rgbc[0] + co[2] * rgbc[1] + co[3] * rgbc[2] - co[4];
    }
  } else {
    if (st.vp) g += co[0] * mean_abs3(rc, st.rp) + co[1] * st.rp[0] + co[2] * st.rp[1] + co[3] * st.rp[2] - co[4];
    if (st.vn) g += co[5] * mean_abs3(rc, st.rn) + co[6] * st.rn[0] + co[7] * st.rn[1] + co[8] * st.rn[2] - co[9];
  }
  g_w[i] = g * ds;
}

__global__ void reproj_layout_kernel(const long long* __restrict__ idx, long long n, int S, int* bad) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n && __ldg(idx + i) != i / S) atomicOr(bad, 1);
}

int64_t ws_floats(const so_reproj_desc& d) {
  return (int64_t)d.n_cam * d.n_rays * (9 + kSums + 2 + kGrad + kCoef);
}

int validate(const so_reproj_desc* d) {
  if (!d) return SO_ERR_INVALID_ARG;
  if (d->variant != SO_REPROJ_COMBINE && d->variant != SO_REPROJ_MONO_MULTI_NEW) return SO_ERR_INVALID_ARG;
  if (d->n_cam < 1 || d->n_rays < 1 || d->n_samples < 1 || d->img_h < 1 || d->img_w < 1) return SO_ERR_INVALID_ARG;
  if (!(d->size_h > 0.f) || !(d->size_w > 0.f)) return SO_ERR_INVALID_ARG;
  if (d->ssim && (d->grid_h < 2 || d->grid_w < 2 || (int64_t)d->grid_h * d->grid_w != d->n_rays)) return SO_ERR_INVALID_ARG;
  if ((int64_t)d->n_cam * d->n_rays >= ((int64_t)1 << 26)) return SO_ERR_UNSUPPORTED;   // warp-per-ray grid in 32 bits
  return SO_OK;
}

ReprojDev make_dev(const so_reproj_desc& d, const float* curr, const float* prev, const float* next, const float* pix,
                   const float* img2prev, const float* img2next, const float* weights, const float* ts, const float* deltas,
                   float* ws) {
  ReprojDev D;
  D.curr = curr; D.prev = prev; D.next = next; D.pix = pix; D.Tp = img2prev; D.Tn = img2next;
  D.w = weights; D.ts = ts; D.deltas = deltas;
  D.N = d.n_cam; D.R = d.n_rays; D.S = d.n_samples; D.H = d.img_h; D.W = d.img_w;
  D.gh = d.grid_h; D.gw = d.grid_w; D.sh = d.size_h; D.sw = d.size_w;
  D.ssim = d.ssim ? 1 : 0; D.automask = d.automask ? 1 : 0;
  const int64_t nr = (int64_t)d.n_cam * d.n_rays;
  D.rc = ws; D.tp = D.rc + 3 * nr; D.tn = D.tp + 3 * nr;
  D.sums = D.tn + 3 * nr;
  D.proj = D.sums + kSums * nr; D.choice = D.proj + nr;
  D.grad = D.choice + nr;
  D.coef = D.grad + kGrad * nr;
  return D;
}

}  // namespace so

using namespace so;

extern "C" int64_t so_reproj_workspace_floats(const so_reproj_desc* desc_host) {
  if (validate(desc_host)) return -1;
  return ws_floats(*desc_host);
}

extern "C" int so_reproj_forward(const so_reproj_desc* desc_host, const float* curr, const float* prev, const float* next,
                                 const float* pix, const float* img2prev, const float* img2next, const float* weights,
                                 const float* ts, const float* deltas, float* loss, float* workspace, void* stream) {
  int rc = validate(desc_host);
  if (rc) return rc;
  if (!curr || !prev || !next || !pix || !img2prev || !img2next || !weights || !ts || !loss || !workspace)
    return SO_ERR_INVALID_ARG;
  const so_reproj_desc& d = *desc_host;
  ReprojDev D = make_dev(d, curr, prev, next, pix, img2prev, img2next, weights, ts, deltas, workspace);
  const int nr = d.n_cam * d.n_rays;
  const unsigned g_ray = (unsigned)ceil_div64(nr, 256), g_warp = (unsigned)ceil_div64((int64_t)nr * 32, 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (d.variant == SO_REPROJ_COMBINE) {
    reproj_ray_kernel<true><<<g_ray, 256, 0, st>>>(D);
    reproj_sample_fwd_kernel<true><<<g_warp, 256, 0, st>>>(D);
    reproj_grid_fwd_kernel<true><<<g_ray, 256, 0, st>>>(D);
  } else {
    reproj_ray_kernel<false><<<g_ray, 256, 0, st>>>(D);
    reproj_sample_fwd_kernel<false><<<g_warp, 256, 0, st>>>(D);
    reproj_grid_fwd_kernel<false><<<g_ray, 256, 0, st>>>(D);
  }
  reproj_mean_kernel<<<1, kMeanThreads, 0, st>>>(D.proj, d.n_cam, d.n_rays, loss);
  note_launch(4);
  return check_launch();
}

extern "C" int so_reproj_backward(const so_reproj_desc* desc_host, const float* curr, const float* prev, const float* next,
                                  const float* pix, const float* img2prev, const float* img2next, const float* weights,
                                  const float* ts, const float* deltas, const float* g_loss, float* g_weights, float* workspace,
                                  void* stream) {
  int rc = validate(desc_host);
  if (rc) return rc;
  if (!curr || !prev || !next || !pix || !img2prev || !img2next || !weights || !ts || !g_loss || !g_weights || !workspace)
    return SO_ERR_INVALID_ARG;
  const so_reproj_desc& d = *desc_host;
  ReprojDev D = make_dev(d, curr, prev, next, pix, img2prev, img2next, weights, ts, deltas, workspace);
  const int nr = d.n_cam * d.n_rays;
  const int64_t ns = (int64_t)nr * d.n_samples;
  const unsigned g_ray = (unsigned)ceil_div64(nr, 256), g_smp = (unsigned)ceil_div64(ns, 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (d.variant == SO_REPROJ_COMBINE) {
    reproj_grid_bwd1_kernel<true><<<g_ray, 256, 0, st>>>(D, g_loss);
    reproj_grid_bwd2_kernel<true><<<g_ray, 256, 0, st>>>(D);
    reproj_sample_bwd_kernel<true><<<g_smp, 256, 0, st>>>(D, g_weights);
  } else {
    reproj_grid_bwd1_kernel<false><<<g_ray, 256, 0, st>>>(D, g_loss);
    reproj_grid_bwd2_kernel<false><<<g_ray, 256, 0, st>>>(D);
    reproj_sample_bwd_kernel<false><<<g_smp, 256, 0, st>>>(D, g_weights);
  }
  note_launch(3);
  return check_launch();
}

extern "C" int so_reproj_check_layout(const int64_t* ray_idx, int64_t n, int32_t n_samples, int32_t* bad, void* stream) {
  if (!ray_idx || !bad || n < 0 || n_samples < 1) return SO_ERR_INVALID_ARG;
  if (n == 0) return SO_OK;
  reproj_layout_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const long long*>(ray_idx), n, n_samples, bad);
  note_launch(1);
  return check_launch();
}
