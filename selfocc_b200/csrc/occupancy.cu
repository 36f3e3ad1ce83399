// Occupancy evaluation on the device (eval_iou.py:206-258, eval_iou_kitti.py:167-196; utils/metric_util.py:66-244,
// utils/scenerf_metric.py).
//
// so_occ_classify: decoded volume -> one uint8 occupancy label (and optionally one semantic label) per output voxel,
// in ONE launch.  The reference materialises the whole get_uniform_sdf lattice (5.12 M points x 25 channels for Occ3D
// at 0.2 m) only to read 640 k voxels out of it with F.grid_sample; here every lattice node an output voxel needs is
// queried on the spot with the field-query device code of so_field_query (render_common.cuh), so the lattice is never
// stored and the 21 semantic channels are gathered only where the voxel is occupied.
//
// so_occ_hist: the joint (gt, pred) label histogram every reference occupancy metric is a function of.  Per-block
// shared-memory counts (warp-aggregated), then one 64-bit atomic per non-empty bin per block: integer counts, so the
// result does not depend on the launch order.
#include "render_common.cuh"

namespace so {

struct OccDev {
  const float* xs;   // lattice node coordinates in metres: x -> lattice W, y -> lattice H, z -> lattice D
  const float* ys;
  const float* zs;
  int nx, ny, nz;
  const float* pts;  // [n][3] normalised (x, y, z) sample points, nullptr = the output grid is the lattice itself
  int n0, n1, n2;
  int z_lo, z_hi, b0lo, b0hi, b1lo, b1hi;
  float thresh;
  const unsigned char* lut;
  int n_sem;
};

// sdf of the lattice node (h, w, d) = the so_field_query value at (xs[w], ys[h], zs[d]), bit for bit
__device__ __forceinline__ Taps node_taps(const VolumeDev& V, const OccDev& O, int h, int w, int d) {
  float kh, kw, kd;
  return field_taps(V, __ldg(O.xs + w), __ldg(O.ys + h), __ldg(O.zs + d), kh, kw, kd);
}
__device__ __forceinline__ float node_sdf(const VolumeDev& V, const Taps& t) {
  float s, dgh, dgw, dgd;
  gather_sdf(V, t, s, dgh, dgw, dgd);
  return s;
}

// grid_sample(align_corners=True) source index of a normalised [0, 1] coordinate, formed as eval_iou.py:221 and ATen do:
// g = u * 2 - 1, then ((g + 1) / 2) * (size - 1)
__device__ __forceinline__ float unnormalise(float u, int size) {
  float g = __fsub_rn(__fmul_rn(u, 2.f), 1.f);
  return __fmul_rn(__fdiv_rn(__fadd_rn(g, 1.f), 2.f), (float)(size - 1));
}

template <bool RESAMPLE, bool SEM>
__global__ void __launch_bounds__(256) occ_classify_kernel(VolumeDev V, OccDev O, long long n, unsigned char* __restrict__ occ_out,
                                                           unsigned char* __restrict__ sem_out) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int i2 = (int)(i % O.n2);
  const long long r = i / O.n2;
  const int i1 = (int)(r % O.n1), i0 = (int)(r / O.n1);
  // border rules (eval_iou.py:228-232, :252-257, eval_iou_kitti.py:182-186): a zeroed voxel needs no field query
  const bool keep = i2 >= O.z_lo && i2 < O.z_hi && i0 >= O.b0lo && i0 < O.n0 - O.b0hi && i1 >= O.b1lo && i1 < O.n1 - O.b1hi;
  bool occ = false;
  int arg = 0;
  if (keep && !RESAMPLE) {
    const Taps t = node_taps(V, O, i0, i1, i2);
    occ = node_sdf(V, t) <= O.thresh;
    if (SEM && occ) {                         // torch.argmax over h[..., 4:]: the first maximum
      float best = -INFINITY;
      for (int c = 0; c < O.n_sem; ++c) {
        float f1[1];
        gather_feat<1>(V, t, 3 + c, f1);
        if (f1[0] > best) { best = f1[0]; arg = c; }
      }
    }
  } else if (keep) {
    // F.grid_sample(lattice[None, None], pts[..., [2, 0, 1]] * 2 - 1, bilinear, align_corners=True, zeros padding):
    // grid x -> lattice D (from z), grid y -> lattice W (from x), grid z -> lattice H (from y)
    const float ix = unnormalise(__ldg(O.pts + 3 * i + 2), O.nz);
    const float iy = unnormalise(__ldg(O.pts + 3 * i + 0), O.nx);
    const float iz = unnormalise(__ldg(O.pts + 3 * i + 1), O.ny);
    const float fx = floorf(ix), fy = floorf(iy), fz = floorf(iz);
    // clamp before the int conversion so far-out points cannot overflow (every corner is then out of range anyway)
    const int d0 = (int)fminf(fmaxf(fx, -2.f), (float)O.nz);
    const int w0 = (int)fminf(fmaxf(fy, -2.f), (float)O.nx);
    const int h0 = (int)fminf(fmaxf(fz, -2.f), (float)O.ny);
    // corner weights in ATen's form (x factor * y factor * z factor), corners in ATen's order tnw, tne, tsw, tse, bnw, ...
    const float wx0 = __fsub_rn(__fadd_rn(fx, 1.f), ix), wx1 = __fsub_rn(ix, fx);
    const float wy0 = __fsub_rn(__fadd_rn(fy, 1.f), iy), wy1 = __fsub_rn(iy, fy);
    const float wz0 = __fsub_rn(__fadd_rn(fz, 1.f), iz), wz1 = __fsub_rn(iz, fz);
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int dh = k >> 2, dw = (k >> 1) & 1, dd = k & 1;
      const int h = h0 + dh, w = w0 + dw, d = d0 + dd;
      if ((unsigned)h < (unsigned)O.ny && (unsigned)w < (unsigned)O.nx && (unsigned)d < (unsigned)O.nz)
        s = fmaf(node_sdf(V, node_taps(V, O, h, w, d)), __fmul_rn(__fmul_rn(dd ? wx1 : wx0, dw ? wy1 : wy0), dh ? wz1 : wz0), s);
    }
    occ = s <= O.thresh;
    if (SEM && occ) {
      float acc[kMaxSem];
#pragma unroll
      for (int c = 0; c < kMaxSem; ++c) acc[c] = 0.f;
      for (int k = 0; k < 8; ++k) {
        const int dh = k >> 2, dw = (k >> 1) & 1, dd = k & 1;
        const int h = h0 + dh, w = w0 + dw, d = d0 + dd;
        if (!((unsigned)h < (unsigned)O.ny && (unsigned)w < (unsigned)O.nx && (unsigned)d < (unsigned)O.nz)) continue;
        const Taps t = node_taps(V, O, h, w, d);
        const float wk = __fmul_rn(__fmul_rn(dd ? wx1 : wx0, dw ? wy1 : wy0), dh ? wz1 : wz0);
#pragma unroll
        for (int c = 0; c < kMaxSem; ++c) {
          if (c < O.n_sem) {
            float f1[1];
            gather_feat<1>(V, t, 3 + c, f1);
            acc[c] = fmaf(f1[0], wk, acc[c]);
          }
        }
      }
      float best = -INFINITY;
#pragma unroll
      for (int c = 0; c < kMaxSem; ++c)
        if (c < O.n_sem && acc[c] > best) { best = acc[c]; arg = c; }
    }
  }
  occ_out[i] = occ ? 1 : 0;
  if (SEM) sem_out[i] = occ ? (O.lut ? __ldg(O.lut + arg) : (unsigned char)arg) : 0;
}

constexpr int kHistBlock = 256;

// hist[g][min(p, P - 1)] += #{i : mask[i] != 0, gt[i] == g, pred[i] == p}
__global__ void __launch_bounds__(kHistBlock) occ_hist_kernel(const unsigned char* __restrict__ pred, const unsigned char* __restrict__ gt,
                                                              const unsigned char* __restrict__ mask, long long n, int P,
                                                              unsigned long long* __restrict__ hist) {
  extern __shared__ unsigned int s_hist[];   // [256 * P]
  const int bins = 256 * P;
  for (int b = threadIdx.x; b < bins; b += blockDim.x) s_hist[b] = 0u;
  __syncthreads();
  const long long stride = (long long)gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  // the loop bound is uniform over the block, so every lane of a warp takes part in the match below
  for (long long base = (long long)blockIdx.x * blockDim.x; base < n; base += stride) {
    const long long i = base + threadIdx.x;
    int key = -1;
    if (i < n && (!mask || __ldg(mask + i))) key = (int)__ldg(gt + i) * P + min((int)__ldg(pred + i), P - 1);
    // most voxels share a handful of bins (empty / empty): one shared atomic per distinct bin per warp
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && lane == __ffs(peers) - 1) atomicAdd(s_hist + key, (unsigned)__popc(peers));
  }
  __syncthreads();
  for (int b = threadIdx.x; b < bins; b += blockDim.x) {
    const unsigned c = s_hist[b];
    if (c) atomicAdd(hist + b, (unsigned long long)c);
  }
}

}  // namespace so

using namespace so;

extern "C" int so_occ_classify(const float* vol_sdf, const float* vol_feat, const so_volume_desc* vol_host, const float* xs,
                               const float* ys, const float* zs, int32_t nx, int32_t ny, int32_t nz, const float* points,
                               const so_occ_grid* grid_host, const uint8_t* lut, int32_t lut_len, uint8_t* occ, uint8_t* sem,
                               void* stream) {
  if (!vol_sdf || !xs || !ys || !zs || !grid_host || !occ) return SO_ERR_INVALID_ARG;
  int rc = validate_volume(vol_host);
  if (rc) return rc;
  const so_occ_grid& g = *grid_host;
  if (nx < 1 || ny < 1 || nz < 1 || g.n0 < 0 || g.n1 < 0 || g.n2 < 0) return SO_ERR_INVALID_ARG;
  if (!points && (g.n0 != ny || g.n1 != nx || g.n2 != nz)) return SO_ERR_INVALID_ARG;   // lattice mode: output = lattice
  for (int k = 0; k < 4; ++k)
    if (g.border[k] < 0) return SO_ERR_INVALID_ARG;
  const int n_sem = vol_host->n_feat - 3;
  if (sem) {
    if (n_sem < 1 || !vol_feat) return SO_ERR_INVALID_ARG;
    if (n_sem > kMaxSem) return SO_ERR_UNSUPPORTED;
    if (lut && lut_len < n_sem) return SO_ERR_INVALID_ARG;
  }
  const long long n = (long long)g.n0 * g.n1 * g.n2;
  if (n == 0) return SO_OK;
  VolumeDev V = make_volume(*vol_host, vol_sdf, vol_feat);
  OccDev O;
  O.xs = xs; O.ys = ys; O.zs = zs; O.nx = nx; O.ny = ny; O.nz = nz; O.pts = points;
  O.n0 = g.n0; O.n1 = g.n1; O.n2 = g.n2;
  O.z_lo = g.z_lo; O.z_hi = g.z_hi;
  O.b0lo = g.border[0]; O.b0hi = g.border[1]; O.b1lo = g.border[2]; O.b1hi = g.border[3];
  O.thresh = g.thresh; O.lut = lut; O.n_sem = sem ? n_sem : 0;
  const unsigned grid = (unsigned)ceil_div64(n, 256);
  cudaStream_t st = (cudaStream_t)stream;
#define SO_OCC(R, S) occ_classify_kernel<R, S><<<grid, 256, 0, st>>>(V, O, n, occ, sem)
  if (points) { if (sem) SO_OCC(true, true); else SO_OCC(true, false); }
  else { if (sem) SO_OCC(false, true); else SO_OCC(false, false); }
#undef SO_OCC
  note_launch(1);
  return check_launch();
}

extern "C" int so_occ_hist(const uint8_t* pred, const uint8_t* gt, const uint8_t* mask, int64_t n, int32_t P, int64_t* hist,
                           void* stream) {
  if (!pred || !gt || !hist || n < 0 || P < 1) return SO_ERR_INVALID_ARG;
  if (P > SO_OCC_HIST_MAX_P) return SO_ERR_UNSUPPORTED;
  if (n == 0) return SO_OK;
  // enough blocks to fill the GPU, few enough that the per-block flush (256 * P bins) stays small next to the counting
  const long long blocks = ceil_div64(n, kHistBlock * 8);
  const unsigned grid = (unsigned)(blocks < 4 * kNumSMs ? blocks : 4 * kNumSMs);
  occ_hist_kernel<<<grid, kHistBlock, 256 * P * sizeof(unsigned int), (cudaStream_t)stream>>>(
      pred, gt, mask, n, P, reinterpret_cast<unsigned long long*>(hist));
  note_launch(1);
  return check_launch();
}
