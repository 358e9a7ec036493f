// pxr_fm_eval.cuh — the residual/Jacobian hot kernels of the featuremetric path.
//
// K0  ba_project_kernel : one thread per observation. WorldToPixel (reference
//     pixsfm/base/src/projection.h:60-75) + FeaturePatch::ToPixelCoordinates
//     (features/src/featurepatch.h:250-255) with analytic d(uv)/d(pose,point,intrinsics)
//     instead of ceres Jets (residuals/src/feature_reference.h:87-96).
// K1  fm_eval_kernel    : one warp per observation, lane <-> C/32 channels.  The 4x4xC tap
//     window of the observation's patch is staged HBM -> shared memory by the TMA bulk-copy
//     engine (cp.async.bulk + mbarrier complete_tx; SASS UBLKCP) through a per-warp ring of
//     kStages slots, so every warp keeps kStages*4 KiB of loads in flight while it computes.
//     Border semantics = per-tap clamp (base/src/grid2d.h:29-35): in-range columns are copied
//     as 4 x (4 taps) contiguous rows, clamped windows fall back to 16 per-tap copies.
//     Bicubic: horizontal pass in the input's SIMD precision (fp32 for f16/f32), vertical pass in
//     fp64, same op order as the reference (base/src/interpolation.h:177-218); L2 normalisation
//     with its chain rule (interpolation.h:648-666); residual r = f - ref
//     (feature_reference.h:132-134).  The C-channel contraction collapses to
//     ||r||^2, G^T r (2) and G^T G (3 uniques) by warp shuffles — the per-observation Jacobian is
//     rank 2 (J = G * d(uv)/d(theta)).
#pragma once
#include "pxr_device.cuh"

namespace pxr {

struct ProjectArgs {
  const int32_t* obs_img; const int64_t* obs_pt; const int64_t* obs_patch;
  const int32_t* img_cam; const int32_t* cam_model;
  const double* cam_params; const double* qvec; const double* tvec; const double* xyz;
  const int32_t* corner; const double* scale; double ups;
  int64_t obs_begin, obs_end;
  const int64_t* item_index;  // optional: process observations item_index[obs_begin..obs_end)
  double* uv;    // [n_obs][2] (u = col, v = row), patch pixel units
  double* xy;    // optional [n_obs][2]
  double* juv;   // optional [n_obs][juv_stride]: 2 x (6 pose | 3 point | K intr), row-major
  int juv_stride;
  int juv_k;     // K columns stored per row
};

// WorldToPixel + ToPixelCoordinates of observation o at the 3D point X: uv in patch pixels, xy in image pixels,
// sc = d(uv)/d(xy) per row; with JAC the derivatives of xy (world_to_pixel)
template <bool JAC>
__device__ __forceinline__ void observe(const ProjectArgs& a, int64_t o, const double X[3], double uv[2], double xy[2],
                                        double sc[2], double Jpose[2][6], double Jpt[2][3], double Jk[2][kMaxK]) {
  const int img = a.obs_img[o];
  const int64_t pi = a.obs_patch ? a.obs_patch[o] : o;
  const int cam = a.img_cam[img];
  const int model = a.cam_model[cam];
  double q[4], t[3], cp[kMaxK];
#pragma unroll
  for (int i = 0; i < 4; ++i) q[i] = a.qvec[4 * (int64_t)img + i];
#pragma unroll
  for (int i = 0; i < 3; ++i) t[i] = a.tvec[3 * (int64_t)img + i];
#pragma unroll
  for (int i = 0; i < kMaxK; ++i) cp[i] = a.cam_params[(int64_t)cam * kMaxK + i];
  world_to_pixel<JAC>(model, cp, q, t, X, xy, Jpose, Jpt, Jk);
  const double sx = a.scale[2 * pi], sy = a.scale[2 * pi + 1];
  const double cx = (double)a.corner[2 * pi], cy = (double)a.corner[2 * pi + 1];
  uv[0] = (xy[0] * sx - 0.5 - cx) * a.ups;
  uv[1] = (xy[1] * sy - 0.5 - cy) * a.ups;
  sc[0] = sx * a.ups; sc[1] = sy * a.ups;
}

// one observation: uv (and xy) to global memory, the 2 x (9 + K) record d(uv)/d(theta) to `out` (global or shared)
template <bool JAC>
__device__ __forceinline__ void project_observation(const ProjectArgs& a, int64_t o, double* out) {
  const int64_t pt = a.obs_pt[o];
  double X[3], uv[2], xy[2], s[2], Jpose[2][6], Jpt[2][3], Jk[2][kMaxK];
#pragma unroll
  for (int i = 0; i < 3; ++i) X[i] = a.xyz[3 * pt + i];
  observe<JAC>(a, o, X, uv, xy, s, Jpose, Jpt, Jk);
  a.uv[2 * o] = uv[0];
  a.uv[2 * o + 1] = uv[1];
  if (a.xy) { a.xy[2 * o] = xy[0]; a.xy[2 * o + 1] = xy[1]; }
  if (JAC && out) {
    const int W = 9 + a.juv_k;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
#pragma unroll
      for (int k = 0; k < 6; ++k) out[r * W + k] = s[r] * Jpose[r][k];
#pragma unroll
      for (int k = 0; k < 3; ++k) out[r * W + 6 + k] = s[r] * Jpt[r][k];
      for (int k = 0; k < a.juv_k; ++k) out[r * W + 9 + k] = s[r] * Jk[r][k];
    }
  }
}

template <bool JAC>
__global__ void __launch_bounds__(128) ba_project_kernel(ProjectArgs a) {
  const int64_t k = a.obs_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= a.obs_end) return;
  const int64_t o = a.item_index ? a.item_index[k] : k;
  project_observation<JAC>(a, o, (JAC && a.juv) ? a.juv + o * (int64_t)a.juv_stride : nullptr);
}

// Full-pass variant (no item list): the 128 records of a CTA are contiguous in `juv`, so they are assembled in shared
// memory (rows padded to an odd number of doubles) and written out with coalesced stores instead of 22 strided
// 8 B stores per thread.  Dynamic shared memory: 128 * (juv_stride | 1) doubles.
static __global__ void __launch_bounds__(128) ba_project_staged_kernel(ProjectArgs a) {
  extern __shared__ double sm_proj[];
  const int tid = threadIdx.x;
  const int64_t o0 = a.obs_begin + (int64_t)blockIdx.x * 128;
  const int n = (int)min((int64_t)128, a.obs_end - o0);
  const int js = a.juv_stride, SP = js | 1;
  if (tid < n) project_observation<true>(a, o0 + tid, sm_proj + tid * SP);
  __syncthreads();
  double* dst = a.juv + o0 * (int64_t)js;
  int r = tid / js, c = tid - r * js;
  const int dr = 128 / js, dcol = 128 - dr * js;
  for (int i = tid; i < n * js; i += 128) {
    dst[i] = sm_proj[r * SP + c];
    r += dr; c += dcol;
    if (c >= js) { c -= js; ++r; }
  }
}

// ---------------------------------------------------------------------------------------------
struct FmEvalArgs {
  const double* uv;            // [n][2]
  const int64_t* item_patch;   // [n] or null (identity)
  const int64_t* item_ref;     // [n] index into refs (point id) or null (identity)
  const uint8_t* patches; int ph, pw;
  const double* refs;          // [n_refs][C] or null -> residual = f
  int64_t begin, end;          // item range
  const int64_t* item_index;   // optional indirection: item k is observation item_index[k] (all per-item arrays use that id)
  double* out;                 // [n][8]: s, b_u, b_v, a_uu, a_uv, a_vv, 0, 0  (JAC) / only s (COST)
  double* residuals;           // optional [n][C]
  double* desc;                // optional [n][C]: interpolated (normalised) descriptor f (reference extraction)
  double* grad = nullptr;      // optional [n][2][C]: d r/d u, d r/d v per channel (Jacobian mode; the cost-functor surface)
  // window residency (pxr_resident.cuh): when set, only the rectangle res_rect[patch] of every patch has been brought
  // to the device; an item whose 4x4 tap window leaves it is appended to viol_list (its outputs are garbage and the
  // host re-runs the pass after fetching the patch)
  const uint32_t* res_rect = nullptr;        // [n_patches] r0 | c0 << 8 | rows << 16 | cols << 24
  unsigned long long* viol_count = nullptr;  // [1]
  int64_t* viol_list = nullptr;              // [viol_capacity]
  long long viol_capacity = 0;               // entries beyond it are dropped (they are reported again by the repeated pass)
  LossParams loss;
  int l2_normalize;
};

// the taps an item reads are rows clamp(row-1 .. row+2) and columns clamp(col-1 .. col+2) (per-tap clamp, grid2d.h:29-35):
// are they all inside the resident rectangle?
__device__ __forceinline__ bool window_resident(uint32_t rect, int row, int col, int ph, int pw) {
  const int r0 = (int)(rect & 255u), c0 = (int)((rect >> 8) & 255u), nr = (int)((rect >> 16) & 255u), ncol = (int)(rect >> 24);
  const int rlo = min(max(row - 1, 0), ph - 1), rhi = min(max(row + 2, 0), ph - 1);
  const int clo = min(max(col - 1, 0), pw - 1), chi = min(max(col + 2, 0), pw - 1);
  return rlo >= r0 && rhi < r0 + nr && clo >= c0 && chi < c0 + ncol;
}

#ifndef PXR_FM_WARPS
#define PXR_FM_WARPS 16
#endif
constexpr int kFmStages = 2;   // TMA ring slots per warp
struct FmAux {                 // per-item window geometry, one entry per lane of a batch (40 B)
  double xc, xr;
  int64_t item;
  const uint8_t* src;
  int col, row;
};
// warps per CTA so that the ring fits in ~128 KiB of shared memory
template <typename T, int C> struct FmCfg {
  static constexpr int kSlot = 16 * C * (int)sizeof(T);
  static constexpr int kWarps = kSlot <= 4096 ? PXR_FM_WARPS : (kSlot <= 8192 ? 8 : (kSlot <= 16384 ? 4 : 2));
  static constexpr int kSmem = kWarps * kFmStages * kSlot + kWarps * kFmStages * 8 + kWarps * 32 * (int)sizeof(FmAux);
};

// One TMA bulk copy of the 4x4 tap window of item x into a ring slot (completes on `bar`), whole warp.  In-range
// columns are 4 contiguous rows of 4 taps; a window clamped at a side border falls back to 16 per-tap copies.
template <int TAP_BYTES>
__device__ __forceinline__ void issue_window(const FmAux& x, uint8_t* dst, uint64_t* bar, int ph, int pw, int lane) {
  const int jc = x.col, jr = x.row;
  if (lane == 0) mbar_expect_tx(bar, 16 * TAP_BYTES);
  __syncwarp();
  const bool contiguous = (jc - 1 >= 0) && (jc + 2 <= pw - 1);
  if (contiguous) {
    if (lane < 4) {
      const int rr = min(max(jr - 1 + lane, 0), ph - 1);
      bulk_g2s(dst + lane * 4 * TAP_BYTES, x.src + ((int64_t)rr * pw + (jc - 1)) * TAP_BYTES, 4 * TAP_BYTES, bar);
    }
  } else if (lane < 16) {
    const int rr = min(max(jr - 1 + (lane >> 2), 0), ph - 1);
    const int cc = min(max(jc - 1 + (lane & 3), 0), pw - 1);
    bulk_g2s(dst + lane * TAP_BYTES, x.src + ((int64_t)rr * pw + cc) * TAP_BYTES, TAP_BYTES, bar);
  }
}

// per-item window geometry of the projection (u, v) into a patch at src
__device__ __forceinline__ FmAux window_geometry(double u, double v, const uint8_t* src, int64_t item, int ph, int pw) {
  const double fu = floor(u), fv = floor(v);
  // guard the int conversion (NaN/huge projections clamp to the border like any far-away tap)
  FmAux x;
  x.item = item;
  x.col = (int)fmin(fmax(fu, -4.0), (double)pw + 4.0);
  x.row = (int)fmin(fmax(fv, -4.0), (double)ph + 4.0);
  x.xc = u - fu; x.xr = v - fv;
  x.src = src;
  return x;
}

template <typename T> struct HorizT { typedef float type; };
template <> struct HorizT<double> { typedef double type; };

// load CPL consecutive channels of one tap from shared memory and widen
template <typename T, int CPL>
__device__ __forceinline__ void load_tap(const uint8_t* p, typename HorizT<T>::type v[CPL]);
template <> __device__ __forceinline__ void load_tap<__half, 4>(const uint8_t* p, float v[4]) {
  const uint2 w = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&w.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&w.y));
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
template <> __device__ __forceinline__ void load_tap<__half, 2>(const uint8_t* p, float v[2]) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(p));
  v[0] = a.x; v[1] = a.y;
}
template <> __device__ __forceinline__ void load_tap<__half, 1>(const uint8_t* p, float v[1]) {
  v[0] = __half2float(*reinterpret_cast<const __half*>(p));
}
template <> __device__ __forceinline__ void load_tap<__half, 8>(const uint8_t* p, float v[8]) {
  const uint4 w = *reinterpret_cast<const uint4*>(p);
  const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&ws[i])); v[2 * i] = a.x; v[2 * i + 1] = a.y; }
}
template <> __device__ __forceinline__ void load_tap<float, 4>(const uint8_t* p, float v[4]) {
  const float4 w = *reinterpret_cast<const float4*>(p); v[0] = w.x; v[1] = w.y; v[2] = w.z; v[3] = w.w;
}
template <> __device__ __forceinline__ void load_tap<float, 2>(const uint8_t* p, float v[2]) {
  const float2 w = *reinterpret_cast<const float2*>(p); v[0] = w.x; v[1] = w.y;
}
template <> __device__ __forceinline__ void load_tap<float, 1>(const uint8_t* p, float v[1]) { v[0] = *reinterpret_cast<const float*>(p); }
template <> __device__ __forceinline__ void load_tap<float, 8>(const uint8_t* p, float v[8]) {
  load_tap<float, 4>(p, v); load_tap<float, 4>(p + 16, v + 4);
}
template <> __device__ __forceinline__ void load_tap<double, 4>(const uint8_t* p, double v[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p); const double2 b = *reinterpret_cast<const double2*>(p + 16);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
template <> __device__ __forceinline__ void load_tap<double, 2>(const uint8_t* p, double v[2]) {
  const double2 a = *reinterpret_cast<const double2*>(p); v[0] = a.x; v[1] = a.y;
}
template <> __device__ __forceinline__ void load_tap<double, 1>(const uint8_t* p, double v[1]) { v[0] = *reinterpret_cast<const double*>(p); }
template <> __device__ __forceinline__ void load_tap<double, 8>(const uint8_t* p, double v[8]) {
  load_tap<double, 4>(p, v); load_tap<double, 4>(p + 32, v + 4);
}

// Bicubic f / dfdr / dfdc for CPL channels from a staged 4x4 window (tap t = 4*i + j at
// win + t*TAP_BYTES), reference op order (interpolation.h:177-218).
// tap address providers: addr(i, j) -> pointer to channel 0 of tap (row i, col j) of the window
template <int TAP_BYTES>
struct SmemWindow {
  const uint8_t* win;
  __device__ __forceinline__ const uint8_t* operator()(int i, int j) const { return win + (4 * i + j) * TAP_BYTES; }
};
struct GlobalWindow {  // clamped rows/cols resolved by the caller (grid2d.h:29-35)
  const uint8_t* rowp[4];
  int coff[4];
  __device__ __forceinline__ const uint8_t* operator()(int i, int j) const { return rowp[i] + coff[j]; }
};

template <typename T, int C, int CPL, bool DERIV, bool FLOAT_SIMD, typename Addr>
__device__ __forceinline__ void bicubic_window(const Addr& addr, int lane, double xc, double xr,
                                               double f[CPL], double fr[CPL], double fc[CPL]) {
  typedef typename HorizT<T>::type H;
  const size_t loff = (size_t)lane * CPL * sizeof(T);
  if (C >= 8) {
    H hf[4][CPL], hd[4][CPL];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      H p0[CPL], p1[CPL], p2[CPL], p3[CPL];
      load_tap<T, CPL>(addr(i, 0) + loff, p0);
      load_tap<T, CPL>(addr(i, 1) + loff, p1);
      load_tap<T, CPL>(addr(i, 2) + loff, p2);
      load_tap<T, CPL>(addr(i, 3) + loff, p3);
      if (sizeof(H) == 4) {
        const SplineCoefF32 cc(xc);
        if (CPL % 2 == 0) {
          // Blackwell packed fp32x2 FMA: two channels per instruction, bit-identical results
#pragma unroll
          for (int k = 0; k < CPL; k += 2) {
            float2 ff, dd = make_float2(0.f, 0.f);
            spline_f32x2<DERIV>(make_float2((float)p0[k], (float)p0[k + 1]), make_float2((float)p1[k], (float)p1[k + 1]),
                                make_float2((float)p2[k], (float)p2[k + 1]), make_float2((float)p3[k], (float)p3[k + 1]), cc, ff, dd);
            hf[i][k] = (H)ff.x; hf[i][k + 1] = (H)ff.y; hd[i][k] = (H)dd.x; hd[i][k + 1] = (H)dd.y;
          }
        } else {
#pragma unroll
          for (int k = 0; k < CPL; ++k) {
            float ff, dd = 0.f;
            spline_f32<DERIV>((float)p0[k], (float)p1[k], (float)p2[k], (float)p3[k], cc, ff, dd);
            hf[i][k] = (H)ff; hd[i][k] = (H)dd;
          }
        }
      } else {
        const SplineCoefF64 cc(xc);
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          double ff, dd = 0.0;
          spline_f64<true, DERIV>((double)p0[k], (double)p1[k], (double)p2[k], (double)p3[k], cc, ff, dd);
          hf[i][k] = (H)ff; hd[i][k] = (H)dd;
        }
      }
    }
    if (FLOAT_SIMD) {
      const SplineCoefF32 cr(xr);
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
        float ff, dd = 0.f;
        spline_f32<DERIV>((float)hf[0][k], (float)hf[1][k], (float)hf[2][k], (float)hf[3][k], cr, ff, dd);
        f[k] = (double)ff;
        if (DERIV) {
          fr[k] = (double)dd;
          float gg, unused = 0.f;
          spline_f32<false>((float)hd[0][k], (float)hd[1][k], (float)hd[2][k], (float)hd[3][k], cr, gg, unused);
          fc[k] = (double)gg;
        }
      }
    } else {
      const SplineCoefF64 cr(xr);
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
        double dd = 0.0;
        spline_f64<true, DERIV>((double)hf[0][k], (double)hf[1][k], (double)hf[2][k], (double)hf[3][k], cr, f[k], dd);
        if (DERIV) {
          fr[k] = dd;
          double unused = 0.0;
          spline_f64<true, false>((double)hd[0][k], (double)hd[1][k], (double)hd[2][k], (double)hd[3][k], cr, fc[k], unused);
        }
      }
    }
  } else {
    // C < 8: ceres::CubicHermiteSpline in double (interpolation.h:230-262)
    double hf[4][CPL], hd[4][CPL];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      H p0[CPL], p1[CPL], p2[CPL], p3[CPL];
      load_tap<T, CPL>(addr(i, 0) + loff, p0);
      load_tap<T, CPL>(addr(i, 1) + loff, p1);
      load_tap<T, CPL>(addr(i, 2) + loff, p2);
      load_tap<T, CPL>(addr(i, 3) + loff, p3);
#pragma unroll
      for (int k = 0; k < CPL; ++k) {
        hd[i][k] = 0.0;
        spline_ceres<DERIV>((double)p0[k], (double)p1[k], (double)p2[k], (double)p3[k], xc, hf[i][k], hd[i][k]);
      }
    }
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      double dd = 0.0, unused = 0.0;
      spline_ceres<DERIV>(hf[0][k], hf[1][k], hf[2][k], hf[3][k], xr, f[k], dd);
      if (DERIV) { fr[k] = dd; spline_ceres<false>(hd[0][k], hd[1][k], hd[2][k], hd[3][k], xr, fc[k], unused); }
    }
  }
}

// PixelInterpolator L2 normalisation + residual + rank-2 reduction for one item, whole warp.
// ALLRED=true : red[0..5] valid in every lane (butterfly all-reduce).
// ALLRED=false: transposed reduction — returns in lane L the total of value ((L>>4)&1)*4+((L>>3)&1)*2+((L>>2)&1)
//               (0:s 1:b_u 2:b_v 3:a_uu 4:a_uv 5:a_vv), 9 double shuffles instead of 30.
template <int CPL, bool DERIV, bool ALLRED>
__device__ __forceinline__ double normalize_and_reduce(bool active, bool l2, const double* refp /*lane's CPL refs or null*/,
                                                       double f[CPL], double fr[CPL], double fc[CPL],
                                                       double r[CPL], double red[6], int lane) {
  if (l2) {
    double n2 = 0.0;
    if (active) {
#pragma unroll
      for (int k = 0; k < CPL; ++k) n2 += f[k] * f[k];
    }
    n2 = warp_sum(n2);
    const double ninv = 1.0 / sqrt(n2);
    double dc = 0.0, dr = 0.0;
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      f[k] *= ninv;
      if (DERIV) { fc[k] *= ninv; fr[k] *= ninv; if (active) { dc += f[k] * fc[k]; dr += f[k] * fr[k]; } }
    }
    if (DERIV) {
      dc = warp_sum(dc); dr = warp_sum(dr);
#pragma unroll
      for (int k = 0; k < CPL; ++k) { fc[k] -= dc * f[k]; fr[k] -= dr * f[k]; }
    }
  }
  double v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (active) {
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      r[k] = refp ? f[k] - refp[k] : f[k];
      v[0] += r[k] * r[k];
      if (DERIV) {
        v[1] += fc[k] * r[k]; v[2] += fr[k] * r[k];
        v[3] += fc[k] * fc[k]; v[4] += fc[k] * fr[k]; v[5] += fr[k] * fr[k];
      }
    }
  }
  if (!DERIV) { red[0] = warp_sum(v[0]); return red[0]; }
  if (ALLRED) {
#pragma unroll
    for (int k = 0; k < 6; ++k) red[k] = warp_sum(v[k]);
    return red[0];
  }
  return warp_reduce8_transposed(v, lane);
}

// MODE 0: cost only (f), MODE 1: value + derivatives
template <typename T, int C, int MODE, bool FLOAT_SIMD>
__global__ void __launch_bounds__(FmCfg<T, C>::kWarps * 32, 1) fm_eval_kernel(FmEvalArgs a) {
  constexpr int kFmWarps = FmCfg<T, C>::kWarps;
  constexpr bool DERIV = MODE == 1;
  constexpr int CPL = C >= 32 ? C / 32 : 1;
  constexpr int ACTIVE = C / CPL;
  constexpr int TAP_BYTES = C * (int)sizeof(T);
  constexpr int SLOT_BYTES = 16 * TAP_BYTES;
  static_assert(TAP_BYTES % 16 == 0, "bulk copies need 16-byte multiples");
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* wbase = smem + (size_t)warp * kFmStages * SLOT_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)kFmWarps * kFmStages * SLOT_BYTES) + warp * kFmStages;
  FmAux* aux = reinterpret_cast<FmAux*>(smem + (size_t)kFmWarps * kFmStages * SLOT_BYTES + kFmWarps * kFmStages * 8) + warp * 32;
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kFmStages; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
  }
  __syncwarp();
  const bool active = lane < ACTIVE;
  const int64_t item_end = a.end;
  const int64_t n_items = item_end - a.begin;
  const int64_t n_batches = (n_items + 31) / 32;
  const int64_t warp_global = (int64_t)blockIdx.x * kFmWarps + warp;
  const int64_t warps_total = (int64_t)gridDim.x * kFmWarps;
  uint32_t phase_bits = 0;
  const int64_t patch_bytes = (int64_t)a.ph * a.pw * TAP_BYTES;
  const bool has_ref = a.refs != nullptr;

  for (int64_t batch = warp_global; batch < n_batches; batch += warps_total) {
    const int nvalid = (int)min((int64_t)32, item_end - (a.begin + batch * 32));
    int64_t o = a.begin + batch * 32 + lane;
    if (a.item_index && lane < nvalid) o = a.item_index[o];
    // ---- phase 1: per-lane window geometry, published to the warp through shared memory
    __syncwarp();
    int64_t ref_idx = 0;
    {
      double u = 0.0, v = 0.0;
      int64_t pidx = 0, ridx = 0;
      if (lane < nvalid) {
        u = a.uv[2 * o]; v = a.uv[2 * o + 1];
        pidx = a.item_patch ? a.item_patch[o] : o;
        ridx = a.item_ref ? a.item_ref[o] : o;
      }
      const FmAux x = window_geometry(u, v, a.patches + pidx * patch_bytes, o, a.ph, a.pw);
      aux[lane] = x;
      ref_idx = ridx;
      if (a.res_rect && lane < nvalid && !window_resident(a.res_rect[pidx], x.row, x.col, a.ph, a.pw)) {
        const unsigned long long slot = atomicAdd(a.viol_count, 1ull);
        if ((long long)slot < a.viol_capacity) a.viol_list[slot] = o;
      }
    }
    __syncwarp();

    auto issue = [&](int j, int slot) {
      issue_window<TAP_BYTES>(aux[j], wbase + (size_t)slot * SLOT_BYTES, &bars[slot], a.ph, a.pw, lane);
    };

    // ---- phase 2: software pipeline over the batch
#pragma unroll
    for (int s = 0; s < kFmStages; ++s)
      if (s < nvalid) issue(s, s);
    for (int j = 0; j < nvalid; ++j) {
      const int slot = j % kFmStages;
      const double jxc = aux[j].xc, jxr = aux[j].xr;
      double refv[CPL];
      if (has_ref) {
        const int64_t jref = __shfl_sync(0xffffffffu, (long long)ref_idx, j);
        const double* rp = a.refs + jref * C + (active ? lane * CPL : 0);
#pragma unroll
        for (int k = 0; k < CPL; ++k) refv[k] = __ldg(rp + k);
      }
      mbar_wait(&bars[slot], (phase_bits >> slot) & 1u);
      phase_bits ^= (1u << slot);
      double f[CPL], fr[CPL], fc[CPL], r[CPL], red[6];
#pragma unroll
      for (int k = 0; k < CPL; ++k) { f[k] = 0; fr[k] = 0; fc[k] = 0; r[k] = 0; }
      if (active) {
        const SmemWindow<TAP_BYTES> win{wbase + (size_t)slot * SLOT_BYTES};
        bicubic_window<T, C, CPL, DERIV, FLOAT_SIMD>(win, lane, jxc, jxr, f, fr, fc);
      }
      __syncwarp();
      if (j + kFmStages < nvalid) issue(j + kFmStages, slot);  // refill the slot just consumed
      const double tot = normalize_and_reduce<CPL, DERIV, false>(active, a.l2_normalize != 0, has_ref ? refv : nullptr, f, fr, fc, r, red, lane);
      const int64_t oj = aux[j].item;
      if (a.residuals && active) {
#pragma unroll
        for (int k = 0; k < CPL; ++k) a.residuals[oj * C + lane * CPL + k] = r[k];
      }
      if (a.desc && active) {
#pragma unroll
        for (int k = 0; k < CPL; ++k) a.desc[oj * C + lane * CPL + k] = f[k];
      }
      if (DERIV && a.grad && active) {
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          a.grad[(oj * 2) * C + lane * CPL + k] = fc[k];
          a.grad[(oj * 2 + 1) * C + lane * CPL + k] = fr[k];
        }
      }
      if (a.out) {
        if (DERIV) {
          // lanes 0,4,..,28 hold s, a_vv?...: value index = bit4*4 + bit3*2 + bit2
          const int idx = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
          if ((lane & 3) == 0 && idx < 6) a.out[oj * 8 + idx] = tot;
        } else if (lane == 0) {
          a.out[oj * 8] = tot;
        }
      }
    }
  }
}

// cost = sum_i 0.5 * rho(s_i) over items (s at out[i*8]); per-block partials, fixed order
static __global__ void __launch_bounds__(256) cost_from_sq_norm_kernel(const double* __restrict__ out, int64_t begin, int64_t end,
                                                                       LossParams loss, double* __restrict__ partials) {
  double acc = 0.0;
  for (int64_t i = begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < end; i += (int64_t)gridDim.x * blockDim.x) {
    double rho[3];
    loss_eval(loss, 1.0, out[i * 8], rho);
    acc += 0.5 * rho[0];
  }
  __shared__ double sh[8];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) { double t = 0; for (int k = 0; k < 8; ++k) t += sh[k]; partials[blockIdx.x] = t; }
}

}  // namespace pxr
