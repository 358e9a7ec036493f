// K1s: featuremetric evaluation for SMALL channel counts (C < 8) — the cost-map path.
//
// Reference: with C < 8 BiCubicInterpolator::Evaluate takes the all-double branch
// (base/src/interpolation.h:224,230-262: ceres::CubicHermiteSpline on every tap row, then on the
// column), and CostMapBundleOptimizer::AddResiduals (bundle_adjustment/src/costmap_bundle_optimizer.h:76-132)
// builds FeatureReferenceCostFunctor<C=3, N_NODES=1> with ref == nullptr, i.e. residual = the three
// interpolated cost-map channels (cost, dcost/dr, dcost/dc).
//
// A window is 16*C*sizeof(T) = 96 B (fp16, C=3): one THREAD per observation, taps read straight
// from global memory (the 4 taps of a row are 4*C contiguous values), all arithmetic in fp64 in the
// reference's order.  Output contract identical to K1 (pxr_fm_eval.cuh): out[o*8+0..5] =
// (s, b_u, b_v, a_uu, a_uv, a_vv), so everything downstream of K1 is shared.
#pragma once
#include "pxr_fm_eval.cuh"

namespace pxr {

template <typename T> __device__ __forceinline__ double small_tap(const T* p);
template <> __device__ __forceinline__ double small_tap<__half>(const __half* p) { return (double)__half2float(*p); }
template <> __device__ __forceinline__ double small_tap<float>(const float* p) { return (double)*p; }
template <> __device__ __forceinline__ double small_tap<double>(const double* p) { return *p; }

// one observation at the projection (u, v): red = (s, b_u, b_v, a_uu, a_uv, a_vv) (DERIV) or s; the optional
// residual / descriptor / gradient outputs of FmEvalArgs are written here
template <typename T, int C, bool DERIV>
__device__ __forceinline__ void fm_small_item(const FmEvalArgs& a, int64_t o, double u, double v, double red[6]) {
  const int64_t pidx = a.item_patch ? a.item_patch[o] : o;
  const double fu = floor(u), fv = floor(v);
  const int col = (int)fmin(fmax(fu, -4.0), (double)a.pw + 4.0);
  const int row = (int)fmin(fmax(fv, -4.0), (double)a.ph + 4.0);
  const double xc = u - fu, xr = v - fv;
  const T* src = reinterpret_cast<const T*>(a.patches) + pidx * (int64_t)a.ph * a.pw * C;
  int cc[4], rr[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    cc[i] = min(max(col - 1 + i, 0), a.pw - 1);     // per-tap clamp, base/src/grid2d.h:29-73
    rr[i] = min(max(row - 1 + i, 0), a.ph - 1);
  }
  double f[C], fr[C], fc[C];
#pragma unroll
  for (int ch = 0; ch < C; ++ch) {
    double fi[4], di[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const T* rowp = src + (int64_t)rr[i] * a.pw * C + ch;
      const double p0 = small_tap<T>(rowp + cc[0] * C), p1 = small_tap<T>(rowp + cc[1] * C);
      const double p2 = small_tap<T>(rowp + cc[2] * C), p3 = small_tap<T>(rowp + cc[3] * C);
      double dd = 0.0;
      spline_ceres<DERIV>(p0, p1, p2, p3, xc, fi[i], dd);
      di[i] = dd;
    }
    double d0 = 0.0, d1 = 0.0;
    spline_ceres<DERIV>(fi[0], fi[1], fi[2], fi[3], xr, f[ch], d0);
    fr[ch] = d0;
    if (DERIV) { double g; spline_ceres<false>(di[0], di[1], di[2], di[3], xr, g, d1); fc[ch] = g; } else fc[ch] = 0.0;
  }
  if (a.l2_normalize) {
    // PixelInterpolator::Evaluate, base/src/interpolation.h:642-667
    double n2 = 0.0;
#pragma unroll
    for (int ch = 0; ch < C; ++ch) n2 += f[ch] * f[ch];
    const double ninv = 1.0 / sqrt(n2);
    double dc = 0.0, dr = 0.0;
#pragma unroll
    for (int ch = 0; ch < C; ++ch) { f[ch] *= ninv; if (DERIV) { fc[ch] *= ninv; fr[ch] *= ninv; } }
    if (DERIV) {
#pragma unroll
      for (int ch = 0; ch < C; ++ch) { dc += f[ch] * fc[ch]; dr += f[ch] * fr[ch]; }
#pragma unroll
      for (int ch = 0; ch < C; ++ch) { fc[ch] -= dc * f[ch]; fr[ch] -= dr * f[ch]; }
    }
  }
  const int64_t ridx = a.item_ref ? a.item_ref[o] : o;
  double s = 0, bu = 0, bv = 0, auu = 0, auv = 0, avv = 0;
#pragma unroll
  for (int ch = 0; ch < C; ++ch) {
    const double r = a.refs ? f[ch] - a.refs[ridx * C + ch] : f[ch];
    if (a.residuals) a.residuals[o * C + ch] = r;
    if (a.desc) a.desc[o * C + ch] = f[ch];
    if (DERIV && a.grad) { a.grad[(o * 2) * C + ch] = fc[ch]; a.grad[(o * 2 + 1) * C + ch] = fr[ch]; }
    s += r * r;
    if (DERIV) { bu += fc[ch] * r; bv += fr[ch] * r; auu += fc[ch] * fc[ch]; auv += fc[ch] * fr[ch]; avv += fr[ch] * fr[ch]; }
  }
  red[0] = s;
  if (DERIV) { red[1] = bu; red[2] = bv; red[3] = auu; red[4] = auv; red[5] = avv; }
}

template <typename T, int C, int MODE>
static __global__ void __launch_bounds__(128) fm_eval_small_kernel(FmEvalArgs a) {
  constexpr bool DERIV = MODE == 1;
  const int64_t k = a.begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= a.end) return;
  const int64_t o = a.item_index ? a.item_index[k] : k;
  double red[6];
  fm_small_item<T, C, DERIV>(a, o, a.uv[2 * o], a.uv[2 * o + 1], red);
  if (a.out) {
    double* op = a.out + o * 8;
    op[0] = red[0];
    if (DERIV) { op[1] = red[1]; op[2] = red[2]; op[3] = red[3]; op[4] = red[4]; op[5] = red[5]; }
  }
}

// ------------------------------------------------------------------------------------------------
// Cost-map extraction: CostMapExtractor::FillPointCostmap (bundle_adjustment/src/costmap_extractor.h:
// 230-358), the upsampling_factor == 1, !compute_cross_derivative branch (":253-279" central
// differences on the raw patch, ":287-322" loss / gradient / optional sqrt; ":330-356" the
// !as_gradientfield single-channel variant).  One warp per output pixel: lanes stride the C input
// channels, the three dot products are reduced with shuffles in a fixed order.
//   in : patches [n_patches][ph][pw][C] (T), refs [n_points][C] f64, item -> (patch, point)
//   out: cost patches [n_patches][ph][pw][OC] (TO), OC = 3 (gradient field) or 1
template <typename T> struct DiffT;
// Eigen evaluates (Map<dtype> - Map<dtype>) in dtype before .cast<double>(): for half that is one
// rounding to fp16 (half.hpp HALF_ROUND_STYLE=1, round-to-nearest-even, third-party/half.hpp:373).
template <> struct DiffT<__half> {
  static __device__ __forceinline__ double diff(__half a, __half b) { return (double)__half2float(__float2half_rn(__half2float(a) - __half2float(b))); }
  static __device__ __forceinline__ double val(__half a) { return (double)__half2float(a); }
};
template <> struct DiffT<float> {
  static __device__ __forceinline__ double diff(float a, float b) { return (double)__fsub_rn(a, b); }
  static __device__ __forceinline__ double val(float a) { return (double)a; }
};
template <> struct DiffT<double> {
  static __device__ __forceinline__ double diff(double a, double b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ double val(double a) { return a; }
};
template <typename TO> __device__ __forceinline__ TO costmap_cast(double v);
// FeaturePatch::SetEntry stores dtype(value) (features/src/featurepatch.h:246-248): half(float(double)) = two roundings
template <> __device__ __forceinline__ __half costmap_cast<__half>(double v) { return __float2half_rn(__double2float_rn(v)); }
template <> __device__ __forceinline__ float costmap_cast<float>(double v) { return (float)v; }
template <> __device__ __forceinline__ double costmap_cast<double>(double v) { return v; }

struct CostmapArgs {
  const uint8_t* patches; int ph, pw, C;
  const double* refs;            // [n_points][C]
  const int64_t* item_patch;     // [n_items] or null (identity)
  const int64_t* item_ref;       // [n_items] point index
  int64_t n_items;
  uint8_t* out; int OC;          // [n_patches][ph][pw][OC]
  LossParams loss;
  int as_gradientfield, apply_sqrt;
};

template <typename T, typename TO>
static __global__ void __launch_bounds__(256) costmap_extract_kernel(CostmapArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t px_per = (int64_t)a.ph * a.pw;
  if (wid >= a.n_items * px_per) return;
  const int64_t item = wid / px_per;
  const int pix = (int)(wid % px_per);
  const int y = pix / a.pw, x = pix % a.pw;
  const int64_t pidx = a.item_patch ? a.item_patch[item] : item;
  const int C = a.C;
  const T* src = reinterpret_cast<const T*>(a.patches) + pidx * px_per * C;
  const double* ref = a.refs + a.item_ref[item] * C;
  const int top = min(a.ph - 1, y + 1), bottom = max(0, y - 1);
  const int right = min(a.pw - 1, x + 1), left = max(0, x - 1);
  const T* pc = src + ((int64_t)y * a.pw + x) * C;
  const T* pt = src + ((int64_t)top * a.pw + x) * C;
  const T* pb = src + ((int64_t)bottom * a.pw + x) * C;
  const T* pr = src + ((int64_t)y * a.pw + right) * C;
  const T* pl = src + ((int64_t)y * a.pw + left) * C;
  double s = 0.0, dr = 0.0, dc = 0.0;
  for (int ch = lane; ch < C; ch += 32) {
    const double r = DiffT<T>::val(pc[ch]) - ref[ch];
    s += r * r;
    if (a.as_gradientfield) {
      dr += r * (DiffT<T>::diff(pt[ch], pb[ch]) * 0.5);
      dc += r * (DiffT<T>::diff(pr[ch], pl[ch]) * 0.5);
    }
  }
  s = warp_sum(s); dr = warp_sum(dr); dc = warp_sum(dc);
  if (lane != 0) return;
  double rho[3];
  loss_eval(a.loss, 1.0, s, rho);
  double cost = rho[0] * 0.5;
  double dcostdr = 0.0, dcostdc = 0.0;
  TO* op = reinterpret_cast<TO*>(a.out) + (pidx * px_per + pix) * a.OC;
  if (a.as_gradientfield) {
    if (cost > 1.0e-8) {
      dcostdr = rho[1] * dr;
      dcostdc = rho[1] * dc;
      if (a.apply_sqrt) {
        cost = sqrt(cost);
        dcostdr *= 0.5 / cost;
        dcostdc *= 0.5 / cost;
      }
    }
    op[0] = costmap_cast<TO>(cost); op[1] = costmap_cast<TO>(dcostdr); op[2] = costmap_cast<TO>(dcostdc);
  } else {
    if (a.apply_sqrt) cost = sqrt(cost);
    op[0] = costmap_cast<TO>(cost);
  }
}

}  // namespace pxr
