// pxr_ba.cu — featuremetric bundle adjustment on the device: problem upload, the fused
// residual/Jacobian evaluation (K0+K1), and the Levenberg-Marquardt driver that replaces
// ceres::Solve for FeatureReferenceBundleOptimizer (reference
// pixsfm/bundle_adjustment/src/bundle_optimizer.h:114-245,
// feature_reference_bundle_optimizer.h:90-149).  The host only orchestrates launches and reads
// back a handful of scalars per LM iteration; all arithmetic runs in the CUDA kernels of
// pxr_fm_eval.cuh / pxr_ba_kernels.cuh / pxr_inner.cuh.
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <limits>
#include <memory>

#include "pxr_ba_host.h"

#include "pxr_resident.cuh"
#include "pxr_chol2.cuh"

namespace pxr {

// -------------------------------------------------------------------------------- fm_eval dispatch
template <typename T, int C, int MODE, bool FS>
static int launch_fm(pxr_ctx* ctx, const FmEvalArgs& a, int* n_partials) {
  typedef FmCfg<T, C> Cfg;
  auto kern = fm_eval_kernel<T, C, MODE, FS>;
  static bool attr_set = false;
  if (!attr_set) {
    PXR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem));
    attr_set = true;
  }
  const int64_t n_batches = cdiv(a.end - a.begin, 32);
  int64_t grid = cdiv(n_batches, Cfg::kWarps);
  const int64_t resident = (int64_t)ctx->sm_count * std::max(1, (int)(200 * 1024 / Cfg::kSmem));
  if (grid > resident) grid = resident;
  if (grid < 1) grid = 1;
  *n_partials = (int)(grid * Cfg::kWarps);
  PXR_LAUNCH(ctx, kern, (unsigned)grid, Cfg::kWarps * 32, Cfg::kSmem, a);
  PXR_CUDA(cudaGetLastError());
  return PXR_OK;
}

template <typename T, int C>
static int launch_fm_tc(pxr_ctx* ctx, const FmEvalArgs& a, int mode, bool fs, int* np) {
  if (mode == 1) return fs ? launch_fm<T, C, 1, true>(ctx, a, np) : launch_fm<T, C, 1, false>(ctx, a, np);
  return fs ? launch_fm<T, C, 0, true>(ctx, a, np) : launch_fm<T, C, 0, false>(ctx, a, np);
}

template <typename T, int C>
static int launch_fm_small(pxr_ctx* ctx, const FmEvalArgs& a, int mode, int* np) {
  const int64_t n = a.end - a.begin;
  *np = 0;
  if (n <= 0) return PXR_OK;
  if (mode == 1) PXR_LAUNCH(ctx, (fm_eval_small_kernel<T, C, 1>), (unsigned)cdiv(n, 128), 128, 0, a);
  else PXR_LAUNCH(ctx, (fm_eval_small_kernel<T, C, 0>), (unsigned)cdiv(n, 128), 128, 0, a);
  PXR_CUDA(cudaGetLastError());
  return PXR_OK;
}

int fm_supported(int dtype, int C) {
  // C < 8: the reference's all-double bicubic branch (interpolation.h:224); 3/4 = cost maps, 1 = scalar maps
  if ((C == 1 || C == 3 || C == 4) && (dtype == PXR_F16 || dtype == PXR_F32 || dtype == PXR_F64)) return 1;
  if (dtype == PXR_F16) return C == 8 || C == 16 || C == 32 || C == 64 || C == 128 || C == 256;
  if (dtype == PXR_F32) return C == 16 || C == 64 || C == 128;
  if (dtype == PXR_F64) return C == 16 || C == 128;
  return 0;
}

int fm_max_partials(pxr_ctx* ctx) { return ctx->sm_count * 16 * 64; }

int launch_fm_eval(pxr_ctx* ctx, int dtype, int C, int mode, bool float_simd, const FmEvalArgs& a, int* np) {
#define PXR_SMALL(T) \
  { if (C == 3) return launch_fm_small<T, 3>(ctx, a, mode, np); if (C == 4) return launch_fm_small<T, 4>(ctx, a, mode, np); \
    if (C == 1) return launch_fm_small<T, 1>(ctx, a, mode, np); }
  if (C < 8) {
    if (dtype == PXR_F16) PXR_SMALL(__half) else if (dtype == PXR_F32) PXR_SMALL(float) else if (dtype == PXR_F64) PXR_SMALL(double)
    return fail(PXR_ERR_UNSUPPORTED, "Unsupported dimensions (CHANNELS=%d, dtype=%d, N_NODES=1).", C, dtype);
  }
#undef PXR_SMALL
#define PXR_CASE(T, CC) \
  if (C == CC) return launch_fm_tc<T, CC>(ctx, a, mode, float_simd, np);
  if (dtype == PXR_F16) {
    PXR_CASE(__half, 128) PXR_CASE(__half, 64) PXR_CASE(__half, 32) PXR_CASE(__half, 16) PXR_CASE(__half, 8)
    PXR_CASE(__half, 256)
  } else if (dtype == PXR_F32) {
    PXR_CASE(float, 128) PXR_CASE(float, 64) PXR_CASE(float, 16)
  } else if (dtype == PXR_F64) {
    PXR_CASE(double, 128) PXR_CASE(double, 16)
  }
#undef PXR_CASE
  return fail(PXR_ERR_UNSUPPORTED, "Unsupported dimensions (CHANNELS=%d, dtype=%d, N_NODES=1).", C, dtype);
}

// -------------------------------------------------------------------------------- inner iterations dispatch
template <typename T, int C, bool FS>
static int launch_inner_k(pxr_ctx* ctx, const InnerArgs& a) {
  typedef InnerCfg<T, C> Cfg;
  auto kern = inner_fused_kernel<T, C, FS>;
  static bool attr_set = false;
  if (!attr_set) {
    PXR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem));
    attr_set = true;
  }
  // two CTAs per SM (the L2 budget of pxr_inner.cuh); fewer when there are fewer points
  const int64_t grid = std::max<int64_t>(1, std::min<int64_t>((int64_t)ctx->sm_count * 2, cdiv(a.n_points, kInnerSlots)));
  PXR_LAUNCH(ctx, kern, (unsigned)grid, Cfg::kWarps * 32, Cfg::kSmem, a);
  PXR_CUDA(cudaGetLastError());
  return PXR_OK;
}

// the (dtype, C) pairs of launch_fm_eval
int launch_inner_fused(pxr_ctx* ctx, int dtype, int C, bool float_simd, const InnerArgs& a) {
#define PXR_SMALL(T) \
  { if (C == 3) return launch_inner_k<T, 3, false>(ctx, a); if (C == 4) return launch_inner_k<T, 4, false>(ctx, a); \
    if (C == 1) return launch_inner_k<T, 1, false>(ctx, a); }
  if (C < 8) {
    if (dtype == PXR_F16) PXR_SMALL(__half) else if (dtype == PXR_F32) PXR_SMALL(float) else if (dtype == PXR_F64) PXR_SMALL(double)
    return fail(PXR_ERR_UNSUPPORTED, "Unsupported dimensions (CHANNELS=%d, dtype=%d, N_NODES=1).", C, dtype);
  }
#undef PXR_SMALL
#define PXR_CASE(T, CC) \
  if (C == CC) return float_simd ? launch_inner_k<T, CC, true>(ctx, a) : launch_inner_k<T, CC, false>(ctx, a);
  if (dtype == PXR_F16) {
    PXR_CASE(__half, 128) PXR_CASE(__half, 64) PXR_CASE(__half, 32) PXR_CASE(__half, 16) PXR_CASE(__half, 8)
    PXR_CASE(__half, 256)
  } else if (dtype == PXR_F32) {
    PXR_CASE(float, 128) PXR_CASE(float, 64) PXR_CASE(float, 16)
  } else if (dtype == PXR_F64) {
    PXR_CASE(double, 128) PXR_CASE(double, 16)
  }
#undef PXR_CASE
  return fail(PXR_ERR_UNSUPPORTED, "Unsupported dimensions (CHANNELS=%d, dtype=%d, N_NODES=1).", C, dtype);
}

// -------------------------------------------------------------------------------- problem upload
static int check_desc(const pxr_ba_desc* d) {
  if (!d) return fail(PXR_ERR_INVALID_ARGUMENT, "desc is NULL");
  if (d->n_cameras <= 0 || d->n_images <= 0 || d->n_points < 0 || d->n_obs < 0)
    return fail(PXR_ERR_INVALID_ARGUMENT, "empty problem");
  if (!d->cam_model || !d->cam_params || !d->cam_const_mask || !d->qvec || !d->tvec || !d->img_cam ||
      !d->pose_const || !d->tvec_const_mask || (d->n_points && (!d->xyz || !d->point_const)) ||
      (d->n_obs && (!d->obs_img || !d->obs_pt)) || (!d->patches && d->n_patch_blocks <= 0) || !d->corner || !d->scale)
    return fail(PXR_ERR_INVALID_ARGUMENT, "a required array is NULL");
  if (!fm_supported(d->patch_dtype, d->channels))
    return fail(PXR_ERR_UNSUPPORTED, "Unsupported dimensions (CHANNELS=%d, dtype=%d, N_NODES=1).", d->channels, d->patch_dtype);
  if (d->ph < 1 || d->pw < 1) return fail(PXR_ERR_INVALID_ARGUMENT, "bad patch size");
  for (int c = 0; c < d->n_cameras; ++c)
    if (cam_num_params(d->cam_model[c]) == 0) return fail(PXR_ERR_UNSUPPORTED, "unsupported camera model id %d", d->cam_model[c]);
  for (int i = 0; i < d->n_images; ++i)
    if (d->img_cam[i] < 0 || d->img_cam[i] >= d->n_cameras) return fail(PXR_ERR_INVALID_ARGUMENT, "img_cam out of range");
  const int64_t np = d->obs_patch ? d->n_patches : d->n_obs;
  for (int64_t o = 0; o < d->n_obs; ++o) {
    if (d->obs_img[o] < 0 || d->obs_img[o] >= d->n_images) return fail(PXR_ERR_INVALID_ARGUMENT, "obs_img out of range");
    if (d->obs_pt[o] < 0 || d->obs_pt[o] >= d->n_points) return fail(PXR_ERR_INVALID_ARGUMENT, "obs_pt out of range");
    if (o && d->obs_pt[o] < d->obs_pt[o - 1]) return fail(PXR_ERR_INVALID_ARGUMENT, "observations must be sorted by point index");
    if (d->obs_patch && (d->obs_patch[o] < 0 || d->obs_patch[o] >= np)) return fail(PXR_ERR_INVALID_ARGUMENT, "obs_patch out of range");
  }
  if (!d->obs_patch && d->n_patches < d->n_obs) return fail(PXR_ERR_INVALID_ARGUMENT, "n_patches < n_obs with identity patch map");
  return PXR_OK;
}

int BA::create(pxr_ctx* c, const pxr_ba_desc* d, const pxr_interp_config* ic, const pxr_solver_options* so, bool for_solve) {
  ctx = c;
  PXR_TRY(check_desc(d));
  if (ic) interp = *ic; else pxr_default_interp_config(&interp);
  if (so) opt = *so; else pxr_default_ba_options(&opt);
  if (interp.check_bounds) return fail(PXR_ERR_UNSUPPORTED, "check_bounds=true is not supported on this path");
  env.pcg_sparse = getenv("PXR_PCG_SPARSE") != nullptr; env.build_atomic = getenv("PXR_BUILD_ATOMIC") != nullptr;
  env.chol_multikernel = getenv("PXR_CHOL_MULTIKERNEL") != nullptr; env.chol_test_abort = getenv("PXR_CHOL_TEST_ABORT") != nullptr;
  env.build_staged = getenv("PXR_BUILD_UNSTAGED") == nullptr;
  env.project_staged = getenv("PXR_PROJECT_UNSTAGED") == nullptr;
  env.cg_multi = getenv("PXR_CG_MULTI") != nullptr; env.no_speculation = getenv("PXR_NO_SPECULATION") != nullptr;
  if (const char* t = getenv("PXR_CHOL_TRACE")) env.chol_trace = t;
  PXR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  n_cameras = d->n_cameras; n_images = d->n_images; n_points = d->n_points; n_obs = d->n_obs;
  C = d->channels; ph = d->ph; pw = d->pw; dtype = d->patch_dtype; ups = d->upsampling_factor;
  n_patches = d->obs_patch ? d->n_patches : std::max(d->n_patches, d->n_obs);
  has_refs = d->refs != nullptr;
  // the big patch upload goes first, on the context's side stream: the host-side layout / co-visibility work below
  // (and the small synchronous uploads it makes on `s`) overlaps with the DMA; joined when create() returns
  cudaStream_t us = nullptr;
  PXR_TRY(upload_stream(ctx, &us));
  struct JoinUpload { BA* ba; cudaStream_t us; ~JoinUpload() { if (ba->res_thread.joinable()) ba->res_thread.join(); cudaStreamSynchronize(us); } } join_upload{this, us};
  double h2d_patch = 0;
  const size_t esz = dtype == PXR_F16 ? 2 : (dtype == PXR_F32 ? 4 : 8);
  const size_t pbytes = (size_t)n_patches * ph * pw * C * esz;
  if (d->n_patch_blocks > 0) {
    if (!d->patch_block_ptrs || !d->patch_block_counts) return fail(PXR_ERR_INVALID_ARGUMENT, "patch block arrays are NULL");
    int64_t tot = 0;
    for (int b = 0; b < d->n_patch_blocks; ++b) tot += d->patch_block_counts[b];
    if (tot < n_patches) return fail(PXR_ERR_INVALID_ARGUMENT, "patch blocks hold %lld patches, %lld needed", (long long)tot, (long long)n_patches);
    PXR_TRY(patches_owned.alloc(ctx, (size_t)tot * ph * pw * C * esz));
    PXR_TRY(resident_setup(d, esz));                      // window residency where it applies (copies issued further down)
    if (!resident) {
      // a block may live in host OR device memory (device-resident feature store): UVA resolves the direction
      std::vector<size_t> seg_bytes((size_t)d->n_patch_blocks);
      for (int b = 0; b < d->n_patch_blocks; ++b) seg_bytes[b] = (size_t)d->patch_block_counts[b] * ph * pw * C * esz;
      PXR_TRY(upload_segments(ctx, patches_owned.p, d->patch_block_ptrs, seg_bytes.data(), d->n_patch_blocks, &h2d_patch, us));
    }
    d_patches = patches_owned.p;
  } else if (d->patches_on_device) {
    d_patches = (const uint8_t*)d->patches;
  } else {
    PXR_TRY(patches_owned.alloc(ctx, pbytes));
    PXR_TRY(resident_setup(d, esz));
    if (!resident) {
      PXR_TRY(upload_bytes(ctx, patches_owned.p, d->patches, pbytes, nullptr, us));
      h2d_patch = (double)pbytes;
    }
    d_patches = patches_owned.p;
  }
  // ---- layout (same rules as BundleOptimizer::Parameterize*, resolved into masks by the caller)
  K = 0;
  for (int i = 0; i < n_cameras; ++i) K = std::max(K, cam_num_params(d->cam_model[i]));
  dcmax = 6 + K;
  juv_stride = 2 * (9 + K);
  h_pose_off.assign(n_images, -1); h_intr_off.assign(n_cameras, -1); h_point_off.assign(n_points, -1);
  int off = 0;
  for (int i = 0; i < n_images; ++i) {
    if (d->pose_const[i]) continue;
    h_pose_off[i] = off;
    off += 3 + (3 - __builtin_popcount(d->tvec_const_mask[i] & 7u));
  }
  std::vector<uint32_t> cmask(n_cameras);
  for (int i = 0; i < n_cameras; ++i) {
    const int k = cam_num_params(d->cam_model[i]);
    const uint32_t full = (1u << k) - 1u;
    cmask[i] = d->cam_const_mask[i] & full;
    if (cmask[i] == full) continue;
    h_intr_off[i] = off;
    off += k - __builtin_popcount(cmask[i]);
  }
  nc = off;
  int64_t po = off;
  for (int64_t p = 0; p < n_points; ++p) if (!d->point_const[p]) { h_point_off[p] = po; po += 3; }
  nl = (int64_t)po;
  h_pt_begin.assign(n_points + 1, 0);
  for (int64_t o = 0; o < n_obs; ++o) h_pt_begin[d->obs_pt[o] + 1]++;
  for (int64_t p = 0; p < n_points; ++p) h_pt_begin[p + 1] += h_pt_begin[p];

  double h2d = h2d_patch;
  auto up = [&](auto& buf, const auto* host, size_t n) -> int { h2d += n * sizeof(*host); return buf.upload(host, n, s); };
  PXR_TRY(up(obs_img, d->obs_img, n_obs));
  PXR_TRY(up(obs_pt, d->obs_pt, n_obs));
  if (d->obs_patch) PXR_TRY(up(obs_patch, d->obs_patch, n_obs));
  PXR_TRY(up(img_cam, d->img_cam, n_images));
  PXR_TRY(up(cam_model, d->cam_model, n_cameras));
  PXR_TRY(up(cam_mask, cmask.data(), n_cameras));
  PXR_TRY(up(tmask, d->tvec_const_mask, n_images));
  PXR_TRY(up(pose_off, h_pose_off.data(), n_images));
  PXR_TRY(up(intr_off, h_intr_off.data(), n_cameras));
  PXR_TRY(up(point_off, h_point_off.data(), n_points));
  PXR_TRY(up(pt_begin, h_pt_begin.data(), n_points + 1));
  PXR_TRY(up(corner, d->corner, (size_t)n_patches * 2));
  PXR_TRY(up(scale, d->scale, (size_t)n_patches * 2));
  if (has_refs) PXR_TRY(up(refs, d->refs, (size_t)n_points * C));
  for (int k = 0; k < 2; ++k) {
    PXR_TRY(cam[k].upload(d->cam_params, (size_t)n_cameras * kMaxK, s));
    PXR_TRY(q[k].upload(d->qvec, (size_t)n_images * 4, s));
    PXR_TRY(t[k].upload(d->tvec, (size_t)n_images * 3, s));
    PXR_TRY(X[k].upload(d->xyz, (size_t)n_points * 3, s));
  }
  h2d += ((size_t)n_cameras * kMaxK + n_images * 7 + n_points * 3) * 8.0;
  cur = 0;
  // per-observation and linearisation buffers
  PXR_TRY(uv.alloc((size_t)n_obs * 2));
  if (resident) { double wbytes = 0; PXR_TRY(resident_begin(us, &wbytes)); h2d += wbytes; }
  PXR_TRY(obs_out.alloc((size_t)n_obs * 8));
  PXR_TRY(juv.alloc((size_t)n_obs * juv_stride));
  if (for_solve) {
    PXR_TRY(uv_alt.alloc((size_t)n_obs * 2)); PXR_TRY(obs_out_alt.alloc((size_t)n_obs * 8)); PXR_TRY(juv_alt.alloc((size_t)n_obs * juv_stride));
    PXR_TRY(obs_out_alt.zero(s));
  }
  // linear solver as BundleOptimizer::SolveProblem picks it (bundle_optimizer.h:181-191): exact factorisation up to
  // 1000 images, ITERATIVE_SCHUR + SCHUR_JACOBI above (or when asked for)
  use_pcg = opt.linear_solver == PXR_SOLVER_ITERATIVE_SCHUR || (opt.linear_solver == PXR_SOLVER_AUTO && n_images > 1000);
  {
    // per-image column tables: an observation's camera columns are [pose columns | intrinsics columns] of its image
    int dc_needed = 0;
    h_img_cols.assign((size_t)n_images * 8, -1); h_img_pd.assign(n_images, 0);
    std::vector<int8_t> h_src((size_t)n_images * 8, -1);     // entry of the Jacobian row [rot3 | t3 | X3 | cam K] per column
    std::vector<int32_t> h_dc(n_images, 0);
    for (int i = 0; i < n_images; ++i) {
      std::vector<int> cols, src;
      if (h_pose_off[i] >= 0) {
        for (int k = 0; k < 3; ++k) { cols.push_back(h_pose_off[i] + k); src.push_back(k); }
        int la = 3;
        for (int k = 0; k < 3; ++k) if (!(d->tvec_const_mask[i] & (1u << k))) { cols.push_back(h_pose_off[i] + la++); src.push_back(3 + k); }
      }
      const int pd = (int)cols.size();
      const int cam_i = d->img_cam[i];
      if (h_intr_off[cam_i] >= 0) {
        const int kc = cam_num_params(d->cam_model[cam_i]);
        int la = 0;
        for (int k = 0; k < kc; ++k) if (!(cmask[cam_i] & (1u << k))) { cols.push_back(h_intr_off[cam_i] + la++); src.push_back(9 + k); }
      }
      dc_needed = std::max(dc_needed, (int)cols.size());
      h_img_pd[i] = pd;
      h_dc[i] = (int32_t)cols.size();
      for (size_t k = 0; k < cols.size() && k < 8; ++k) { h_img_cols[(size_t)i * 8 + k] = cols[k]; h_src[(size_t)i * 8 + k] = (int8_t)src[k]; }
    }
    img_dc_max = dc_needed;
    if (dc_needed <= 8) {
      PXR_TRY(img_cols8.upload(h_img_cols.data(), h_img_cols.size(), s));
      PXR_TRY(img_src8.upload(h_src.data(), h_src.size(), s));
      PXR_TRY(img_dc8.upload(h_dc.data(), h_dc.size(), s));
      PXR_CUDA(cudaStreamSynchronize(s));   // h_src / h_dc are locals
    }
    h_img_cam.assign(d->img_cam, d->img_cam + n_images);
    // implicit block-sparse reduced system: on request, or when the dense one would not fit comfortably
    sparse_schur = for_solve && use_pcg && dc_needed <= 8 && (n_obs > 0 || ctx->world > 1) &&
                   (env.pcg_sparse || (int64_t)nc * nc * 8 > (int64_t)4e9);
    // block mode: image-block assembly + ONE all-reduce per LM iteration (pxr_block.cuh).  Always on with several ranks
    // (the image tables are replicated, so every rank takes the same decision); PXR_BLOCK_ASSEMBLY=1 runs the same code on
    // one GPU (tests).  Images with more than 8 camera columns keep the dense multi-collective path.
    deterministic = for_solve && opt.deterministic != 0;
    if (deterministic && dc_needed > 8)
      return fail(PXR_ERR_UNSUPPORTED, "deterministic assembly needs <= 8 camera columns per image (pose 6 + intrinsics), got %d", dc_needed);
    block_mode = for_solve && dc_needed <= 8 && (ctx->world > 1 || deterministic || getenv("PXR_BLOCK_ASSEMBLY") != nullptr);
    if (ctx->world > 1 && sparse_schur && !block_mode) sparse_schur = false;
    if (!sparse_schur && (int64_t)nc * nc * 8 > (int64_t)40e9)
      return fail(PXR_ERR_UNSUPPORTED, "reduced camera system too large for the dense path (nc=%d) and the block-sparse path needs ITERATIVE_SCHUR with <= 8 camera columns per image", nc);
  }
  if (!sparse_schur && !block_mode) PXR_TRY(Hcc.alloc((size_t)nc * nc));
  PXR_TRY(gc.alloc(nc));
  PXR_TRY(Hpp.alloc((size_t)n_points * 9)); PXR_TRY(gp.alloc((size_t)n_points * 3));
  h_obs_img.assign(d->obs_img, d->obs_img + n_obs);
  if (for_solve) PXR_TRY(build_schur_pairs());
  if (block_mode) PXR_TRY(block_setup());
  if (for_solve && n_obs > 0 && n_obs < ((int64_t)1 << 31)) {
    // per-image observation chunks for the camera-block build (ba_build_cam_kernel): images whose pose and
    // intrinsics are both constant contribute nothing and are left out; usable when every image has <= 8 columns
    int dc_needed = 0;
    std::vector<int> img_dc(n_images, 0);
    for (int i = 0; i < n_images; ++i) {
      int dc = 0;
      if (h_pose_off[i] >= 0) dc += 3 + (3 - __builtin_popcount(d->tvec_const_mask[i] & 7u));
      const int cam_i = d->img_cam[i];
      if (h_intr_off[cam_i] >= 0) dc += cam_num_params(d->cam_model[cam_i]) - __builtin_popcount(cmask[cam_i]);
      img_dc[i] = dc;
      dc_needed = std::max(dc_needed, dc);
    }
    if (dc_needed <= 8) {
      std::vector<int64_t> cnt(n_images + 1, 0);
      for (int64_t o = 0; o < n_obs; ++o) if (img_dc[d->obs_img[o]] > 0) cnt[d->obs_img[o] + 1]++;
      for (int i = 0; i < n_images; ++i) cnt[i + 1] += cnt[i];
      std::vector<int32_t> list(cnt[n_images]);
      {
        std::vector<int64_t> cur_pos(cnt.begin(), cnt.end() - 1);
        for (int64_t o = 0; o < n_obs; ++o) if (img_dc[d->obs_img[o]] > 0) list[cur_pos[d->obs_img[o]]++] = (int32_t)o;
      }
      std::vector<int64_t> cb;
      h_img_chunk_begin.assign((size_t)n_images + 1, 0);
      for (int i = 0; i < n_images; ++i) {
        h_img_chunk_begin[i] = (int64_t)cb.size();
        for (int64_t b = cnt[i]; b < cnt[i + 1]; b += 128) cb.push_back(b);
      }
      h_img_chunk_begin[n_images] = (int64_t)cb.size();
      cb.push_back(cnt[n_images]);
      io_n_chunks = (int64_t)cb.size() - 1;
      if (io_n_chunks > 0) {
        PXR_TRY(io_obs.upload(list.data(), list.size(), s));
        PXR_TRY(io_chunk_begin.upload(cb.data(), cb.size(), s));
        PXR_CUDA(cudaStreamSynchronize(s));   // host vectors go out of scope
      }
      if (deterministic) {                    // fixed-order reduction of the camera-block chunk partials (pxr_block.cuh)
        PXR_TRY(det_cam_part.alloc((size_t)std::max<int64_t>(io_n_chunks, 1) * 48));
        PXR_TRY(det_img_chunk_begin.upload(h_img_chunk_begin.data(), h_img_chunk_begin.size(), s));
        PXR_CUDA(cudaStreamSynchronize(s));
      }
    }
  }
  PXR_TRY(W.alloc((size_t)n_obs * dcmax * 3)); PXR_TRY(Wcols.alloc((size_t)n_obs * dcmax)); PXR_TRY(Wdc.alloc(n_obs));
  if (!sparse_schur) PXR_TRY(S.alloc((size_t)(nc + 1) * nc));   // block mode: filled from the global blocks (blk_gather_kernel)
  PXR_TRY(rhs.alloc(nc));
  PXR_TRY(diag.alloc(nl)); PXR_TRY(jscale.alloc(nl)); PXR_TRY(D2.alloc(nl)); PXR_TRY(delta.alloc(nl));
  PXR_TRY(partials.alloc(fm_max_partials(ctx)));
  if (deterministic) {
    const int64_t big = std::max<int64_t>({n_obs, n_points * 3, (int64_t)n_images * 4, (int64_t)n_cameras * kMaxK});
    PXR_TRY(det_scal_part.alloc((size_t)(cdiv(big, 128) * 4 + 16)));
    if (io_n_chunks == 0 && n_obs > 0) return fail(PXR_ERR_UNSUPPORTED, "deterministic assembly needs the per-image chunk lists (problem too large for 32-bit observation ids)");
  }
  PXR_TRY(scalars.alloc(16));
  PXR_TRY(flags.alloc(4));
  PXR_TRY(rdiag.alloc(kNB));
  PXR_TRY(Hpp.zero(s)); PXR_TRY(gp.zero(s)); PXR_TRY(obs_out.zero(s));
  PXR_CUDA(cudaStreamSynchronize(s));
  if (res_thread.joinable()) {       // the window upload runs beside all of the above
    res_thread.join();
    if (res_thread_rc != PXR_OK) return fail(res_thread_rc, "%s", res_thread_err.c_str());
  }
  h2d_bytes = h2d;
  return PXR_OK;
}

// Static structure of the Schur complement: every pair of observations (i >= j) of a variable point,
// grouped by the (image_i, image_j) pair they address in the reduced camera system; long groups are
// split into chunks of at most kChunk entries (one warp each).
int BA::build_schur_pairs() {
  if (sp_built) return PXR_OK;
  PXR_TRY(Tbuf.alloc((size_t)n_obs * dcmax * 3));
  PXR_TRY(Hinv.alloc((size_t)std::max<int64_t>(n_points, 1) * 6));
  const int64_t kChunk = 128;
  const int64_t ni = n_images;
  auto key_of = [&](int ia, int ib, bool self) -> int64_t {  // ia >= ib
    return ((int64_t)ia * (ia + 1) / 2 + ib) * 2 + (self ? 1 : 0);
  };
  const int64_t n_keys = (ni * (ni + 1) / 2) * 2;
  std::vector<int64_t> count(n_keys + 1, 0);
  int64_t total = 0;
  for (int64_t p = 0; p < n_points; ++p) {
    if (h_point_off[p] < 0) continue;
    for (int64_t i = h_pt_begin[p]; i < h_pt_begin[p + 1]; ++i)
      for (int64_t j = h_pt_begin[p]; j <= i; ++j) {
        const int a = h_obs_img[i], b = h_obs_img[j];
        count[key_of(std::max(a, b), std::min(a, b), i == j) + 1]++;
        ++total;
      }
  }
  if (total >= ((int64_t)1 << 31) || n_obs >= ((int64_t)1 << 31) || n_points >= ((int64_t)1 << 31))
    return fail(PXR_ERR_UNSUPPORTED, "too many observation pairs for 32-bit pair indices");
  for (int64_t k = 0; k < n_keys; ++k) count[k + 1] += count[k];
  std::vector<int32_t> px(total), py(total), pp(total);
  {
    std::vector<int64_t> cursor(count.begin(), count.end() - 1);
    for (int64_t p = 0; p < n_points; ++p) {
      if (h_point_off[p] < 0) continue;
      for (int64_t i = h_pt_begin[p]; i < h_pt_begin[p + 1]; ++i)
        for (int64_t j = h_pt_begin[p]; j <= i; ++j) {
          const int a = h_obs_img[i], b = h_obs_img[j];
          const int64_t k = cursor[key_of(std::max(a, b), std::min(a, b), i == j)]++;
          // x = the observation in the image with the larger index
          if (a >= b) { px[k] = (int32_t)i; py[k] = (int32_t)j; } else { px[k] = (int32_t)j; py[k] = (int32_t)i; }
          pp[k] = (int32_t)p;
        }
    }
  }
  std::vector<int64_t> cb;
  std::vector<uint8_t> cself;
  std::vector<int32_t> ckey, ka, kbv;      // sparse path: compact id of every non-empty (image pair, self) key
  std::vector<uint8_t> kself;
  {
    int64_t k = 0;
    for (int64_t ia = 0; ia < ni; ++ia)
      for (int64_t ib = 0; ib <= ia; ++ib)
        for (int self = 0; self < 2; ++self, ++k) {
          if (count[k + 1] == count[k]) continue;
          if (sparse_schur || block_mode) { ka.push_back((int32_t)ia); kbv.push_back((int32_t)ib); kself.push_back((uint8_t)self); h_key_code_local.push_back(k); }
          for (int64_t s = count[k]; s < count[k + 1]; s += kChunk) {
            cb.push_back(s); cself.push_back((uint8_t)self);
            if (sparse_schur || block_mode) ckey.push_back((int32_t)ka.size() - 1);
          }
        }
  }
  cb.push_back(total);
  if (block_mode) {
    // the key list becomes the union over the ranks, the blocks live in the packed buffer (block_setup)
    h_key_a = ka; h_key_b = kbv; h_key_self = kself;
    PXR_TRY(ss_chunk_key.upload(ckey.data(), ckey.size(), ctx->stream));     // local ids for now; block_setup remaps them
    PXR_CUDA(cudaStreamSynchronize(ctx->stream));
    h_chunk_key_local = ckey;
  } else if (sparse_schur) {
    ss_n_keys = (int)ka.size();
    PXR_TRY(ss_key_a.upload(ka.data(), ka.size(), ctx->stream)); PXR_TRY(ss_key_b.upload(kbv.data(), kbv.size(), ctx->stream));
    PXR_TRY(ss_key_self.upload(kself.data(), kself.size(), ctx->stream));
    PXR_TRY(ss_chunk_key.upload(ckey.data(), ckey.size(), ctx->stream));
    PXR_TRY(ss_Bk.alloc((size_t)std::max(ss_n_keys, 1) * 64));
    PXR_TRY(ss_Himg.alloc((size_t)n_images * 64));
    PXR_TRY(ss_img_cols.upload(h_img_cols.data(), h_img_cols.size(), ctx->stream));
    PXR_TRY(ss_img_pd.upload(h_img_pd.data(), h_img_pd.size(), ctx->stream));
    PXR_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  sp_n_chunks = (int64_t)cself.size();
  cudaStream_t s = ctx->stream;
  PXR_TRY(sp_px.upload(px.data(), px.size(), s));
  PXR_TRY(sp_py.upload(py.data(), py.size(), s));
  PXR_TRY(sp_pp.upload(pp.data(), pp.size(), s));
  PXR_TRY(sp_chunk_begin.upload(cb.data(), cb.size(), s));
  PXR_TRY(sp_chunk_self.upload(cself.data(), cself.size(), s));
  PXR_CUDA(cudaStreamSynchronize(s));  // host vectors go out of scope
  sp_built = true;
  return PXR_OK;
}

SchurPairs BA::schur_pairs() {
  SchurPairs sp;
  sp.px = sp_px.p; sp.py = sp_py.p; sp.pp = sp_pp.p; sp.chunk_begin = sp_chunk_begin.p; sp.chunk_self = sp_chunk_self.p;
  sp.n_chunks = sp_n_chunks;
  return sp;
}

// -------------------------------------------------------------------------------- evaluation
int BA::project(int set, bool jac, double* xy_out) {
  ProjectArgs a;
  a.obs_img = obs_img.p; a.obs_pt = obs_pt.p; a.obs_patch = obs_patch.p;
  a.img_cam = img_cam.p; a.cam_model = cam_model.p;
  a.cam_params = cam[set].p; a.qvec = q[set].p; a.tvec = t[set].p; a.xyz = X[set].p;
  a.corner = corner.p; a.scale = scale.p; a.ups = ups;
  a.obs_begin = 0; a.obs_end = n_obs; a.item_index = nullptr;
  a.uv = uv.p; a.xy = xy_out; a.juv = jac ? juv.p : nullptr; a.juv_stride = juv_stride; a.juv_k = K;
  if (n_obs == 0) return PXR_OK;
  StageScope st(this, 2);
  const size_t staged_smem = (size_t)128 * (juv_stride | 1) * sizeof(double);
  if (jac && env.project_staged && staged_smem <= 48 * 1024)
    PXR_LAUNCH(ctx, ba_project_staged_kernel, (unsigned)cdiv(n_obs, 128), 128, staged_smem, a);
  else if (jac) PXR_LAUNCH(ctx, ba_project_kernel<true>, (unsigned)cdiv(n_obs, 128), 128, 0, a);
  else PXR_LAUNCH(ctx, ba_project_kernel<false>, (unsigned)cdiv(n_obs, 128), 128, 0, a);
  PXR_CUDA(cudaGetLastError());
  return PXR_OK;
}

// ---- window residency -----------------------------------------------------------------------------------------
int BA::resident_setup(const pxr_ba_desc* d, size_t esz) {
  resident = false;
  if (!allow_resident || n_obs == 0) return PXR_OK;
  if (const char* v = getenv("PXR_RESIDENT_WINDOW")) { const int e = std::atoi(v); if (e == 0 || !res_window_fixed) res_window = e; }
  const int W = res_window;
  if (W < 4 || C < 8 || ph > 255 || pw > 255 || ph < W + 2 || pw < W + 2) return PXR_OK;       // nothing to gain / not representable
  if ((size_t)ph * pw * C * esz > staged_chunk_bytes()) return PXR_OK;      // a whole (shared) patch must fit a staging buffer
  // the blocks must be HOST memory (a device-resident block needs no upload at all)
  auto is_device = [](const void* ptr) -> bool {
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
    return pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged;
  };
  res_srcs.clear(); res_block_first.assign(1, 0);
  if (d->n_patch_blocks > 0) {
    for (int b = 0; b < d->n_patch_blocks; ++b) {
      if (is_device(d->patch_block_ptrs[b])) return PXR_OK;
      res_srcs.push_back(d->patch_block_ptrs[b]);
      res_block_first.push_back(res_block_first.back() + d->patch_block_counts[b]);
    }
  } else {
    if (is_device(d->patches)) return PXR_OK;
    res_srcs.push_back(d->patches);
    res_block_first.push_back(n_patches);
  }
  res_esz = esz;
  cudaStream_t s = ctx->stream;
  // patches several observations read are brought over whole
  std::vector<uint8_t> shared((size_t)n_patches, 0);
  if (d->obs_patch) {
    h_obs_patch.assign(d->obs_patch, d->obs_patch + n_obs);
    std::vector<uint8_t> seen((size_t)n_patches, 0);
    for (int64_t o = 0; o < n_obs; ++o) { const int64_t p = d->obs_patch[o]; if (seen[p]) shared[p] = 1; seen[p] = 1; }
  }
  PXR_TRY(res_shared.upload(shared.data(), shared.size(), s));
  PXR_CUDA(cudaStreamSynchronize(s));             // `shared` is a local
  PXR_TRY(res_rect.alloc((size_t)n_patches)); PXR_TRY(res_rect.zero(s));
  PXR_TRY(res_viol_count.alloc(1)); PXR_TRY(res_viol_count.zero(s));
  PXR_TRY(res_viol_list.alloc((size_t)n_obs)); PXR_TRY(res_fix_list.alloc((size_t)n_obs));
  resident = true;
  return PXR_OK;
}

// K0 at the initial parameters -> rectangle of every patch -> packed window upload on its own thread (joined when
// create() returns), so the host-side layout work of create() overlaps it as it overlaps the plain slab upload
int BA::resident_begin(cudaStream_t us, double* h2d_patch) {
  cudaStream_t s = ctx->stream;
  ProjectArgs pa;
  pa.obs_img = obs_img.p; pa.obs_pt = obs_pt.p; pa.obs_patch = obs_patch.p; pa.img_cam = img_cam.p; pa.cam_model = cam_model.p;
  pa.cam_params = cam[0].p; pa.qvec = q[0].p; pa.tvec = t[0].p; pa.xyz = X[0].p;
  pa.corner = corner.p; pa.scale = scale.p; pa.ups = ups; pa.obs_begin = 0; pa.obs_end = n_obs; pa.item_index = nullptr;
  pa.uv = uv.p; pa.xy = nullptr; pa.juv = nullptr; pa.juv_stride = juv_stride; pa.juv_k = K;
  PXR_LAUNCH(ctx, ba_project_kernel<false>, (unsigned)cdiv(n_obs, 128), 128, 0, pa);
  PXR_LAUNCH(ctx, resident_rect_kernel, (unsigned)cdiv(n_obs, 256), 256, 0, uv.p, obs_patch.p, res_shared.p, n_obs, ph, pw, res_window, res_rect.p);
  PXR_CUDA(cudaGetLastError());
  auto h_rect = std::make_shared<std::vector<uint32_t>>((size_t)n_patches);
  PXR_CUDA(cudaMemcpyAsync(h_rect->data(), res_rect.p, (size_t)n_patches * 4, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  double bytes = 0;
  for (uint32_t rc : *h_rect) bytes += (double)((rc >> 16) & 255u) * (double)(rc >> 24) * C * (double)res_esz;
  *h2d_patch = bytes;
  res_thread_rc = PXR_OK;
  pxr_ctx* c = ctx;
  uint8_t* slab = patches_owned.p;
  const uint32_t* d_rect = res_rect.p;
  const int64_t np = n_patches; const int ph_ = ph, pw_ = pw, tap = C * (int)res_esz;
  res_thread = std::thread([this, c, slab, d_rect, np, ph_, pw_, tap, us, h_rect]() {
    cudaSetDevice(c->device);
    res_thread_rc = upload_windows(c, slab, res_srcs.data(), res_block_first.data(), (int)res_srcs.size(), h_rect->data(), d_rect,
                                   np, ph_, pw_, tap, nullptr, us);
    if (res_thread_rc != PXR_OK) res_thread_err = pxr_last_error();
  });
  return PXR_OK;
}

void BA::resident_args(FmEvalArgs& a) {
  if (!resident) return;
  a.res_rect = res_rect.p; a.viol_count = res_viol_count.p; a.viol_list = res_viol_list.p; a.viol_capacity = (long long)n_obs;
}

// Called after an evaluation pass: did any observation read outside its resident rectangle?  Then fetch those
// patches whole; the caller evaluates the listed observations (res_fix_list[0 .. n_fixed)) again.
int BA::resident_fix(int64_t* n_fixed) {
  *n_fixed = 0;
  if (!resident) return PXR_OK;
  cudaStream_t s = ctx->stream;
  unsigned long long n = 0;
  PXR_CUDA(cudaMemcpyAsync(&n, res_viol_count.p, sizeof(n), cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  if (n == 0) return PXR_OK;
  n = std::min<unsigned long long>(n, (unsigned long long)n_obs);      // entries beyond the capacity were dropped (reported again later)
  std::vector<int64_t> list((size_t)n);
  PXR_CUDA(cudaMemcpyAsync(list.data(), res_viol_list.p, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaMemcpyAsync(res_fix_list.p, res_viol_list.p, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
  PXR_CUDA(cudaMemsetAsync(res_viol_count.p, 0, sizeof(unsigned long long), s));
  PXR_CUDA(cudaStreamSynchronize(s));
  const size_t patch_bytes = (size_t)ph * pw * C * res_esz;
  // an observation is reported by every evaluation of it before its patch is whole (the inner iterations evaluate it
  // many times before the list is looked at): fetch each patch once
  if (res_whole.size() != (size_t)n_patches) res_whole.assign((size_t)n_patches, 0);
  int64_t fetched = 0;
  for (int64_t o : list) {
    const int64_t p = h_obs_patch.empty() ? o : h_obs_patch[(size_t)o];
    if (res_whole[(size_t)p]) continue;
    res_whole[(size_t)p] = 1; ++fetched;
    const size_t blk = (size_t)(std::upper_bound(res_block_first.begin(), res_block_first.end(), p) - res_block_first.begin()) - 1;
    const uint8_t* src = (const uint8_t*)res_srcs[blk] + (size_t)(p - res_block_first[blk]) * patch_bytes;
    PXR_CUDA(cudaMemcpyAsync(patches_owned.p + (size_t)p * patch_bytes, src, patch_bytes, cudaMemcpyHostToDevice, s));
  }
  PXR_LAUNCH(ctx, resident_mark_full_kernel, (unsigned)cdiv((int64_t)n, 256), 256, 0, res_fix_list.p, (int64_t)n, obs_patch.p, ph, pw, res_rect.p);
  PXR_CUDA(cudaGetLastError());
  res_refetched += fetched; res_passes_repeated++;
  h2d_bytes += (double)fetched * (double)patch_bytes;
  *n_fixed = (int64_t)n;
  return PXR_OK;
}

int BA::fm(int mode, double* residuals_out, double* cost_dev, double* grad_out) {
  PXR_TRY(fm_k1(mode, residuals_out, grad_out, nullptr, n_obs));
  for (;;) {      // window residency: observations that left their window are evaluated again once their patch is whole
    int64_t n_fixed = 0;
    PXR_TRY(resident_fix(&n_fixed));
    if (n_fixed == 0) break;
    PXR_TRY(fm_k1(mode, residuals_out, grad_out, res_fix_list.p, n_fixed));
  }
  return fm_cost(cost_dev);
}

int BA::fm_k1(int mode, double* residuals_out, double* grad_out, const int64_t* list, int64_t n) {
  if (n <= 0 || n_obs == 0) return PXR_OK;
  FmEvalArgs a;
  a.uv = uv.p; a.item_patch = obs_patch.p; a.item_ref = obs_pt.p;
  a.patches = d_patches; a.ph = ph; a.pw = pw;
  a.refs = has_refs ? refs.p : nullptr;
  a.begin = 0; a.end = n; a.item_index = list;
  a.out = obs_out.p; a.residuals = residuals_out; a.desc = nullptr; a.grad = grad_out;
  a.loss.type = opt.loss_type; a.loss.a = opt.loss_scale;
  a.l2_normalize = interp.l2_normalize;
  resident_args(a);
  int np = 0;
  StageScope st(this, mode ? 1 : 0);
  return launch_fm_eval(ctx, dtype, C, mode, interp.use_float_simd != 0, a, &np);
}

int BA::fm_cost(double* cost_dev /* device scalar */) {
  if (n_obs > 0) {
    StageScope st2(this, 10);
    LossParams loss; loss.type = opt.loss_type; loss.a = opt.loss_scale;
    const int cb = std::min<int>(fm_max_partials(ctx), ctx->sm_count * 8);
    PXR_LAUNCH(ctx, cost_from_sq_norm_kernel, cb, 256, 0, obs_out.p, (int64_t)0, n_obs, loss, partials.p);
    PXR_LAUNCH(ctx, reduce_partials_kernel, 1, 1024, 0, partials.p, (int64_t)cb, cost_dev);
  } else {
    PXR_CUDA(cudaMemsetAsync(cost_dev, 0, 8, ctx->stream));
  }
  return PXR_OK;
}

// cost (and with jac the full linearisation) at parameter set `set`; returns the global cost
int BA::evaluate(int set, bool jac, double* cost_out) {
  PXR_TRY(project(set, jac, nullptr));
  PXR_TRY(fm(jac ? 1 : 0, nullptr, scalars.p + 0));
  if (jac) PXR_TRY(build());
  return read_cost(cost_out);
}

// the global cost from this rank's part in scalars[0]
int BA::read_cost(double* cost_out) {
  if (block_mode) return global_cost_block(cost_out);
  PXR_TRY(allreduce_f64(ctx, scalars.p + 0, 1));
  double c = 0;
  PXR_CUDA(cudaMemcpyAsync(&c, scalars.p + 0, 8, cudaMemcpyDeviceToHost, ctx->stream));
  PXR_CUDA(cudaStreamSynchronize(ctx->stream));
  *cost_out = c;
  return PXR_OK;
}

BADev BA::dev() {
  BADev d;
  d.n_cameras = n_cameras; d.n_images = n_images; d.K = K; d.n_points = n_points; d.n_obs = n_obs;
  d.nc = nc; d.nl = (int)nl; d.dcmax = dcmax; d.juv_stride = juv_stride;
  d.obs_img = obs_img.p; d.obs_pt = obs_pt.p; d.img_cam = img_cam.p; d.cam_model = cam_model.p;
  d.cam_mask = cam_mask.p; d.tmask = tmask.p; d.pose_off = pose_off.p; d.intr_off = intr_off.p;
  d.point_off = point_off.p; d.pt_begin = pt_begin.p; d.obs_out = obs_out.p; d.juv = juv.p;
  d.img_cols8 = img_cols8.p; d.img_src8 = img_src8.p; d.img_dc8 = img_dc8.p;
  d.Hcc = Hcc.p; d.Hpp = Hpp.p; d.gp = gp.p; d.W = W.p; d.Wcols = Wcols.p; d.Wdc = Wdc.p;
  d.gc = block_mode ? pack_local.p + pk_off_gc : gc.p;   // block mode: the partial gradient lives in the packed buffer
  d.loss.type = opt.loss_type; d.loss.a = opt.loss_scale;
  return d;
}

int BA::build() {
  if (block_mode) return build_block();
  StageScope st(this, 3);
  if (!sparse_schur) PXR_TRY(Hcc.zero(ctx->stream));
  PXR_TRY(gc.zero(ctx->stream));
  PXR_TRY(Hpp.zero(ctx->stream));
  PXR_TRY(gp.zero(ctx->stream));
  const bool chunked = io_n_chunks > 0 && (sparse_schur || !env.build_atomic);
  if (sparse_schur && !chunked && n_obs > 0) return fail(PXR_ERR_INTERNAL, "block-sparse path without per-image chunks");
  if (sparse_schur) PXR_TRY(ss_Himg.zero(ctx->stream));
  if (n_obs > 0) {
    const BADev dv = dev();
    const size_t staged_smem = (size_t)128 * ((std::max(dv.juv_stride, dv.dcmax * 3) | 1) + 9) * sizeof(double);
    if (img_src8.p && chunked && env.build_staged && staged_smem <= 48 * 1024)
      PXR_LAUNCH(ctx, ba_build_staged_kernel, (unsigned)cdiv(n_obs, 128), 128, staged_smem, dv);
    else if (img_src8.p) PXR_LAUNCH(ctx, ba_build_kernel<true>, (unsigned)cdiv(n_obs, 128), 128, 0, dv, chunked ? 0 : 1);
    else PXR_LAUNCH(ctx, ba_build_kernel<false>, (unsigned)cdiv(n_obs, 128), 128, 0, dv, chunked ? 0 : 1);
  }
  if (n_obs > 0 && chunked)
    PXR_LAUNCH(ctx, ba_build_cam_kernel, (unsigned)cdiv(io_n_chunks * 32, 256), 256, 0, dev(), io_obs.p, io_chunk_begin.p, io_n_chunks,
               sparse_schur ? ss_Himg.p : nullptr);
  const int64_t n = std::max<int64_t>(nc, n_points);
  if (sparse_schur && nc > 0) PXR_CUDA(cudaMemsetAsync(diag.p, 0, (size_t)nc * 8, ctx->stream));
  if (n > 0) PXR_LAUNCH(ctx, ba_diag_kernel, (unsigned)cdiv(n, 256), 256, 0, dev(), diag.p);
  if (sparse_schur && nc > 0) PXR_LAUNCH(ctx, sp_diag_kernel, (unsigned)cdiv((int64_t)n_images * 8, 256), 256, 0, sparse(), diag.p);
  if (ctx->world > 1 && nc > 0) {
    // multi-GPU: Hcc stays a per-rank partial sum (it only ever enters the reduced system, which is all-reduced
    // anyway); globally needed are its diagonal (Jacobi scaling / LM damping) and the gradient
    if (!gc_local.p) { PXR_TRY(gc_local.alloc(nc)); PXR_TRY(ar_buf.alloc((size_t)2 * nc)); }
    PXR_CUDA(cudaMemcpyAsync(gc_local.p, gc.p, (size_t)nc * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    // one collective for [diag(Hcc) | gc]
    PXR_CUDA(cudaMemcpyAsync(ar_buf.p, diag.p, (size_t)nc * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    PXR_CUDA(cudaMemcpyAsync(ar_buf.p + nc, gc.p, (size_t)nc * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    PXR_TRY(allreduce_f64(ctx, ar_buf.p, (size_t)2 * nc));
    PXR_CUDA(cudaMemcpyAsync(diag.p, ar_buf.p, (size_t)nc * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    PXR_CUDA(cudaMemcpyAsync(gc.p, ar_buf.p + nc, (size_t)nc * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  }
  PXR_CUDA(cudaGetLastError());
  return PXR_OK;
}

SparseSchur BA::sparse() {
  SparseSchur q;
  q.n_images = n_images; q.n_keys = ss_n_keys; q.nc = nc;
  q.img_cols = ss_img_cols.p; q.img_pd = ss_img_pd.p; q.img_pose_blk = ss_img_pose_blk.p; q.img_cam_blk = ss_img_cam_blk.p;
  q.key_a = ss_key_a.p; q.key_b = ss_key_b.p; q.key_self = ss_key_self.p;
  q.Himg = ss_Himg.p; q.Bk = ss_Bk.p;
  return q;
}

// Dense Cholesky of [S; rhs] + both substitutions (pxr_chol.cuh) -> delta[0..nc): captured once into a CUDA graph.
int BA::chol_launch() {
  cudaStream_t s = ctx->stream;
    // The factorisation + back-substitution is a fixed sequence of ~3*nc/32 dependent launches: it is
    // captured once into a CUDA graph and replayed, which removes the per-launch gaps.
    if (!chol_graph_exec) {
      chol_multikernel = chol_force_multikernel || env.chol_multikernel;
      if (!chol_multikernel) {
        // every CTA of the persistent kernel must be resident at once: grid = occupancy x SMs
        int per_sm = 0, sms = 0, dev = 0;
        PXR_CUDA(cudaGetDevice(&dev));
        PXR_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        chol_band = getenv("PXR_CHOL_BAND") != nullptr;     // the band design (pxr_chol2.cuh) is opt-in: see DESIGN.md section 3
        if (chol_band) {
          PXR_CUDA(cudaFuncSetAttribute(pxr_chol2::chol_band_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pxr_chol2::smem_bytes()));
          PXR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pxr_chol2::chol_band_kernel, pxr_chol::kThreads, pxr_chol2::smem_bytes()));
        } else {
          PXR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pxr_chol::chol_persistent_kernel, pxr_chol::kThreads, 0));
        }
        if (per_sm < 1) return pxr::fail(PXR_ERR_CUDA, "persistent Cholesky kernel does not fit on an SM");
        const int nbt = (int)cdiv(nc, kNB);
        const int64_t tiles = (int64_t)(nbt + 1) * nbt / 2 + nbt;
        chol_grid = (int)std::min<int64_t>((int64_t)per_sm * sms, std::max<int64_t>(2, tiles + 1));
        PXR_TRY(chol_sync.alloc(pxr_chol::sync_ints(nbt)));
        if (!env.chol_trace.empty()) { PXR_TRY(chol_trace.alloc((size_t)(nbt + 3) * 8 + nbt)); PXR_TRY(chol_trace.zero(s)); }
      }
      cudaGraph_t graph = nullptr;
      PXR_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
      // an error between Begin and EndCapture must not leave the context's stream capturing
      struct CaptureGuard { cudaStream_t s; bool armed = true; ~CaptureGuard() { if (armed) { cudaGraph_t g = nullptr; cudaStreamEndCapture(s, &g); if (g) cudaGraphDestroy(g); } } } cap_guard{s};
      const int nb = (int)cdiv(nc, kNB);
      int64_t captured = 0;
      if (!chol_multikernel) {
        // one persistent kernel: tile DAG with flags (pxr_chol.cuh); the memset of the flags is part of the graph
        PXR_CUDA(cudaMemsetAsync(chol_sync.p, 0, chol_sync.n * sizeof(int), s));
        PXR_CUDA(cudaMemsetAsync(delta.p, 0xFF, (size_t)nc * 8, s));   // x doubles as its own ready flag (pxr_chol.cuh)
        pxr_chol::Args ca;
        ca.A = S.p; ca.x = delta.p; ca.n = nc; ca.nb = nb;
        ca.diag_ready = chol_sync.p; ca.ready = ca.diag_ready + nb; ca.upd = ca.ready + (size_t)(nb + 1) * nb;
        ca.xready = ca.upd + (size_t)(nb + 1) * nb; ca.abort = ca.xready + nb; ca.fail_flag = flags.p + 1; ca.trace = chol_trace.p;
        if (chol_band) pxr_chol2::chol_band_kernel<<<chol_grid, pxr_chol::kThreads, pxr_chol2::smem_bytes(), s>>>(ca);
        else pxr_chol::chol_persistent_kernel<<<chol_grid, pxr_chol::kThreads, 0, s>>>(ca);
        ++captured;
      } else {
      for (int k = 0; k < nb; ++k) {
        const int k0 = k * kNB, kb = std::min(kNB, nc - k0);
        const int rows_below = nc + 1 - (k0 + kb);               // includes the rhs row
        chol_diag_kernel<<<1, 32, 0, s>>>(S.p, nc, k, rdiag.p, flags.p + 1); ++captured;
        if (rows_below > 0) { chol_panel_kernel<<<(unsigned)cdiv(rows_below, kNB), kPanelThreads, 0, s>>>(S.p, nc, nc + 1, k, rdiag.p); ++captured; }
        const int nrb = (int)cdiv(nc + 1, kNB);
        const int rem = nrb - (k + 1);
        if (rem > 0 && kb == kNB) { chol_update_kernel<<<rem * (rem + 1) / 2, kNB * kNB, 0, s>>>(S.p, nc, nc + 1, k); ++captured; }
      }
      chol_backsolve_kernel<<<1, 1024, 0, s>>>(S.p, S.p + (size_t)nc * nc, delta.p, nc); ++captured;
      }
      cap_guard.armed = false;
      PXR_CUDA(cudaStreamEndCapture(s, &graph));
      PXR_CUDA(cudaGraphInstantiate(&chol_graph_exec, graph, 0));
      cudaGraphDestroy(graph);
      chol_graph_kernels = captured;
    }
    PXR_CUDA(cudaGraphLaunch(chol_graph_exec, s));
    ctx->launches += chol_graph_kernels;
    if (chol_trace.p) {   // debugging aid: dump the panel CTA's time line of this factorisation
      std::vector<long long> h(chol_trace.n);
      PXR_CUDA(cudaMemcpyAsync(h.data(), chol_trace.p, h.size() * 8, cudaMemcpyDeviceToHost, s));
      PXR_CUDA(cudaStreamSynchronize(s));
      if (FILE* f = fopen(env.chol_trace.c_str(), "w")) {
        const int nbt = (int)cdiv(nc, kNB);
        const int rows = chol_band ? nbt + 1 : nbt;      // the band kernel also walks the rhs row
        for (int k = 0; k < rows; ++k) { for (int q = 0; q < 7; ++q) fprintf(f, "%lld ", h[(size_t)k * 8 + q] - h[0]); fprintf(f, "\n"); }
        const size_t tail = (size_t)(chol_band ? nbt + 1 : nbt) * 8;
        fprintf(f, "backsolve_start %lld\n", h[tail] - h[0]);
        for (int c = nbt - 1; c >= 0; --c) fprintf(f, "x %d %lld\n", c, h[tail + 8 + c] - h[0]);
        fclose(f);
      }
    }
    return PXR_OK;
}

// S -= sum over observation pairs T_x W_y^T, rhs += sum T gp: the staged pair kernel when every image has at most 8
// columns (the usual case: pose + up to two intrinsics, or pose only), the direct kernels otherwise
int BA::launch_schur_pairs(const BADev& d) {
  if (sp_n_chunks <= 0) return PXR_OK;
  const unsigned pair_grid = (unsigned)cdiv(sp_n_chunks * 32, kPairThreads);
  const bool small = img_dc_max <= 8 && dcmax >= 9;   // dcmax = 6 + K >= 9 for every camera model: row 8 of a record exists
  if (small && schur_kernel == 0) {                   // fused tensor-core walk: no T buffer
    if (schur_ctas == 3) PXR_LAUNCH(ctx, (ba_schur_pairs_mma_kernel<3, true>), pair_grid, kPairThreads, 0, d, schur_pairs(), Hinv.p, S.p, rhs.p);
    else PXR_LAUNCH(ctx, (ba_schur_pairs_mma_kernel<4, true>), pair_grid, kPairThreads, 0, d, schur_pairs(), Hinv.p, S.p, rhs.p);
    return PXR_OK;
  }
  PXR_LAUNCH(ctx, ba_schur_prep_kernel, (unsigned)cdiv(n_obs * dcmax, 256), 256, 0, d, Hinv.p, Tbuf.p);
  if (small && schur_kernel == 3) {
    if (schur_ctas == 4) PXR_LAUNCH(ctx, (ba_schur_pairs_mma_kernel<4, false>), pair_grid, kPairThreads, 0, d, schur_pairs(), Tbuf.p, S.p, rhs.p);
    else PXR_LAUNCH(ctx, (ba_schur_pairs_mma_kernel<3, false>), pair_grid, kPairThreads, 0, d, schur_pairs(), Tbuf.p, S.p, rhs.p);
  } else if (small && schur_kernel == 1) {
    const bool vec = dcmax % 2 == 0;               // 16-byte gathers need 16-byte records
    if (schur_ctas == 3) {
      if (vec) PXR_LAUNCH(ctx, (ba_schur_pairs_staged_kernel<true, 3>), pair_grid, kPairThreads, 0, d, schur_pairs(), Tbuf.p, S.p, rhs.p);
      else PXR_LAUNCH(ctx, (ba_schur_pairs_staged_kernel<false, 3>), pair_grid, kPairThreads, 0, d, schur_pairs(), Tbuf.p, S.p, rhs.p);
    } else {
      if (vec) PXR_LAUNCH(ctx, (ba_schur_pairs_staged_kernel<true, 4>), pair_grid, kPairThreads, 0, d, schur_pairs(), Tbuf.p, S.p, rhs.p);
      else PXR_LAUNCH(ctx, (ba_schur_pairs_staged_kernel<false, 4>), pair_grid, kPairThreads, 0, d, schur_pairs(), Tbuf.p, S.p, rhs.p);
    }
  } else if (img_dc_max <= 8) PXR_LAUNCH(ctx, ba_schur_pairs_kernel<true>, pair_grid, kPairThreads, 0, d, schur_pairs(), Tbuf.p, S.p, rhs.p);
  else PXR_LAUNCH(ctx, ba_schur_pairs_kernel<false>, pair_grid, kPairThreads, 0, d, schur_pairs(), Tbuf.p, S.p, rhs.p);
  return PXR_OK;
}

// the same walk with the image-pair blocks as the sink (block-sparse ITERATIVE_SCHUR, block mode); these paths only
// exist for images of at most 8 columns
int BA::launch_sp_schur_pairs(const BADev& d, double* Bk, double* rhs_out, double* part) {
  if (sp_n_chunks <= 0) return PXR_OK;
  const unsigned pair_grid = (unsigned)cdiv(sp_n_chunks * 32, kPairThreads);
  if (dcmax >= 9 && schur_kernel == 0) {
    PXR_LAUNCH(ctx, sp_schur_pairs_kernel<4>, pair_grid, kPairThreads, 0, d, schur_pairs(), ss_chunk_key.p, Hinv.p, Bk, rhs_out, part);
    return PXR_OK;
  }
  PXR_LAUNCH(ctx, ba_schur_prep_kernel, (unsigned)cdiv(n_obs * dcmax, 256), 256, 0, d, Hinv.p, Tbuf.p);
  if (dcmax >= 9 && schur_kernel == 3) PXR_LAUNCH(ctx, sp_schur_pairs_kernel<3>, pair_grid, kPairThreads, 0, d, schur_pairs(), ss_chunk_key.p, Tbuf.p, Bk, rhs_out, part);
  else if (dcmax >= 9 && schur_kernel == 1) {
    if (dcmax % 2 == 0) PXR_LAUNCH(ctx, sp_schur_pairs_kernel<1>, pair_grid, kPairThreads, 0, d, schur_pairs(), ss_chunk_key.p, Tbuf.p, Bk, rhs_out, part);
    else PXR_LAUNCH(ctx, sp_schur_pairs_kernel<2>, pair_grid, kPairThreads, 0, d, schur_pairs(), ss_chunk_key.p, Tbuf.p, Bk, rhs_out, part);
  } else PXR_LAUNCH(ctx, sp_schur_pairs_kernel<0>, pair_grid, kPairThreads, 0, d, schur_pairs(), ss_chunk_key.p, Tbuf.p, Bk, rhs_out, part);
  return PXR_OK;
}

// One LM step attempt at the current linearisation: fills delta, returns validity and model cost change
int BA::compute_step(double radius, bool* valid, double* model_cost_change) {
  cudaStream_t s = ctx->stream;
  PXR_TRY(build_schur_pairs());
  if (block_mode) return compute_step_block_sync(radius, valid, model_cost_change);
  BADev d = dev();
  std::unique_ptr<StageScope> st(new StageScope(this, 4));   // RAII: an early error return still closes the stage
  if (nl > 0) PXR_LAUNCH(ctx, ba_d2_kernel, (unsigned)cdiv(nl, 256), 256, 0, diag.p, jscale.p, D2.p, nl, radius,
                         opt.min_lm_diagonal, opt.max_lm_diagonal);
  PXR_CUDA(cudaMemsetAsync(flags.p, 0, 4 * sizeof(int), s));
  if (sparse_schur) {
    // image-block form (pxr_sparse_schur.cuh): rhs = -gc + sum T gp, B_ab = sum T_x W_y^T; nothing of size nc^2
    if (nc > 0) PXR_LAUNCH(ctx, sp_init_rhs_kernel, (unsigned)cdiv(nc, 256), 256, 0, ctx->world > 1 ? gc_local.p : gc.p, rhs.p, nc);
    PXR_TRY(ss_Bk.zero(s));
    if (n_points > 0) {
      PXR_LAUNCH(ctx, ba_point_inverse_kernel, (unsigned)cdiv(n_points, 256), 256, 0, d, D2.p, Hinv.p, flags.p);
      PXR_TRY(launch_sp_schur_pairs(d, ss_Bk.p, rhs.p, nullptr));   // T = W Hinv first, unless the walk forms it itself
    }
    if (ctx->world > 1 && nc > 0) PXR_TRY(allreduce_f64(ctx, rhs.p, nc));
  } else {
  // multi-GPU: every rank starts from ITS partial Hcc / gc (rank 0 adds the damping), subtracts its points' Schur
  // contributions, and ONE all-reduce of [S | rhs] (rhs is row nc of the same array) yields the reduced system
  if (nc > 0) PXR_LAUNCH(ctx, ba_init_reduced_kernel, (unsigned)cdiv((int64_t)nc * nc, 256), 256, 0, Hcc.p,
                         ctx->world > 1 ? gc_local.p : gc.p, D2.p, S.p, rhs.p, nc, (ctx->world <= 1 || ctx->rank == 0) ? 1 : 0);
  if (n_points > 0) {
    PXR_LAUNCH(ctx, ba_point_inverse_kernel, (unsigned)cdiv(n_points, 256), 256, 0, d, D2.p, Hinv.p, flags.p);
    PXR_TRY(launch_schur_pairs(d));
  }
  // rhs rides along as row nc of S: the factorisation performs the forward substitution
  if (nc > 0) PXR_CUDA(cudaMemcpyAsync(S.p + (size_t)nc * nc, rhs.p, (size_t)nc * 8, cudaMemcpyDeviceToDevice, s));
  if (ctx->world > 1 && nc > 0) {
    PXR_TRY(allreduce_f64(ctx, S.p, (size_t)(nc + 1) * nc));
    PXR_CUDA(cudaMemcpyAsync(rhs.p, S.p + (size_t)nc * nc, (size_t)nc * 8, cudaMemcpyDeviceToDevice, s));   // PCG / debug read rhs
  }
  }
  st.reset(); st.reset(new StageScope(this, 5));
  last_linear_iterations = 1;
  if (nc > 0 && sparse_schur) {
    PXR_TRY(pcg_solve_sparse());
  } else if (nc > 0 && use_pcg) {
    PXR_TRY(pcg_solve());
  } else if (nc > 0) {
    PXR_TRY(chol_launch());
  }
  st.reset(); st.reset(new StageScope(this, 7));
  PXR_CUDA(cudaMemsetAsync(scalars.p + 4, 0, 4 * 8, s));  // acc[0..3]
  if (n_points > 0) PXR_LAUNCH(ctx, ba_backsub_kernel, (unsigned)cdiv(n_points * 32, 256), 256, 0, d, D2.p, delta.p);
  if (n_obs > 0) {
    if (img_src8.p) PXR_LAUNCH(ctx, ba_model_cost_kernel<true>, (unsigned)cdiv(n_obs, 256), 256, 0, d, delta.p, scalars.p + 4);
    else PXR_LAUNCH(ctx, ba_model_cost_kernel<false>, (unsigned)cdiv(n_obs, 256), 256, 0, d, delta.p, scalars.p + 4);
  }
  PXR_CUDA(cudaGetLastError());
  st.reset();
  double acc = 0, fld = 0;
  if (chol_graph_exec && !chol_multikernel && !use_pcg && env.chol_test_abort) {
    // test hook: pretend the persistent kernel bailed out of a wait (abort word + failure flag)
    const int one = 1;
    PXR_CUDA(cudaMemcpyAsync(chol_sync.p + (pxr_chol::sync_ints((int)cdiv(nc, kNB)) - 1), &one, sizeof(int), cudaMemcpyHostToDevice, s));
    PXR_CUDA(cudaMemcpyAsync(flags.p + 1, &one, sizeof(int), cudaMemcpyHostToDevice, s));
    PXR_CUDA(cudaStreamSynchronize(s));
  }
  PXR_LAUNCH(ctx, flags_to_double_kernel, 1, 1, 0, flags.p, scalars.p + 5);
  PXR_TRY(allreduce_f64(ctx, scalars.p + 4, 2));   // model cost change + failure flag: every rank takes the same branch
  double two[2] = {0, 0};
  PXR_CUDA(cudaMemcpyAsync(two, scalars.p + 4, 16, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  acc = two[0]; fld = two[1];
  if (fld != 0.0 && chol_graph_exec && !chol_multikernel && !use_pcg && ctx->world <= 1) {
    // Did the persistent Cholesky bail out of a wait?  That only happens when its CTAs were not all resident at
    // once (GPU shared with another client, MPS/MIG partition smaller than queried): switch, for the rest of this
    // handle's life, to the launch-per-panel path, which needs no co-residency, and redo this step.
    int aborted = 0;
    const int nbt = (int)cdiv(nc, kNB);
    PXR_CUDA(cudaMemcpyAsync(&aborted, chol_sync.p + (pxr_chol::sync_ints(nbt) - 1), sizeof(int), cudaMemcpyDeviceToHost, s));
    PXR_CUDA(cudaStreamSynchronize(s));
    if (aborted) {
      cudaGraphExecDestroy(chol_graph_exec); chol_graph_exec = nullptr;
      chol_force_multikernel = true;
      return compute_step(radius, valid, model_cost_change);
    }
  }
  const bool solved = fld == 0.0 && std::isfinite(acc);
  *model_cost_change = -acc;
  *valid = solved && (*model_cost_change > 0.0);
  return PXR_OK;
}

// candidate (other set) = Plus(current, delta); returns ||step|| and ||x|| (ambient)
int BA::apply_step(double* step_norm, double* x_norm) {
  PlusArgs a;
  a.n_cameras = n_cameras; a.n_images = n_images; a.n_points = n_points;
  a.cam_model = cam_model.p; a.cam_mask = cam_mask.p; a.tmask = tmask.p;
  a.pose_off = pose_off.p; a.intr_off = intr_off.p; a.point_off = point_off.p;
  a.cam = cam[cur].p; a.q = q[cur].p; a.t = t[cur].p; a.X = X[cur].p;
  a.cam_o = cam[1 - cur].p; a.q_o = q[1 - cur].p; a.t_o = t[1 - cur].p; a.X_o = X[1 - cur].p;
  a.delta = delta.p; a.acc = scalars.p + 4;
  StageScope st(this, 8);
  PXR_CUDA(cudaMemsetAsync(scalars.p + 5, 0, 4 * 8, ctx->stream));
  const int64_t n = std::max<int64_t>(std::max<int64_t>(n_points, n_images), n_cameras);
  if (deterministic) a.part = det_scal_part.p;
  PXR_LAUNCH(ctx, ba_plus_kernel, (unsigned)cdiv(n, 128), 128, 0, a);
  if (deterministic)
    for (int k = 0; k < 4; ++k) PXR_LAUNCH(ctx, det_reduce_add_kernel, 1, 1024, 0, det_scal_part.p, cdiv(n, 128), 4, k, a.acc + 1 + k);
  PXR_CUDA(cudaGetLastError());
  if (!block_mode) PXR_TRY(allreduce_f64(ctx, scalars.p + 5, 2));  // point parts are sharded, camera parts replicated (block mode: scalar exchange)
  if (step_norm || x_norm) {
    double v[4];
    PXR_CUDA(cudaMemcpyAsync(v, scalars.p + 5, 32, cudaMemcpyDeviceToHost, ctx->stream));
    PXR_CUDA(cudaStreamSynchronize(ctx->stream));
    if (step_norm) *step_norm = std::sqrt(v[0] + v[2]);
    if (x_norm) *x_norm = std::sqrt(v[1] + v[3]);
  }
  return PXR_OK;
}

// Inner iterations: one launch of inner_fused_kernel (pxr_inner.cuh) solves every variable point with the cameras
// of parameter set `set` fixed.  It leaves in obs_out[o*8] the squared norm of every observation of those points at
// the point's final position, so the cost after the inner iterations is fm_cost() over obs_out.
int BA::inner_iterations(int set) {
  if (n_points == 0 || n_obs == 0) return PXR_OK;
  StageScope stg(this, 9);
  cudaStream_t s = ctx->stream;
  if (!inner_rec.p) { PXR_TRY(inner_rec.alloc((size_t)n_obs * kInnerRec)); PXR_TRY(inner_next.alloc(1)); }
  InnerArgs a;
  a.n_points = n_points; a.point_off = point_off.p; a.pt_begin = pt_begin.p;
  a.geo.obs_img = obs_img.p; a.geo.obs_pt = obs_pt.p; a.geo.obs_patch = obs_patch.p;
  a.geo.img_cam = img_cam.p; a.geo.cam_model = cam_model.p;
  a.geo.cam_params = cam[set].p; a.geo.qvec = q[set].p; a.geo.tvec = t[set].p; a.geo.xyz = X[set].p;
  a.geo.corner = corner.p; a.geo.scale = scale.p; a.geo.ups = ups;
  a.geo.obs_begin = 0; a.geo.obs_end = n_obs; a.geo.item_index = nullptr;
  a.geo.uv = nullptr; a.geo.xy = nullptr; a.geo.juv = nullptr; a.geo.juv_stride = juv_stride; a.geo.juv_k = K;
  a.fm.uv = nullptr; a.fm.item_patch = obs_patch.p; a.fm.item_ref = obs_pt.p;
  a.fm.patches = d_patches; a.fm.ph = ph; a.fm.pw = pw;
  a.fm.refs = has_refs ? refs.p : nullptr;
  a.fm.begin = 0; a.fm.end = n_obs; a.fm.item_index = nullptr;
  a.fm.out = obs_out.p; a.fm.residuals = nullptr; a.fm.desc = nullptr;
  a.fm.loss.type = opt.loss_type; a.fm.loss.a = opt.loss_scale;
  a.fm.l2_normalize = interp.l2_normalize;
  resident_args(a.fm);
  a.xyz = X[set].p; a.rec = inner_rec.p; a.next_point = inner_next.p;
  // window residency: an observation may leave its window in any evaluation and nobody looks before the kernel is
  // over — keep the starting points, and if something was reported fetch those patches and run again from the start
  if (resident) {
    if (!inner_snapshot.p) PXR_TRY(inner_snapshot.alloc((size_t)n_points * 3));
    PXR_CUDA(cudaMemcpyAsync(inner_snapshot.p, X[set].p, (size_t)n_points * 24, cudaMemcpyDeviceToDevice, s));
  }
  for (;;) {
    PXR_CUDA(cudaMemsetAsync(inner_next.p, 0, sizeof(unsigned long long), s));
    PXR_TRY(launch_inner_fused(ctx, dtype, C, interp.use_float_simd != 0, a));
    int64_t n_fixed = 0;
    PXR_TRY(resident_fix(&n_fixed));
    if (n_fixed == 0) break;
    PXR_CUDA(cudaMemcpyAsync(X[set].p, inner_snapshot.p, (size_t)n_points * 24, cudaMemcpyDeviceToDevice, s));
  }
  return PXR_OK;
}

int BA::step_norm_between_sets(double* out) {
  cudaStream_t s = ctx->stream;
  PXR_CUDA(cudaMemsetAsync(scalars.p + 11, 0, 16, s));
  auto run = [&](const double* a, const double* b, int64_t n, double* acc) {
    if (n > 0) PXR_LAUNCH(ctx, diff_norm_kernel, (unsigned)cdiv(n, 256), 256, 0, a, b, n, acc);
  };
  run(cam[0].p, cam[1].p, (int64_t)n_cameras * kMaxK, scalars.p + 12);
  run(q[0].p, q[1].p, (int64_t)n_images * 4, scalars.p + 12);
  run(t[0].p, t[1].p, (int64_t)n_images * 3, scalars.p + 12);
  run(X[0].p, X[1].p, n_points * 3, scalars.p + 11);
  PXR_TRY(allreduce_f64(ctx, scalars.p + 11, 1));
  double v[2] = {0, 0};
  PXR_CUDA(cudaMemcpyAsync(v, scalars.p + 11, 16, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  *out = std::sqrt(v[0] + v[1]);
  return PXR_OK;
}

// S delta_c = rhs by Schur-Jacobi preconditioned CG (pxr_pcg.cuh); result in delta[0..nc)
int BA::pcg_setup_blocks() {
  if (cg_state.p) return PXR_OK;
  cudaStream_t s = ctx->stream;
  // SCHUR_JACOBI blocks = the camera-side parameter blocks (one per variable pose, one per variable intrinsics)
  std::vector<int32_t> off;
  for (int i = 0; i < n_images; ++i) if (h_pose_off[i] >= 0) off.push_back(h_pose_off[i]);
  for (int c = 0; c < n_cameras; ++c) if (h_intr_off[c] >= 0) off.push_back(h_intr_off[c]);
  std::sort(off.begin(), off.end());
  std::vector<int32_t> sd(off.size());
  for (size_t k = 0; k < off.size(); ++k) sd[k] = (k + 1 < off.size() ? off[k + 1] : nc) - off[k];
  cg_nblk = (int)off.size();
  PXR_TRY(cg_blk_off.upload(off.data(), off.size(), s)); PXR_TRY(cg_blk_dim.upload(sd.data(), sd.size(), s));
  PXR_TRY(cg_Minv.alloc((size_t)nc * 12)); PXR_TRY(cg_row_off.alloc(nc)); PXR_TRY(cg_row_dim.alloc(nc));
  PXR_TRY(cg_z.alloc(nc)); PXR_TRY(cg_p.alloc(nc)); PXR_TRY(cg_q.alloc(nc)); PXR_TRY(cg_r.alloc(nc)); PXR_TRY(cg_x.alloc(nc)); PXR_TRY(cg_tmp.alloc(nc));
  PXR_TRY(cg_state.alloc(1));
  if (sparse_schur) {
    auto blk_of = [&](int offset) -> int32_t { return (int32_t)(std::lower_bound(off.begin(), off.end(), offset) - off.begin()); };
    h_img_pose_blk.assign(n_images, -1); h_img_cam_blk.assign(n_images, -1);
    for (int i = 0; i < n_images; ++i) {
      if (h_pose_off[i] >= 0) h_img_pose_blk[i] = blk_of(h_pose_off[i]);
      const int io = h_intr_off[h_img_cam[i]];
      if (io >= 0) h_img_cam_blk[i] = blk_of(io);
    }
    PXR_TRY(ss_img_pose_blk.upload(h_img_pose_blk.data(), h_img_pose_blk.size(), s));
    PXR_TRY(ss_img_cam_blk.upload(h_img_cam_blk.data(), h_img_cam_blk.size(), s));
    PXR_TRY(ss_Dblk.alloc((size_t)std::max(cg_nblk, 1) * 144));
  }
  PXR_CUDA(cudaStreamSynchronize(s));
  return PXR_OK;
}

// ITERATIVE_SCHUR on the implicit block-sparse reduced system (pxr_sparse_schur.cuh).  Same CG recurrences and
// termination as pcg_solve(); the mat-vec gathers/scatters through the image blocks, and in the multi-GPU path the
// product (nc doubles) is all-reduced per iteration instead of the matrix once.
int BA::pcg_solve_sparse() {
  cudaStream_t s = ctx->stream;
  PXR_TRY(pcg_setup_blocks());
  const int n = nc;
  const SparseSchur sp = sparse();
  const int64_t nthreads = std::max<int64_t>(((int64_t)n_images + ss_n_keys) * 8, n);
  const unsigned gs = (unsigned)cdiv(nthreads, 256);
  const int add_d2 = (ctx->world <= 1 || ctx->rank == 0) ? 1 : 0;
  auto spmv = [&](const double* x, double* y) -> int {
    PXR_CUDA(cudaMemsetAsync(y, 0, (size_t)n * 8, s));
    PXR_LAUNCH(ctx, sp_spmv_kernel, gs, 256, 0, sp, D2.p, x, y, add_d2, cg_state.p);
    if (ctx->world > 1) PXR_TRY(allreduce_f64(ctx, y, n));
    return PXR_OK;
  };
  PXR_TRY(ss_Dblk.zero(s));
  PXR_LAUNCH(ctx, sp_blockdiag_kernel, (unsigned)cdiv(((int64_t)n_images + ss_n_keys) * 8, 256), 256, 0, sp, ss_Dblk.p);
  if (ctx->world > 1) PXR_TRY(allreduce_f64(ctx, ss_Dblk.p, (size_t)cg_nblk * 144));
  PXR_LAUNCH(ctx, sp_block_inverse_kernel, (unsigned)cdiv(cg_nblk, 64), 64, 0, ss_Dblk.p, D2.p, 1, cg_blk_off.p, cg_blk_dim.p, cg_nblk,
             cg_Minv.p, cg_row_off.p, cg_row_dim.p, flags.p + 1);
  return run_cg(spmv);
}

int BA::pcg_solve() {
  cudaStream_t s = ctx->stream;
  PXR_TRY(pcg_setup_blocks());
  const int n = nc;
  const unsigned gv = (unsigned)cdiv((int64_t)n * 32, 256);
  PXR_LAUNCH(ctx, cg_mirror_kernel, (unsigned)cdiv((int64_t)n * n, 256), 256, 0, S.p, n);
  PXR_LAUNCH(ctx, cg_block_inverse_kernel, (unsigned)cdiv(cg_nblk, 64), 64, 0, S.p, n, cg_blk_off.p, cg_blk_dim.p, cg_nblk, cg_Minv.p,
             cg_row_off.p, cg_row_dim.p, flags.p + 1);
  auto spmv = [&](const double* x, double* y) -> int {
    PXR_LAUNCH(ctx, cg_gemv_kernel, gv, 256, 0, S.p, x, y, n, cg_state.p);
    return PXR_OK;
  };
  return run_cg(spmv);
}

// Preconditioned CG on the reduced system given its product; Ceres' ConjugateGradientsSolver recurrences and
// termination (Q-decrease ratio, residual refresh every 10 iterations).  Small systems run the single-CTA vector
// kernels (deterministic sums); from 4096 unknowns the multi-CTA variants.
int BA::run_cg(const std::function<int(const double*, double*)>& spmv) {
  cudaStream_t s = ctx->stream;
  const int n = nc;
  const bool multi = n >= 4096 || env.cg_multi;
  const unsigned gn = (unsigned)cdiv(n, 256);
  CGState hs;
  if (multi) {
    if (cg_part.n < (size_t)3 * gn) PXR_TRY(cg_part.alloc((size_t)3 * gn));
    PXR_LAUNCH(ctx, cgm_init_state_kernel, 1, 1, 0, cg_state.p, opt.max_linear_solver_iterations, 0.1);
    PXR_LAUNCH(ctx, cgm_init_kernel, gn, 256, 0, rhs.p, cg_x.p, cg_r.p, n, cg_state.p, cg_part.p);
    PXR_LAUNCH(ctx, cgm_init_done_kernel, 1, 32, 0, cg_state.p, cg_part.p, (int)gn);
  } else {
    PXR_LAUNCH(ctx, cg_init_kernel, 1, 1024, 0, rhs.p, cg_x.p, cg_r.p, n, cg_state.p, opt.max_linear_solver_iterations, 0.1);
  }
  for (int it = 0; it < opt.max_linear_solver_iterations; ++it) {
    const bool refresh = (it + 1) % 10 == 0;   // residual_reset_period
    if (multi) {
      PXR_LAUNCH(ctx, cgm_precond_kernel, gn, 256, 0, cg_Minv.p, cg_row_off.p, cg_row_dim.p, cg_r.p, cg_z.p, n, cg_state.p, cg_part.p);
      PXR_LAUNCH(ctx, cgm_beta_kernel, 1, 32, 0, cg_state.p, cg_part.p, (int)gn);
      PXR_LAUNCH(ctx, cgm_dir_kernel, gn, 256, 0, cg_z.p, cg_p.p, n, cg_state.p);
      PXR_TRY(spmv(cg_p.p, cg_q.p));
      PXR_LAUNCH(ctx, cgm_pq_kernel, gn, 256, 0, cg_p.p, cg_q.p, n, cg_state.p, cg_part.p);
      PXR_LAUNCH(ctx, cgm_alpha_kernel, 1, 32, 0, cg_state.p, cg_part.p, (int)gn);
      PXR_LAUNCH(ctx, cgm_update_kernel, gn, 256, 0, rhs.p, cg_p.p, cg_q.p, cg_x.p, cg_r.p, n, cg_state.p, cg_part.p);
      if (refresh) {
        PXR_TRY(spmv(cg_x.p, cg_tmp.p));
        PXR_LAUNCH(ctx, cgm_refresh_kernel, gn, 256, 0, rhs.p, cg_tmp.p, cg_x.p, cg_r.p, n, cg_state.p, cg_part.p);
      }
      PXR_LAUNCH(ctx, cgm_check_kernel, 1, 32, 0, cg_state.p, cg_part.p, (int)gn);
    } else {
      PXR_LAUNCH(ctx, cg_precond_kernel, 1, 1024, 0, cg_Minv.p, cg_row_off.p, cg_row_dim.p, cg_r.p, cg_z.p, cg_p.p, n, cg_state.p);
      PXR_TRY(spmv(cg_p.p, cg_q.p));
      PXR_LAUNCH(ctx, cg_update_kernel, 1, 1024, 0, rhs.p, cg_p.p, cg_q.p, cg_x.p, cg_r.p, n, cg_state.p);
      if (refresh) {
        PXR_TRY(spmv(cg_x.p, cg_tmp.p));
        PXR_LAUNCH(ctx, cg_refresh_kernel, 1, 1024, 0, rhs.p, cg_tmp.p, cg_r.p, n, cg_state.p);
      }
      PXR_LAUNCH(ctx, cg_check_kernel, 1, 1024, 0, rhs.p, cg_x.p, cg_r.p, n, cg_state.p);
    }
    if ((it + 1) % 8 == 0 || it + 1 == opt.max_linear_solver_iterations) {
      PXR_CUDA(cudaMemcpyAsync(&hs, cg_state.p, sizeof(hs), cudaMemcpyDeviceToHost, s));
      PXR_CUDA(cudaStreamSynchronize(s));
      if (hs.done) break;
    }
  }
  PXR_CUDA(cudaMemcpyAsync(&hs, cg_state.p, sizeof(hs), cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaMemcpyAsync(delta.p, cg_x.p, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  last_linear_iterations = hs.it;
  if (hs.failed) { int one = 1; PXR_CUDA(cudaMemcpyAsync(flags.p + 1, &one, sizeof(int), cudaMemcpyHostToDevice, s)); }
  return PXR_OK;
}

int BA::gradient_max_norm(double* out) {
  PXR_CUDA(cudaMemsetAsync(scalars.p + 10, 0, 8, ctx->stream));
  const int64_t n = std::max<int64_t>(std::max<int64_t>(n_images, n_cameras), n_points);
  const BADev d = dev();
  if (n > 0) PXR_LAUNCH(ctx, ba_gradmax_kernel, (unsigned)cdiv(n, 256), 256, 0, d, d.gc, q[cur].p, 1, scalars.p + 10);
  PXR_TRY(allreduce_f64(ctx, scalars.p + 10, 1, true));
  PXR_CUDA(cudaMemcpyAsync(out, scalars.p + 10, 8, cudaMemcpyDeviceToHost, ctx->stream));
  PXR_CUDA(cudaStreamSynchronize(ctx->stream));
  return PXR_OK;
}

// -------------------------------------------------------------------------------- LM driver
// Mirrors ceres::internal::TrustRegionMinimizer::Minimize (Ceres 2.1) with
// LevenbergMarquardtStrategy, monotonic steps, Jacobi scaling, inner iterations.  The loop state
// lives in the BA object so that a solve can be continued (pxr_ba_iterate) — bench.py times K
// consecutive iterations of one trajectory after W warm-up iterations.
int BA::lm_begin() {
  if (block_mode) return lm_begin_block();
  PXR_CUDA(cudaSetDevice(ctx->device));
  lm = LMState();
  lm.radius = opt.initial_trust_region_radius;
  lm.inner_enabled = opt.use_inner_iterations != 0;
  // ---- IterationZero
  PXR_TRY(evaluate(cur, true, &lm.x_cost));
  if (!std::isfinite(lm.x_cost)) return fail(PXR_ERR_NUMERIC, "initial cost is not finite");
  if (nl > 0) PXR_LAUNCH(ctx, ba_scale_kernel, (unsigned)cdiv(nl, 256), 256, 0, diag.p, jscale.p, nl, opt.jacobi_scaling);
  std::memset(&lm.it, 0, sizeof(lm.it));
  lm.it.cost = lm.x_cost;
  PXR_TRY(gradient_max_norm(&lm.it.gradient_max_norm));
  lm.initial_cost = lm.minimum_cost = lm.x_cost;
  lm.ev.init(lm.x_cost, opt.use_nonmonotonic_steps ? opt.max_consecutive_nonmonotonic_steps : 0);
  lm.best_is_current = true;
  lm.started = true;
  lm.pending_finalize = true;
  lm.term = 1;
  lm.message = "Maximum number of iterations reached.";
  return PXR_OK;
}

// FinalizeIterationAndCheckIfMinimizerCanContinue
bool BA::lm_finalize(int max_iteration) {
  pxr_iteration_summary& it = lm.it;
  if (lm.pending_finalize) {
    if (it.step_is_successful) {
      // ceres copies x into the user's parameters only when it is the best iterate so far; with monotonic steps every
      // accepted iterate is, with use_nonmonotonic_steps the best one is snapshotted on the device
      ++lm.n_succ;
      if (lm.x_cost < lm.minimum_cost) lm.minimum_cost = lm.x_cost;
    } else if (it.iteration > 0) ++lm.n_unsucc;
    it.trust_region_radius = lm.radius;
    it.iteration_time_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - lm.it_start).count();
    lm.its.push_back(it);
    lm.pending_finalize = false;
  }
  if (it.iteration >= max_iteration) { lm.term = 1; lm.message = "Maximum number of iterations reached."; return false; }
  if (it.gradient_max_norm <= opt.gradient_tolerance) { lm.term = 0; lm.message = "Gradient tolerance reached."; lm.finished = true; return false; }
  if (lm.radius < opt.min_trust_region_radius) { lm.term = 0; lm.message = "Minimum trust region radius reached."; lm.finished = true; return false; }
  return true;
}

// Runs LM iterations until iteration index `max_iteration` (absolute) or termination.
int BA::lm_iterate(int max_iteration) {
  if (block_mode) return lm_iterate_block(max_iteration);
  using clk = std::chrono::steady_clock;
  if (!lm.started) PXR_TRY(lm_begin());
  lm.it_start = clk::now();
  while (!lm.finished && lm_finalize(max_iteration)) {
    if (interrupt_pending()) {     // Ctrl-C in the host (util/src/py_interrupt.h:29-38): stop between iterations
      lm.finished = true; lm.term = 3;
      lm.message = "interrupted by the host";
      return fail(PXR_ERR_INTERRUPTED, "interrupted by the host after LM iteration %d", lm.it.iteration);
    }
    lm.it_start = clk::now();
    pxr_iteration_summary& it = lm.it;
    const double prev_gmax = it.gradient_max_norm;
    const int iteration = it.iteration + 1;
    std::memset(&it, 0, sizeof(it));
    it.iteration = iteration;
    lm.pending_finalize = true;

    bool valid = false;
    double model_cost_change = 0;
    PXR_TRY(compute_step(lm.radius, &valid, &model_cost_change));
    it.linear_solver_iterations = last_linear_iterations;
    it.step_is_valid = valid;
    if (!valid) {
      if (++lm.num_invalid >= opt.max_num_consecutive_invalid_steps) {
        lm.term = 2; lm.finished = true;
        lm.message = "Number of consecutive invalid steps more than Solver::Options::max_num_consecutive_invalid_steps";
        break;
      }
      lm.radius /= lm.decrease_factor; lm.decrease_factor *= 2.0;
      it.cost = lm.x_cost; it.gradient_max_norm = prev_gmax;
      continue;
    }
    lm.num_invalid = 0;

    double step_norm = 0, x_norm = 0, candidate_cost = 0;
    const bool speculate = !lm.inner_enabled && !env.no_speculation;
    // the norms of the step are read back together with the trial cost (one host round trip instead of two)
    if (speculate) PXR_TRY(apply_step(nullptr, nullptr)); else PXR_TRY(apply_step(&step_norm, &x_norm));
    // Trial point.  Ceres evaluates the cost here and, if the step is accepted, evaluates residuals AND Jacobians
    // again at the same point.  Both passes stream the same patch windows, so when no inner iterations will move
    // the point afterwards the Jacobian-mode pass is run right away into the alternate buffer set (0.52 ms instead
    // of 0.37 + 0.52 ms at S3); a rejected step merely discards it.
    swap_sets();
    int rc = PXR_OK;
    if (speculate) {
      rc = project(1 - cur, true, nullptr);
      if (rc == PXR_OK) rc = fm(1, nullptr, scalars.p + 0);
      if (rc == PXR_OK) rc = allreduce_f64(ctx, scalars.p + 0, 1);
      if (rc == PXR_OK) {
        double nv[4] = {0, 0, 0, 0};
        cudaError_t e = cudaMemcpyAsync(&candidate_cost, scalars.p + 0, 8, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(nv, scalars.p + 5, 32, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(PXR_ERR_CUDA, "trial evaluation failed: %s", cudaGetErrorString(e));
        step_norm = std::sqrt(nv[0] + nv[2]); x_norm = std::sqrt(nv[1] + nv[3]);
      }
    } else {
      rc = evaluate(1 - cur, false, &candidate_cost);
    }
    if (rc != PXR_OK) { swap_sets(); return rc; }
    if (!std::isfinite(candidate_cost)) candidate_cost = std::numeric_limits<double>::max();

    bool inner_useful = false;
    if (lm.inner_enabled && candidate_cost < std::numeric_limits<double>::max()) {
      ++lm.n_inner;
      rc = inner_iterations(1 - cur);
      double inner_cost = 0;
      if (rc == PXR_OK) rc = fm_cost(scalars.p + 0);
      if (rc == PXR_OK) rc = read_cost(&inner_cost);
      if (rc != PXR_OK) { swap_sets(); return rc; }
      if (std::isfinite(inner_cost)) {
        model_cost_change += candidate_cost - inner_cost;
        inner_useful = inner_cost < lm.x_cost;
        const double rel = 1.0 - inner_cost / candidate_cost;
        lm.inner_enabled = rel > opt.inner_iteration_tolerance;
        candidate_cost = inner_cost;
        rc = step_norm_between_sets(&step_norm);
        if (rc != PXR_OK) { swap_sets(); return rc; }
      }
    }
    swap_sets();   // back: uv/obs_out/juv = linearisation at the current point again
    it.step_norm = step_norm;
    if (step_norm <= opt.parameter_tolerance * (x_norm + opt.parameter_tolerance)) {
      lm.term = 0; lm.message = "Parameter tolerance reached."; lm.finished = true; break;
    }
    it.cost_change = lm.x_cost - candidate_cost;
    if (std::fabs(it.cost_change) <= opt.function_tolerance * lm.x_cost) {
      lm.term = 0; lm.message = "Function tolerance reached."; lm.finished = true; break;
    }
    it.relative_decrease = lm.ev.quality(candidate_cost, model_cost_change);
    const bool ok = inner_useful || it.relative_decrease > opt.min_relative_decrease;
    if (ok) {
      cur = 1 - cur;
      if (speculate && candidate_cost < std::numeric_limits<double>::max()) {
        swap_sets();                 // the speculative pass IS the linearisation at the new point
        PXR_TRY(build());
        lm.x_cost = candidate_cost;
      } else {
        PXR_TRY(evaluate(cur, true, &lm.x_cost));
      }
      it.cost = lm.x_cost;
      PXR_TRY(gradient_max_norm(&it.gradient_max_norm));
      it.step_is_successful = 1;
      lm.radius = lm.radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * it.relative_decrease - 1.0, 3));
      lm.radius = std::min(opt.max_trust_region_radius, lm.radius);
      lm.decrease_factor = 2.0;
      lm.ev.accepted(candidate_cost, model_cost_change);
      if (opt.use_nonmonotonic_steps) {
        // ceres copies x into the user's parameter blocks only when it is the best iterate so far
        // (FinalizeIterationAndCheckIfMinimizerCanContinue); a non-monotonic acceptance moves away from it, so the
        // iterate being left (still intact in the other parameter set) is snapshotted on the device
        if (lm.x_cost < lm.minimum_cost) lm.best_is_current = true;
        else if (lm.best_is_current) { PXR_TRY(save_best(1 - cur)); lm.best_is_current = false; }
      }
    } else {
      it.step_is_successful = 0;
      it.cost = candidate_cost;
      it.gradient_max_norm = prev_gmax;
      lm.radius /= lm.decrease_factor; lm.decrease_factor *= 2.0;
    }
  }
  if (lm.x_cost < lm.minimum_cost) lm.minimum_cost = lm.x_cost;
  PXR_CUDA(cudaStreamSynchronize(ctx->stream));
  return PXR_OK;
}

void BA::fill_summary(pxr_summary* sum, double seconds, int64_t launches) {
  if (!sum) return;
  sum->initial_cost = lm.initial_cost; sum->final_cost = lm.minimum_cost;
  sum->num_residual_blocks = (int32_t)n_obs; sum->num_residuals = n_obs * C;
  sum->num_successful_steps = lm.n_succ; sum->num_unsuccessful_steps = lm.n_unsucc;
  sum->num_inner_iteration_steps = lm.n_inner; sum->termination_type = lm.term;
  sum->solve_time_s = seconds; sum->total_time_s = seconds;
  sum->h2d_bytes = h2d_bytes; sum->d2h_bytes = 0;
  sum->num_iterations = (int32_t)lm.its.size();
  const int m = std::min<int>((int)lm.its.size(), sum->iterations ? sum->iterations_capacity : 0);
  for (int i = 0; i < m; ++i) sum->iterations[i] = lm.its[i];
  sum->kernel_launches = launches;
  std::snprintf(sum->message, sizeof(sum->message), "%s", lm.message.c_str());
  sum->resident_window = resident ? res_window : 0;
  sum->resident_passes_repeated = (int32_t)res_passes_repeated; sum->resident_refetched = res_refetched;
}

int BA::solve(pxr_summary* sum) {
  const auto t0 = std::chrono::steady_clock::now();
  const int64_t l0 = ctx->launches;
  PXR_TRY(lm_begin());
  PXR_TRY(lm_iterate(opt.max_num_iterations));
  if (block_mode) PXR_TRY(finish_gmax_block());
  fill_summary(sum, std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(), ctx->launches - l0);
  return PXR_OK;
}

int BA::save_best(int set) {
  cudaStream_t s = ctx->stream;
  if (!best_cam.p) {
    PXR_TRY(best_cam.alloc((size_t)n_cameras * kMaxK)); PXR_TRY(best_q.alloc((size_t)n_images * 4));
    PXR_TRY(best_t.alloc((size_t)n_images * 3)); PXR_TRY(best_X.alloc((size_t)n_points * 3));
  }
  PXR_CUDA(cudaMemcpyAsync(best_cam.p, cam[set].p, best_cam.n * 8, cudaMemcpyDeviceToDevice, s));
  PXR_CUDA(cudaMemcpyAsync(best_q.p, q[set].p, best_q.n * 8, cudaMemcpyDeviceToDevice, s));
  PXR_CUDA(cudaMemcpyAsync(best_t.p, t[set].p, best_t.n * 8, cudaMemcpyDeviceToDevice, s));
  if (best_X.n) PXR_CUDA(cudaMemcpyAsync(best_X.p, X[set].p, best_X.n * 8, cudaMemcpyDeviceToDevice, s));
  return PXR_OK;
}

int BA::read_params(double* cam_o, double* q_o, double* t_o, double* X_o) {
  cudaStream_t s = ctx->stream;
  // the lowest-cost iterate, as ceres leaves it in the user's parameter blocks
  const bool best = lm.started && !lm.best_is_current && best_cam.p;
  const double* pc = best ? best_cam.p : cam[cur].p; const double* pq = best ? best_q.p : q[cur].p;
  const double* pt = best ? best_t.p : t[cur].p; const double* pX = best ? best_X.p : X[cur].p;
  if (cam_o) PXR_CUDA(cudaMemcpyAsync(cam_o, pc, (size_t)n_cameras * kMaxK * 8, cudaMemcpyDeviceToHost, s));
  if (q_o) PXR_CUDA(cudaMemcpyAsync(q_o, pq, (size_t)n_images * 4 * 8, cudaMemcpyDeviceToHost, s));
  if (t_o) PXR_CUDA(cudaMemcpyAsync(t_o, pt, (size_t)n_images * 3 * 8, cudaMemcpyDeviceToHost, s));
  if (X_o) PXR_CUDA(cudaMemcpyAsync(X_o, pX, (size_t)n_points * 3 * 8, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  return PXR_OK;
}

}  // namespace pxr

using namespace pxr;

extern "C" {

int pxr_ba_create(pxr_ctx* ctx, const pxr_ba_desc* desc, const pxr_interp_config* interp,
                  const pxr_solver_options* opt, pxr_ba** out) {
  if (!ctx || !out) return fail(PXR_ERR_INVALID_ARGUMENT, "ctx/out is NULL");
  BA* b = new BA();
  const int rc = b->create(ctx, desc, interp, opt, true);
  if (rc != PXR_OK) { delete b; return rc; }
  *out = reinterpret_cast<pxr_ba*>(b);
  return PXR_OK;
}
int pxr_ba_destroy(pxr_ba* ba) {
  if (ba) { BA* b = reinterpret_cast<BA*>(ba); cudaSetDevice(b->ctx->device); delete b; }
  return PXR_OK;
}
int pxr_ba_solve(pxr_ba* ba, pxr_summary* summary) {
  if (!ba) return fail(PXR_ERR_INVALID_ARGUMENT, "ba is NULL");
  return reinterpret_cast<BA*>(ba)->solve(summary);
}
int pxr_ba_iterate(pxr_ba* ba, int n_iterations, pxr_summary* summary) {
  if (!ba || n_iterations < 0) return fail(PXR_ERR_INVALID_ARGUMENT, "bad arguments");
  BA* b = reinterpret_cast<BA*>(ba);
  const auto t0 = std::chrono::steady_clock::now();
  const int64_t l0 = b->ctx->launches;
  if (!b->lm.started) PXR_TRY(b->lm_begin());
  PXR_TRY(b->lm_iterate(b->lm.it.iteration + n_iterations));
  b->fill_summary(summary, std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(), b->ctx->launches - l0);
  return PXR_OK;
}
int pxr_ba_kernel_timing(pxr_ba* ba, int enable, int which, double* total_ms, int* count) {
  if (!ba) return fail(PXR_ERR_INVALID_ARGUMENT, "ba is NULL");
  BA* b = reinterpret_cast<BA*>(ba);
  PXR_CUDA(cudaSetDevice(b->ctx->device));
  if (total_ms || count) {
    PXR_CUDA(cudaStreamSynchronize(b->ctx->stream));
    double tot = 0; int n = 0;
    if (which < 0 || which >= BA::kNumStages) return fail(PXR_ERR_INVALID_ARGUMENT, "bad stage id");
    for (auto& pr : b->timed[which]) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) { tot += ms; ++n; }
    }
    if (total_ms) *total_ms = tot;
    if (count) *count = n;
  }
  if (enable >= 0) {
    for (int k = 0; k < BA::kNumStages; ++k) { for (auto& pr : b->timed[k]) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); } b->timed[k].clear(); }
    b->time_kernels = enable != 0;
  }
  return PXR_OK;
}
int pxr_ba_read_params(pxr_ba* ba, double* cam_params, double* qvec, double* tvec, double* xyz) {
  if (!ba) return fail(PXR_ERR_INVALID_ARGUMENT, "ba is NULL");
  return reinterpret_cast<BA*>(ba)->read_params(cam_params, qvec, tvec, xyz);
}
int pxr_ba_reset(pxr_ba* ba, const double* cam_params, const double* qvec, const double* tvec, const double* xyz) {
  if (!ba || !cam_params || !qvec || !tvec) return fail(PXR_ERR_INVALID_ARGUMENT, "NULL argument");
  BA* b = reinterpret_cast<BA*>(ba);
  PXR_CUDA(cudaSetDevice(b->ctx->device));
  cudaStream_t s = b->ctx->stream;
  if (b->n_points > 0 && !xyz) return fail(PXR_ERR_INVALID_ARGUMENT, "xyz is NULL");
  for (int k = 0; k < 2; ++k) {
    PXR_CUDA(cudaMemcpyAsync(b->cam[k].p, cam_params, (size_t)b->n_cameras * kMaxK * 8, cudaMemcpyHostToDevice, s));
    PXR_CUDA(cudaMemcpyAsync(b->q[k].p, qvec, (size_t)b->n_images * 4 * 8, cudaMemcpyHostToDevice, s));
    PXR_CUDA(cudaMemcpyAsync(b->t[k].p, tvec, (size_t)b->n_images * 3 * 8, cudaMemcpyHostToDevice, s));
    if (b->n_points > 0) PXR_CUDA(cudaMemcpyAsync(b->X[k].p, xyz, (size_t)b->n_points * 3 * 8, cudaMemcpyHostToDevice, s));
  }
  PXR_CUDA(cudaStreamSynchronize(s));
  b->cur = 0;
  b->lm = LMState();
  return PXR_OK;
}
int pxr_ba_run(pxr_ctx* ctx, const pxr_ba_desc* desc, const pxr_interp_config* interp,
               const pxr_solver_options* opt, pxr_summary* summary) {
  const auto t0 = std::chrono::steady_clock::now();
  if (!ctx) return fail(PXR_ERR_INVALID_ARGUMENT, "ctx is NULL");
  // one-shot call: the caller's patch buffer outlives the solve, so the slab may stay partially resident
  // (pxr_resident.cuh) — only the tap windows the solve touches cross PCIe
  BA* b = new BA();
  b->allow_resident = true;
  {
    const int rc0 = b->create(ctx, desc, interp, opt, true);
    if (rc0 != PXR_OK) { delete b; return rc0; }
  }
  pxr_ba* h = reinterpret_cast<pxr_ba*>(b);
  int rc = b->solve(summary);
  if (rc == PXR_OK) rc = b->read_params(desc->cam_params, desc->qvec, desc->tvec, desc->xyz);
  pxr_ba_destroy(h);      // inside the timed call: what the caller waits for
  if (summary) {
    summary->d2h_bytes = ((double)desc->n_cameras * kMaxK + desc->n_images * 7.0 + desc->n_points * 3.0) * 8.0;
    summary->total_time_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  }
  return rc;
}

int pxr_ba_evaluate(pxr_ba* ba, double* sq_norm, double* gtr, double* gtg, double* xy, double* residuals,
                    double* cost) {
  if (!ba) return fail(PXR_ERR_INVALID_ARGUMENT, "ba is NULL");
  BA* b = reinterpret_cast<BA*>(ba);
  pxr_ctx* ctx = b->ctx;
  PXR_CUDA(cudaSetDevice(ctx->device));
  DevBuf<double> dxy, dres;
  if (xy) PXR_TRY(dxy.alloc((size_t)b->n_obs * 2));
  if (residuals) PXR_TRY(dres.alloc((size_t)b->n_obs * b->C));
  PXR_TRY(b->project(b->cur, true, dxy.p));
  PXR_TRY(b->fm(1, dres.p, b->scalars.p + 0));
  std::vector<double> out((size_t)b->n_obs * 8);
  double c = 0;
  PXR_CUDA(cudaMemcpyAsync(out.data(), b->obs_out.p, out.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
  PXR_CUDA(cudaMemcpyAsync(&c, b->scalars.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (xy) PXR_CUDA(cudaMemcpyAsync(xy, dxy.p, (size_t)b->n_obs * 16, cudaMemcpyDeviceToHost, ctx->stream));
  if (residuals) PXR_CUDA(cudaMemcpyAsync(residuals, dres.p, (size_t)b->n_obs * b->C * 8, cudaMemcpyDeviceToHost, ctx->stream));
  PXR_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int64_t o = 0; o < b->n_obs; ++o) {
    const double* r = &out[(size_t)o * 8];
    if (sq_norm) sq_norm[o] = r[0];
    if (gtr) { gtr[2 * o] = r[1]; gtr[2 * o + 1] = r[2]; }
    if (gtg) { gtg[3 * o] = r[3]; gtg[3 * o + 1] = r[4]; gtg[3 * o + 2] = r[5]; }
  }
  if (cost) *cost = c;
  return PXR_OK;
}

// The cost-functor surface (residuals/bindings.cc:14-30): residual vectors and the two factors of every block's
// Jacobian, J = G * P.
int pxr_ba_evaluate_jacobians(pxr_ba* ba, double* residuals, double* grad, double* juv, int32_t* juv_cols, double* xy) {
  if (!ba) return fail(PXR_ERR_INVALID_ARGUMENT, "ba is NULL");
  BA* b = reinterpret_cast<BA*>(ba);
  pxr_ctx* ctx = b->ctx;
  PXR_CUDA(cudaSetDevice(ctx->device));
  const size_t n = (size_t)b->n_obs, C = (size_t)b->C;
  const int W = 9 + b->K;
  if (juv_cols) *juv_cols = W;
  DevBuf<double> dxy, dres, dgrad;
  if (xy) PXR_TRY(dxy.alloc(n * 2));
  if (residuals) PXR_TRY(dres.alloc(n * C));
  if (grad) PXR_TRY(dgrad.alloc(n * 2 * C));
  PXR_TRY(b->project(b->cur, true, dxy.p));
  PXR_TRY(b->fm(1, dres.p, b->scalars.p + 0, dgrad.p));
  cudaStream_t s = ctx->stream;
  if (xy) PXR_CUDA(cudaMemcpyAsync(xy, dxy.p, n * 16, cudaMemcpyDeviceToHost, s));
  if (residuals) PXR_CUDA(cudaMemcpyAsync(residuals, dres.p, n * C * 8, cudaMemcpyDeviceToHost, s));
  if (grad) PXR_CUDA(cudaMemcpyAsync(grad, dgrad.p, n * 2 * C * 8, cudaMemcpyDeviceToHost, s));
  if (juv && n > 0)     // device rows are juv_stride doubles apart, 2 x W of them used
    PXR_CUDA(cudaMemcpy2DAsync(juv, (size_t)2 * W * 8, b->juv.p, (size_t)b->juv_stride * 8, (size_t)2 * W * 8, n, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  return PXR_OK;
}


// Introspection for parity tests: linearise at the current parameters and compute one LM step at
// `radius` (Jacobi scaling from this linearisation, as in iteration 0).  Any output may be NULL.
int pxr_ba_debug_linearize(pxr_ba* ba, double radius, double* cost, double* Hcc, double* gc, double* Hpp,
                           double* gp, double* S, double* rhs, double* delta, double* model_cost_change) {
  if (!ba) return fail(PXR_ERR_INVALID_ARGUMENT, "ba is NULL");
  BA* b = reinterpret_cast<BA*>(ba);
  pxr_ctx* ctx = b->ctx;
  cudaStream_t s = ctx->stream;
  PXR_CUDA(cudaSetDevice(ctx->device));
  if ((b->sparse_schur || b->block_mode) && (Hcc || S)) return fail(PXR_ERR_UNSUPPORTED, "the block-sparse path has no dense Hcc / S to return");
  double c = 0;
  PXR_TRY(b->evaluate(b->cur, true, &c));
  if (cost) *cost = c;
  if (b->block_mode) {   // point columns now, camera columns after the all-reduce inside compute_step
    if (b->nl - b->nc > 0) PXR_LAUNCH(ctx, ba_scale_kernel, (unsigned)cdiv(b->nl - b->nc, 256), 256, 0, b->diag.p + b->nc, b->jscale.p + b->nc, b->nl - b->nc, b->opt.jacobi_scaling);
    b->jscale_c_pending = true;
  } else if (b->nl > 0) PXR_LAUNCH(ctx, ba_scale_kernel, (unsigned)cdiv(b->nl, 256), 256, 0, b->diag.p, b->jscale.p, b->nl, b->opt.jacobi_scaling);
  const size_t nc = b->nc;
  if (Hcc) PXR_CUDA(cudaMemcpyAsync(Hcc, b->Hcc.p, nc * nc * 8, cudaMemcpyDeviceToHost, s));
  if (gc) PXR_CUDA(cudaMemcpyAsync(gc, b->block_mode ? b->pack_local.p + b->pk_off_gc : b->gc.p, nc * 8, cudaMemcpyDeviceToHost, s));   // block mode: this rank's partial
  if (Hpp) PXR_CUDA(cudaMemcpyAsync(Hpp, b->Hpp.p, (size_t)b->n_points * 72, cudaMemcpyDeviceToHost, s));
  if (gp) PXR_CUDA(cudaMemcpyAsync(gp, b->gp.p, (size_t)b->n_points * 24, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  if (S || rhs) {
    // the damped Schur system before factorisation: rerun the assembly part only
    PXR_TRY(b->build_schur_pairs());
    BADev d = b->dev();
    if (b->nl > 0) PXR_LAUNCH(ctx, ba_d2_kernel, (unsigned)cdiv(b->nl, 256), 256, 0, b->diag.p, b->jscale.p, b->D2.p, b->nl, radius,
                              b->opt.min_lm_diagonal, b->opt.max_lm_diagonal);
    if (nc > 0) PXR_LAUNCH(ctx, ba_init_reduced_kernel, (unsigned)cdiv((int64_t)nc * nc, 256), 256, 0, b->Hcc.p, b->gc.p, b->D2.p, b->S.p, b->rhs.p, (int)nc, 1);
    PXR_CUDA(cudaMemsetAsync(b->flags.p, 0, 4 * sizeof(int), s));
    if (b->n_points > 0) {
      PXR_LAUNCH(ctx, ba_point_inverse_kernel, (unsigned)cdiv(b->n_points, 256), 256, 0, d, b->D2.p, b->Hinv.p, b->flags.p);
      PXR_TRY(b->launch_schur_pairs(d));
    }
    if (S) PXR_CUDA(cudaMemcpyAsync(S, b->S.p, nc * nc * 8, cudaMemcpyDeviceToHost, s));
    if (rhs) PXR_CUDA(cudaMemcpyAsync(rhs, b->rhs.p, nc * 8, cudaMemcpyDeviceToHost, s));
    PXR_CUDA(cudaStreamSynchronize(s));
  }
  bool valid = false;
  double mcc = 0;
  PXR_TRY(b->compute_step(radius, &valid, &mcc));
  if (delta) PXR_CUDA(cudaMemcpyAsync(delta, b->delta.p, (size_t)b->nl * 8, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  if (model_cost_change) *model_cost_change = mcc;
  return PXR_OK;
}

// Runs inner iterations on the current parameter set (parity tests).
int pxr_ba_debug_inner_iterations(pxr_ba* ba) {
  if (!ba) return fail(PXR_ERR_INVALID_ARGUMENT, "ba is NULL");
  BA* b = reinterpret_cast<BA*>(ba);
  PXR_CUDA(cudaSetDevice(b->ctx->device));
  PXR_TRY(b->inner_iterations(b->cur));
  PXR_CUDA(cudaStreamSynchronize(b->ctx->stream));
  return PXR_OK;
}

int pxr_ba_time_stage(pxr_ba* ba, int stage, int iters, double* ms_per_launch) {
  if (!ba || iters < 1 || !ms_per_launch) return fail(PXR_ERR_INVALID_ARGUMENT, "bad arguments");
  BA* b = reinterpret_cast<BA*>(ba);
  pxr_ctx* ctx = b->ctx;
  cudaStream_t s = ctx->stream;
  PXR_CUDA(cudaSetDevice(ctx->device));
  cudaEvent_t e0, e1;
  PXR_CUDA(cudaEventCreate(&e0)); PXR_CUDA(cudaEventCreate(&e1));
  double c;
  PXR_TRY(b->project(b->cur, true, nullptr));  // uv for the current parameters
  PXR_CUDA(cudaStreamSynchronize(s));
  PXR_CUDA(cudaEventRecord(e0, s));
  for (int i = 0; i < iters; ++i) {
    if (stage == 0) PXR_TRY(b->fm(1, nullptr, b->scalars.p));
    else if (stage == 1) PXR_TRY(b->fm(0, nullptr, b->scalars.p));
    else if (stage == 3) PXR_TRY(b->project(b->cur, true, nullptr));
    else if (stage == 4) PXR_TRY(b->build());
    else if (stage == 5) PXR_TRY(b->inner_iterations(1 - b->cur));
    else PXR_TRY(b->evaluate(b->cur, true, &c));
  }
  PXR_CUDA(cudaEventRecord(e1, s));
  PXR_CUDA(cudaEventSynchronize(e1));
  float ms = 0;
  PXR_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *ms_per_launch = (double)ms / iters;
  return PXR_OK;
}

}  // extern "C"
