// pxr_ba_host.h — host-side state of one featuremetric BA problem resident on the device.
#pragma once
#include <cstdlib>
#include <chrono>
#include <string>
#include <functional>
#include <thread>
#include <limits>
#include <algorithm>
#include <utility>
#include <vector>

#include "pxr_ba_kernels.cuh"
#include "pxr_chol.cuh"
#include "pxr_fm_eval.cuh"
#include "pxr_fm_small.cuh"
#include "pxr_inner.cuh"
#include "pxr_internal.h"
#include "pxr_pcg.cuh"
#include "pxr_sparse_schur.cuh"
#include "pxr_block.cuh"

namespace pxr {

int fm_supported(int dtype, int C);
int fm_max_partials(pxr_ctx* ctx);
int launch_fm_eval(pxr_ctx* ctx, int dtype, int C, int mode, bool float_simd, const FmEvalArgs& a, int* n_partials);
int launch_inner_fused(pxr_ctx* ctx, int dtype, int C, bool float_simd, const InnerArgs& a);

// ceres::internal::TrustRegionStepEvaluator (Conn, Gould & Toint, algorithm 10.1.2); max_nonmonotonic == 0 is the
// monotonic minimizer.  Same arithmetic as oracle/orc_trust_region.h::StepEvaluator.
struct StepEvaluator {
  int max_nonmonotonic = 0, num_consecutive_nonmonotonic_steps = 0;
  double minimum_cost = 0, current_cost = 0, reference_cost = 0, candidate_cost = 0;
  double acc_reference = 0, acc_candidate = 0;
  void init(double c, int max_nm) { *this = StepEvaluator(); max_nonmonotonic = max_nm; minimum_cost = current_cost = reference_cost = candidate_cost = c; }
  double quality(double cost, double mcc) const {
    if (cost >= std::numeric_limits<double>::max()) return std::numeric_limits<double>::lowest();
    return std::max((current_cost - cost) / mcc, (reference_cost - cost) / (acc_reference + mcc));
  }
  void accepted(double cost, double mcc) {
    current_cost = cost; acc_candidate += mcc; acc_reference += mcc;
    if (current_cost < minimum_cost) { minimum_cost = current_cost; num_consecutive_nonmonotonic_steps = 0; candidate_cost = current_cost; acc_candidate = 0; }
    else { ++num_consecutive_nonmonotonic_steps; if (current_cost > candidate_cost) { candidate_cost = current_cost; acc_candidate = 0; } }
    if (num_consecutive_nonmonotonic_steps == max_nonmonotonic) { reference_cost = candidate_cost; acc_reference = acc_candidate; }
  }
};

struct LMState {
  bool started = false, finished = false, pending_finalize = false, inner_enabled = false;
  StepEvaluator ev;
  bool gmax_pending = false;       // block mode, several ranks: max |g| of the current point arrives with the next all-reduce
  bool best_is_current = true;     // non-monotonic steps: the lowest-cost iterate lives in BA::best_* when false
  double x_cost = 0, radius = 1e4, decrease_factor = 2.0, initial_cost = 0, minimum_cost = 0;
  int num_invalid = 0, n_succ = 0, n_unsucc = 0, n_inner = 0, term = 1;
  pxr_iteration_summary it;
  std::vector<pxr_iteration_summary> its;
  std::string message;
  std::chrono::steady_clock::time_point it_start;
};

struct BA {
  pxr_ctx* ctx = nullptr;
  LMState lm;
  // optional CUDA-event timing of the LM stages (pxr_ba_kernel_timing): 0 K1 cost-only, 1 K1 Jacobian,
  // 2 projection K0, 3 block build, 4 damping+Schur assembly, 5 Cholesky factor, 6 Cholesky solve,
  // 7 back-substitution+model cost, 8 manifold plus, 9 inner iterations, 10 cost reduction, 11 misc
  static constexpr int kNumStages = 12;
  bool time_kernels = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timed[kNumStages];
  struct StageScope {
    BA* b; int id; cudaEvent_t e0 = nullptr, e1 = nullptr;
    StageScope(BA* b_, int id_) : b(b_), id(id_) {
      if (b->time_kernels && cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess) cudaEventRecord(e0, b->ctx->stream);
    }
    ~StageScope() { if (e0 && e1) { cudaEventRecord(e1, b->ctx->stream); b->timed[id].push_back({e0, e1}); } }
  };
  pxr_interp_config interp;
  pxr_solver_options opt;
  // sizes
  int n_cameras = 0, n_images = 0, K = 0, C = 0, ph = 0, pw = 0, dtype = 0;
  int64_t n_points = 0, n_obs = 0, n_patches = 0, nl = 0;
  int nc = 0, dcmax = 0, juv_stride = 0, img_dc_max = 0;
  double ups = 1.0;
  bool has_refs = false;
  double h2d_bytes = 0;
  // host layout
  std::vector<int32_t> h_pose_off, h_intr_off;
  std::vector<int64_t> h_point_off, h_pt_begin;
  // device: topology
  DevBuf<int32_t> obs_img, img_cam, cam_model, pose_off, intr_off, corner, Wcols, Wdc;
  DevBuf<int64_t> obs_pt, obs_patch, point_off, pt_begin;
  DevBuf<uint32_t> cam_mask;
  DevBuf<uint8_t> tmask;
  PatchSlab patches_owned;
  DevBuf<double> scale, refs;
  const uint8_t* d_patches = nullptr;
  // device: parameters (two sets: current / candidate)
  DevBuf<double> cam[2], q[2], t[2], X[2];
  DevBuf<double> best_cam, best_q, best_t, best_X;   // use_nonmonotonic_steps: snapshot of the lowest-cost iterate
  int save_best(int set);
  int cur = 0;
  // device: per-observation and linearisation
  // uv/obs_out/juv hold the linearisation at the CURRENT point; every trial-point evaluation (cost-only,
  // speculative Jacobian, inner iterations) runs on the *_alt set (swap_sets()) so a rejected step never
  // clobbers what the next compute_step reads.
  DevBuf<double> uv_alt, obs_out_alt, juv_alt;
  void swap_sets() { std::swap(uv.p, uv_alt.p); std::swap(uv.n, uv_alt.n); std::swap(obs_out.p, obs_out_alt.p); std::swap(obs_out.n, obs_out_alt.n); std::swap(juv.p, juv_alt.p); std::swap(juv.n, juv_alt.n); }
  DevBuf<double> ar_buf;             // staging for the fused [diag | gc] all-reduce
  DevBuf<double> gc_local;           // multi-GPU: this rank's partial gradient (gc holds the global one)
  DevBuf<double> uv, obs_out, juv, Hcc, gc, Hpp, gp, W, S, rhs, diag, jscale, D2, delta, partials, scalars;
  DevBuf<int> flags;
  DevBuf<double> rdiag;
  // ITERATIVE_SCHUR (PCG) workspace
  bool use_pcg = false;
  DevBuf<double> cg_Minv, cg_z, cg_p, cg_q, cg_r, cg_x, cg_tmp, cg_part;   // cg_part: per-CTA dot-product partials (fixed-order sums)
  DevBuf<int32_t> cg_blk_off, cg_blk_dim, cg_row_off, cg_row_dim;
  DevBuf<CGState> cg_state;
  int cg_nblk = 0, last_linear_iterations = 1;
  int pcg_solve();
  int run_cg(const std::function<int(const double*, double*)>& spmv);
  // implicit block-sparse reduced system (pxr_sparse_schur.cuh): no nc x nc array is ever allocated
  // debugging / A-B switches, read from the environment once in create()
  struct EnvFlags { bool pcg_sparse = false, build_atomic = false, chol_multikernel = false, chol_test_abort = false,
                         cg_multi = false, no_speculation = false, build_staged = true, project_staged = true; std::string chol_trace; } env;
  bool sparse_schur = false;
  int ss_n_keys = 0;
  std::vector<int32_t> h_img_cols, h_img_pd, h_img_pose_blk, h_img_cam_blk, h_img_cam;
  DevBuf<int32_t> ss_img_cols, ss_img_pd, ss_img_pose_blk, ss_img_cam_blk, ss_key_a, ss_key_b, ss_chunk_key;
  DevBuf<uint8_t> ss_key_self;
  DevBuf<double> ss_Himg, ss_Bk, ss_Dblk;
  SparseSchur sparse();
  int pcg_solve_sparse();
  // ---- block mode (pxr_block.cuh, pxr_ba_block.cu): image-block assembly into ONE packed buffer, ONE all-reduce per
  // LM iteration, everything after it deterministic; scalar decisions travel through the peer mailboxes
  bool block_mode = false;
  DevBuf<double> pack_local, pack_global;          // world == 1: pack_global stays empty and aliases pack_local
  size_t pk_off_B = 0, pk_off_rhs = 0, pk_off_gc = 0, pk_off_slots = 0, pk_n = 0;
  double* pk(bool global) { return (global && pack_global.p) ? pack_global.p : pack_local.p; }
  SparseSchur sparse_blk(bool global);
  std::vector<int32_t> h_key_a, h_key_b; std::vector<uint8_t> h_key_self;     // global key list (host copy)
  DevBuf<int64_t> gmS_dest, gmS_ptr, dg_ptr, gmD_dest, gmD_ptr, br_chunk_begin, br_cols_ptr;
  DevBuf<int32_t> gmS_src, dg_src, gmD_src, br_chunk_img, br_ent_key, br_cols_src;
  DevBuf<uint8_t> br_chunk_first;
  DevBuf<double> br_ypart, mb_in, mb_out;
  int64_t gmS_rows = 0, gmD_rows = 0, br_n_chunks = 0;
  // deterministic assembly (pxr_solver_options.deterministic): block mode + fixed-order reductions of the chunk partials
  bool deterministic = false;
  std::vector<int64_t> h_img_chunk_begin;           // [n_images+1] chunks of every image in io order (create())
  DevBuf<int64_t> det_img_chunk_begin, det_key_chunk_begin;
  DevBuf<double> det_cam_part, det_pair_part, det_gimg, det_rimg, det_scal_part;
  bool jscale_c_pending = false;
  bool blk_lag_gmax = false;                       // world > 1: max |g| of the current point is known after the next all-reduce
  int block_setup();                               // global keys, gather maps, block rows
  int build_block();
  int compute_step_block(double radius);
  int compute_step_block_sync(double radius, bool* valid, double* model_cost_change);   // + exchange + read-back (debug entry points)
  int global_cost_block(double* cost_out);         // scalars[0] summed over the ranks
  int pcg_solve_block();
  int lm_begin_block();
  int lm_iterate_block(int max_iteration);
  int finish_gmax_block();
  int exchange_scalars(int n_sum);                 // mb_in -> mb_out (peer mailboxes, or NCCL when they are unavailable)
  std::vector<int32_t> h_chunk_key_local;
  std::vector<int64_t> h_key_code_local;           // local key codes in build order (set by build_schur_pairs)
  int pcg_setup_blocks();
  int launch_schur_pairs(const BADev& d);
  int launch_sp_schur_pairs(const BADev& d, double* Bk, double* rhs_out, double* part);
  cudaGraphExec_t chol_graph_exec = nullptr;
  int64_t chol_graph_kernels = 0;
  bool chol_multikernel = false, chol_force_multikernel = false, chol_band = false; int chol_grid = 0;
  // pair-walk kernel of the Schur assembly (images of <= 8 columns): 0 fused tensor-core walk (default), 3 tensor-core walk
  // on a precomputed T, 1 staged, 2 direct.  PXR_SCHUR_KERNEL=fused|mma|staged|direct and PXR_SCHUR_CTAS=3|4 (register
  // budget) are A/B switches for measurements.
  int schur_kernel = [] { const char* e = getenv("PXR_SCHUR_KERNEL"); return !e ? 0 : (e[0] == 'm' ? 3 : (e[0] == 's' ? 1 : (e[0] == 'd' ? 2 : 0))); }();
  int schur_ctas = getenv("PXR_SCHUR_CTAS") ? atoi(getenv("PXR_SCHUR_CTAS")) : 0;   // 0: the kernel's default (fused 4, mma 3, staged 4)
  DevBuf<int32_t> img_cols8, img_dc8; DevBuf<int8_t> img_src8;   // per-image column tables (<= 8 columns per image)
  DevBuf<int32_t> io_obs;           // observations grouped by image, chunks of <= 128 (camera-block build)
  DevBuf<int64_t> io_chunk_begin; int64_t io_n_chunks = 0;
  DevBuf<long long> chol_trace;     // PXR_CHOL_TRACE=<file>: panel-CTA time stamps
  DevBuf<int> chol_sync;            // flags of the persistent tile-DAG Cholesky (pxr_chol.cuh)
  ~BA() { if (res_thread.joinable()) res_thread.join(); if (chol_graph_exec) cudaGraphExecDestroy(chol_graph_exec); for (int k = 0; k < kNumStages; ++k) for (auto& pr : timed[k]) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); } }
  // static co-visibility structure for the Schur complement (see ba_schur_pairs_kernel)
  DevBuf<int32_t> sp_px, sp_py, sp_pp;
  DevBuf<int64_t> sp_chunk_begin;
  DevBuf<uint8_t> sp_chunk_self;
  DevBuf<double> Tbuf, Hinv;
  int64_t sp_n_chunks = 0;
  bool sp_built = false;
  std::vector<int32_t> h_obs_img;
  int build_schur_pairs();
  SchurPairs schur_pairs();

  int create(pxr_ctx* c, const pxr_ba_desc* d, const pxr_interp_config* ic, const pxr_solver_options* so, bool for_solve);
  // ---- window residency of the patch slab (pxr_resident.cuh): only in the one-shot pxr_ba_run (the host source must
  // outlive the solve), mapped pinned host source, C >= 8.  A repeated pass is local to the rank, so it composes with the
  // multi-GPU block mode (it only adds a host look at the violation counter after each evaluation).
  bool allow_resident = false, resident = false;
  int res_window = 8;
  bool res_window_fixed = false;                   // the caller knows the exact window (reference extraction: the points do not move)
  DevBuf<uint32_t> res_rect;
  DevBuf<unsigned long long> res_viol_count;
  DevBuf<int64_t> res_viol_list, res_fix_list;
  DevBuf<uint8_t> res_shared;
  std::vector<const void*> res_srcs;               // host blocks of whole patches (one entry for a contiguous source)
  std::vector<int64_t> res_block_first;            // [n_blocks+1]
  std::vector<int64_t> h_obs_patch;                // host copy (which patch an observation reads), empty = identity
  std::vector<uint8_t> res_whole;                  // patches already fetched whole
  int64_t res_refetched = 0, res_passes_repeated = 0;
  size_t res_esz = 2;
  std::thread res_thread;                          // packs and uploads the windows while create() goes on
  int res_thread_rc = 0; std::string res_thread_err;
  int resident_setup(const pxr_ba_desc* d, size_t esz);                    // decides and allocates
  int resident_begin(cudaStream_t us, double* h2d_patch);                  // K0 + rectangles + the window upload (own thread)
  int resident_fix(int64_t* n_fixed);               // after an evaluation: fetch the patches of reported observations
  void resident_args(FmEvalArgs& a);                // hooks the guard into an evaluation launch
  BADev dev();
  int project(int set, bool jac, double* xy_out);
  int fm(int mode, double* residuals_out, double* cost_dev, double* grad_out = nullptr);
  int fm_k1(int mode, double* residuals_out, double* grad_out, const int64_t* list, int64_t n);   // K1 over all observations or a list
  int fm_cost(double* cost_dev);                                                                   // robustified cost from obs_out
  int build();
  int evaluate(int set, bool jac, double* cost_out);
  int read_cost(double* cost_out);                 // global cost from scalars[0] (all-reduce + read-back)
  int compute_step(double radius, bool* valid, double* model_cost_change);
  int chol_launch();
  int apply_step(double* step_norm, double* x_norm);
  int gradient_max_norm(double* out);
  int inner_iterations(int set);
  DevBuf<double> inner_rec;                        // [n_obs][kInnerRec]: the evaluations of a round (pxr_inner.cuh)
  DevBuf<unsigned long long> inner_next;           // next point a slot of inner_fused_kernel takes
  DevBuf<double> inner_snapshot;                   // window residency: the points before the inner iterations (redo after a refetch)
  int step_norm_between_sets(double* out);
  int lm_begin();
  bool lm_finalize(int max_iteration);
  int lm_iterate(int max_iteration);
  void fill_summary(pxr_summary* sum, double seconds, int64_t launches);
  int solve(pxr_summary* sum);
  int read_params(double* cam_o, double* q_o, double* t_o, double* X_o);
};

}  // namespace pxr
