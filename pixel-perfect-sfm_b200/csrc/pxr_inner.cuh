// pxr_inner.cuh — inner iterations: every 3D point solved with everything else fixed, in one kernel.
//
// Replaces ceres' CoordinateDescentMinimizer (enabled by the reference through
// use_inner_iterations=True, pixsfm/bundle_adjustment/main.py:41-44 and
// bundle_optimizer.h:131-134,350-355: all non-constant points form independent set 0).  Each
// point runs a Levenberg-Marquardt loop with Ceres' DEFAULT Solver::Options
// (CoordinateDescentMinimizer::Solve builds Minimizer::Options from defaults):
// max 50 iterations, function_tolerance 1e-6, gradient_tolerance 1e-10,
// parameter_tolerance 1e-8, Jacobi scaling, monotonic steps, 5 consecutive invalid steps.
//
// inner_fused_kernel: a CTA iterates kInnerSlots points at a time.  One round evaluates every observation of its
// slots — one warp per observation through the K1 window ring (pxr_fm_eval.cuh), one thread per observation for
// C < 8 (pxr_fm_small.cuh) — spread over all warps, so a lone long-running point still costs about one
// observation's latency per LM step.  Then one warp per slot sums cost, J^T J and J^T r in observation order and one
// thread applies the LM step.  A slot whose point is done takes the next point from a global counter: CTAs never
// wait for each other and nothing assumes they are co-resident.
// L2 budget: every evaluation reads the point's 4x4-tap windows again.  With 4 slots and 2 CTAs per SM the points
// being iterated own 148 * 2 * 4 * (track length) windows: 48 MB at 10 observations of 128 fp16 channels (4 KiB per
// window), well inside the 126 MB L2, so a point's windows come from HBM about once per call.
#pragma once
#include "pxr_ba_kernels.cuh"
#include "pxr_fm_eval.cuh"
#include "pxr_fm_small.cuh"

namespace pxr {

struct InnerState {
  double x[3];        // last accepted point
  double cand[3];     // candidate being evaluated
  double cost, current_cost, H[6], g[3], sc[3];
  double radius, decf, xnorm, gmax, mcc;
  int iter, invalid;
};

__device__ __forceinline__ bool inner_propose(InnerState& s) {
  // ceres Solver::Options defaults (CoordinateDescentMinimizer::Solve)
  const int max_iter = 50, max_invalid = 5;
  const double gtol = 1e-10, min_radius = 1e-32, min_diag = 1e-6, max_diag = 1e32;
  for (;;) {
    s.iter += 1;
    if (s.iter - 1 >= max_iter) return false;
    if (s.gmax <= gtol) return false;
    if (s.radius < min_radius) return false;
    const double diag[3] = {s.H[0], s.H[3], s.H[5]};
    double D2[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double s2 = s.sc[k] * s.sc[k];
      D2[k] = fmin(fmax(diag[k] * s2, min_diag), max_diag) / (s.radius * s2);
    }
    const double Hf[9] = {s.H[0], s.H[1], s.H[2], s.H[1], s.H[3], s.H[4], s.H[2], s.H[4], s.H[5]};
    double inv[9];
    bool valid = inv3_sym(Hf, D2, inv);
    double d[3] = {0, 0, 0}, mcc = 0;
    if (valid) {
#pragma unroll
      for (int k = 0; k < 3; ++k) d[k] = -(inv[k * 3] * s.g[0] + inv[k * 3 + 1] * s.g[1] + inv[k * 3 + 2] * s.g[2]);
      double gd = 0, dHd = 0;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        gd += s.g[k] * d[k];
        dHd += d[k] * (Hf[k * 3] * d[0] + Hf[k * 3 + 1] * d[1] + Hf[k * 3 + 2] * d[2]);
      }
      mcc = -gd - 0.5 * dHd;
      valid = isfinite(d[0]) && isfinite(d[1]) && isfinite(d[2]) && mcc > 0.0;
    }
    if (!valid) {
      if (++s.invalid >= max_invalid) return false;
      s.radius /= s.decf; s.decf *= 2.0;
      continue;
    }
    s.invalid = 0;
    s.mcc = mcc;
#pragma unroll
    for (int k = 0; k < 3; ++k) s.cand[k] = s.x[k] + d[k];
    return true;
  }
}

// adds one observation to its point's cost, J^T J (6 uniques: 00 01 02 11 12 22) and J^T r; oo = K1's
// (s, b_u, b_v, a_uu, a_uv, a_vv), pu / pv = d(u)/dX, d(v)/dX
__device__ __forceinline__ void inner_add(const LossParams& loss, const double* oo, const double* pu, const double* pv,
                                          double& cost, double H[6], double g[3]) {
  double rho[3];
  loss_eval(loss, 1.0, oo[0], rho);
  cost += 0.5 * rho[0];
  const double bu = rho[1] * oo[1], bv = rho[1] * oo[2];
  const double auu = rho[1] * oo[3], auv = rho[1] * oo[4], avv = rho[1] * oo[5];
  double apu[3], apv[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { apu[k] = auu * pu[k] + auv * pv[k]; apv[k] = auv * pu[k] + avv * pv[k]; }
  H[0] += pu[0] * apu[0] + pv[0] * apv[0];
  H[1] += pu[0] * apu[1] + pv[0] * apv[1];
  H[2] += pu[0] * apu[2] + pv[0] * apv[2];
  H[3] += pu[1] * apu[1] + pv[1] * apv[1];
  H[4] += pu[1] * apu[2] + pv[1] * apv[2];
  H[5] += pu[2] * apu[2] + pv[2] * apv[2];
#pragma unroll
  for (int k = 0; k < 3; ++k) g[k] += pu[k] * bu + pv[k] * bv;
}

// One LM decision of a point after an evaluation (cost, H, g): with `first` at its start s.x (state set up from it),
// otherwise at the candidate s.cand (accepted or rejected).  Returns true with the next candidate in s.cand, false when
// the point is done at s.x.  *accepted: the evaluated position is now s.x.
__device__ __forceinline__ bool inner_step(InnerState& s, bool first, double cost, const double H[6], const double g[3],
                                           bool* accepted) {
  const double ftol = 1e-6, ptol = 1e-8, min_rel_dec = 1e-3, max_radius = 1e16;
  *accepted = first;
  if (first) {
    s.iter = 0; s.invalid = 0;
    s.cost = s.current_cost = cost;
#pragma unroll
    for (int k = 0; k < 6; ++k) s.H[k] = H[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) s.g[k] = g[k];
    s.sc[0] = 1.0 / (1.0 + sqrt(H[0])); s.sc[1] = 1.0 / (1.0 + sqrt(H[3])); s.sc[2] = 1.0 / (1.0 + sqrt(H[5]));
    s.radius = 1e4; s.decf = 2.0;
    s.xnorm = sqrt(s.x[0] * s.x[0] + s.x[1] * s.x[1] + s.x[2] * s.x[2]);
    s.gmax = fmax(fabs(g[0]), fmax(fabs(g[1]), fabs(g[2])));
    if (!isfinite(cost)) return false;
  } else {
    const double candidate_cost = isfinite(cost) ? cost : 1.7976931348623157e308;
    const double dx = s.cand[0] - s.x[0], dy = s.cand[1] - s.x[1], dz = s.cand[2] - s.x[2];
    const double step_norm = sqrt(dx * dx + dy * dy + dz * dz);
    if (step_norm <= ptol * (s.xnorm + ptol)) return false;                    // parameter tolerance
    if (fabs(s.cost - candidate_cost) <= ftol * s.cost) return false;          // function tolerance
    const double rel = (s.current_cost - candidate_cost) / s.mcc;
    if (rel > min_rel_dec) {
      *accepted = true;
#pragma unroll
      for (int k = 0; k < 3; ++k) { s.x[k] = s.cand[k]; s.g[k] = g[k]; }
#pragma unroll
      for (int k = 0; k < 6; ++k) s.H[k] = H[k];
      s.xnorm = sqrt(s.x[0] * s.x[0] + s.x[1] * s.x[1] + s.x[2] * s.x[2]);
      s.cost = cost; s.current_cost = candidate_cost;
      s.gmax = fmax(fabs(g[0]), fmax(fabs(g[1]), fabs(g[2])));
      s.radius = s.radius / fmax(1.0 / 3.0, 1.0 - pow(2.0 * rel - 1.0, 3.0));
      s.radius = fmin(max_radius, s.radius);
      s.decf = 2.0;
    } else {
      s.radius /= s.decf; s.decf *= 2.0;
    }
  }
  return inner_propose(s);
}

constexpr int kInnerSlots = 4;   // points a CTA iterates at once (L2 budget above)
constexpr int kInnerRec = 12;    // per-observation record: s, b_u, b_v, a_uu, a_uv, a_vv | d(u)/dX | d(v)/dX

struct InnerArgs {
  int64_t n_points;
  const int64_t* point_off; const int64_t* pt_begin;
  ProjectArgs geo;                 // cameras of the parameter set (the points come from the slots)
  FmEvalArgs fm;                   // patches, refs, loss, normalisation, residency guard; out = obs_out of the set
  double* xyz;                     // in/out: the points of the parameter set
  double* rec;                     // [n_obs][kInnerRec] scratch
  unsigned long long* next_point;  // zero at launch
};

struct InnerSlot {
  InnerState st;
  double x[3];      // position evaluated this round
  int64_t p, ob;    // point (-1: none left), its first observation
  int n;            // its observations (0: slot empty)
  int first;        // x is the start point
};

// K1's shared-memory ring for C >= 8; 4 warps for windows above 4 KiB, whose evaluation needs more than the 128
// registers a thread has at 2 x 256 threads per SM
template <typename T, int C> struct InnerCfg {
  static constexpr bool kSmall = C < 8;
  static constexpr int kSlot = 16 * C * (int)sizeof(T);
  static constexpr int kWarps = (kSmall || kSlot <= 4096) ? 8 : 4;
  static constexpr int kSmem = kSmall ? 0 : kWarps * kFmStages * kSlot + kWarps * kFmStages * 8 + kWarps * 32 * (int)sizeof(FmAux);
};

// takes the next point that has something to solve (one thread)
__device__ __forceinline__ void inner_claim(const InnerArgs& a, InnerSlot& sl) {
  for (;;) {
    const int64_t p = (int64_t)atomicAdd(a.next_point, 1ull);
    if (p >= a.n_points) { sl.p = -1; sl.n = 0; return; }
    const int64_t ob = a.pt_begin[p], oe = a.pt_begin[p + 1];
    if (a.point_off[p] < 0 || oe == ob) continue;
    sl.p = p; sl.ob = ob; sl.n = (int)(oe - ob); sl.first = 1;
#pragma unroll
    for (int k = 0; k < 3; ++k) sl.st.x[k] = sl.x[k] = a.xyz[3 * p + k];
    return;
  }
}

// item k of a round: slot and observation (pre = exclusive prefix of the slots' observation counts)
__device__ __forceinline__ const InnerSlot& inner_item(const InnerSlot* slots, const int pre[kInnerSlots + 1], int k, int64_t* o) {
  int s = 0, start = 0;
#pragma unroll
  for (int i = 1; i < kInnerSlots; ++i)
    if (k >= pre[i]) { s = i; start = pre[i]; }
  *o = slots[s].ob + (k - start);
  return slots[s];
}

// projection of item k: uv, and d(u)/dX, d(v)/dX into its record
__device__ __forceinline__ void inner_project(const InnerArgs& a, const InnerSlot& sl, int64_t o, double uv[2]) {
  const double X[3] = {sl.x[0], sl.x[1], sl.x[2]};
  double xy[2], sc[2], Jpose[2][6], Jpt[2][3], Jk[2][kMaxK];
  observe<true>(a.geo, o, X, uv, xy, sc, Jpose, Jpt, Jk);
  double* r = a.rec + o * kInnerRec;
#pragma unroll
  for (int k = 0; k < 3; ++k) { r[6 + k] = sc[0] * Jpt[0][k]; r[9 + k] = sc[1] * Jpt[1][k]; }
}

// C >= 8: one warp per observation; item k = base + lane * W + warp, so a round's items spread over all warps
template <typename T, int C, bool FS>
__device__ __forceinline__ void inner_eval_warps(const InnerArgs& a, const InnerSlot* slots, const int pre[kInnerSlots + 1],
                                                 int n_items, uint8_t* smem, uint32_t& phase_bits) {
  constexpr int W = InnerCfg<T, C>::kWarps;
  constexpr int CPL = C >= 32 ? C / 32 : 1;
  constexpr int ACTIVE = C / CPL;
  constexpr int TAP_BYTES = C * (int)sizeof(T);
  constexpr int SLOT_BYTES = 16 * TAP_BYTES;
  static_assert(TAP_BYTES % 16 == 0, "bulk copies need 16-byte multiples");
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* wbase = smem + (size_t)warp * kFmStages * SLOT_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)W * kFmStages * SLOT_BYTES) + warp * kFmStages;
  FmAux* aux = reinterpret_cast<FmAux*>(smem + (size_t)W * kFmStages * SLOT_BYTES + W * kFmStages * 8) + warp * 32;
  const FmEvalArgs& f = a.fm;
  const bool active = lane < ACTIVE;
  const int64_t patch_bytes = (int64_t)f.ph * f.pw * TAP_BYTES;
  for (int base = 0; base < n_items; base += 32 * W) {
    const int nvalid = min(32, (n_items - base - warp + W - 1) / W);
    if (nvalid <= 0) break;
    int64_t pt = 0;
    __syncwarp();
    if (lane < nvalid) {
      int64_t o;
      const InnerSlot& sl = inner_item(slots, pre, base + lane * W + warp, &o);
      pt = sl.p;
      double uv[2];
      inner_project(a, sl, o, uv);
      const int64_t pidx = f.item_patch ? f.item_patch[o] : o;
      const FmAux x = window_geometry(uv[0], uv[1], f.patches + pidx * patch_bytes, o, f.ph, f.pw);
      aux[lane] = x;
      if (f.res_rect && !window_resident(f.res_rect[pidx], x.row, x.col, f.ph, f.pw)) {
        const unsigned long long slot = atomicAdd(f.viol_count, 1ull);
        if ((long long)slot < f.viol_capacity) f.viol_list[slot] = o;
      }
    }
    __syncwarp();
#pragma unroll
    for (int s = 0; s < kFmStages; ++s)
      if (s < nvalid) issue_window<TAP_BYTES>(aux[s], wbase + (size_t)s * SLOT_BYTES, &bars[s], f.ph, f.pw, lane);
    for (int j = 0; j < nvalid; ++j) {
      const int slot = j % kFmStages;
      double refv[CPL];
      if (f.refs) {
        const int64_t jp = __shfl_sync(0xffffffffu, (long long)pt, j);
        const double* rp = f.refs + jp * C + (active ? lane * CPL : 0);
#pragma unroll
        for (int k = 0; k < CPL; ++k) refv[k] = __ldg(rp + k);
      }
      mbar_wait(&bars[slot], (phase_bits >> slot) & 1u);
      phase_bits ^= (1u << slot);
      double fv[CPL], fr[CPL], fc[CPL], r[CPL], red[6];
#pragma unroll
      for (int k = 0; k < CPL; ++k) { fv[k] = 0; fr[k] = 0; fc[k] = 0; r[k] = 0; }
      if (active) {
        const SmemWindow<TAP_BYTES> win{wbase + (size_t)slot * SLOT_BYTES};
        bicubic_window<T, C, CPL, true, FS>(win, lane, aux[j].xc, aux[j].xr, fv, fr, fc);
      }
      __syncwarp();
      if (j + kFmStages < nvalid)
        issue_window<TAP_BYTES>(aux[j + kFmStages], wbase + (size_t)slot * SLOT_BYTES, &bars[slot], f.ph, f.pw, lane);
      // lane 0 holds s exactly as the cost-only K1 pass computes it (same butterfly order)
      const double tot = normalize_and_reduce<CPL, true, false>(active, f.l2_normalize != 0, f.refs ? refv : nullptr, fv, fr, fc, r, red, lane);
      const int idx = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
      if ((lane & 3) == 0 && idx < 6) a.rec[aux[j].item * kInnerRec + idx] = tot;
    }
  }
}

// C < 8 (cost maps): one thread per observation
template <typename T, int C>
__device__ __forceinline__ void inner_eval_threads(const InnerArgs& a, const InnerSlot* slots, const int pre[kInnerSlots + 1], int n_items) {
  for (int k = threadIdx.x; k < n_items; k += blockDim.x) {
    int64_t o;
    const InnerSlot& sl = inner_item(slots, pre, k, &o);
    double uv[2], red[6];
    inner_project(a, sl, o, uv);
    fm_small_item<T, C, true>(a.fm, o, uv[0], uv[1], red);
    double* r = a.rec + o * kInnerRec;
#pragma unroll
    for (int i = 0; i < 6; ++i) r[i] = red[i];
  }
}

// the LM step of one slot after its evaluation, whole warp
__device__ __forceinline__ void inner_slot_step(const InnerArgs& a, InnerSlot& sl, int lane) {
  double cost = 0, H[6] = {0, 0, 0, 0, 0, 0}, g[3] = {0, 0, 0};
  for (int base = 0; base < sl.n; base += 32) {
    const int m = min(32, sl.n - base);
    double v[kInnerRec];
#pragma unroll
    for (int i = 0; i < kInnerRec; ++i) v[i] = lane < m ? a.rec[(sl.ob + base + lane) * kInnerRec + i] : 0.0;
    for (int j = 0; j < m; ++j) {           // in observation order, identically in every lane
      double w[kInnerRec];
#pragma unroll
      for (int i = 0; i < kInnerRec; ++i) w[i] = __shfl_sync(0xffffffffu, v[i], j);
      inner_add(a.fm.loss, w, w + 6, w + 9, cost, H, g);
    }
  }
  bool accepted = false, go = false;
  if (lane == 0) {
    InnerState s = sl.st;
    go = inner_step(s, sl.first != 0, cost, H, g, &accepted);
#pragma unroll
    for (int k = 0; k < 3; ++k) sl.x[k] = go ? s.cand[k] : s.x[k];
    if (!go) {
#pragma unroll
      for (int k = 0; k < 3; ++k) a.xyz[3 * sl.p + k] = s.x[k];
    }
    sl.st = s; sl.first = 0;
  }
  accepted = __shfl_sync(0xffffffffu, accepted, 0);
  go = __shfl_sync(0xffffffffu, go, 0);
  // the squared norms at the point's accepted position: obs_out then holds what a cost-only pass would compute
  if (accepted)
    for (int i = lane; i < sl.n; i += 32) a.fm.out[(sl.ob + i) * 8] = a.rec[(sl.ob + i) * kInnerRec];
  __syncwarp();
  if (!go && lane == 0) inner_claim(a, sl);
}

template <typename T, int C, bool FS>
__global__ void __launch_bounds__(InnerCfg<T, C>::kWarps * 32, 2) inner_fused_kernel(InnerArgs a) {
  typedef InnerCfg<T, C> Cfg;
  static_assert(kInnerSlots <= Cfg::kWarps, "one warp per slot runs its step");
  __shared__ InnerSlot slots[kInnerSlots];
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x < kInnerSlots) inner_claim(a, slots[threadIdx.x]);
  if (!Cfg::kSmall && lane == 0) {
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)Cfg::kWarps * kFmStages * Cfg::kSlot) + warp * kFmStages;
#pragma unroll
    for (int s = 0; s < kFmStages; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
  }
  __syncthreads();
  uint32_t phase_bits = 0;
  for (;;) {
    int pre[kInnerSlots + 1];
    pre[0] = 0;
#pragma unroll
    for (int s = 0; s < kInnerSlots; ++s) pre[s + 1] = pre[s] + slots[s].n;
    const int n_items = pre[kInnerSlots];
    if (n_items == 0) break;
    if constexpr (Cfg::kSmall) inner_eval_threads<T, C>(a, slots, pre, n_items);
    else inner_eval_warps<T, C, FS>(a, slots, pre, n_items, smem, phase_bits);
    __syncthreads();
    if (warp < kInnerSlots && slots[warp].n > 0) inner_slot_step(a, slots[warp], lane);
    __syncthreads();
  }
}

// ||a - b|| over two parameter sets (ambient), for step_norm after inner iterations
static __global__ void __launch_bounds__(256) diff_norm_kernel(const double* a, const double* b, int64_t n, double* acc, double* part = nullptr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double v = 0.0;
  if (i < n) { const double d = a[i] - b[i]; v = d * d; }
  __shared__ double sh[8];
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0; for (int k = 0; k < 8; ++k) s += sh[k];
    if (part) part[blockIdx.x] = s;          // deterministic mode (det_reduce_add_kernel)
    else atomicAdd(acc, s);
  }
}

// multi-GPU: S += lower(Hcc) + diag(D2c), rhs += -gc after the allreduce of the Schur parts
static __global__ void ba_add_reduced_kernel(const double* Hcc, const double* gc, const double* D2, double* S,
                                      double* rhs, int nc) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n2 = (int64_t)nc * nc;
  if (i < n2) {
    const int r = (int)(i / nc), c = (int)(i % nc);
    double v = c <= r ? Hcc[i] : 0.0;
    if (r == c) v += D2[r];
    S[i] += v;
  }
  if (i < nc) rhs[i] -= gc[i];
}

}  // namespace pxr
