// pxr_ba_block.cu — the multi-GPU LM iteration of featuremetric BA: image-block assembly, ONE NCCL all-reduce of the
// packed reduced-camera blocks per LM iteration, a deterministic replicated solve, and the accept/reject scalars
// exchanged through peer mailboxes over NVLink (pxr_api.cu).  Layout and invariants: pxr_block.cuh.
//
// Same trust-region logic as BA::lm_iterate (ceres TrustRegionMinimizer 2.1, reference call site
// bundle_adjustment/src/bundle_optimizer.h:224); what differs is WHEN the host learns the scalars: every LM iteration
// enqueues  assemble -> all-reduce -> solve -> back-substitute -> plus -> trial evaluation (-> inner iterations)
// without looking at anything, then exchanges all partial sums at once and synchronises ONCE.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <memory>
#include <numeric>

#include "pxr_ba_host.h"

namespace pxr {

namespace {

// CSR of "dest <- signed sources" built from an unordered contribution list: counting sort by destination ROW
// (dest / row_len) then a stable sort inside each row, so that equal inputs give equal maps on every rank.
struct Contribution { int64_t dest; int32_t src; };

struct HostGatherMap { std::vector<int64_t> dest, ptr; std::vector<int32_t> src; };

HostGatherMap make_gather_map(std::vector<Contribution>& c, int64_t n_dest_rows, int64_t row_len, bool all_rows) {
  HostGatherMap m;
  // bucket by dest / row_len
  std::vector<int64_t> cnt((size_t)n_dest_rows + 1, 0);
  for (const auto& e : c) cnt[(size_t)(e.dest / row_len) + 1]++;
  for (int64_t r = 0; r < n_dest_rows; ++r) cnt[r + 1] += cnt[r];
  std::vector<Contribution> sorted(c.size());
  {
    std::vector<int64_t> cur(cnt.begin(), cnt.end() - 1);
    for (const auto& e : c) sorted[(size_t)cur[(size_t)(e.dest / row_len)]++] = e;
  }
  for (int64_t r = 0; r < n_dest_rows; ++r)
    std::stable_sort(sorted.begin() + cnt[r], sorted.begin() + cnt[r + 1],
                     [](const Contribution& a, const Contribution& b) { return a.dest < b.dest; });
  m.src.resize(sorted.size());
  if (all_rows) {
    // one map row per destination 0..n_dest_rows*row_len-1 is only used with row_len == 1 (vectors)
    m.ptr.assign((size_t)n_dest_rows + 1, 0);
    for (size_t i = 0; i < sorted.size(); ++i) { m.src[i] = sorted[i].src; m.ptr[(size_t)sorted[i].dest + 1]++; }
    for (int64_t r = 0; r < n_dest_rows; ++r) m.ptr[r + 1] += m.ptr[r];
    return m;
  }
  m.ptr.push_back(0);
  for (size_t i = 0; i < sorted.size(); ++i) {
    if (i == 0 || sorted[i].dest != sorted[i - 1].dest) { if (i) m.ptr.push_back((int64_t)i); m.dest.push_back(sorted[i].dest); }
    m.src[i] = sorted[i].src;
  }
  if (!sorted.empty()) m.ptr.push_back((int64_t)sorted.size()); else m.ptr.assign(1, 0);
  return m;
}

__global__ void blk_pack_scalars_kernel(const double* __restrict__ scalars, const int* __restrict__ flags, double* mb_in, int stage,
                                        int is_rank0, int interrupted) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (stage == 0) {            // after the step: model cost accumulator, failure flags
    mb_in[0] = scalars[4]; mb_in[1] = (double)(flags[0] + flags[1]);
    mb_in[10] = (double)interrupted;
    mb_in[11] = scalars[13];   // max |g_p| of this rank's points at the current linearisation (MAX slot)
  } else if (stage == 1) {     // after Plus + trial evaluation
    mb_in[2] = scalars[0]; mb_in[3] = scalars[5]; mb_in[4] = scalars[6];
    mb_in[5] = is_rank0 ? scalars[7] : 0.0; mb_in[6] = is_rank0 ? scalars[8] : 0.0;      // replicated camera parts: rank 0's copy
    mb_in[7] = 0.0; mb_in[8] = 0.0; mb_in[9] = 0.0;
  } else if (stage == 2) {     // after the inner iterations
    mb_in[7] = scalars[0]; mb_in[8] = scalars[11]; mb_in[9] = is_rank0 ? scalars[12] : 0.0;
  } else {                     // a single cost (+ the MAX slot)
    mb_in[0] = scalars[0]; mb_in[11] = scalars[13];
  }
}

// a failed factorisation leaves NaNs in the camera step: neutralise it (the step is declared invalid on the host)
__global__ void blk_guard_delta_kernel(const int* __restrict__ flags, double* delta, int nc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nc && (flags[0] | flags[1])) delta[i] = 0.0;
}

}  // namespace

SparseSchur BA::sparse_blk(bool global) {
  SparseSchur q;
  q.n_images = n_images; q.n_keys = ss_n_keys; q.nc = nc;
  q.img_cols = ss_img_cols.p; q.img_pd = ss_img_pd.p; q.img_pose_blk = ss_img_pose_blk.p; q.img_cam_blk = ss_img_cam_blk.p;
  q.key_a = ss_key_a.p; q.key_b = ss_key_b.p; q.key_self = ss_key_self.p;
  q.Himg = pk(global); q.Bk = pk(global) + pk_off_B;
  return q;
}

// mb_in[0 .. n_sum) are summed over the ranks, mb_in[11] is maximised; results in mb_out (same slots)
int BA::exchange_scalars(int n_sum) {
  cudaStream_t s = ctx->stream;
  if (ctx->world <= 1) {
    PXR_CUDA(cudaMemcpyAsync(mb_out.p, mb_in.p, (size_t)kMboxSlots * 8, cudaMemcpyDeviceToDevice, s));
    return PXR_OK;
  }
  (void)n_sum;
  if (ctx->mbox_ready) return mailbox_exchange(ctx, mb_in.p, 11, 1, mb_out.p, flags.p + 3);
  // no peer access on this box: two more (tiny) NCCL calls
  PXR_CUDA(cudaMemcpyAsync(mb_out.p, mb_in.p, (size_t)kMboxSlots * 8, cudaMemcpyDeviceToDevice, s));
  PXR_TRY(allreduce_f64(ctx, mb_out.p, 11));
  return allreduce_f64(ctx, mb_out.p + 11, 1, true);
}

// -------------------------------------------------------------------------------- set-up
int BA::block_setup() {
  cudaStream_t s = ctx->stream;
  const int world = ctx->world;
  // ---- 1. the key list of the packed buffer = union of the ranks' co-visible image pairs
  std::vector<int64_t> gcode;
  if (world > 1) {
    int64_t mine = (int64_t)h_key_code_local.size();
    DevBuf<int64_t> d_cnt, d_cnt_all;
    PXR_TRY(d_cnt.upload(&mine, 1, s)); PXR_TRY(d_cnt_all.alloc(world));
    PXR_TRY(allgather_bytes(ctx, d_cnt.p, d_cnt_all.p, sizeof(int64_t)));
    std::vector<int64_t> counts(world);
    PXR_CUDA(cudaMemcpyAsync(counts.data(), d_cnt_all.p, world * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    PXR_CUDA(cudaStreamSynchronize(s));
    const int64_t maxc = *std::max_element(counts.begin(), counts.end());
    if (maxc > 0) {
      std::vector<int64_t> padded((size_t)maxc, -1);
      std::copy(h_key_code_local.begin(), h_key_code_local.end(), padded.begin());
      DevBuf<int64_t> d_keys, d_all;
      PXR_TRY(d_keys.upload(padded.data(), padded.size(), s)); PXR_TRY(d_all.alloc((size_t)maxc * world));
      PXR_TRY(allgather_bytes(ctx, d_keys.p, d_all.p, (size_t)maxc * sizeof(int64_t)));
      std::vector<int64_t> all((size_t)maxc * world);
      PXR_CUDA(cudaMemcpyAsync(all.data(), d_all.p, all.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
      PXR_CUDA(cudaStreamSynchronize(s));
      for (int r = 0; r < world; ++r) gcode.insert(gcode.end(), all.begin() + (size_t)r * maxc, all.begin() + (size_t)r * maxc + counts[r]);
      std::sort(gcode.begin(), gcode.end());
      gcode.erase(std::unique(gcode.begin(), gcode.end()), gcode.end());
    }
  } else {
    gcode = h_key_code_local;      // already ascending
  }
  if ((int64_t)gcode.size() * 64 + (int64_t)n_images * 64 >= ((int64_t)1 << 31))
    return fail(PXR_ERR_UNSUPPORTED, "too many co-visible image pairs for 32-bit block indices (%lld)", (long long)gcode.size());
  ss_n_keys = (int)gcode.size();
  h_key_a.resize(gcode.size()); h_key_b.resize(gcode.size()); h_key_self.resize(gcode.size());
  for (size_t k = 0; k < gcode.size(); ++k) {
    const int64_t pair = gcode[k] >> 1;
    int64_t ia = (int64_t)((std::sqrt(8.0 * (double)pair + 1.0) - 1.0) * 0.5);
    while ((ia + 1) * (ia + 2) / 2 <= pair) ++ia;
    while (ia * (ia + 1) / 2 > pair) --ia;
    h_key_a[k] = (int32_t)ia; h_key_b[k] = (int32_t)(pair - ia * (ia + 1) / 2); h_key_self[k] = (uint8_t)(gcode[k] & 1);
  }
  // local key -> global id, chunk keys remapped
  {
    std::vector<int32_t> l2g(h_key_code_local.size());
    for (size_t k = 0; k < h_key_code_local.size(); ++k)
      l2g[k] = (int32_t)(std::lower_bound(gcode.begin(), gcode.end(), h_key_code_local[k]) - gcode.begin());
    std::vector<int32_t> ck(h_chunk_key_local.size());
    for (size_t c = 0; c < ck.size(); ++c) ck[c] = l2g[(size_t)h_chunk_key_local[c]];
    PXR_TRY(ss_chunk_key.upload(ck.data(), ck.size(), s));
    if (deterministic) {
      // the pair chunks of one key are consecutive (the pair list is grouped by image pair): chunk range per key
      std::vector<int64_t> kb((size_t)gcode.size() + 1, 0);
      for (size_t c = 0; c < ck.size(); ++c) {
        if (c && ck[c] < ck[c - 1]) return fail(PXR_ERR_INTERNAL, "pair chunks are not grouped by key");
        kb[(size_t)ck[c] + 1]++;
      }
      for (size_t k = 0; k < gcode.size(); ++k) kb[k + 1] += kb[k];
      PXR_TRY(det_key_chunk_begin.upload(kb.data(), kb.size(), s));
      PXR_TRY(det_pair_part.alloc(std::max<size_t>(ck.size(), 1) * 72));
      PXR_TRY(det_gimg.alloc((size_t)n_images * 8)); PXR_TRY(det_rimg.alloc((size_t)n_images * 8));
      PXR_TRY(det_gimg.zero(s)); PXR_TRY(det_rimg.zero(s));
    }
    PXR_CUDA(cudaStreamSynchronize(s));
  }
  PXR_TRY(ss_key_a.upload(h_key_a.data(), h_key_a.size(), s)); PXR_TRY(ss_key_b.upload(h_key_b.data(), h_key_b.size(), s));
  PXR_TRY(ss_key_self.upload(h_key_self.data(), h_key_self.size(), s));
  PXR_TRY(ss_img_cols.upload(h_img_cols.data(), h_img_cols.size(), s));
  PXR_TRY(ss_img_pd.upload(h_img_pd.data(), h_img_pd.size(), s));
  // ---- 2. the packed buffer
  pk_off_B = (size_t)n_images * 64;
  pk_off_rhs = pk_off_B + (size_t)ss_n_keys * 64;
  pk_off_gc = pk_off_rhs + (size_t)nc;
  pk_off_slots = pk_off_gc + (size_t)nc;
  pk_n = pk_off_slots + kPackSlots;
  PXR_TRY(pack_local.alloc(pk_n)); PXR_TRY(pack_local.zero(s));
  if (world > 1) { PXR_TRY(pack_global.alloc(pk_n)); PXR_TRY(pack_global.zero(s)); }
  PXR_TRY(mb_in.alloc(kMboxSlots)); PXR_TRY(mb_out.alloc(kMboxSlots));
  PXR_TRY(mb_in.zero(s)); PXR_TRY(mb_out.zero(s));
  blk_lag_gmax = world > 1;
  // ---- 3. per-image column counts
  std::vector<int> dc(n_images, 0);
  for (int i = 0; i < n_images; ++i) for (int a = 0; a < 8; ++a) if (h_img_cols[(size_t)i * 8 + a] >= 0) dc[i] = a + 1;
  auto col = [&](int img, int a) { return (int64_t)h_img_cols[(size_t)img * 8 + a]; };
  // ---- 4. diag(H_cc): column <- H_img[a][a] of every image that owns the column
  {
    std::vector<Contribution> c;
    for (int i = 0; i < n_images; ++i) for (int a = 0; a < dc[i]; ++a) c.push_back({col(i, a), (int32_t)(i * 64 + a * 9)});
    HostGatherMap m = make_gather_map(c, std::max(nc, 1), 1, true);
    PXR_TRY(dg_ptr.upload(m.ptr.data(), m.ptr.size(), s)); PXR_TRY(dg_src.upload(m.src.data(), m.src.size(), s));
    PXR_CUDA(cudaStreamSynchronize(s));
  }
  // ---- 5. dense S (lower triangle) from the blocks, for the exact solve and the dense PCG
  if (!sparse_schur && nc > 0) {
    std::vector<Contribution> c;
    c.reserve((size_t)n_images * 36 + (size_t)ss_n_keys * 64);
    for (int i = 0; i < n_images; ++i)
      for (int a = 0; a < dc[i]; ++a) for (int b = 0; b <= a; ++b) c.push_back({col(i, a) * nc + col(i, b), (int32_t)(i * 64 + a * 8 + b)});
    for (int k = 0; k < ss_n_keys; ++k) {
      const int ia = h_key_a[k], ib = h_key_b[k]; const bool self = h_key_self[k] != 0;
      for (int a = 0; a < dc[ia]; ++a)
        for (int b = 0; b < dc[ib]; ++b) {
          const int64_t ca = col(ia, a), cb = col(ib, b);
          const int32_t src = ~(int32_t)(pk_off_B + (size_t)k * 64 + a * 8 + b);      // subtracted
          if (self) { if (a >= b) c.push_back({ca * nc + cb, src}); }
          else if (ca > cb) c.push_back({ca * nc + cb, src});
          else if (ca < cb) c.push_back({cb * nc + ca, src});
          else { c.push_back({ca * nc + ca, src}); c.push_back({ca * nc + ca, src}); }   // entry and its transpose coincide
        }
    }
    HostGatherMap m = make_gather_map(c, nc, nc, false);
    gmS_rows = (int64_t)m.dest.size();
    PXR_TRY(gmS_dest.upload(m.dest.data(), m.dest.size(), s)); PXR_TRY(gmS_ptr.upload(m.ptr.data(), m.ptr.size(), s));
    PXR_TRY(gmS_src.upload(m.src.data(), m.src.size(), s));
    PXR_CUDA(cudaStreamSynchronize(s));
  }
  // ---- 6. implicit PCG: SCHUR_JACOBI blocks and the deterministic block-row product
  if (sparse_schur && nc > 0) {
    PXR_TRY(pcg_setup_blocks());     // cg_* work space, h_img_pose_blk / h_img_cam_blk
    {
      std::vector<Contribution> c;
      for (int i = 0; i < n_images; ++i) {
        const int pd = h_img_pd[i], pb = h_img_pose_blk[i], cb = h_img_cam_blk[i];
        for (int a = 0; a < dc[i]; ++a)
          for (int b = 0; b < dc[i]; ++b) {
            const int32_t src = (int32_t)(i * 64 + (a >= b ? a * 8 + b : b * 8 + a));
            if (a < pd && b < pd) { if (pb >= 0) c.push_back({(int64_t)pb * 144 + a * 12 + b, src}); }
            else if (a >= pd && b >= pd) { if (cb >= 0) c.push_back({(int64_t)cb * 144 + (a - pd) * 12 + (b - pd), src}); }
          }
      }
      for (int k = 0; k < ss_n_keys; ++k) {
        const int ia = h_key_a[k], ib = h_key_b[k]; const bool self = h_key_self[k] != 0;
        const int pda = h_img_pd[ia], pdb = h_img_pd[ib];
        const bool same_img = ia == ib;
        const bool same_cam = h_img_cam_blk[ia] >= 0 && h_img_cam_blk[ia] == h_img_cam_blk[ib];
        if (!same_img && !same_cam) continue;
        for (int a = 0; a < dc[ia]; ++a)
          for (int b = 0; b < dc[ib]; ++b) {
            const int32_t src = ~(int32_t)(pk_off_B + (size_t)k * 64 + a * 8 + b);
            if (a < pda && b < pdb && same_img && h_img_pose_blk[ia] >= 0) {
              const int64_t D = (int64_t)h_img_pose_blk[ia] * 144;
              c.push_back({D + a * 12 + b, src});
              if (!self) c.push_back({D + b * 12 + a, src});
            }
            if (a >= pda && b >= pdb && same_cam) {
              const int64_t D = (int64_t)h_img_cam_blk[ia] * 144;
              c.push_back({D + (a - pda) * 12 + (b - pdb), src});
              if (!self) c.push_back({D + (b - pdb) * 12 + (a - pda), src});
            }
          }
      }
      HostGatherMap m = make_gather_map(c, std::max(cg_nblk, 1), 144, false);
      gmD_rows = (int64_t)m.dest.size();
      PXR_TRY(gmD_dest.upload(m.dest.data(), m.dest.size(), s)); PXR_TRY(gmD_ptr.upload(m.ptr.data(), m.ptr.size(), s));
      PXR_TRY(gmD_src.upload(m.src.data(), m.src.size(), s));
      PXR_CUDA(cudaStreamSynchronize(s));
    }
    {
      // block rows: entries of image a = (k, plain) for keys with key_a == a, (k, transposed) for non-self keys with key_b == a
      std::vector<int64_t> cnt((size_t)n_images + 1, 0);
      // (an image without camera columns has no row: its entries would never be read)
      for (int k = 0; k < ss_n_keys; ++k) {
        if (dc[h_key_a[k]] > 0) cnt[(size_t)h_key_a[k] + 1]++;
        if (!h_key_self[k] && dc[h_key_b[k]] > 0) cnt[(size_t)h_key_b[k] + 1]++;
      }
      for (int i = 0; i < n_images; ++i) cnt[i + 1] += cnt[i];
      std::vector<int32_t> ent((size_t)cnt[n_images]);
      {
        std::vector<int64_t> cur(cnt.begin(), cnt.end() - 1);
        for (int k = 0; k < ss_n_keys; ++k) {
          if (dc[h_key_a[k]] > 0) ent[(size_t)cur[h_key_a[k]]++] = k;
          if (!h_key_self[k] && dc[h_key_b[k]] > 0) ent[(size_t)cur[h_key_b[k]]++] = (int32_t)((uint32_t)k | 0x80000000u);
        }
      }
      std::vector<int64_t> cbeg; std::vector<int32_t> cimg; std::vector<uint8_t> cfirst;
      std::vector<Contribution> cols;
      for (int i = 0; i < n_images; ++i) {
        if (dc[i] == 0) continue;
        bool first = true;
        int64_t e = cnt[i];
        do {
          const int64_t chunk = (int64_t)cimg.size();
          cbeg.push_back(e); cimg.push_back(i); cfirst.push_back(first ? 1 : 0);
          for (int a = 0; a < dc[i]; ++a) cols.push_back({col(i, a), (int32_t)(chunk * 8 + a)});
          e = std::min<int64_t>(e + kRowChunk, cnt[i + 1]);
          first = false;
        } while (e < cnt[i + 1]);
      }
      // chunk c covers entries [cbeg[c], cbeg[c+1]) only within its image: close every image's last chunk explicitly
      std::vector<int64_t> cb2(cbeg.size() + 1);
      for (size_t c = 0; c < cbeg.size(); ++c) cb2[c] = cbeg[c];
      cb2[cbeg.size()] = cnt[n_images];
      // (entries are laid out image after image, so the next chunk's begin IS this chunk's end — also across images,
      //  because an image's first chunk starts at cnt[i] == end of the previous image's entries)
      br_n_chunks = (int64_t)cimg.size();
      if ((int64_t)br_n_chunks * 8 >= ((int64_t)1 << 31)) return fail(PXR_ERR_UNSUPPORTED, "too many block-row chunks");
      HostGatherMap m = make_gather_map(cols, std::max(nc, 1), 1, true);
      PXR_TRY(br_chunk_begin.upload(cb2.data(), cb2.size(), s)); PXR_TRY(br_chunk_img.upload(cimg.data(), cimg.size(), s));
      PXR_TRY(br_chunk_first.upload(cfirst.data(), cfirst.size(), s)); PXR_TRY(br_ent_key.upload(ent.data(), ent.size(), s));
      PXR_TRY(br_cols_ptr.upload(m.ptr.data(), m.ptr.size(), s)); PXR_TRY(br_cols_src.upload(m.src.data(), m.src.size(), s));
      PXR_TRY(br_ypart.alloc((size_t)std::max<int64_t>(br_n_chunks, 1) * 8));
      PXR_CUDA(cudaStreamSynchronize(s));
    }
  }
  return PXR_OK;
}

// -------------------------------------------------------------------------------- linearisation (local, no collective)
int BA::build_block() {
  StageScope st(this, 3);
  cudaStream_t s = ctx->stream;
  double* L = pack_local.p;
  PXR_CUDA(cudaMemsetAsync(L, 0, pk_off_B * 8, s));                                   // H_img
  PXR_CUDA(cudaMemsetAsync(L + pk_off_gc, 0, ((size_t)nc + kPackSlots) * 8, s));      // g_c, slots
  PXR_TRY(Hpp.zero(s)); PXR_TRY(gp.zero(s));
  if (n_obs > 0) {
    const BADev dv = dev();
    const size_t staged_smem = (size_t)128 * ((std::max(dv.juv_stride, dv.dcmax * 3) | 1) + 9) * sizeof(double);
    if (io_n_chunks > 0 && env.build_staged && staged_smem <= 48 * 1024)
      PXR_LAUNCH(ctx, ba_build_staged_kernel, (unsigned)cdiv(n_obs, 128), 128, staged_smem, dv);
    else PXR_LAUNCH(ctx, ba_build_kernel<true>, (unsigned)cdiv(n_obs, 128), 128, 0, dv, 0);
    if (io_n_chunks > 0)
      PXR_LAUNCH(ctx, ba_build_cam_kernel, (unsigned)cdiv(io_n_chunks * 32, 256), 256, 0, dv, io_obs.p, io_chunk_begin.p, io_n_chunks, L,
                 deterministic ? det_cam_part.p : nullptr);
    if (deterministic) {
      // fixed-order sums: chunk partials -> image blocks and image gradients -> columns; point blocks observation by observation
      PXR_LAUNCH(ctx, det_cam_reduce_kernel, (unsigned)cdiv((int64_t)n_images * 48, 256), 256, 0, det_cam_part.p, det_img_chunk_begin.p,
                 n_images, L, det_gimg.p);
      if (nc > 0) {
        GatherMap dg{nullptr, dg_ptr.p, dg_src.p, nc};
        PXR_LAUNCH(ctx, det_gather_cols_kernel, (unsigned)cdiv(nc, 256), 256, 0, dg, det_gimg.p, L + pk_off_gc, nc);
      }
      if (n_points > 0) PXR_LAUNCH(ctx, det_point_blocks_kernel, (unsigned)cdiv(n_points, 128), 128, 0, dv);
    }
  }
  if (n_points > 0) {
    BADev dv = dev(); dv.Hcc = nullptr;
    PXR_LAUNCH(ctx, ba_diag_kernel, (unsigned)cdiv(n_points, 256), 256, 0, dv, diag.p);               // point part only
  }
  PXR_CUDA(cudaMemsetAsync(scalars.p + 13, 0, 8, s));
  if (n_points > 0) PXR_LAUNCH(ctx, blk_gpmax_kernel, (unsigned)cdiv(n_points, 256), 256, 0, gp.p, point_off.p, n_points, scalars.p + 13);
  PXR_CUDA(cudaGetLastError());
  return PXR_OK;
}

// -------------------------------------------------------------------------------- one LM step attempt (enqueue only)
// Leaves: delta (camera + point step), scalars[4] = model cost accumulator of THIS rank's observations,
// scalars[10] = max |g| at the current point (global), flags.
int BA::compute_step_block(double radius) {
  cudaStream_t s = ctx->stream;
  BADev d = dev();
  double* L = pack_local.p;
  std::unique_ptr<StageScope> st(new StageScope(this, 4));
  const int64_t npl = nl - nc;
  if (npl > 0) PXR_LAUNCH(ctx, ba_d2_kernel, (unsigned)cdiv(npl, 256), 256, 0, diag.p + nc, jscale.p + nc, D2.p + nc, npl, radius,
                          opt.min_lm_diagonal, opt.max_lm_diagonal);
  PXR_CUDA(cudaMemsetAsync(flags.p, 0, 4 * sizeof(int), s));
  PXR_CUDA(cudaMemsetAsync(L + pk_off_B, 0, ((size_t)ss_n_keys * 64 + nc) * 8, s));               // B_key, rhsS
  if (n_points > 0 && n_obs > 0) {
    PXR_LAUNCH(ctx, ba_point_inverse_kernel, (unsigned)cdiv(n_points, 256), 256, 0, d, D2.p, Hinv.p, flags.p);
    PXR_TRY(launch_sp_schur_pairs(d, L + pk_off_B, L + pk_off_rhs, deterministic ? det_pair_part.p : nullptr));
    if (deterministic) {
      PXR_CUDA(cudaMemsetAsync(det_rimg.p, 0, (size_t)n_images * 8 * 8, s));
      if (ss_n_keys > 0)
        PXR_LAUNCH(ctx, det_pair_reduce_kernel, (unsigned)cdiv((int64_t)ss_n_keys * 72, 256), 256, 0, det_pair_part.p, det_key_chunk_begin.p,
                   ss_n_keys, ss_key_a.p, ss_key_self.p, L + pk_off_B, det_rimg.p);
      if (nc > 0) {
        GatherMap dg{nullptr, dg_ptr.p, dg_src.p, nc};
        PXR_LAUNCH(ctx, det_gather_cols_kernel, (unsigned)cdiv(nc, 256), 256, 0, dg, det_rimg.p, L + pk_off_rhs, nc);
      }
    }
  }
  st.reset();
  if (nc > 0) {
    // ---- THE collective of this LM iteration
    if (ctx->world > 1) { StageScope sc(this, 11); PXR_TRY(allreduce_f64_oop(ctx, pack_local.p, pack_global.p, pk_n)); }
    st.reset(new StageScope(this, 4));
    const double* G = pk(true);
    PXR_CUDA(cudaMemsetAsync(scalars.p + 10, 0, 8, s));
    PXR_CUDA(cudaMemsetAsync(scalars.p + 14, 0, 8, s));
    GatherMap dg{nullptr, dg_ptr.p, dg_src.p, nc};
    PXR_LAUNCH(ctx, blk_post_kernel, (unsigned)cdiv(nc, 256), 256, 0, dg, G, G + pk_off_gc, G + pk_off_rhs, diag.p, jscale.p,
               jscale_c_pending ? 1 : 0, opt.jacobi_scaling, D2.p, radius, opt.min_lm_diagonal, opt.max_lm_diagonal, rhs.p, nc, scalars.p + 14);
    {   // camera part of ceres' gradient_max_norm from the GLOBAL gradient (quaternion blocks through the manifold)
      const int64_t n = std::max<int64_t>(n_images, n_cameras);
      PXR_LAUNCH(ctx, ba_gradmax_kernel, (unsigned)cdiv(n, 256), 256, 0, d, G + pk_off_gc, q[cur].p, 0, scalars.p + 10);
    }
    jscale_c_pending = false;
    last_linear_iterations = 1;
    if (sparse_schur) {
      st.reset(); st.reset(new StageScope(this, 5));
      PXR_TRY(pcg_solve_block());
    } else {
      PXR_CUDA(cudaMemsetAsync(S.p, 0, (size_t)(nc + 1) * nc * 8, s));
      GatherMap gm{gmS_dest.p, gmS_ptr.p, gmS_src.p, gmS_rows};
      if (gmS_rows > 0) PXR_LAUNCH(ctx, blk_gather_kernel, (unsigned)cdiv(gmS_rows, 256), 256, 0, gm, G, S.p, D2.p, nc);
      PXR_CUDA(cudaMemcpyAsync(S.p + (size_t)nc * nc, rhs.p, (size_t)nc * 8, cudaMemcpyDeviceToDevice, s));
      st.reset(); st.reset(new StageScope(this, 5));
      if (use_pcg) PXR_TRY(pcg_solve()); else PXR_TRY(chol_launch());
    }
    PXR_LAUNCH(ctx, blk_guard_delta_kernel, (unsigned)cdiv(nc, 256), 256, 0, flags.p, delta.p, nc);
  } else {
    PXR_CUDA(cudaMemsetAsync(scalars.p + 10, 0, 8, s));        // no camera columns: max |g| is the point part alone
  }
  st.reset(); st.reset(new StageScope(this, 7));
  PXR_CUDA(cudaMemsetAsync(scalars.p + 4, 0, 4 * 8, s));
  if (n_points > 0) PXR_LAUNCH(ctx, ba_backsub_kernel, (unsigned)cdiv(n_points * 32, 256), 256, 0, d, D2.p, delta.p);
  if (n_obs > 0) {
    double* part = deterministic ? det_scal_part.p : nullptr;
    if (img_src8.p) PXR_LAUNCH(ctx, ba_model_cost_kernel<true>, (unsigned)cdiv(n_obs, 256), 256, 0, d, delta.p, scalars.p + 4, part);
    else PXR_LAUNCH(ctx, ba_model_cost_kernel<false>, (unsigned)cdiv(n_obs, 256), 256, 0, d, delta.p, scalars.p + 4, part);
    if (part) PXR_LAUNCH(ctx, det_reduce_add_kernel, 1, 1024, 0, part, cdiv(n_obs, 256), 1, 0, scalars.p + 4);
  }
  PXR_CUDA(cudaGetLastError());
  return PXR_OK;
}

int BA::global_cost_block(double* cost_out) {
  cudaStream_t s = ctx->stream;
  PXR_CUDA(cudaMemsetAsync(flags.p + 3, 0, sizeof(int), s));
  PXR_LAUNCH(ctx, blk_pack_scalars_kernel, 1, 1, 0, scalars.p, flags.p, mb_in.p, 3, ctx->rank == 0 ? 1 : 0, 0);
  PXR_TRY(exchange_scalars(1));
  double c = 0; int mfail = 0;
  PXR_CUDA(cudaMemcpyAsync(&c, mb_out.p, 8, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaMemcpyAsync(&mfail, flags.p + 3, sizeof(int), cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  if (mfail) return fail(PXR_ERR_NCCL, "a peer rank did not deliver its scalars (mailbox time-out)");
  *cost_out = c;
  return PXR_OK;
}

int BA::compute_step_block_sync(double radius, bool* valid, double* model_cost_change) {
  cudaStream_t s = ctx->stream;
  PXR_TRY(compute_step_block(radius));
  PXR_LAUNCH(ctx, blk_pack_scalars_kernel, 1, 1, 0, scalars.p, flags.p, mb_in.p, 0, ctx->rank == 0 ? 1 : 0, 0);
  PXR_TRY(exchange_scalars(2));
  double o[2] = {0, 0}; int mfail = 0;
  PXR_CUDA(cudaMemcpyAsync(o, mb_out.p, 16, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaMemcpyAsync(&mfail, flags.p + 3, sizeof(int), cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  if (mfail) return fail(PXR_ERR_NCCL, "a peer rank did not deliver its scalars (mailbox time-out)");
  *model_cost_change = -o[0];
  *valid = o[1] == 0.0 && std::isfinite(o[0]) && *model_cost_change > 0.0;
  return PXR_OK;
}

// ITERATIVE_SCHUR on the GLOBAL image blocks, run redundantly and deterministically by every rank: no communication
int BA::pcg_solve_block() {
  cudaStream_t s = ctx->stream;
  PXR_TRY(pcg_setup_blocks());
  const SparseSchur sp = sparse_blk(true);
  const double* G = pk(true);
  PXR_TRY(ss_Dblk.zero(s));
  GatherMap gd{gmD_dest.p, gmD_ptr.p, gmD_src.p, gmD_rows};
  if (gmD_rows > 0) PXR_LAUNCH(ctx, blk_gather_kernel, (unsigned)cdiv(gmD_rows, 256), 256, 0, gd, G, ss_Dblk.p, (const double*)nullptr, 1);
  PXR_LAUNCH(ctx, sp_block_inverse_kernel, (unsigned)cdiv(cg_nblk, 64), 64, 0, ss_Dblk.p, D2.p, 1, cg_blk_off.p, cg_blk_dim.p, cg_nblk,
             cg_Minv.p, cg_row_off.p, cg_row_dim.p, flags.p + 1);
  BlockRows br;
  br.chunk_begin = br_chunk_begin.p; br.chunk_img = br_chunk_img.p; br.chunk_first = br_chunk_first.p; br.ent_key = br_ent_key.p;
  br.n_chunks = br_n_chunks; br.cols = GatherMap{nullptr, br_cols_ptr.p, br_cols_src.p, nc};
  const int n = nc;
  auto spmv = [&](const double* x, double* y) -> int {
    if (br_n_chunks > 0) PXR_LAUNCH(ctx, blk_rows_kernel, (unsigned)cdiv(br_n_chunks * 8, 256), 256, 0, sp, br, x, br_ypart.p, cg_state.p);
    PXR_LAUNCH(ctx, blk_cols_kernel, (unsigned)cdiv(n, 256), 256, 0, br.cols, br_ypart.p, D2.p, x, y, n, cg_state.p);
    return PXR_OK;
  };
  return run_cg(spmv);
}

// -------------------------------------------------------------------------------- LM driver (block mode)
int BA::lm_begin_block() {
  PXR_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  lm = LMState();
  lm.radius = opt.initial_trust_region_radius;
  lm.inner_enabled = opt.use_inner_iterations != 0;
  // ---- IterationZero
  PXR_TRY(project(cur, true, nullptr));
  PXR_TRY(fm(1, nullptr, scalars.p + 0));
  PXR_TRY(build_block());
  PXR_TRY(global_cost_block(&lm.x_cost));
  if (!std::isfinite(lm.x_cost)) return fail(PXR_ERR_NUMERIC, "initial cost is not finite");
  // Jacobi scaling: point columns now, camera columns right after the first all-reduce (they need the global diagonal)
  if (nl - nc > 0) PXR_LAUNCH(ctx, ba_scale_kernel, (unsigned)cdiv(nl - nc, 256), 256, 0, diag.p + nc, jscale.p + nc, nl - nc, opt.jacobi_scaling);
  jscale_c_pending = true;
  std::memset(&lm.it, 0, sizeof(lm.it));
  lm.it.cost = lm.x_cost;
  if (blk_lag_gmax) { lm.it.gradient_max_norm = std::numeric_limits<double>::quiet_NaN(); lm.gmax_pending = true; }
  else { PXR_TRY(gradient_max_norm(&lm.it.gradient_max_norm)); lm.gmax_pending = false; }
  lm.initial_cost = lm.minimum_cost = lm.x_cost;
  lm.ev.init(lm.x_cost, opt.use_nonmonotonic_steps ? opt.max_consecutive_nonmonotonic_steps : 0);
  lm.best_is_current = true;
  lm.started = true;
  lm.pending_finalize = true;
  lm.term = 1;
  lm.message = "Maximum number of iterations reached.";
  return PXR_OK;
}

// max |g| of the current point when no further LM iteration will deliver it: one small all-reduce of g_c, and the
// per-rank point maxima through the scalar exchange
int BA::finish_gmax_block() {
  if (!lm.gmax_pending) return PXR_OK;
  cudaStream_t s = ctx->stream;
  PXR_CUDA(cudaMemsetAsync(scalars.p + 10, 0, 8, s));
  if (nc > 0) {
    PXR_TRY(allreduce_f64_oop(ctx, pack_local.p + pk_off_gc, pk(true) + pk_off_gc, (size_t)nc));
    const int64_t n = std::max<int64_t>(n_images, n_cameras);
    PXR_LAUNCH(ctx, ba_gradmax_kernel, (unsigned)cdiv(n, 256), 256, 0, dev(), pk(true) + pk_off_gc, q[cur].p, 0, scalars.p + 10);
  }
  PXR_CUDA(cudaMemsetAsync(flags.p + 3, 0, sizeof(int), s));
  PXR_LAUNCH(ctx, blk_pack_scalars_kernel, 1, 1, 0, scalars.p, flags.p, mb_in.p, 3, ctx->rank == 0 ? 1 : 0, 0);
  PXR_TRY(exchange_scalars(1));
  double gcm = 0, gpm = 0;
  PXR_CUDA(cudaMemcpyAsync(&gcm, scalars.p + 10, 8, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaMemcpyAsync(&gpm, mb_out.p + 11, 8, cudaMemcpyDeviceToHost, s));
  PXR_CUDA(cudaStreamSynchronize(s));
  const double g = std::max(gcm, gpm);
  lm.it.gradient_max_norm = g;
  if (!lm.its.empty() && !(lm.its.back().gradient_max_norm == lm.its.back().gradient_max_norm)) lm.its.back().gradient_max_norm = g;
  lm.gmax_pending = false;
  return PXR_OK;
}

int BA::lm_iterate_block(int max_iteration) {
  using clk = std::chrono::steady_clock;
  cudaStream_t s = ctx->stream;
  if (!lm.started) PXR_TRY(lm_begin_block());
  lm.it_start = clk::now();
  const double kMax = std::numeric_limits<double>::max();
  while (!lm.finished && lm_finalize(max_iteration)) {
    const int interrupted = interrupt_pending() ? 1 : 0;      // agreed on through the scalar exchange (a rank must not leave alone)
    lm.it_start = clk::now();
    pxr_iteration_summary& it = lm.it;
    const pxr_iteration_summary prev_it = it;
    const double prev_gmax = it.gradient_max_norm;
    const int iteration = it.iteration + 1;
    std::memset(&it, 0, sizeof(it));
    it.iteration = iteration;
    lm.pending_finalize = true;

    // ---- enqueue the whole iteration
    PXR_TRY(compute_step_block(lm.radius));
    it.linear_solver_iterations = last_linear_iterations;
    PXR_LAUNCH(ctx, blk_pack_scalars_kernel, 1, 1, 0, scalars.p, flags.p, mb_in.p, 0, ctx->rank == 0 ? 1 : 0, interrupted);
    PXR_TRY(apply_step(nullptr, nullptr));
    swap_sets();
    const bool speculate = !lm.inner_enabled && !env.no_speculation;
    const bool ran_inner = lm.inner_enabled;
    int rc = project(1 - cur, speculate, nullptr);
    if (rc == PXR_OK) rc = fm(speculate ? 1 : 0, nullptr, scalars.p + 0);
    if (rc != PXR_OK) { swap_sets(); return rc; }
    PXR_LAUNCH(ctx, blk_pack_scalars_kernel, 1, 1, 0, scalars.p, flags.p, mb_in.p, 1, ctx->rank == 0 ? 1 : 0, 0);
    if (ran_inner) {
      // ceres skips them when the trial cost is not finite — a GLOBAL fact that is only known after the exchange; they are
      // per-point and local, so they run regardless and their result is ignored in that case (the step is rejected)
      rc = inner_iterations(1 - cur);
      if (rc == PXR_OK) rc = fm_cost(scalars.p + 0);
      if (rc != PXR_OK) { swap_sets(); return rc; }
      PXR_CUDA(cudaMemsetAsync(scalars.p + 11, 0, 16, s));
      auto run = [&](const double* a, const double* b, int64_t n, double* acc) {
        if (n <= 0) return;
        PXR_LAUNCH(ctx, diff_norm_kernel, (unsigned)cdiv(n, 256), 256, 0, a, b, n, acc, deterministic ? det_scal_part.p : nullptr);
        if (deterministic) PXR_LAUNCH(ctx, det_reduce_add_kernel, 1, 1024, 0, det_scal_part.p, cdiv(n, 256), 1, 0, acc);
      };
      run(cam[0].p, cam[1].p, (int64_t)n_cameras * kMaxK, scalars.p + 12);
      run(q[0].p, q[1].p, (int64_t)n_images * 4, scalars.p + 12);
      run(t[0].p, t[1].p, (int64_t)n_images * 3, scalars.p + 12);
      run(X[0].p, X[1].p, n_points * 3, scalars.p + 11);
      PXR_LAUNCH(ctx, blk_pack_scalars_kernel, 1, 1, 0, scalars.p, flags.p, mb_in.p, 2, ctx->rank == 0 ? 1 : 0, 0);
    }
    PXR_TRY(exchange_scalars(11));
    double o[12]; double gmax_here = 0; int mfail = 0;
    PXR_CUDA(cudaMemcpyAsync(o, mb_out.p, sizeof(o), cudaMemcpyDeviceToHost, s));
    PXR_CUDA(cudaMemcpyAsync(&gmax_here, scalars.p + 10, 8, cudaMemcpyDeviceToHost, s));
    PXR_CUDA(cudaMemcpyAsync(&mfail, flags.p + 3, sizeof(int), cudaMemcpyDeviceToHost, s));
    PXR_CUDA(cudaStreamSynchronize(s));                         // the ONE host synchronisation of the iteration
    swap_sets();   // back: uv/obs_out/juv = linearisation at the current point again
    if (mfail) { lm.finished = true; lm.term = 2; return fail(PXR_ERR_NCCL, "a peer rank did not deliver its scalars (mailbox time-out)"); }
    gmax_here = std::max(gmax_here, o[11]);    // camera part (global g_c) | point part (max over the ranks)

    // ---- what the host would have known earlier on one GPU
    if (lm.gmax_pending) {
      // max |g| at the CURRENT point arrives with this iteration's all-reduce; ceres tests it before starting the
      // iteration: when it already meets the tolerance, this iteration never happened
      lm.gmax_pending = false;
      if (!lm.its.empty()) lm.its.back().gradient_max_norm = gmax_here;
      if (gmax_here <= opt.gradient_tolerance) {
        it = prev_it; it.gradient_max_norm = gmax_here;
        lm.pending_finalize = false;
        lm.term = 0; lm.message = "Gradient tolerance reached."; lm.finished = true;
        break;
      }
    }
    const double known_gmax = blk_lag_gmax ? gmax_here : prev_gmax;
    if (o[10] > 0.0) {
      it = prev_it; lm.pending_finalize = false;
      lm.finished = true; lm.term = 3; lm.message = "interrupted by the host";
      return fail(PXR_ERR_INTERRUPTED, "interrupted by the host after LM iteration %d", it.iteration);
    }
    double model_cost_change = -o[0];
    const bool valid = o[1] == 0.0 && std::isfinite(o[0]) && model_cost_change > 0.0;
    it.step_is_valid = valid;
    if (!valid) {
      if (++lm.num_invalid >= opt.max_num_consecutive_invalid_steps) {
        lm.term = 2; lm.finished = true;
        lm.message = "Number of consecutive invalid steps more than Solver::Options::max_num_consecutive_invalid_steps";
        break;
      }
      lm.radius /= lm.decrease_factor; lm.decrease_factor *= 2.0;
      it.cost = lm.x_cost; it.gradient_max_norm = known_gmax;
      continue;
    }
    lm.num_invalid = 0;
    double candidate_cost = o[2];
    if (!std::isfinite(candidate_cost)) candidate_cost = kMax;
    double step_norm = std::sqrt(o[3] + o[5]);
    const double x_norm = std::sqrt(o[4] + o[6]);
    bool inner_useful = false;
    if (ran_inner && candidate_cost < kMax) {
      ++lm.n_inner;
      const double inner_cost = o[7];
      if (std::isfinite(inner_cost)) {
        model_cost_change += candidate_cost - inner_cost;
        inner_useful = inner_cost < lm.x_cost;
        const double rel = 1.0 - inner_cost / candidate_cost;
        lm.inner_enabled = rel > opt.inner_iteration_tolerance;
        candidate_cost = inner_cost;
        step_norm = std::sqrt(o[8] + o[9]);
      }
    }
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
      if (speculate && candidate_cost < kMax) {
        swap_sets();                 // the speculative pass IS the linearisation at the new point
        PXR_TRY(build_block());
      } else {
        PXR_TRY(project(cur, true, nullptr));
        PXR_TRY(fm(1, nullptr, scalars.p + 0));
        PXR_TRY(build_block());
      }
      lm.x_cost = candidate_cost;    // same point, same residuals: the trial cost is the new cost
      it.cost = lm.x_cost;
      if (blk_lag_gmax) { it.gradient_max_norm = std::numeric_limits<double>::quiet_NaN(); lm.gmax_pending = true; }
      else PXR_TRY(gradient_max_norm(&it.gradient_max_norm));
      it.step_is_successful = 1;
      lm.radius = lm.radius / std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * it.relative_decrease - 1.0, 3));
      lm.radius = std::min(opt.max_trust_region_radius, lm.radius);
      lm.decrease_factor = 2.0;
      lm.ev.accepted(candidate_cost, model_cost_change);
      if (opt.use_nonmonotonic_steps) {
        if (lm.x_cost < lm.minimum_cost) lm.best_is_current = true;
        else if (lm.best_is_current) { PXR_TRY(save_best(1 - cur)); lm.best_is_current = false; }
      }
    } else {
      it.step_is_successful = 0;
      it.cost = candidate_cost;
      it.gradient_max_norm = known_gmax;
      lm.radius /= lm.decrease_factor; lm.decrease_factor *= 2.0;
    }
  }
  if (lm.x_cost < lm.minimum_cost) lm.minimum_cost = lm.x_cost;
  if (lm.finished) PXR_TRY(finish_gmax_block());
  PXR_CUDA(cudaStreamSynchronize(s));
  return PXR_OK;
}

}  // namespace pxr
