// Batched NMF solver: all (k, seed) restarts of cNMF.factorize (cnmf.py:735-745) advance together.
//
// One outer iteration of sklearn's solvers (MU: _nmf.py:826-879, CD: _nmf.py:491-516) becomes
//   NUM_r = Fc * X^T            tensor-core GEMM, M = sum k (all restarts), N = n_r, reduce over n_c
//   Fr   <- update(Fr, NUM_r, Gram(Fc))       elementwise, K x K Gram from smem
//   NUM_c = Fr * X              tensor-core GEMM, split-K over n_r
//   Fc   <- update(Fc, NUM_c, Gram(Fr))
// with Fr = W^T (SK x cells) and Fc = H (SK x genes), so the data matrix is streamed once per
// product for ALL restarts.  Convergence is evaluated on the device per restart (trace-form
// Frobenius error for MU, projected-gradient violation for CD); converged restarts are frozen
// (their blocks exit) and the host only polls the flags.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "engine.h"
#include "gemm.h"
#include "nmf_kernels.cuh"

namespace cnmf {

DataView make_view(const cnmf_dataset_s* d, bool transposed) {
  Operand X{d->X, d->X_hi, d->X_lo, d->f16 ? d->X_h16 : nullptr, d->n_rows, d->n_cols, d->ld_c};
  Operand Xt{d->Xt, d->Xt_hi, d->Xt_lo, d->f16 ? d->Xt_h16 : nullptr, d->n_cols, d->n_rows, d->ld_r};
  DataView v;
  if (!transposed) {
    v.B_rows = X; v.B_cols = Xt;
    v.n_r = d->n_rows; v.n_c = d->n_cols; v.ld_r = d->ld_r; v.ld_c = d->ld_c;
  } else {
    v.B_rows = Xt; v.B_cols = X;
    v.n_r = d->n_cols; v.n_c = d->n_rows; v.ld_r = d->ld_c; v.ld_c = d->ld_r;
  }
  v.sum = d->sum;
  v.sum_sq = d->sum_sq;
  v.exact = d->exact;
  v.f16 = d->f16;
  v.scale_r = transposed ? d->col_scale : d->row_scale;
  v.scale_c = transposed ? d->row_scale : d->col_scale;
  return v;
}

namespace {

// C[z] (SK x B.rows) = A (SK x B.cols) * B^T, counted and profiled as one GEMM launch
int run_gemm(cnmf_handle_s* h, bool tc, const GemmA& A, int SK, const Operand& B, float* C, int ldc,
             const GemmPlan& plan, bool exact, const float* out_scale, cudaStream_t s) {
  h->launches += 1;
  const int slot = h->prof_begin(s, 2.0 * (double)SK * (double)B.rows * (double)B.cols);
  const int rc = gemm_run(tc, exact, out_scale, SK, A, B, C, ldc, plan, s);
  h->prof_end(s, slot);
  return rc;
}

}  // namespace

int solve_batched(cnmf_handle_s* h, const DataView& v, SolveIO& io, const cnmf_nmf_params& p, cudaStream_t s) {
  const int R0 = io.R;
  if (p.beta_loss != CNMF_LOSS_FROBENIUS) return solve_batched_beta(h, v, io, p, s);
  CNMF_REQUIRE(R0 > 0 && (int)io.ks.size() == R0, "solve: bad restart list");
  CNMF_REQUIRE(p.solver == CNMF_SOLVER_MU || p.solver == CNMF_SOLVER_CD, "solve: unknown solver");
  CNMF_REQUIRE(p.max_iter >= 1, "solve: max_iter must be >= 1");
  const bool tf32 = p.precision == CNMF_PRECISION_TF32X3;
  const bool f16 = tf32 && v.f16;       // exact-count dataset created with CNMF_PRECISION_F16X2: kind::f16 products
  const bool mu = p.solver == CNMF_SOLVER_MU;

  // ---- slot tables (host mirrors); slot s holds restart rid[s] at packed rows [off[s], off[s]+k[s])
  std::vector<int> off0(R0), s_off(R0), s_k(io.ks), s_rid(R0);
  int SK0 = 0, kmax = 0;
  for (int r = 0; r < R0; ++r) {
    CNMF_REQUIRE(io.ks[r] >= 1 && io.ks[r] <= KMAX, "solve: n_components must be in [1, 32] on the CUDA path");
    off0[r] = s_off[r] = SK0;
    s_rid[r] = r;
    SK0 += io.ks[r];
    kmax = std::max(kmax, io.ks[r]);
  }
  int R = R0, SK = SK0;     // live slots / live packed rows
  const int kp = kmax <= 16 ? 16 : 32;
  // block granularity of the streaming kernels, fixed for the whole solve (partial buffers are sized by it)
  // update kernels: 3 blocks of 128 threads per SM resident, a block walks 1-4 tiles -> aim for >= 8 blocks per SM;
  // stand-alone Gram kernel: 1 block/SM resident and a fixed-cost block reduction -> long blocks, about two waves
  const int tile = upd_tile_cols(kp);
  // the update kernels' chunking follows the number of LIVE restarts (re-planned after every compaction): with few
  // restarts left a block should hold one tile, so that the work spreads over many SMs
  int cpb_r = 0, cpb_c = 0, chunks_r = 0, chunks_c = 0;
  auto plan_blocks = [&](int r_live) {
    cpb_r = pick_cols_per_block(v.n_r, r_live, 4 * tile, tile, 148 * 8);
    cpb_c = pick_cols_per_block(v.n_c, r_live, 4 * tile, tile, 148 * 8);
    chunks_r = (v.n_r + cpb_r - 1) / cpb_r;
    chunks_c = (v.n_c + cpb_c - 1) / cpb_c;
  };
  const int gcpb_r = pick_cols_per_block(v.n_r, R0, 8192, 1024, 148 * 2), gcpb_c = pick_cols_per_block(v.n_c, R0, 8192, 1024, 148 * 2);
  const int chunks_cap = std::max((v.n_r + tile - 1) / tile, (v.n_c + tile - 1) / tile);   // finest chunking possible
  const int gchunks_max = std::max((v.n_r + gcpb_r - 1) / gcpb_r, (v.n_c + gcpb_c - 1) / gcpb_c);
  size_t fused_part_slots = 0;      // slot-indexed partials of the fused kernels: max over live counts of R * chunks
  for (int r = 1; r <= R0; ++r) {
    plan_blocks(r);
    fused_part_slots = std::max(fused_part_slots, (size_t)r * std::max(chunks_r, chunks_c));
  }
  plan_blocks(R0);
  const bool fuse = kp == 16;   // the update kernels emit the Gram of the factor they write (nmf_kernels.cu)

  // ---- workspace
  int* d_meta = static_cast<int*>(h->dev_buf("solve.meta", sizeof(int) * 8 * R0));
  double* d_state = static_cast<double*>(h->dev_buf("solve.state", sizeof(double) * 8 * R0));
  double* d_gram = static_cast<double*>(h->dev_buf("solve.gram", sizeof(double) * 2 * R0 * KMAX * KMAX));
  // per-block Gram partials of each factor (summed by the last block of the producing launch)
  const size_t gpart_elems = std::max((size_t)R0 * std::max(gchunks_max, std::max((v.n_r + 1023) / 1024, (v.n_c + 1023) / 1024)),
                                     fused_part_slots) * kp * kp;
  double* d_gram_part = static_cast<double*>(h->dev_buf("solve.gram_part", sizeof(double) * 2 * gpart_elems));
  double* d_scal_part = static_cast<double*>(h->dev_buf("solve.scal_part", sizeof(double) * 2 * (size_t)R0 * chunks_cap));
  if (!d_meta || !d_state || !d_gram || !d_gram_part || !d_scal_part) return -2;

  GemmPlan plan_r, plan_c;   // plan_r: NUM_r = Fc * B_rows^T (reduce over n_c); plan_c: NUM_c = Fr * B_cols^T
  float *NUMr = nullptr, *NUMc = nullptr;
  auto plan_one = [&](int sk, int n, int kd, GemmPlan* pl) {
    if (tf32) {
      gemm_plan(sk, n, kd, h->sm_count, &pl->splits, &pl->bn, f16 ? 1 : 0);
    } else {
      pl->splits = gemm_fixed_splits(kd, 0);
      pl->bn = 0;
    }
  };
  auto plan_gemms = [&]() -> int {
    plan_one(SK, v.n_r, v.n_c, &plan_r);
    plan_r.split_stride = (long long)SK * v.ld_r;
    plan_one(SK, v.n_c, v.n_r, &plan_c);
    plan_c.split_stride = (long long)SK * v.ld_c;
    return 0;
  };
  plan_gemms();
  // size the product buffers: the split-K factor depends on the reduction length only, the rows never exceed SK0
  {
    const size_t need_r = (size_t)plan_r.splits * (size_t)SK0 * v.ld_r;
    const size_t need_c = (size_t)plan_c.splits * (size_t)SK0 * v.ld_c;
    NUMr = static_cast<float*>(h->dev_buf("solve.NUMr", sizeof(float) * need_r));
    NUMc = io.update_cols ? static_cast<float*>(h->dev_buf("solve.NUMc", sizeof(float) * need_c)) : nullptr;
    if (!NUMr || (io.update_cols && !NUMc)) return -2;
  }

  int* d_off = d_meta;             // [slots]
  int* d_k = d_meta + R0;          // [slots]
  int* d_rid = d_meta + 2 * R0;    // [slots]
  int* d_done = d_meta + 3 * R0;   // [rid]
  int* d_niter = d_meta + 4 * R0;  // [rid]
  int* d_ticket = d_meta + 5 * R0; // [rid] last-block tickets of the fused update kernels (self-resetting)
  auto upload_slots = [&]() -> int {
    std::vector<int> hm(3 * R0, 0);
    std::memcpy(hm.data(), s_off.data(), sizeof(int) * R);
    std::memcpy(hm.data() + R0, s_k.data(), sizeof(int) * R);
    std::memcpy(hm.data() + 2 * R0, s_rid.data(), sizeof(int) * R);
    CNMF_CUDA_CHECK(cudaMemcpyAsync(d_meta, hm.data(), sizeof(int) * 3 * R0, cudaMemcpyHostToDevice, s));
    CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
    return 0;
  };
  CNMF_TRY(upload_slots());
  CNMF_CUDA_CHECK(cudaMemsetAsync(d_done, 0, sizeof(int) * 3 * R0, s));   // done, n_iter, tickets
  CNMF_CUDA_CHECK(cudaMemsetAsync(d_state, 0, sizeof(double) * 8 * R0, s));
  ConvState st{d_state, d_state + R0, d_state + 2 * R0, d_done, d_niter};
  double* d_crossA = d_state + 3 * R0;   // finalised scalars: cross / violation of the row half
  double* d_crossB = d_state + 4 * R0;   // ... of the column half
  double* d_gramR = d_gram;                            // Gram of Fr (e.g. W^T W), by rid
  double* d_gramC = d_gram + (size_t)R0 * KMAX * KMAX; // Gram of Fc (e.g. H H^T), by rid
  double* d_scalA = d_scal_part;
  double* d_scalB = d_scal_part + (size_t)R0 * chunks_cap;
  double* d_gpartR = d_gram_part;                      // partials of Gram(Fr)
  double* d_gpartC = d_gram_part + gpart_elems;        // partials of Gram(Fc)

  // working factor arrays (start in the caller's buffers; compaction ping-pongs to "solve.alt.*")
  float *wFr = io.Fr, *wFr_hi = io.Fr_hi, *wFr_lo = io.Fr_lo, *wFc = io.Fc, *wFc_hi = io.Fc_hi, *wFc_lo = io.Fc_lo;
  float *aFr = nullptr, *aFr_hi = nullptr, *aFr_lo = nullptr, *aFc = nullptr, *aFc_hi = nullptr, *aFc_lo = nullptr;
  float *resFr = nullptr, *resFc = nullptr;   // final factors of restarts that were compacted away (original offsets)
  bool compacted = false;

  auto bm = [&]() { return BatchMeta{d_off, d_k, d_rid, d_done, R, kp}; };
  float* d_rs_r = nullptr;   // f16: power-of-two scales of the Fr / Fc pieces, [packed row][512-element group]
  float* d_rs_c = nullptr;
  if (f16) {
    d_rs_r = static_cast<float*>(h->dev_buf("solve.rowscale_r", sizeof(float) * (size_t)SK0 * ((v.ld_r + 511) / 512)));
    d_rs_c = static_cast<float*>(h->dev_buf("solve.rowscale_c", sizeof(float) * (size_t)SK0 * ((v.ld_c + 511) / 512)));
    if (!d_rs_r || !d_rs_c) return -2;
  }
  // tf32 pieces are written by the update kernels; the fp16 pieces need the row maximum first and come from
  // emit_pieces() after the update (the hi / lo buffers then hold halves)
  const bool upd_pieces = tf32 && !f16;
  // f16: the Gram-fused update kernels (K <= 16, factor being iterated) emit the fp16 pieces themselves, per 512-column
  // tile; everything else (initial factors, compaction, K > 16) goes through emit_pieces() with one scale per row
  const int ktiles_r = (v.ld_r + 511) / 512, ktiles_c = (v.ld_c + 511) / 512;
  const bool emit_in_update = f16 && kp == 16 && io.update_cols;
  auto fr = [&]() {
    FactorView f{};
    f.F = wFr; f.F_hi = upd_pieces ? wFr_hi : nullptr; f.F_lo = upd_pieces ? wFr_lo : nullptr;
    f.n = v.n_r; f.ld = v.ld_r; f.piece_scale = v.exact ? v.scale_r : nullptr;
    if (emit_in_update) { f.P_hi = wFr_hi; f.P_mid = wFr_lo; f.tile_scale = d_rs_r; f.n_ktiles = ktiles_r; }
    f.cpb = cpb_r; f.gcpb = gcpb_r;
    return f;
  };
  auto fc = [&]() {
    FactorView f{};
    f.F = wFc; f.F_hi = upd_pieces ? wFc_hi : nullptr; f.F_lo = upd_pieces ? wFc_lo : nullptr;
    f.n = v.n_c; f.ld = v.ld_c; f.piece_scale = v.exact ? v.scale_c : nullptr;
    if (emit_in_update) { f.P_hi = wFc_hi; f.P_mid = wFc_lo; f.tile_scale = d_rs_c; f.n_ktiles = ktiles_c; }
    f.cpb = cpb_c; f.gcpb = gcpb_c;
    if (!io.update_cols) { f.F_hi = nullptr; f.F_lo = nullptr; }   // never rewritten
    return f;
  };
  // side: 0 = row factor Fr, 1 = column factor Fc.  Stand-alone Gram: partial launch + finalize (initial factors,
  // fixed factors of a refit, batches with K > 16).
  auto gram_full = [&](const FactorView& f, int side_is_c) -> int {
    h->launches += 2;
    double* part = side_is_c ? d_gpartC : d_gpartR;
    CNMF_TRY(launch_gram_partial(f, bm(), part, s));
    return launch_finalize(part, side_is_c ? d_gramC : d_gramR, nullptr, nullptr, gram_chunks(f), bm(), s);
  };
  auto gram_after = [&](const FactorView& f, int side_is_c) -> int {   // Gram of a factor the update kernel just wrote
    return fuse ? 0 : gram_full(f, side_is_c);
  };
  auto emit_pieces = [&](int side_is_c) -> int {   // fp16 pieces + row scales of a factor that was just (re)written
    if (!f16) return 0;
    h->launches += 1;
    const int n = side_is_c ? v.n_c : v.n_r;
    const int slot = h->prof_begin(s, 8.0 * (double)SK * (double)n, 1);   // fp32 in, two fp16 pieces out
    const int rc = side_is_c
        ? launch_emit_f16(wFc, SK, v.n_c, v.ld_c, v.exact ? v.scale_c : nullptr, wFc_hi, wFc_lo, d_rs_c, ktiles_c, s)
        : launch_emit_f16(wFr, SK, v.n_r, v.ld_r, v.exact ? v.scale_r : nullptr, wFr_hi, wFr_lo, d_rs_r, ktiles_r, s);
    h->prof_end(s, slot);
    return rc;
  };
  // algorithmic bytes of one update launch: factor read, product slices read, factor (+ tf32 pieces) written
  // (pieces: two tf32 pieces = 2 floats per element, two fp16 pieces = 1)
  auto upd_bytes = [&](int n_items, int nsplit, int piece_floats) {
    return 4.0 * (double)SK * (double)n_items * (double)(2 + nsplit + piece_floats);
  };
  auto update = [&](bool cd, const FactorView& f, const float* NUM, const GemmPlan& pl, const double* gram_in, float l1,
                    float l2, const FusedOut& out) -> int {
    h->launches += 1;
    const int slot = h->prof_begin(s, upd_bytes(f.n, pl.splits, f.F_hi ? 2 : ((f.P_hi && out.gram_part) ? 1 : 0)), 1);
    const int rc = cd ? launch_cd_update(f, NUM, pl.splits, pl.split_stride, gram_in, bm(), l1, l2, out, s)
                      : launch_mu_update(f, NUM, pl.splits, pl.split_stride, gram_in, bm(), l1, l2, out, s);
    h->prof_end(s, slot);
    if (rc != 0 || !io.update_cols) return rc;   // a refit never multiplies by the factor it updates
    if (f.P_hi && out.gram_part) return 0;       // the Gram-fused kernel emitted the pieces of every tile it wrote
    return emit_pieces(f.F == wFc ? 1 : 0);
  };
  auto fused_out = [&](int side_is_c, bool want_gram, double* scal_part, double* scal) {
    FusedOut o{};
    if (want_gram && fuse) {
      o.gram_part = side_is_c ? d_gpartC : d_gpartR;
      o.gram = side_is_c ? d_gramC : d_gramR;
    }
    o.scal_part = scal_part;
    o.scal = scal;
    o.counter = d_ticket;
    return o;
  };
  auto finalize_scal = [&](const double* part, double* out, int chunks) -> int {
    h->launches += 1;
    return launch_finalize(nullptr, nullptr, part, out, chunks, bm(), s);
  };
  auto gemm_rows = [&]() -> int {   // NUM_r = Fc * B_rows^T
    return run_gemm(h, tf32, {wFc, wFc_hi, wFc_lo, d_rs_c, v.ld_c}, SK, v.B_rows, NUMr, v.ld_r, plan_r, v.exact,
                    v.scale_r, s);
  };
  auto gemm_cols = [&]() -> int {   // NUM_c = Fr * B_cols^T
    return run_gemm(h, tf32, {wFr, wFr_hi, wFr_lo, d_rs_r, v.ld_r}, SK, v.B_cols, NUMc, v.ld_c, plan_c, v.exact,
                    v.scale_c, s);
  };

  // gathers `cnt` restarts' rows: dst[dst_off[i] ..] <- src[src_off[i] ..].  Index triples go through a pinned
  // ring of GATHER_SLOTS entries so that consecutive gathers need no host synchronisation in between; the
  // caller synchronises the stream before the ring wraps (upload_slots / the final sync do).
  constexpr int GATHER_SLOTS = 12;
  int* h_gidx = static_cast<int*>(h->host_buf("solve.gather_idx", sizeof(int) * 3 * (size_t)R0 * GATHER_SLOTS));
  int* d_gidx = static_cast<int*>(h->dev_buf("solve.gather_didx", sizeof(int) * 3 * (size_t)R0 * GATHER_SLOTS));
  if (!h_gidx || !d_gidx) return -2;
  int gslot = 0;
  auto gather = [&](const float* src, float* dst, const std::vector<int>& so, const std::vector<int>& dof,
                    const std::vector<int>& kk, int ld) -> int {
    const int cnt = (int)kk.size();
    if (cnt == 0 || !src || !dst) return 0;
    if (gslot == GATHER_SLOTS) {
      CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
      gslot = 0;
    }
    int* hm = h_gidx + (size_t)gslot * 3 * R0;
    int* dm = d_gidx + (size_t)gslot * 3 * R0;
    ++gslot;
    std::memcpy(hm, so.data(), sizeof(int) * cnt);
    std::memcpy(hm + R0, dof.data(), sizeof(int) * cnt);
    std::memcpy(hm + 2 * R0, kk.data(), sizeof(int) * cnt);
    CNMF_CUDA_CHECK(cudaMemcpyAsync(dm, hm, sizeof(int) * 3 * R0, cudaMemcpyHostToDevice, s));
    h->launches += 1;
    return launch_gather_rows(src, dm, dst, dm + R0, dm + 2 * R0, cnt, ld, s);
  };

  const double normX2 = v.sum_sq;
  double* d_cd_err = d_state + 7 * R0;
  auto cd_final_error = [&]() -> int {
    int* d_zero = static_cast<int*>(h->dev_buf("solve.zero", sizeof(int) * 2 * R0));
    if (!d_zero) return -2;
    CNMF_CUDA_CHECK(cudaMemsetAsync(d_zero, 0, sizeof(int) * 2 * R0, s));
    BatchMeta bm0{d_off, d_k, d_rid, d_zero, R, kp};
    h->launches += 7;
    CNMF_TRY(launch_gram_partial(fr(), bm0, d_gpartR, s));
    CNMF_TRY(launch_gram_partial(fc(), bm0, d_gpartC, s));
    CNMF_TRY(launch_finalize(d_gpartR, d_gramR, nullptr, nullptr, gram_chunks(fr()), bm0, s));
    CNMF_TRY(launch_finalize(d_gpartC, d_gramC, nullptr, nullptr, gram_chunks(fc()), bm0, s));
    if (io.update_cols) {
      CNMF_TRY(launch_cross(fc(), NUMc, plan_c.splits, plan_c.split_stride, bm0, d_scalB, s));
      CNMF_TRY(launch_finalize(nullptr, nullptr, d_scalB, d_crossB, chunks_c, bm0, s));
    } else {
      CNMF_TRY(launch_cross(fr(), NUMr, plan_r.splits, plan_r.split_stride, bm0, d_scalA, s));
      CNMF_TRY(launch_finalize(nullptr, nullptr, d_scalA, d_crossB, chunks_r, bm0, s));
    }
    ConvState scratch{d_state + 5 * R0, d_state + 6 * R0, d_cd_err, d_zero, d_zero + R0};
    return launch_mu_check(scratch, d_crossB, d_gramR, d_gramC, normX2, bm0, 0, 0.0, p.max_iter, s);
  };

  std::vector<int> h_done(R0, 0);
  // Drop converged restarts from the packed arrays when that saves a 128-row GEMM tile (or >= 1/8 of the rows).
  auto maybe_compact = [&]() -> int {
    if (!io.update_cols) return 0;
    int live_rows = 0;
    for (int sl = 0; sl < R; ++sl)
      if (!h_done[s_rid[sl]]) live_rows += s_k[sl];
    if (live_rows == SK || live_rows == 0) return 0;
    const bool saves_tile = (live_rows + 127) / 128 < (SK + 127) / 128;
    if (!saves_tile && live_rows > SK - SK / 8) return 0;
    if (!mu) CNMF_TRY(cd_final_error());    // restarts leaving the packed arrays get their ||X - WH||_F now
    if (!aFr) {
      const size_t nr = (size_t)SK0 * v.ld_r, nc = (size_t)SK0 * v.ld_c;
      aFr = static_cast<float*>(h->dev_buf("solve.alt.Fr", nr * 4));
      aFc = static_cast<float*>(h->dev_buf("solve.alt.Fc", nc * 4));
      resFr = static_cast<float*>(h->dev_buf("solve.res.Fr", nr * 4));
      resFc = static_cast<float*>(h->dev_buf("solve.res.Fc", nc * 4));
      if (!aFr || !aFc || !resFr || !resFc) return -2;
      if (tf32) {
        aFr_hi = static_cast<float*>(h->dev_buf("solve.alt.Fr_hi", nr * 4));
        aFr_lo = static_cast<float*>(h->dev_buf("solve.alt.Fr_lo", nr * 4));
        aFc_hi = static_cast<float*>(h->dev_buf("solve.alt.Fc_hi", nc * 4));
        aFc_lo = static_cast<float*>(h->dev_buf("solve.alt.Fc_lo", nc * 4));
        if (!aFr_hi || !aFr_lo || !aFc_hi || !aFc_lo) return -2;
      }
    }
    std::vector<int> f_src, f_dst, f_k, l_src, l_dst, l_k, l_rid;
    int pos = 0;
    for (int sl = 0; sl < R; ++sl) {
      const int rid = s_rid[sl];
      if (h_done[rid]) {
        f_src.push_back(s_off[sl]); f_dst.push_back(off0[rid]); f_k.push_back(s_k[sl]);
      } else {
        l_src.push_back(s_off[sl]); l_dst.push_back(pos); l_k.push_back(s_k[sl]); l_rid.push_back(rid);
        pos += s_k[sl];
      }
    }
    CNMF_TRY(gather(wFr, resFr, f_src, f_dst, f_k, v.ld_r));       // finished restarts -> result slabs
    CNMF_TRY(gather(wFc, resFc, f_src, f_dst, f_k, v.ld_c));
    CNMF_TRY(gather(wFr, aFr, l_src, l_dst, l_k, v.ld_r));          // live restarts -> packed front of the alt buffers
    CNMF_TRY(gather(wFc, aFc, l_src, l_dst, l_k, v.ld_c));
    if (tf32 && !f16) {
      CNMF_TRY(gather(wFr_hi, aFr_hi, l_src, l_dst, l_k, v.ld_r));
      CNMF_TRY(gather(wFr_lo, aFr_lo, l_src, l_dst, l_k, v.ld_r));
      CNMF_TRY(gather(wFc_hi, aFc_hi, l_src, l_dst, l_k, v.ld_c));
      CNMF_TRY(gather(wFc_lo, aFc_lo, l_src, l_dst, l_k, v.ld_c));
    }
    std::swap(wFr, aFr); std::swap(wFr_hi, aFr_hi); std::swap(wFr_lo, aFr_lo);
    std::swap(wFc, aFc); std::swap(wFc_hi, aFc_hi); std::swap(wFc_lo, aFc_lo);
    R = (int)l_k.size();
    SK = pos;
    std::copy(l_dst.begin(), l_dst.end(), s_off.begin());
    std::copy(l_k.begin(), l_k.end(), s_k.begin());
    std::copy(l_rid.begin(), l_rid.end(), s_rid.begin());
    CNMF_TRY(upload_slots());      // synchronises the stream: the gather ring can be reused
    gslot = 0;
    plan_gemms();
    plan_blocks(R);
    CNMF_TRY(emit_pieces(0));      // f16: pieces and row scales follow the new packing
    CNMF_TRY(emit_pieces(1));
    compacted = true;
    return 0;
  };

  auto poll_all_done = [&]() -> int {   // 1 = all done, 0 = not yet, <0 error
    CNMF_CUDA_CHECK(cudaMemcpyAsync(h_done.data(), d_done, sizeof(int) * R0, cudaMemcpyDeviceToHost, s));
    CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
    for (int sl = 0; sl < R; ++sl)
      if (!h_done[s_rid[sl]]) return maybe_compact();
    return 1;
  };

  const float l1W = (float)p.l1_reg_W, l2W = (float)p.l2_reg_W, l1H = (float)p.l1_reg_H, l2H = (float)p.l2_reg_H;
  int it = 0;
  CNMF_TRY(emit_pieces(0));        // f16: the callers' tf32 pieces are replaced by fp16 pieces of the initial factors
  CNMF_TRY(emit_pieces(1));

  if (mu) {
    // ---------------- multiplicative update (sklearn _nmf.py:726-888) ----------------
    CNMF_TRY(gram_full(fc(), 1));
    CNMF_TRY(gram_full(fr(), 0));
    if (io.update_cols) {
      CNMF_TRY(gemm_cols());
      h->launches += 1;
      CNMF_TRY(launch_cross(fc(), NUMc, plan_c.splits, plan_c.split_stride, bm(), d_scalB, s));
      CNMF_TRY(finalize_scal(d_scalB, d_crossB, chunks_c));
    } else {
      CNMF_TRY(gemm_rows());          // H fixed: X H^T is computed once (sklearn caches XHt, _nmf.py:537-548)
      h->launches += 1;
      CNMF_TRY(launch_cross(fr(), NUMr, plan_r.splits, plan_r.split_stride, bm(), d_scalA, s));
      CNMF_TRY(finalize_scal(d_scalA, d_crossB, chunks_r));
    }
    h->launches += 1;
    CNMF_TRY(launch_mu_check(st, d_crossB, d_gramR, d_gramC, normX2, bm(), 0, p.tol, p.max_iter, s));

    // one iteration = GEMM, update(+Gram), GEMM, update(+Gram): the update kernels leave the finalised Gram of the
    // factor they wrote (and, at check iterations, <NUM, F>) behind, so nothing else sits between the GEMMs
    for (it = 1; it <= p.max_iter; ++it) {
      const bool check = (p.tol > 0 && it % 10 == 0) || it == p.max_iter;
      if (io.update_cols) {
        CNMF_TRY(gemm_rows());
        CNMF_TRY(update(false, fr(), NUMr, plan_r, d_gramC, l1W, l2W, fused_out(0, true, nullptr, nullptr)));
        CNMF_TRY(gram_after(fr(), 0));
        CNMF_TRY(gemm_cols());
        CNMF_TRY(update(false, fc(), NUMc, plan_c, d_gramR, l1H, l2H, fused_out(1, true, check ? d_scalB : nullptr, d_crossB)));
        CNMF_TRY(gram_after(fc(), 1));
      } else {
        CNMF_TRY(update(false, fr(), NUMr, plan_r, d_gramC, l1W, l2W, fused_out(0, check, check ? d_scalA : nullptr, d_crossB)));
        if (check) CNMF_TRY(gram_after(fr(), 0));
      }
      if (check) {
        h->launches += 1;
        // at it == max_iter with it % 10 != 0 sklearn does not test; tol = -1 makes the test never fire
        const double tol_eff = (p.tol > 0 && it % 10 == 0) ? p.tol : -1.0;
        CNMF_TRY(launch_mu_check(st, d_crossB, d_gramR, d_gramC, normX2, bm(), it, tol_eff, p.max_iter, s));
        const int all = poll_all_done();
        if (all < 0) return all;
        if (all) break;
      }
    }
  } else {
    // ---------------- coordinate descent (sklearn _nmf.py:399-518, shuffle=False) ----------------
    const int poll_every = 4;
    for (it = 1; it <= p.max_iter; ++it) {
      if (it == 1) CNMF_TRY(gram_full(fc(), 1));     // afterwards: left behind by the sweep over Fc
      if (io.update_cols || it == 1) CNMF_TRY(gemm_rows());
      CNMF_TRY(update(true, fr(), NUMr, plan_r, d_gramC, l1W, l2W, fused_out(0, io.update_cols, d_scalA, d_crossA)));
      if (io.update_cols) {
        CNMF_TRY(gram_after(fr(), 0));
        CNMF_TRY(gemm_cols());
        CNMF_TRY(update(true, fc(), NUMc, plan_c, d_gramR, l1H, l2H, fused_out(1, true, d_scalB, d_crossB)));
        CNMF_TRY(gram_after(fc(), 1));
      }
      h->launches += 1;
      CNMF_TRY(launch_cd_check(st, d_crossA, io.update_cols ? d_crossB : nullptr, bm(), it, p.tol, p.max_iter, s));
      if (it % poll_every == 0 || it == p.max_iter) {
        const int all = poll_all_done();
        if (all < 0) return all;
        if (all) break;
      }
    }
  }

  // final ||X - Fr^T Fc||_F: MU holds it in st.last from each restart's last check; CD tracks the
  // projected-gradient violation instead, so the trace form is evaluated here for the restarts still
  // packed (those compacted away earlier were evaluated just before they left)
  double* d_err = st.last;
  if (!mu) {
    CNMF_TRY(cd_final_error());
    d_err = d_cd_err;
  }

  // ---- put every restart's final factors back at its original rows of the caller's buffers
  if (compacted) {
    std::vector<int> so(s_off.begin(), s_off.begin() + R), ko(s_k.begin(), s_k.begin() + R), dof(R);
    for (int sl = 0; sl < R; ++sl) dof[sl] = off0[s_rid[sl]];
    CNMF_TRY(gather(wFr, resFr, so, dof, ko, v.ld_r));
    CNMF_TRY(gather(wFc, resFc, so, dof, ko, v.ld_c));
    CNMF_CUDA_CHECK(cudaMemcpyAsync(io.Fr, resFr, (size_t)SK0 * v.ld_r * 4, cudaMemcpyDeviceToDevice, s));
    CNMF_CUDA_CHECK(cudaMemcpyAsync(io.Fc, resFc, (size_t)SK0 * v.ld_c * 4, cudaMemcpyDeviceToDevice, s));
  }

  io.n_iter.assign(R0, 0);
  io.last.assign(R0, 0.0);
  io.err.assign(R0, 0.0);
  CNMF_CUDA_CHECK(cudaMemcpyAsync(io.n_iter.data(), d_niter, sizeof(int) * R0, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaMemcpyAsync(io.last.data(), st.last, sizeof(double) * R0, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaMemcpyAsync(io.err.data(), d_err, sizeof(double) * R0, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  // per-launch event pairs are folded into the totals lazily (cnmf_profile_get*), not inside the solve
  return 0;
}

}  // namespace cnmf
