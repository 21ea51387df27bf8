// extern "C": NNLS refits (cNMF.refit_usage / refit_spectra, cnmf.py:776-820), prediction error
// (cnmf.py:926-930), left projections for the OLS step (cnmf.py:98-119), column statistics,
// column-subset datasets (cnmf.py:965-969) and a raw GEMM hook used by tests / micro-benchmarks.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <vector>

#include "engine.h"
#include "gemm.h"
#include "nmf_kernels.cuh"

using namespace cnmf;

namespace {

__global__ void fill_kernel(float* p, float v, int rows, int n, int ld) {
  const long long total = (long long)rows * n;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    p[(i / n) * ld + (i % n)] = v;
}

// column sums of v and v^2 with v = X[r, c] * (row_scale ? row_scale[r] : 1), fp64.  Threads own columns (coalesced),
// blockIdx.y owns a fixed strip of rows: partial[y][c], reduced in strip order by col_stats_reduce_kernel
// (deterministic: the HVG ranking of prepare() is a sort of these numbers).
__global__ void col_stats_kernel(const float* __restrict__ X, int rows, int cols, int ld,
                                 const double* __restrict__ row_scale, double* __restrict__ part) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const int per = (rows + gridDim.y - 1) / gridDim.y;
  const int r0 = blockIdx.y * per, r1 = min(rows, r0 + per);
  double s = 0.0, q = 0.0;
  for (int r = r0; r < r1; ++r) {
    double v = X[(long long)r * ld + c];
    if (row_scale) v *= row_scale[r];
    s += v;
    q += v * v;
  }
  part[((long long)blockIdx.y * 2) * cols + c] = s;
  part[((long long)blockIdx.y * 2 + 1) * cols + c] = q;
}

__global__ void col_stats_reduce_kernel(const double* __restrict__ part, int strips, int cols, double* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  double s = 0.0, q = 0.0;
  for (int y = 0; y < strips; ++y) {
    s += part[((long long)y * 2) * cols + c];
    q += part[((long long)y * 2 + 1) * cols + c];
  }
  out[c] = s;
  out[cols + c] = q;
}

// one warp per row: fp64 sum of the row (cell totals: the TPM denominators of cnmf.py:245-251)
__global__ void row_sums_kernel(const float* __restrict__ X, int rows, int cols, int ld, double* __restrict__ out) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* row = X + (long long)r * ld;
  double s = 0.0;
  for (int c = lane; c < cols; c += 32) s += (double)row[c];
  s = warp_sum(s);
  if (lane == 0) out[r] = s;
}

__global__ void scale_rows_kernel(const float* __restrict__ src, int rows, int cols, int ld, const float* __restrict__ rs,
                                  float* __restrict__ dst) {
  const long long total = (long long)rows * (ld / 4);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / (ld / 4));
    float4 v = reinterpret_cast<const float4*>(src)[i];
    const float f = rs[r];
    v.x *= f; v.y *= f; v.z *= f; v.w *= f;
    reinterpret_cast<float4*>(dst)[i] = v;
  }
}

__global__ void combine_scale_kernel(const float* __restrict__ scale, const float* __restrict__ src_cs,
                                     const int* __restrict__ cols, int n, int n_pad, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_pad) return;
  out[c] = (c < n) ? scale[c] * (src_cs ? src_cs[cols[c]] : 1.f) : 0.f;
}

__global__ void gather_cols_kernel(const float* __restrict__ src, int rows, int ld_src, const int* __restrict__ cols,
                                   const float* __restrict__ scale, int n_cols, float* __restrict__ dst, int ld_dst) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cols) return;
  const int sc = cols[c];
  const float f = scale[c];
  for (int r = blockIdx.y; r < rows; r += gridDim.y) dst[(long long)r * ld_dst + c] = src[(long long)r * ld_src + sc] * f;
}

// out (M x N, row stride N) = the sum in fp64 of the `slices` split-K slices of the device GEMM output C (M x ldc each,
// contiguous); synchronises the stream
int download_split_sum(const float* C, int slices, int M, int N, int ldc, float* out, cudaStream_t s) {
  std::vector<float> tmp((size_t)slices * M * ldc);
  CNMF_CUDA_CHECK(cudaMemcpyAsync(tmp.data(), C, tmp.size() * 4, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  for (int m = 0; m < M; ++m)
    for (int n = 0; n < N; ++n) {
      double a = 0.0;
      for (int z = 0; z < slices; ++z) a += tmp[(size_t)z * M * ldc + (size_t)m * ldc + n];
      out[(size_t)m * N + n] = (float)a;
    }
  return 0;
}

}  // namespace

extern "C" {

static int col_stats_impl(cnmf_dataset_t d, const double* row_scale_host, double* mean_host, double* var_host, void* stream) {
  CNMF_REQUIRE(d && mean_host && var_host, "col_stats: NULL argument");
  cnmf_handle_s* h = d->h;
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  const int strips = std::max(1, std::min(64, d->n_rows / 64));
  double* part = static_cast<double*>(h->dev_buf("colstats.part", sizeof(double) * 2 * (size_t)strips * d->n_cols));
  double* buf = static_cast<double*>(h->dev_buf("colstats", sizeof(double) * 2 * d->n_cols));
  double* d_rs = nullptr;
  if (row_scale_host) {
    d_rs = static_cast<double*>(h->dev_buf("colstats.rs", sizeof(double) * d->n_rows));
    if (!d_rs) return -2;
    CNMF_CUDA_CHECK(cudaMemcpyAsync(d_rs, row_scale_host, sizeof(double) * d->n_rows, cudaMemcpyHostToDevice, s));
  }
  if (!part || !buf) return -2;
  dim3 grid((d->n_cols + 127) / 128, strips);
  col_stats_kernel<<<grid, 128, 0, s>>>(d->X, d->n_rows, d->n_cols, d->ld_c, d_rs, part);
  col_stats_reduce_kernel<<<(d->n_cols + 127) / 128, 128, 0, s>>>(part, strips, d->n_cols, buf);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 2;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(mean_host, buf, sizeof(double) * d->n_cols, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaMemcpyAsync(var_host, buf + d->n_cols, sizeof(double) * d->n_cols, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  const double n = d->n_rows;
  for (int c = 0; c < d->n_cols; ++c) {
    const double m = mean_host[c] / n;
    mean_host[c] = m;
    var_host[c] = std::max(var_host[c] / n - m * m, 0.0);
  }
  return 0;
}

int cnmf_dataset_col_stats(cnmf_dataset_t d, double* mean_host, double* var_host, void* stream) {
  return col_stats_impl(d, nullptr, mean_host, var_host, stream);
}

int cnmf_dataset_scaled_col_stats(cnmf_dataset_t d, const double* row_scale_host, double* mean_host, double* var_host,
                                  void* stream) {
  CNMF_REQUIRE(row_scale_host, "scaled_col_stats: NULL row scale");
  return col_stats_impl(d, row_scale_host, mean_host, var_host, stream);
}

int cnmf_dataset_row_sums(cnmf_dataset_t d, double* row_sums_host, void* stream) {
  CNMF_REQUIRE(d && row_sums_host, "row_sums: NULL argument");
  cnmf_handle_s* h = d->h;
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  double* buf = static_cast<double*>(h->dev_buf("rowsums", sizeof(double) * d->n_rows));
  if (!buf) return -2;
  row_sums_kernel<<<(d->n_rows + 7) / 8, 256, 0, s>>>(d->X, d->n_rows, d->n_cols, d->ld_c, buf);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 1;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(row_sums_host, buf, sizeof(double) * d->n_rows, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  return 0;
}

int cnmf_dataset_from_columns(cnmf_dataset_t src, const int32_t* cols_host, const float* col_scale_host, int n_cols,
                              void* stream, cnmf_dataset_t* out) {
  CNMF_REQUIRE(src && cols_host && col_scale_host && out && n_cols > 0, "dataset_from_columns: bad arguments");
  for (int c = 0; c < n_cols; ++c)
    CNMF_REQUIRE(cols_host[c] >= 0 && cols_host[c] < src->n_cols, "dataset_from_columns: column index out of range");
  cnmf_handle_s* h = src->h;
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  int* d_cols = static_cast<int*>(h->dev_buf("fromcols.idx", sizeof(int) * n_cols));
  float* d_scale = static_cast<float*>(h->dev_buf("fromcols.scale", sizeof(float) * n_cols));
  if (!d_cols || !d_scale) return -2;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(d_cols, cols_host, sizeof(int) * n_cols, cudaMemcpyHostToDevice, s));
  CNMF_CUDA_CHECK(cudaMemcpyAsync(d_scale, col_scale_host, sizeof(float) * n_cols, cudaMemcpyHostToDevice, s));
  cnmf_dataset_s* d = nullptr;
  CNMF_TRY(dataset_new(h, src, 0, src->n_rows, n_cols, &d));
  int rc = cudaMemsetAsync(d->X, 0, (size_t)d->n_rows * d->ld_c * sizeof(float), s) == cudaSuccess ? 0 : -2;
  if (rc == 0) {
    dim3 grid((n_cols + 127) / 128, std::min(d->n_rows, 16384));
    gather_cols_kernel<<<grid, 128, 0, s>>>(src->X, d->n_rows, src->ld_c, d_cols, d_scale, n_cols, d->X, d->ld_c);
    h->launches += 1;
    if (cudaGetLastError() != cudaSuccess) rc = -2;
  }
  if (rc == 0 && src->exact) {
    // an exact-count source stays exact: same integer matrix (the selected columns), same row scale, and the
    // column scale becomes scale[c] * src.col_scale[cols[c]]; finish() rebuilds C from the scaled values
    d->exact = true;
    rc = dataset_alloc(d, &d->col_scale, (size_t)d->ld_c);
    if (rc == 0) {
      combine_scale_kernel<<<(d->ld_c + 255) / 256, 256, 0, s>>>(d_scale, src->col_scale, d_cols, n_cols, d->ld_c, d->col_scale);
      h->launches += 1;
      if (cudaGetLastError() != cudaSuccess) rc = -2;
    }
    if (rc == 0 && src->row_scale) {
      rc = dataset_alloc(d, &d->row_scale, (size_t)d->ld_r);
      if (rc == 0 && cudaMemcpyAsync(d->row_scale, src->row_scale, sizeof(float) * d->ld_r, cudaMemcpyDeviceToDevice, s) != cudaSuccess)
        rc = -2;
    }
  }
  return finish_or_destroy(d, rc, s, out);
}

int cnmf_dataset_scale_rows(cnmf_dataset_t src, const float* row_scale_host, void* stream, cnmf_dataset_t* out) {
  CNMF_REQUIRE(src && row_scale_host && out, "dataset_scale_rows: bad arguments");
  cnmf_handle_s* h = src->h;
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  float* d_rs = static_cast<float*>(h->dev_buf("scalerows.rs", sizeof(float) * src->n_rows));
  if (!d_rs) return -2;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(d_rs, row_scale_host, sizeof(float) * src->n_rows, cudaMemcpyHostToDevice, s));
  cnmf_dataset_s* d = nullptr;
  CNMF_TRY(dataset_new(h, src, 0, src->n_rows, src->n_cols, &d));
  scale_rows_kernel<<<148 * 8, 256, 0, s>>>(src->X, d->n_rows, d->n_cols, d->ld_c, d_rs, d->X);
  h->launches += 1;
  // exact-count detection runs from scratch in finish(): counts x (1e6 / cell total) is again scaled integers
  return finish_or_destroy(d, cudaGetLastError() == cudaSuccess ? 0 : -2, s, out);
}

// --------------------------------------------------------------------------------- refit
int cnmf_refit(cnmf_dataset_t d, int transposed, int k, const float* fixed_host, const cnmf_nmf_params* p,
               float* out_host, int32_t* n_iter_host, double* err_host, void* stream) {
  CNMF_REQUIRE(d && fixed_host && p && out_host, "refit: NULL argument");
  CNMF_REQUIRE(p->precision == d->precision, "params.precision must match the precision the dataset was created with");
  CNMF_REQUIRE(k >= 1 && k <= KMAX, "refit: n_components must be in [1, 32] on the CUDA path");
  const auto t_enter = std::chrono::steady_clock::now();
  cnmf_handle_s* h = d->h;
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  const bool tf32 = p->precision == CNMF_PRECISION_TF32X3;
  if (p->beta_loss != CNMF_LOSS_FROBENIUS) CNMF_TRY(dataset_ensure_full_transpose(d, s));
  DataView v = make_view(d, transposed != 0);

  SolveIO io;
  CNMF_TRY(alloc_factors(h, "refit.", k, v.ld_r, v.ld_c, tf32, &io));
  float* Fr = io.Fr;
  CNMF_CUDA_CHECK(cudaMemsetAsync(Fr, 0, (size_t)k * v.ld_r * 4, s));
  CNMF_CUDA_CHECK(cudaMemsetAsync(io.Fc, 0, (size_t)k * v.ld_c * 4, s));
  CNMF_CUDA_CHECK(cudaMemcpy2DAsync(io.Fc, (size_t)v.ld_c * 4, fixed_host, (size_t)v.n_c * 4, (size_t)v.n_c * 4, k,
                                    cudaMemcpyHostToDevice, s));
  if (p->solver == CNMF_SOLVER_MU) {
    // sklearn _nmf.py:1223-1226: W = full(sqrt(X.mean() / k))
    const double mean = v.sum / ((double)v.n_r * (double)v.n_c);
    fill_kernel<<<148 * 4, 256, 0, s>>>(Fr, (float)std::sqrt(mean / k), k, v.n_r, v.ld_r);
    CNMF_CUDA_CHECK(cudaGetLastError());
    h->launches += 1;
  }  // 'cd': zeros (sklearn _nmf.py:1227-1228)
  CNMF_TRY(split_factors(h, v, io, k, tf32, s));
  io.R = 1;
  io.ks = {k};
  io.update_cols = false;
  auto t_solve = std::chrono::steady_clock::now();
  if (h->profile) {
    CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
    h->t_h2d_ms = std::chrono::duration<double, std::milli>(t_solve - t_enter).count();
    t_solve = std::chrono::steady_clock::now();
  }
  CNMF_TRY(solve_batched(h, v, io, *p, s));
  if (h->profile) h->t_solve_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_solve).count();

  // Fr is k x n_r; the caller wants n_r x k (row-major).  Transposed on the device into a COMPACT n_r x k array and
  // copied back in one contiguous transfer through pinned memory: a pitched 2-D copy of 50 000 rows of ~40 bytes to
  // pageable memory took 10 ms on a good day and 80 ms on a bad one -- ten times the solve itself.
  float* T = static_cast<float*>(h->dev_buf("refit.T", (size_t)v.n_r * k * 4));
  float* T_host = static_cast<float*>(h->host_buf("refit.T_host", (size_t)v.n_r * k * 4));
  if (!T || !T_host) return -2;
  CNMF_TRY(launch_transpose(Fr, k, v.n_r, v.ld_r, T, nullptr, nullptr, k, s));
  h->launches += 1;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(T_host, T, (size_t)v.n_r * k * 4, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  std::memcpy(out_host, T_host, (size_t)v.n_r * k * 4);
  if (n_iter_host) *n_iter_host = io.n_iter[0];
  if (err_host) *err_host = io.err[0];
  return 0;
}

// --------------------------------------------------------------------------------- projections
// out (k x n_cols) = Ut (k x n_rows) * X  -- the X^T Y accumulator of efficient_ols_all_cols (cnmf.py:119)
int cnmf_project_rows(cnmf_dataset_t d, int k, const float* Ut_host, float* out_host, void* stream) {
  CNMF_REQUIRE(d && Ut_host && out_host && k >= 1, "project_rows: bad arguments");
  cnmf_handle_s* h = d->h;
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  const bool tf32 = d->precision == CNMF_PRECISION_TF32X3;
  const size_t nr = (size_t)k * d->ld_r;
  float* A = static_cast<float*>(h->dev_buf("proj.A", nr * 4));
  float *A_hi = nullptr, *A_lo = nullptr;
  if (!A) return -2;
  CNMF_CUDA_CHECK(cudaMemsetAsync(A, 0, nr * 4, s));
  CNMF_CUDA_CHECK(cudaMemcpy2DAsync(A, (size_t)d->ld_r * 4, Ut_host, (size_t)d->n_rows * 4, (size_t)d->n_rows * 4, k,
                                    cudaMemcpyHostToDevice, s));
  float* A_rs = nullptr;
  const int a_tiles = (d->ld_r + 511) / 512;
  if (tf32) {
    A_hi = static_cast<float*>(h->dev_buf("proj.A_hi", nr * 4));
    A_lo = static_cast<float*>(h->dev_buf("proj.A_lo", nr * 4));
    if (!A_hi || !A_lo) return -2;
    if (d->f16) {            // f16 datasets keep C^T as fp16 only: two fp16 pieces of the (signed) rows, group scales
      A_rs = static_cast<float*>(h->dev_buf("proj.A_rs", sizeof(float) * (size_t)k * a_tiles));
      if (!A_rs) return -2;
      CNMF_TRY(launch_emit_f16(A, k, d->n_rows, d->ld_r, d->exact ? d->row_scale : nullptr, A_hi, A_lo, A_rs, a_tiles, s));
    } else {
      CNMF_TRY(launch_split_scaled(A, A_hi, A_lo, k, d->ld_r, d->exact ? d->row_scale : nullptr, s));
    }
    h->launches += 1;
  }
  int splits = 1;
  {
    const int tiles = ((k + 127) / 128) * ((d->n_cols + 255) / 256);
    if (tiles < 2 * h->sm_count) splits = (2 * h->sm_count + tiles - 1) / tiles;
    splits = std::min(splits, std::max(1, ((d->n_rows + 31) / 32) / 8));
    splits = std::min(splits, 32);
    splits = gemm_effective_splits(d->n_rows, splits, d->f16 ? 1 : 0);
  }
  float* C = static_cast<float*>(h->dev_buf("proj.C", (size_t)splits * k * d->ld_c * 4));
  if (!C) return -2;
  CNMF_TRY(gemm_run(tf32, d->exact, d->col_scale, k, {A, A_hi, A_lo, A_rs, d->ld_r}, make_view(d, false).B_cols, C,
                    d->ld_c, {splits, 0, (long long)k * d->ld_c}, s));
  h->launches += 1;
  return download_split_sum(C, splits, k, d->n_cols, d->ld_c, out_host, s);
}

// --------------------------------------------------------------------------------- raw GEMM hook
// C (M x N) = A (M x Kd) * B (N x Kd)^T on host buffers; reps > 1 re-runs the kernel and reports the
// mean device time per launch in *ms_out (CUDA events).  Used by tests and by the roofline micro-bench.
int cnmf_gemm_abt_host(cnmf_handle_t h, int precision, const float* A, const float* B, int M, int N, int Kd, int splits,
                       float* C, int reps, float* ms_out, void* stream) {
  CNMF_REQUIRE(h && A && B && C && M > 0 && N > 0 && Kd > 0, "gemm_abt_host: bad arguments");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  const int lda = pad_ld(Kd), ldc = pad_ld(N);
  const size_t na = (size_t)M * lda, nb = (size_t)N * lda;
  float* dA = static_cast<float*>(h->dev_buf("gemmtest.A", na * 4));
  float* dB = static_cast<float*>(h->dev_buf("gemmtest.B", nb * 4));
  float* dAh = static_cast<float*>(h->dev_buf("gemmtest.Ah", na * 4));
  float* dAl = static_cast<float*>(h->dev_buf("gemmtest.Al", na * 4));
  float* dBh = static_cast<float*>(h->dev_buf("gemmtest.Bh", nb * 4));
  float* dBl = static_cast<float*>(h->dev_buf("gemmtest.Bl", nb * 4));
  const int se = gemm_effective_splits(Kd, splits, precision == CNMF_PRECISION_F16X2 ? 1 : 0);
  float* dC = static_cast<float*>(h->dev_buf("gemmtest.C", (size_t)se * M * ldc * 4));
  if (!dA || !dB || !dAh || !dAl || !dBh || !dBl || !dC) return -2;
  CNMF_CUDA_CHECK(cudaMemsetAsync(dA, 0, na * 4, s));
  CNMF_CUDA_CHECK(cudaMemsetAsync(dB, 0, nb * 4, s));
  CNMF_CUDA_CHECK(cudaMemcpy2DAsync(dA, (size_t)lda * 4, A, (size_t)Kd * 4, (size_t)Kd * 4, M, cudaMemcpyHostToDevice, s));
  CNMF_CUDA_CHECK(cudaMemcpy2DAsync(dB, (size_t)lda * 4, B, (size_t)Kd * 4, (size_t)Kd * 4, N, cudaMemcpyHostToDevice, s));
  CNMF_TRY(launch_split_tf32(dA, dAh, dAl, (long long)na, s));
  CNMF_TRY(launch_split_tf32(dB, dBh, dBl, (long long)nb, s));
  CNMF_CUDA_CHECK(cudaMemsetAsync(dC, 0xff, (size_t)se * M * ldc * 4, s));   // NaN pattern: unwritten outputs show up
  const bool f16 = precision == CNMF_PRECISION_F16X2;    // B must hold integers <= 2048 (exact in fp16)
  const int tiles = (lda + 511) / 512;
  float* dRs = nullptr;
  if (f16) {
    dRs = static_cast<float*>(h->dev_buf("gemmtest.rs", sizeof(float) * (size_t)M * tiles));
    if (!dRs) return -2;
    CNMF_TRY(launch_emit_f16(dA, M, Kd, lda, nullptr, dAh, dAl, dRs, tiles, s));
    CNMF_TRY(launch_to_half(dB, dBh, (long long)nb, s));
  }
  const bool tc = f16 || precision == CNMF_PRECISION_TF32X3;
  const GemmA a{dA, dAh, dAl, dRs, lda};
  const Operand b{dB, dBh, f16 ? nullptr : dBl, f16 ? dBh : nullptr, N, Kd, lda};
  auto gemm = [&] { return gemm_run(tc, f16, nullptr, M, a, b, dC, ldc, {se, 0, (long long)M * ldc}, s); };
  cudaEvent_t e0, e1;
  CNMF_CUDA_CHECK(cudaEventCreate(&e0));
  CNMF_CUDA_CHECK(cudaEventCreate(&e1));
  if (reps < 1) reps = 1;
  int rc = gemm();   // warm-up + result
  if (rc == 0 && reps > 1) {
    cudaEventRecord(e0, s);
    for (int i = 0; i < reps && rc == 0; ++i) rc = gemm();
    cudaEventRecord(e1, s);
  }
  h->launches += reps;
  if (rc != 0) return rc;
  CNMF_TRY(download_split_sum(dC, se, M, N, ldc, C, s));
  if (ms_out) {
    float ms = 0.f;
    if (reps > 1) cudaEventElapsedTime(&ms, e0, e1);
    *ms_out = reps > 1 ? ms / reps : 0.f;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return 0;
}

}  // extern "C"
