// Host-side engine objects behind the C ABI (handle, dataset, workspace).
#pragma once
#include <cuda_runtime.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/cnmf_b200.h"
#include "common.cuh"
#include "gemm.h"

struct cnmf_handle_s {
  int device = 0;
  int sm_count = 148;
  long long launches = 0;                       // kernels launched by this library (bench: gpu_launches)
  // optional per-launch timing of the hot kernels (batched GEMM, fused update) with CUDA events on the
  // launching stream; read back by bench.py for the roofline lines
  bool profile = false;
  std::vector<cudaEvent_t> ev_pool;
  struct Pending { int begin; int end; int cls; double work; };   // indices of the start / end events in ev_pool
  // a profiled launch that directly follows another profiled launch (no other counted launch in between, same
  // stream) takes the predecessor's end event as its start: one event record per kernel boundary instead of two
  int prof_last_end = -1;
  long long prof_last_launches = -1;
  cudaStream_t prof_last_stream = nullptr;
  std::vector<Pending> ev_pending;
  size_t ev_used = 0;
  // kernel classes: 0 = batched GEMM (work = algorithmic FLOPs), 1 = fused update kernels (work = algorithmic bytes)
  static constexpr int PROF_CLASSES = 2;
  double prof_ms[PROF_CLASSES] = {0.0, 0.0}, prof_work[PROF_CLASSES] = {0.0, 0.0};
  long long prof_launches[PROF_CLASSES] = {0, 0};
  double t_rng_ms = 0, t_h2d_ms = 0, t_solve_ms = 0, t_d2h_ms = 0;   // host wall-clock phases of the last factorize
  int prof_begin(cudaStream_t s, double work, int cls = 0);    // start event (recorded or shared); returns slot or -1
  void prof_end(cudaStream_t s, int slot);
  void prof_collect();                              // after a stream sync: fold pending pairs into the totals
  std::map<std::string, std::pair<void*, size_t>> ws;   // named grow-only device buffers
  std::map<std::string, std::pair<void*, size_t>> pinned;  // named grow-only pinned host buffers

  // size-keyed pool of dataset buffers: cudaMalloc / cudaFree of several 160 MB arrays per dataset
  // cost tens of ms (cudaFree synchronises); datasets of a repeated shape reuse their buffers
  std::multimap<size_t, void*> pool;
  size_t pool_bytes = 0;
  void* pool_take(size_t bytes);
  void pool_give(void* p, size_t bytes);
  void* dev_buf(const std::string& name, size_t bytes);      // nullptr on failure (error set)
  void* host_buf(const std::string& name, size_t bytes);
  void release_all();
};

// A cells x genes matrix resident on the device in the forms the two GEMM orientations need.
//   X   (n_rows x ld_c)  : K-major over columns  -> B operand of  NUM_rows = F_cols * X^T
//   Xt  (n_cols x ld_r)  : K-major over rows     -> B operand of  NUM_cols = F_rows * X
// fp32 mode keeps X and Xt; tf32x3 mode keeps X (full, for column ops) + the hi/lo pieces of both.
struct cnmf_dataset_s {
  cnmf_handle_s* h = nullptr;
  int n_rows = 0, n_cols = 0;
  int ld_c = 0;   // row stride of X  (>= n_cols)
  int ld_r = 0;   // row stride of Xt (>= n_rows)
  int precision = 0;
  float *X = nullptr, *Xt = nullptr;
  float *X_hi = nullptr, *X_lo = nullptr, *Xt_hi = nullptr, *Xt_lo = nullptr;
  // "exact" datasets (tf32x3 only): X = diag(row_scale) * C * diag(col_scale) with C small non-negative integers
  // (what HVG-normalised counts and TPM are).  Then X_hi / Xt_hi hold C / C^T -- exactly representable in tf32,
  // no lo piece -- the scales are folded into the factor pieces / applied to the GEMM output, and every big
  // product needs 2 tensor-core passes instead of 3.  Either scale may be nullptr (= 1).
  bool exact = false;
  bool allow_exact = true;
  // f16x2 precision: requested at creation (want_f16); active (f16) once the dataset turned out exact.  X_h16 / Xt_h16
  // hold the integer matrices C / C^T as fp16 (same shapes and element strides as X_hi / Xt_hi)
  bool want_f16 = false, f16 = false;
  bool drop_tf32 = false;       // f16 datasets: X_hi / Xt_hi are released once the fp16 matrices exist
  void *X_h16 = nullptr, *Xt_h16 = nullptr;
  float *row_scale = nullptr, *col_scale = nullptr;    // lengths ld_r / ld_c, zero padded
  double sum = 0.0, sum_sq = 0.0;
  std::vector<std::pair<void*, size_t>> owned;
};

namespace cnmf {

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// View of a dataset for one solve: "rows" are the items of the row factor (Fr: SK x n_r),
// "cols" the items of the column factor (Fc: SK x n_c).  transposed swaps the roles.
struct DataView {
  Operand B_rows;   // n_r x n_c : B operand when updating Fr (reduction over n_c)
  Operand B_cols;   // n_c x n_r : B operand when updating Fc (reduction over n_r)
  int n_r, n_c, ld_r, ld_c;
  double sum, sum_sq;
  bool exact;               // both operands hold exact integers; scales below complete X
  bool f16;                 // fp16 operand path active (exact datasets created with CNMF_PRECISION_F16X2)
  const float* scale_r;     // per row-item scale (length ld_r) or nullptr
  const float* scale_c;     // per column-item scale (length ld_c) or nullptr
};

DataView make_view(const cnmf_dataset_s* d, bool transposed);

struct SolveIO {
  int R = 0;
  std::vector<int> ks;      // per restart
  // packed device factors (SK x ld): row factor Fr (e.g. W^T), column factor Fc (e.g. H)
  float *Fr = nullptr, *Fr_hi = nullptr, *Fr_lo = nullptr;
  float *Fc = nullptr, *Fc_hi = nullptr, *Fc_lo = nullptr;
  bool update_cols = true;  // false: Fc fixed (refit)
  std::vector<int> n_iter;  // out
  std::vector<double> last; // out: last convergence statistic (mu: error, cd: violation)
  std::vector<double> err;  // out: final ||X - Fr^T Fc||_F
};

// Device buffers for SK packed rows of both factors, plus their tf32 pieces when `tf32`, into io.  The buffers are the
// handle's workspace entries prefix + "Fr", "Fr_hi", ...: each caller keeps its own by its prefix.
int alloc_factors(cnmf_handle_s* h, const char* prefix, int SK, int ld_r, int ld_c, bool tf32, SolveIO* io);
// tf32 pieces of both factors with the view's scales folded in (exact datasets).  Nothing to do unless `tf32`, nor for
// f16 datasets: the solver emits fp16 pieces itself, tf32 pieces would be dead work.
int split_factors(cnmf_handle_s* h, const DataView& v, const SolveIO& io, int SK, bool tf32, cudaStream_t s);

// Runs the batched solver in place on io.Fr / io.Fc.
int solve_batched(cnmf_handle_s* h, const DataView& v, SolveIO& io, const cnmf_nmf_params& p, cudaStream_t s);
// beta_loss = kullback-leibler / itakura-saito (nmf_beta.cu); reached through solve_batched
int solve_batched_beta(cnmf_handle_s* h, const DataView& v, SolveIO& io, const cnmf_nmf_params& p, cudaStream_t s);
int matrix_min(cnmf_handle_s* h, const float* X, int rows, int cols, int ld, float* out_host, cudaStream_t s);
// the streaming beta-divergence kernels read X in both orientations in full fp32: builds d->Xt if the dataset
// (tf32x3 mode) only holds the pieces
int dataset_ensure_full_transpose(cnmf_dataset_s* d, cudaStream_t s);

// A new dataset of n_rows x n_cols on h with X allocated (contents undefined).  Its precision settings are copied from
// `like`, or derived from the CNMF_PRECISION_* code `precision` when `like` is nullptr.
int dataset_new(cnmf_handle_s* h, const cnmf_dataset_s* like, int precision, int n_rows, int n_cols,
                cnmf_dataset_s** out);
// device memory owned by d (from the handle's pool), at least 64 floats
int dataset_alloc(cnmf_dataset_s* d, float** p, size_t elems);
// builds Xt / tf32 pieces / sums from d->X (already resident, padding zeroed)
int dataset_finish(cnmf_dataset_s* d, cudaStream_t s);
// the last step of every dataset constructor: dataset_finish when rc == 0, *out = d on success, d destroyed on failure
int finish_or_destroy(cnmf_dataset_s* d, int rc, cudaStream_t s, cnmf_dataset_t* out);

}  // namespace cnmf
