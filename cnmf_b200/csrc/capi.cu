// extern "C" entry points declared in include/cnmf_b200.h (handle, dataset, factorize, refit).
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstring>
#include <functional>
#include <string>
#include <thread>
#include <vector>

#include "engine.h"
#include "gemm.h"
#include "legacy_rng.h"
#include "nmf_kernels.cuh"

namespace cnmf {

int launch_rng_init(const uint32_t* seeds_host, const int* ks_host, const int* offs_host, const double* avgs_host, int R,
                    int n_samples, int n_features, float* Wt, long long ldW, float* H, long long ldH, cnmf_handle_s* h,
                    cudaStream_t s);

static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }

}  // namespace cnmf

using namespace cnmf;

// ----------------------------------------------------------------------------- handle
void* cnmf_handle_s::dev_buf(const std::string& name, size_t bytes) {
  auto& e = ws[name];
  if (e.second >= bytes && e.first) return e.first;
  if (e.first) cudaFree(e.first);
  e.first = nullptr;
  e.second = 0;
  const size_t want = std::max<size_t>(bytes, 256);
  cudaError_t err = cudaMalloc(&e.first, want);
  if (err != cudaSuccess) {
    set_last_error("cudaMalloc(" + name + ", " + std::to_string(want) + " bytes) failed: " + cudaGetErrorString(err));
    e.first = nullptr;
    return nullptr;
  }
  e.second = want;
  return e.first;
}

void* cnmf_handle_s::host_buf(const std::string& name, size_t bytes) {
  auto& e = pinned[name];
  if (e.second >= bytes && e.first) return e.first;
  if (e.first) cudaFreeHost(e.first);
  e.first = nullptr;
  e.second = 0;
  const size_t want = std::max<size_t>(bytes, 256);
  cudaError_t err = cudaMallocHost(&e.first, want);
  if (err != cudaSuccess) {
    set_last_error("cudaMallocHost(" + name + ", " + std::to_string(want) + " bytes) failed: " + cudaGetErrorString(err));
    e.first = nullptr;
    return nullptr;
  }
  e.second = want;
  return e.first;
}

int cnmf_handle_s::prof_begin(cudaStream_t s, double work, int cls) {
  if (!profile) return -1;
  while (ev_pool.size() < ev_used + 2) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return -1;
    ev_pool.push_back(e);
  }
  int begin;
  // call sites count their launch (launches += 1) before prof_begin: exactly one more than at the last prof_end
  // means nothing else was enqueued by the library in between
  if (prof_last_end >= 0 && prof_last_stream == s && launches == prof_last_launches + 1) {
    begin = prof_last_end;
  } else {
    begin = (int)ev_used++;
    cudaEventRecord(ev_pool[begin], s);
  }
  const int end = (int)ev_used++;
  ev_pending.push_back(Pending{begin, end, cls, work});
  return (int)ev_pending.size() - 1;
}

void cnmf_handle_s::prof_end(cudaStream_t s, int slot) {
  if (slot < 0) return;
  const int end = ev_pending[slot].end;
  cudaEventRecord(ev_pool[end], s);
  prof_last_end = end;
  prof_last_launches = launches;
  prof_last_stream = s;
}

void cnmf_handle_s::prof_collect() {
  for (auto& pr : ev_pending) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev_pool[pr.begin], ev_pool[pr.end]) == cudaSuccess) {
      prof_ms[pr.cls] += ms;
      prof_work[pr.cls] += pr.work;
      prof_launches[pr.cls] += 1;
    }
  }
  ev_pending.clear();
  ev_used = 0;
  prof_last_end = -1;
}

void* cnmf_handle_s::pool_take(size_t bytes) {
  auto it = pool.find(bytes);
  if (it == pool.end()) return nullptr;
  void* p = it->second;
  pool.erase(it);
  pool_bytes -= bytes;
  return p;
}

void cnmf_handle_s::pool_give(void* p, size_t bytes) {
  constexpr size_t POOL_CAP = (size_t)16 << 30;     // keep at most 16 GB parked
  if (pool_bytes + bytes > POOL_CAP) {
    cudaFree(p);
    return;
  }
  pool.emplace(bytes, p);
  pool_bytes += bytes;
}

void cnmf_handle_s::release_all() {
  for (auto& kv : pool) cudaFree(kv.second);
  pool.clear();
  pool_bytes = 0;
  for (auto e : ev_pool) cudaEventDestroy(e);
  ev_pool.clear();
  for (auto& kv : ws)
    if (kv.second.first) cudaFree(kv.second.first);
  ws.clear();
  for (auto& kv : pinned)
    if (kv.second.first) cudaFreeHost(kv.second.first);
  pinned.clear();
}

extern "C" {

int cnmf_abi_version(void) { return CNMF_B200_ABI_VERSION; }
const char* cnmf_last_error(void) { return g_last_error.c_str(); }

int cnmf_create(cnmf_handle_t* out, int device) {
  CNMF_REQUIRE(out != nullptr, "cnmf_create: out is NULL");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    set_last_error(std::string("no CUDA device available (") + cudaGetErrorString(e) +
                   "); cnmf_b200 has no CPU fallback");
    return -2;
  }
  CNMF_REQUIRE(device >= 0 && device < n, "cnmf_create: bad device index");
  CNMF_CUDA_CHECK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CNMF_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_last_error("cnmf_b200 is built for sm_100a only; device reports sm_" + std::to_string(prop.major) +
                   std::to_string(prop.minor));
    return -3;
  }
  auto* h = new cnmf_handle_s();
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  *out = h;
  return 0;
}

int cnmf_destroy(cnmf_handle_t h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  h->release_all();
  delete h;
  return 0;
}

long long cnmf_launch_count(cnmf_handle_t h) { return h ? h->launches : 0; }

int cnmf_mem_info(cnmf_handle_t h, long long* free_bytes, long long* total_bytes, long long* cached_bytes) {
  CNMF_REQUIRE(h, "mem_info: NULL handle");
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  size_t fr = 0, tot = 0;
  CNMF_CUDA_CHECK(cudaMemGetInfo(&fr, &tot));
  size_t cached = h->pool_bytes;
  for (auto& kv : h->ws) cached += kv.second.second;
  if (free_bytes) *free_bytes = (long long)fr;
  if (total_bytes) *total_bytes = (long long)tot;
  if (cached_bytes) *cached_bytes = (long long)cached;
  return 0;
}

long long cnmf_solve_bytes_per_row(cnmf_dataset_t d) {
  if (!d) return 0;
  // Floats per packed row along the cells (ld_r): the factor Fr and its 2 pieces (alloc_factors), their 3 compaction
  // alternates and the result slab (solve_batched), one slice of the product NUM_r per split-K slice -- 7 + splits_r;
  // along the genes (ld_c) the same for Fc -- 7 + splits_c.  The constants 11 and 10 count 4 and 3 rows more than
  // that; the value stays as it is because callers size their restart groups from it.
  const long long splits_c = gemm_fixed_splits(d->n_rows, d->f16 ? 1 : 0);
  const long long splits_r = gemm_fixed_splits(d->n_cols, d->f16 ? 1 : 0);
  return 4LL * ((11 + splits_r) * (long long)d->ld_r + (10 + splits_c) * (long long)d->ld_c);
}

int cnmf_profile_enable(cnmf_handle_t h, int on) {
  CNMF_REQUIRE(h, "profile_enable: NULL handle");
  h->profile = on != 0;
  for (int c = 0; c < cnmf_handle_s::PROF_CLASSES; ++c) {
    h->prof_ms[c] = h->prof_work[c] = 0.0;
    h->prof_launches[c] = 0;
  }
  h->ev_pending.clear();
  h->ev_used = 0;
  h->prof_last_end = -1;
  if (on) {       // event creation is kept out of the timed region: a pool for ~32 000 launches up front
    while (h->ev_pool.size() < 65536) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) break;
      h->ev_pool.push_back(e);
    }
  }
  return 0;
}

int cnmf_profile_get(cnmf_handle_t h, double* gemm_ms, long long* gemm_launches, double* gemm_flops) {
  CNMF_REQUIRE(h, "profile_get: NULL handle");
  return cnmf_profile_get_class(h, 0, gemm_ms, gemm_launches, gemm_flops);
}

int cnmf_profile_get_class(cnmf_handle_t h, int cls, double* ms, long long* launches, double* work) {
  CNMF_REQUIRE(h, "profile_get_class: NULL handle");
  CNMF_REQUIRE(cls >= 0 && cls < cnmf_handle_s::PROF_CLASSES, "profile_get_class: unknown kernel class");
  CNMF_CUDA_CHECK(cudaDeviceSynchronize());     // every recorded event has completed
  h->prof_collect();
  if (ms) *ms = h->prof_ms[cls];
  if (launches) *launches = h->prof_launches[cls];
  if (work) *work = h->prof_work[cls];
  return 0;
}

}  // extern "C"

// ----------------------------------------------------------------------------- dataset
namespace cnmf {

int dataset_alloc(cnmf_dataset_s* d, float** p, size_t elems) {
  const size_t bytes = std::max<size_t>(elems, 64) * sizeof(float);
  void* q = d->h->pool_take(bytes);
  if (!q) {
    cudaError_t e = cudaMalloc(&q, bytes);
    if (e != cudaSuccess) {
      set_last_error(std::string("dataset cudaMalloc failed: ") + cudaGetErrorString(e));
      return -2;
    }
  }
  d->owned.emplace_back(q, bytes);
  *p = static_cast<float*>(q);
  return 0;
}

int dataset_finish(cnmf_dataset_s* d, cudaStream_t s) {
  cnmf_handle_s* h = d->h;
  const size_t nx = (size_t)d->n_rows * d->ld_c, nxt = (size_t)d->n_cols * d->ld_r;
  if (d->precision == CNMF_PRECISION_TF32X3) {
    // ---- exact-count detection: is X = diag(r) C diag(s) with C integer <= 2048 ?  (column scale first,
    //      then row scale; datasets derived by cnmf_dataset_from_columns arrive with `exact` already decided)
    if (d->allow_exact && !d->exact && d->n_rows <= 65535 * 64) {
      float* cmin = nullptr;
      float* rmin = nullptr;
      CNMF_TRY(dataset_alloc(d, &cmin, (size_t)d->ld_c));
      CNMF_TRY(dataset_alloc(d, &rmin, (size_t)d->ld_r));
      int* n_bad = static_cast<int*>(h->dev_buf("dataset.nbad", sizeof(int) * 2));
      if (!n_bad) return -2;
      CNMF_TRY(launch_min_positive(d->X, d->n_rows, d->n_cols, d->ld_c, cmin, rmin, s));
      CNMF_TRY(launch_fix_scale(cmin, d->n_cols, d->ld_c, s));
      CNMF_TRY(launch_fix_scale(rmin, d->n_rows, d->ld_r, s));
      CNMF_CUDA_CHECK(cudaMemsetAsync(n_bad, 0, sizeof(int) * 2, s));
      CNMF_TRY(launch_check_scaled_int(d->X, d->n_rows, d->n_cols, d->ld_c, nullptr, cmin, n_bad, s));
      CNMF_TRY(launch_check_scaled_int(d->X, d->n_rows, d->n_cols, d->ld_c, rmin, nullptr, n_bad + 1, s));
      h->launches += 5;
      int bad[2] = {1, 1};
      CNMF_CUDA_CHECK(cudaMemcpyAsync(bad, n_bad, sizeof(int) * 2, cudaMemcpyDeviceToHost, s));
      CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
      if (bad[0] == 0) { d->exact = true; d->col_scale = cmin; d->row_scale = nullptr; }
      else if (bad[1] == 0) { d->exact = true; d->row_scale = rmin; d->col_scale = nullptr; }
    }
    if (d->exact) {
      CNMF_TRY(dataset_alloc(d, &d->X_hi, nx));
      CNMF_TRY(dataset_alloc(d, &d->Xt_hi, nxt));
      CNMF_CUDA_CHECK(cudaMemsetAsync(d->X_hi, 0, nx * sizeof(float), s));
      CNMF_CUDA_CHECK(cudaMemsetAsync(d->Xt_hi, 0, nxt * sizeof(float), s));
      CNMF_TRY(launch_build_counts(d->X, d->n_rows, d->n_cols, d->ld_c, d->row_scale, d->col_scale, d->X_hi, s));
      CNMF_TRY(launch_transpose(d->X_hi, d->n_rows, d->n_cols, d->ld_c, d->Xt_hi, nullptr, nullptr, d->ld_r, s));
      h->launches += 2;
      if (d->want_f16) {       // counts <= 2048 are exact in fp16: the B operands of the kind::f16 products
        float *xh = nullptr, *xth = nullptr;
        CNMF_TRY(dataset_alloc(d, &xh, (nx + 1) / 2));
        CNMF_TRY(dataset_alloc(d, &xth, (nxt + 1) / 2));
        d->X_h16 = xh;
        d->Xt_h16 = xth;
        CNMF_TRY(launch_to_half(d->X_hi, d->X_h16, (long long)nx, s));
        CNMF_TRY(launch_to_half(d->Xt_hi, d->Xt_h16, (long long)nxt, s));
        h->launches += 2;
        d->f16 = true;
        // every product of an f16 dataset reads the fp16 count matrices: the fp32 copies of C / C^T were scaffolding.
        // Resident forms are then X (fp32, column operations and derived datasets) + C and C^T as fp16: 2 x the
        // bytes of X instead of 4 x.  (Released after the stream has drained, below.)
        d->drop_tf32 = true;
      }
    } else {
      CNMF_TRY(dataset_alloc(d, &d->X_hi, nx));
      CNMF_TRY(dataset_alloc(d, &d->X_lo, nx));
      CNMF_TRY(dataset_alloc(d, &d->Xt_hi, nxt));
      CNMF_TRY(dataset_alloc(d, &d->Xt_lo, nxt));
      CNMF_CUDA_CHECK(cudaMemsetAsync(d->Xt_hi, 0, nxt * sizeof(float), s));
      CNMF_CUDA_CHECK(cudaMemsetAsync(d->Xt_lo, 0, nxt * sizeof(float), s));
      CNMF_TRY(launch_split_tf32(d->X, d->X_hi, d->X_lo, (long long)nx, s));
      CNMF_TRY(launch_transpose(d->X, d->n_rows, d->n_cols, d->ld_c, nullptr, d->Xt_hi, d->Xt_lo, d->ld_r, s));
      h->launches += 2;
    }
  } else {
    CNMF_TRY(dataset_alloc(d, &d->Xt, nxt));
    CNMF_CUDA_CHECK(cudaMemsetAsync(d->Xt, 0, nxt * sizeof(float), s));
    CNMF_TRY(launch_transpose(d->X, d->n_rows, d->n_cols, d->ld_c, d->Xt, nullptr, nullptr, d->ld_r, s));
    h->launches += 1;
  }
  const int scratch_len = 2 * 148 * 8 + 2;
  double* scratch = static_cast<double*>(h->dev_buf("dataset.sums", sizeof(double) * (scratch_len + 2)));
  if (!scratch) return -2;
  CNMF_TRY(launch_matrix_sums(d->X, d->n_rows, d->n_cols, d->ld_c, scratch + scratch_len, scratch, scratch_len, s));
  h->launches += 2;
  double out2[2];
  CNMF_CUDA_CHECK(cudaMemcpyAsync(out2, scratch + scratch_len, 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  d->sum = out2[0];
  d->sum_sq = out2[1];
  if (d->drop_tf32) {          // the conversions above have completed: hand the fp32 count matrices back
    for (float** pp : {&d->X_hi, &d->Xt_hi}) {
      for (auto it = d->owned.begin(); it != d->owned.end(); ++it)
        if (it->first == *pp) {
          h->pool_give(it->first, it->second);
          d->owned.erase(it);
          break;
        }
      *pp = nullptr;
    }
    d->drop_tf32 = false;
  }
  return 0;
}

int dataset_new(cnmf_handle_s* h, const cnmf_dataset_s* like, int precision, int n_rows, int n_cols,
                cnmf_dataset_s** out) {
  auto* d = new cnmf_dataset_s();
  d->h = h;
  d->n_rows = n_rows;
  d->n_cols = n_cols;
  d->ld_c = pad_ld(n_cols);
  d->ld_r = pad_ld(n_rows);
  d->allow_exact = like ? like->allow_exact : precision != CNMF_PRECISION_TF32X3_GENERAL;
  d->want_f16 = like ? like->want_f16 : precision == CNMF_PRECISION_F16X2;
  // GENERAL and F16X2 are TF32X3 datasets that differ in these two flags
  d->precision = like ? like->precision : (d->allow_exact && !d->want_f16 ? precision : CNMF_PRECISION_TF32X3);
  const int rc = dataset_alloc(d, &d->X, (size_t)n_rows * d->ld_c);
  if (rc != 0) {
    cnmf_dataset_destroy(d);
    return rc;
  }
  *out = d;
  return 0;
}

int finish_or_destroy(cnmf_dataset_s* d, int rc, cudaStream_t s, cnmf_dataset_t* out) {
  if (rc == 0) rc = dataset_finish(d, s);
  if (rc != 0) {
    cnmf_dataset_destroy(d);
    return rc;
  }
  *out = d;
  return 0;
}

int dataset_ensure_full_transpose(cnmf_dataset_s* d, cudaStream_t s) {
  if (d->Xt) return 0;
  CNMF_CUDA_CHECK(cudaSetDevice(d->h->device));
  const size_t nxt = (size_t)d->n_cols * d->ld_r;
  CNMF_TRY(dataset_alloc(d, &d->Xt, nxt));
  CNMF_CUDA_CHECK(cudaMemsetAsync(d->Xt, 0, nxt * sizeof(float), s));
  CNMF_TRY(launch_transpose(d->X, d->n_rows, d->n_cols, d->ld_c, d->Xt, nullptr, nullptr, d->ld_r, s));
  d->h->launches += 1;
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  return 0;
}

// ----------------------------------------------------------------------------- factorize
int alloc_factors(cnmf_handle_s* h, const char* prefix, int SK, int ld_r, int ld_c, bool tf32, SolveIO* io) {
  const std::string pre(prefix);
  const size_t nr = (size_t)SK * ld_r, nc = (size_t)SK * ld_c;
  io->Fr = static_cast<float*>(h->dev_buf(pre + "Fr", nr * 4));
  io->Fc = static_cast<float*>(h->dev_buf(pre + "Fc", nc * 4));
  if (!io->Fr || !io->Fc) return -2;
  if (tf32) {
    io->Fr_hi = static_cast<float*>(h->dev_buf(pre + "Fr_hi", nr * 4));
    io->Fr_lo = static_cast<float*>(h->dev_buf(pre + "Fr_lo", nr * 4));
    io->Fc_hi = static_cast<float*>(h->dev_buf(pre + "Fc_hi", nc * 4));
    io->Fc_lo = static_cast<float*>(h->dev_buf(pre + "Fc_lo", nc * 4));
    if (!io->Fr_hi || !io->Fr_lo || !io->Fc_hi || !io->Fc_lo) return -2;
  }
  return 0;
}

int split_factors(cnmf_handle_s* h, const DataView& v, const SolveIO& io, int SK, bool tf32, cudaStream_t s) {
  if (!tf32 || v.f16) return 0;
  CNMF_TRY(launch_split_scaled(io.Fr, io.Fr_hi, io.Fr_lo, SK, v.ld_r, v.exact ? v.scale_r : nullptr, s));
  CNMF_TRY(launch_split_scaled(io.Fc, io.Fc_hi, io.Fc_lo, SK, v.ld_c, v.exact ? v.scale_c : nullptr, s));
  h->launches += 2;
  return 0;
}

}  // namespace cnmf

namespace {

using clk = std::chrono::steady_clock;
double ms_since(clk::time_point t0) { return std::chrono::duration<double, std::milli>(clk::now() - t0).count(); }

// The restarts of one call: K of each, their packed row offsets, the total rows SK and the scale of sklearn's random
// init, sqrt(mean(X) / k)
struct RestartTable {
  std::vector<int> ks, off;
  std::vector<double> avgs;
  int SK = 0;
};

int restart_table(const cnmf_dataset_s* d, int n_restarts, const int32_t* ks_in, RestartTable* t) {
  const double mean = d->sum / ((double)d->n_rows * (double)d->n_cols);
  t->ks.assign(ks_in, ks_in + n_restarts);
  t->off.resize(n_restarts);
  t->avgs.resize(n_restarts);
  for (int r = 0; r < n_restarts; ++r) {
    CNMF_REQUIRE(t->ks[r] >= 1 && t->ks[r] <= KMAX, "n_components must be in [1, 32] on the CUDA path");
    t->off[r] = t->SK;
    t->SK += t->ks[r];
    t->avgs[r] = std::sqrt(mean / t->ks[r]);
  }
  return 0;
}

// the legacy MT19937 / polar-gauss stream of every restart, generated in place on the GPU into packed padded factors
int device_rng(cnmf_dataset_s* d, const RestartTable& t, const uint32_t* seeds, float* Fr, float* Fc, cudaStream_t s) {
  CNMF_CUDA_CHECK(cudaMemsetAsync(Fr, 0, (size_t)t.SK * d->ld_r * 4, s));
  CNMF_CUDA_CHECK(cudaMemsetAsync(Fc, 0, (size_t)t.SK * d->ld_c * 4, s));
  return launch_rng_init(seeds, t.ks.data(), t.off.data(), t.avgs.data(), (int)t.ks.size(), d->n_rows, d->n_cols, Fr,
                         d->ld_r, Fc, d->ld_c, d->h, s);
}

void parallel_for(int n, const std::function<void(int)>& fn) {
  int nt = (int)std::thread::hardware_concurrency();
  if (nt < 1) nt = 1;
  nt = std::min(nt, n);
  if (nt <= 1) {
    for (int i = 0; i < n; ++i) fn(i);
    return;
  }
  std::atomic<int> next{0};
  std::vector<std::thread> th;
  th.reserve(nt);
  for (int t = 0; t < nt; ++t)
    th.emplace_back([&] {
      for (;;) {
        const int i = next.fetch_add(1);
        if (i >= n) break;
        fn(i);
      }
    });
  for (auto& t : th) t.join();
}

// the same stream on the host (bit-exact numpy), in groups through a pinned staging buffer
int host_rng(cnmf_dataset_s* d, const RestartTable& t, const uint32_t* seeds, float* Fr, float* Fc, cudaStream_t s) {
  cnmf_handle_s* h = d->h;
  const std::vector<int>& ks = t.ks;
  const std::vector<int>& off = t.off;
  const int n_restarts = (int)ks.size();
  const size_t group_budget = (size_t)256 << 20;   // bytes of W^T staged per group
  int r0 = 0;
  while (r0 < n_restarts) {
    int r1 = r0;
    size_t bytes = 0;
    while (r1 < n_restarts && (r1 == r0 || bytes + (size_t)ks[r1] * d->ld_r * 4 <= group_budget)) {
      bytes += (size_t)ks[r1] * d->ld_r * 4;
      ++r1;
    }
    const int rows = off[r1 - 1] + ks[r1 - 1] - off[r0];
    float* stW = static_cast<float*>(h->host_buf("stage.W", (size_t)rows * d->ld_r * 4));
    float* stH = static_cast<float*>(h->host_buf("stage.H", (size_t)rows * d->ld_c * 4));
    if (!stW || !stH) return -2;
    auto t_rng = clk::now();
    parallel_for(r1 - r0, [&](int i) {
      const int r = r0 + i;
      float* w = stW + (size_t)(off[r] - off[r0]) * d->ld_r;
      float* hh = stH + (size_t)(off[r] - off[r0]) * d->ld_c;
      nmf_random_init(seeds[r], t.avgs[r], d->n_rows, d->n_cols, ks[r], w, d->ld_r, hh, d->ld_c);
      for (int c = 0; c < ks[r]; ++c) {                  // zero the row padding (each worker its own rows)
        std::memset(w + (size_t)c * d->ld_r + d->n_rows, 0, (size_t)(d->ld_r - d->n_rows) * 4);
        std::memset(hh + (size_t)c * d->ld_c + d->n_cols, 0, (size_t)(d->ld_c - d->n_cols) * 4);
      }
    });
    h->t_rng_ms += ms_since(t_rng);
    auto t_h2d = clk::now();
    CNMF_CUDA_CHECK(cudaMemcpyAsync(Fr + (size_t)off[r0] * d->ld_r, stW, (size_t)rows * d->ld_r * 4,
                                    cudaMemcpyHostToDevice, s));
    CNMF_CUDA_CHECK(cudaMemcpyAsync(Fc + (size_t)off[r0] * d->ld_c, stH, (size_t)rows * d->ld_c * 4,
                                    cudaMemcpyHostToDevice, s));
    CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
    h->t_h2d_ms += ms_since(t_h2d);
    r0 = r1;
  }
  return 0;
}

// Where the starting factors of a factorize come from: the seeded generator on the device or on the host, or packed
// factors of the caller (host: rows of n_rows / n_cols floats; device: rows padded to the dataset's ld)
struct Starts {
  enum Kind { DEVICE_RNG, HOST_RNG, HOST_FACTORS, DEVICE_FACTORS } kind;
  const uint32_t* seeds;
  const float* Wt0;
  const float* H0;
};

Starts seeded(const cnmf_nmf_params& p, const uint32_t* seeds) {
  return {(p.reserved & 1) ? Starts::HOST_RNG : Starts::DEVICE_RNG, seeds, nullptr, nullptr};
}

// Where the results go: spectra (and usages, if set) to the host as packed rows of n_cols (n_rows) floats, or spectra
// to the device as the first `width` floats of rows `ld` apart; per-restart statistics to the host
struct Outputs {
  float* spectra_host;
  float* usages_host;
  float* spectra_dev;
  long long ld, width;
  int32_t* n_iter_host;
  double* err_host;
};

// The one host path of every factorize entry point: starting factors into the "fac." workspace, tf32 pieces, the
// batched solve, results out.  Resets and fills the handle's phase timings.
int factorize_run(cnmf_dataset_s* d, int n_restarts, const int32_t* ks_in, const cnmf_nmf_params& p, const Starts& in,
                  const Outputs& out, void* stream) {
  cnmf_handle_s* h = d->h;
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  RestartTable t;
  CNMF_TRY(restart_table(d, n_restarts, ks_in, &t));
  const int SK = t.SK;
  const bool tf32 = p.precision == CNMF_PRECISION_TF32X3;
  SolveIO io;
  CNMF_TRY(alloc_factors(h, "fac.", SK, d->ld_r, d->ld_c, tf32, &io));
  h->t_rng_ms = h->t_h2d_ms = h->t_solve_ms = h->t_d2h_ms = 0;
  switch (in.kind) {
    case Starts::DEVICE_RNG: {
      // no host synchronisation: launch_rng_init stages its arguments itself, and the solve is enqueued behind the
      // generator on the same stream (t_rng_ms = enqueue time; the kernel's time is part of t_solve_ms)
      const auto t_rng = clk::now();
      CNMF_TRY(device_rng(d, t, in.seeds, io.Fr, io.Fc, s));
      h->t_rng_ms = ms_since(t_rng);
      break;
    }
    case Starts::HOST_RNG:
      CNMF_TRY(host_rng(d, t, in.seeds, io.Fr, io.Fc, s));
      break;
    case Starts::HOST_FACTORS:
      CNMF_CUDA_CHECK(cudaMemsetAsync(io.Fr, 0, (size_t)SK * d->ld_r * 4, s));
      CNMF_CUDA_CHECK(cudaMemsetAsync(io.Fc, 0, (size_t)SK * d->ld_c * 4, s));
      CNMF_CUDA_CHECK(cudaMemcpy2DAsync(io.Fr, (size_t)d->ld_r * 4, in.Wt0, (size_t)d->n_rows * 4,
                                        (size_t)d->n_rows * 4, SK, cudaMemcpyHostToDevice, s));
      CNMF_CUDA_CHECK(cudaMemcpy2DAsync(io.Fc, (size_t)d->ld_c * 4, in.H0, (size_t)d->n_cols * 4,
                                        (size_t)d->n_cols * 4, SK, cudaMemcpyHostToDevice, s));
      break;
    case Starts::DEVICE_FACTORS:
      CNMF_CUDA_CHECK(cudaMemcpyAsync(io.Fr, in.Wt0, (size_t)SK * d->ld_r * 4, cudaMemcpyDeviceToDevice, s));
      CNMF_CUDA_CHECK(cudaMemcpyAsync(io.Fc, in.H0, (size_t)SK * d->ld_c * 4, cudaMemcpyDeviceToDevice, s));
      break;
  }
  const DataView v = make_view(d, false);
  CNMF_TRY(split_factors(h, v, io, SK, tf32, s));
  io.R = n_restarts;
  io.ks = t.ks;
  io.update_cols = true;
  const auto t_solve = clk::now();
  CNMF_TRY(solve_batched(h, v, io, p, s));
  h->t_solve_ms = ms_since(t_solve);
  const auto t_d2h = clk::now();
  if (out.spectra_dev)
    CNMF_CUDA_CHECK(cudaMemcpy2DAsync(out.spectra_dev, (size_t)out.ld * 4, io.Fc, (size_t)d->ld_c * 4,
                                      (size_t)out.width * 4, SK, cudaMemcpyDeviceToDevice, s));
  if (out.spectra_host)
    CNMF_CUDA_CHECK(cudaMemcpy2DAsync(out.spectra_host, (size_t)d->n_cols * 4, io.Fc, (size_t)d->ld_c * 4,
                                      (size_t)d->n_cols * 4, SK, cudaMemcpyDeviceToHost, s));
  if (out.usages_host)
    CNMF_CUDA_CHECK(cudaMemcpy2DAsync(out.usages_host, (size_t)d->n_rows * 4, io.Fr, (size_t)d->ld_r * 4,
                                      (size_t)d->n_rows * 4, SK, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  h->t_d2h_ms = ms_since(t_d2h);
  for (int r = 0; r < n_restarts; ++r) {
    if (out.n_iter_host) out.n_iter_host[r] = io.n_iter[r];
    if (out.err_host) out.err_host[r] = io.err[r];
  }
  return 0;
}

int check_params(cnmf_dataset_s* d, const cnmf_nmf_params* p) {
  CNMF_REQUIRE(d && p, "NULL dataset or params");
  CNMF_REQUIRE(p->precision == d->precision, "params.precision must match the precision the dataset was created with");
  CNMF_REQUIRE(p->reserved2 == 0, "params.reserved2 must be 0");
  if (p->beta_loss != CNMF_LOSS_FROBENIUS) CNMF_TRY(cnmf::dataset_ensure_full_transpose(d, nullptr));
  return 0;
}

}  // namespace

extern "C" {

int cnmf_dataset_create(cnmf_handle_t h, const float* X, int n_rows, int n_cols, long long ld, int src_is_device,
                        int precision, void* stream, cnmf_dataset_t* out) {
  CNMF_REQUIRE(h && X && out, "dataset_create: NULL argument");
  CNMF_REQUIRE(n_rows > 0 && n_cols > 0 && ld >= n_cols, "dataset_create: bad shape");
  CNMF_REQUIRE(precision == CNMF_PRECISION_FP32 || precision == CNMF_PRECISION_TF32X3 ||
                   precision == CNMF_PRECISION_TF32X3_GENERAL || precision == CNMF_PRECISION_F16X2,
               "dataset_create: bad precision");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  cnmf_dataset_s* d = nullptr;
  CNMF_TRY(dataset_new(h, nullptr, precision, n_rows, n_cols, &d));
  int rc = 0;
  cudaError_t e = cudaMemsetAsync(d->X, 0, (size_t)n_rows * d->ld_c * sizeof(float), s);
  if (e == cudaSuccess)
    e = cudaMemcpy2DAsync(d->X, (size_t)d->ld_c * sizeof(float), X, (size_t)ld * sizeof(float),
                          (size_t)n_cols * sizeof(float), n_rows,
                          src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s);
  if (e != cudaSuccess) {
    set_last_error(std::string("dataset upload failed: ") + cudaGetErrorString(e));
    rc = -2;
  }
  return finish_or_destroy(d, rc, s, out);
}

int cnmf_dataset_min(cnmf_dataset_t d, float* min_host, void* stream) {
  CNMF_REQUIRE(d && min_host, "dataset_min: NULL argument");
  CNMF_CUDA_CHECK(cudaSetDevice(d->h->device));
  return cnmf::matrix_min(d->h, d->X, d->n_rows, d->n_cols, d->ld_c, min_host, as_stream(stream));
}

int cnmf_dataset_destroy(cnmf_dataset_t d) {
  if (!d) return 0;
  for (auto& pr : d->owned) d->h->pool_give(pr.first, pr.second);
  delete d;
  return 0;
}

int cnmf_dataset_shape(cnmf_dataset_t d, int* n_rows, int* n_cols) {
  CNMF_REQUIRE(d, "dataset_shape: NULL dataset");
  if (n_rows) *n_rows = d->n_rows;
  if (n_cols) *n_cols = d->n_cols;
  return 0;
}

int cnmf_dataset_is_exact(cnmf_dataset_t d) { return (d && d->exact) ? (d->f16 ? 2 : 1) : 0; }

int cnmf_dataset_sums(cnmf_dataset_t d, double* sum, double* sum_sq) {
  CNMF_REQUIRE(d, "dataset_sums: NULL dataset");
  if (sum) *sum = d->sum;
  if (sum_sq) *sum_sq = d->sum_sq;
  return 0;
}

// ----------------------------------------------------------------------------- random init
int cnmf_random_init_host(uint32_t seed, double avg, int n_samples, int n_features, int k, float* Wt, long long ldW,
                          float* H, long long ldH) {
  CNMF_REQUIRE(Wt && H && n_samples > 0 && n_features > 0 && k > 0, "random_init: bad arguments");
  CNMF_REQUIRE(ldW >= n_samples && ldH >= n_features, "random_init: leading dimension too small");
  nmf_random_init(seed, avg, n_samples, n_features, k, Wt, ldW, H, ldH);
  return 0;
}

int cnmf_factorize(cnmf_dataset_t d, int n_restarts, const int32_t* ks_in, const uint32_t* seeds,
                   const cnmf_nmf_params* p, float* spectra_host, float* usages_host, int32_t* n_iter_host,
                   double* err_host, void* stream) {
  CNMF_REQUIRE(spectra_host, "factorize: spectra_host is NULL");
  CNMF_TRY(check_params(d, p));
  CNMF_REQUIRE(n_restarts > 0 && ks_in && seeds, "factorize: bad arguments");
  return factorize_run(d, n_restarts, ks_in, *p, seeded(*p, seeds),
                       {spectra_host, usages_host, nullptr, 0, 0, n_iter_host, err_host}, stream);
}

int cnmf_factorize_seeds_dev(cnmf_dataset_t d, int n_restarts, const int32_t* ks_in, const uint32_t* seeds,
                             const cnmf_nmf_params* p, float* spectra_dev, long long ld_out, int32_t* n_iter_host,
                             double* err_host, void* stream) {
  CNMF_REQUIRE(spectra_dev, "factorize_seeds_dev: spectra_dev is NULL");
  CNMF_TRY(check_params(d, p));
  CNMF_REQUIRE(n_restarts > 0 && ks_in && seeds, "factorize: bad arguments");
  CNMF_REQUIRE(ld_out >= d->n_cols, "factorize: device output row stride too small");
  return factorize_run(d, n_restarts, ks_in, *p, seeded(*p, seeds),
                       {nullptr, nullptr, spectra_dev, ld_out, d->n_cols, n_iter_host, err_host}, stream);
}

int cnmf_last_timing(cnmf_handle_t h, double* rng_ms, double* h2d_ms, double* solve_ms, double* d2h_ms) {
  CNMF_REQUIRE(h, "last_timing: NULL handle");
  if (rng_ms) *rng_ms = h->t_rng_ms;
  if (h2d_ms) *h2d_ms = h->t_h2d_ms;
  if (solve_ms) *solve_ms = h->t_solve_ms;
  if (d2h_ms) *d2h_ms = h->t_d2h_ms;
  return 0;
}

int cnmf_factorize_init(cnmf_dataset_t d, int n_restarts, const int32_t* ks_in, const float* Wt0_host,
                        const float* H0_host, const cnmf_nmf_params* p, float* spectra_host, float* usages_host,
                        int32_t* n_iter_host, double* err_host, void* stream) {
  CNMF_TRY(check_params(d, p));
  CNMF_REQUIRE(n_restarts > 0 && ks_in && Wt0_host && H0_host && spectra_host, "factorize_init: bad arguments");
  return factorize_run(d, n_restarts, ks_in, *p, {Starts::HOST_FACTORS, nullptr, Wt0_host, H0_host},
                       {spectra_host, usages_host, nullptr, 0, 0, n_iter_host, err_host}, stream);
}

int cnmf_factorize_dev(cnmf_dataset_t d, int n_restarts, const int32_t* ks_in, const float* Wt0_dev,
                       const float* H0_dev, const cnmf_nmf_params* p, float* spectra_dev, int32_t* n_iter_host,
                       double* err_host, void* stream) {
  CNMF_TRY(check_params(d, p));
  CNMF_REQUIRE(n_restarts > 0 && ks_in && Wt0_dev && H0_dev && spectra_dev, "factorize_dev: bad arguments");
  return factorize_run(d, n_restarts, ks_in, *p, {Starts::DEVICE_FACTORS, nullptr, Wt0_dev, H0_dev},
                       {nullptr, nullptr, spectra_dev, d->ld_c, d->ld_c, n_iter_host, err_host}, stream);
}

int cnmf_random_init_dev(cnmf_dataset_t d, int n_restarts, const int32_t* ks_in, const uint32_t* seeds, float* Wt_dev,
                         float* H_dev, void* stream) {
  CNMF_REQUIRE(d && n_restarts > 0 && ks_in && seeds && Wt_dev && H_dev, "random_init_dev: bad arguments");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(d->h->device));
  RestartTable t;
  CNMF_TRY(restart_table(d, n_restarts, ks_in, &t));
  CNMF_TRY(device_rng(d, t, seeds, Wt_dev, H_dev, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  return 0;
}

int cnmf_dataset_ld(cnmf_dataset_t d, int* ld_rows, int* ld_cols) {
  CNMF_REQUIRE(d, "dataset_ld: NULL dataset");
  if (ld_rows) *ld_rows = d->ld_r;
  if (ld_cols) *ld_cols = d->ld_c;
  return 0;
}

}  // extern "C"
