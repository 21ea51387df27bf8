// Consensus-stage kernels: the numeric steps of cNMF.consensus (cnmf.py:882-916) on the stacked
// spectra matrix S (R x G, fp32, row stride ld).  R <= ~6000, G <= ~5000 at the BASELINE configs, so
// S (<= 120 MB) lives in L2 and every kernel here is a streaming / reduction kernel:
//   C1  l2_normalize_rows          cnmf.py:882
//   C2  pairwise distances         cnmf.py:891  (direct sum (x-y)^2: no ||x||^2+||y||^2-2xy cancellation)
//   C3  k-NN local density         cnmf.py:893-896 (exact radix select of the n+1 smallest per row)
//   C5  Lloyd E+M step             sklearn _k_means_lloyd.pyx:168-219 (k-means++ draws stay on the host)
//   C6  per-cluster median         cnmf.py:913-916
#include <algorithm>
#include <vector>

#include "engine.h"

using namespace cnmf;

namespace {

template <typename T>
__device__ __forceinline__ T block_sum_all(T v, T* smem /* >= 33 entries */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  T r = (threadIdx.x < nw) ? smem[threadIdx.x] : T(0);
  if (warp == 0) {
    r = warp_sum(r);
    if (lane == 0) smem[32] = r;
  }
  __syncthreads();
  return smem[32];   // broadcast to every thread
}

// ---------------------------------------------------------------- C1
__global__ void l2_normalize_kernel(float* __restrict__ S, int R, int G, int ld) {
  __shared__ double sm[33];
  const int r = blockIdx.x;
  float* row = S + (long long)r * ld;
  double q = 0.0;
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    const double v = row[g];
    q += v * v;
  }
  q = block_sum_all(q, sm);
  const double inv = 1.0 / sqrt(q);
  for (int g = threadIdx.x; g < G; g += blockDim.x) row[g] = (float)((double)row[g] * inv);
}

// ---------------------------------------------------------------- C2: D[i][j] = sqrt(sum_g (A_i - B_j)^2)
// 64 x 64 output tile per block, 16 x 16 threads, 4 x 4 per thread, k-tiles of 16 through smem.  The inner product
// runs on packed fp32 (FADD2 with a broadcast operand, FFMA2): one instruction per element pair instead of two --
// this kernel is FP32-issue bound, not HBM-bound (profiles/r1h_ncu_consensus_summary.txt).  SYM (A == B, the R x R
// matrix of cnmf.py:891): only tiles on or above the diagonal are computed, each is also written transposed, so the
// matrix is exactly symmetric with an exactly zero diagonal at half the work.
template <bool SQRT, bool SYM>
__global__ void __launch_bounds__(256)
pair_dist_kernel(const float* __restrict__ A, int RA, int lda, const float* __restrict__ B, int RB, int ldb, int G,
                 float* __restrict__ D, int ldd) {
  constexpr int T = 64, TK = 16;
  if (SYM && blockIdx.x < blockIdx.y) return;
  __shared__ __align__(16) float As[TK][T + 4];
  __shared__ __align__(16) float Bs[TK][T + 4];
  const int i0 = blockIdx.y * T, j0 = blockIdx.x * T;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int lrow = threadIdx.x >> 2, lk = (threadIdx.x & 3) * 4;
  float2 acc[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = make_float2(0.f, 0.f);
  for (int k0 = 0; k0 < G; k0 += TK) {
    {
      float va[4] = {0.f, 0.f, 0.f, 0.f}, vb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int g = k0 + lk + e;
        if (g < G) {
          if (i0 + lrow < RA) va[e] = A[(long long)(i0 + lrow) * lda + g];
          if (j0 + lrow < RB) vb[e] = B[(long long)(j0 + lrow) * ldb + g];
        }
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        As[lk + e][lrow] = va[e];
        Bs[lk + e][lrow] = vb[e];
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w};
      const float2 nb0 = make_float2(-b.x, -b.y), nb1 = make_float2(-b.z, -b.w);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 d0 = add2(bcast2(av[i]), nb0), d1 = add2(bcast2(av[i]), nb1);
        acc[i][0] = fma2(d0, d0, acc[i][0]);
        acc[i][1] = fma2(d1, d1, acc[i][1]);
      }
    }
    __syncthreads();
  }
  float o[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    o[i][0] = acc[i][0].x; o[i][1] = acc[i][0].y; o[i][2] = acc[i][1].x; o[i][3] = acc[i][1].y;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (SQRT) o[i][j] = sqrtf(o[i][j]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = i0 + ty * 4 + i;
    if (r >= RA) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = j0 + tx * 4 + j;
      if (c < RB) D[(long long)r * ldd + c] = o[i][j];
    }
  }
  if (SYM && blockIdx.x != blockIdx.y) {             // mirror image of an off-diagonal tile
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = j0 + tx * 4 + j;
      if (c >= RB) continue;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = i0 + ty * 4 + i;
        if (r < RA) D[(long long)c * ldd + r] = o[i][j];
      }
    }
  }
}

// k-means++ candidate scoring (sklearn _kmeans.py:231-262): squared distances from every row of S to a handful of
// candidate rows of S.  HBM-bound form: one warp per row streams it once with 16-byte loads against the (L1-hot)
// candidate rows, differences in fp32, squares accumulated in fp64 (sklearn scores candidates in float64).  The
// 64 x 64-tile kernel above needed 200 us for this shape (60 blocks, latency-bound); 19 calls per init made the
// seeding, not Lloyd, the cost of KMeans (profiles/r1h_ncu_consensus_summary.txt).
template <int NC>
__global__ void __launch_bounds__(256)
cand_dist_kernel(const float* __restrict__ S, int R, int G, int ld, const int32_t* __restrict__ idx, int n_c,
                 float* __restrict__ out /* n_c x R */) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= R) return;
  const float4* row = reinterpret_cast<const float4*>(S + (long long)r * ld);
  const float4* cand[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) cand[c] = reinterpret_cast<const float4*>(S + (long long)idx[c < n_c ? c : 0] * ld);
  double acc[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) acc[c] = 0.0;
  const int g4 = G / 4;
  for (int q = lane; q < g4; q += 32) {
    const float4 x = row[q];
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const float4 y = cand[c][q];
      const float d0 = x.x - y.x, d1 = x.y - y.y, d2 = x.z - y.z, d3 = x.w - y.w;
      acc[c] += (double)d0 * d0 + (double)d1 * d1 + (double)d2 * d2 + (double)d3 * d3;
    }
  }
  for (int g = 4 * g4 + lane; g < G; g += 32) {      // ragged tail
    const float x = S[(long long)r * ld + g];
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const float d = x - S[(long long)idx[c < n_c ? c : 0] * ld + g];
      acc[c] += (double)d * d;
    }
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const double v = warp_sum(acc[c]);
    if (lane == 0 && c < n_c) out[(long long)c * R + r] = (float)v;
  }
}

// ---------------------------------------------------------------- C3: sum of the m smallest entries of each row
// Exact MSB-first radix select on the (non-negative) float bit patterns, one block per row.
__global__ void __launch_bounds__(256)
knn_density_kernel(const float* __restrict__ D, int R, int ldd, int m /* n_neighbors + 1 */, int n_neighbors,
                   float* __restrict__ density) {
  __shared__ int smi[33];
  __shared__ double smd[33];
  const int r = blockIdx.x;
  const float* row = D + (long long)r * ldd;
  uint32_t prefix = 0;
  int k = m - 1;   // 0-based rank of the threshold element
  for (int bit = 30; bit >= 0; --bit) {
    const uint32_t mask_hi = ~((1u << (bit + 1)) - 1u) & 0x7fffffffu;   // bits above `bit`
    int cnt = 0;
    for (int j = threadIdx.x; j < R; j += blockDim.x) {
      const uint32_t u = __float_as_uint(row[j]);
      cnt += ((u & mask_hi) == prefix) && !((u >> bit) & 1u);
    }
    cnt = block_sum_all(cnt, smi);
    if (k >= cnt) {
      k -= cnt;
      prefix |= (1u << bit);
    }
  }
  const float tau = __uint_as_float(prefix);   // the m-th smallest value
  double s = 0.0;
  int less = 0;
  for (int j = threadIdx.x; j < R; j += blockDim.x) {
    const float v = row[j];
    if (v < tau) {
      s += (double)v;
      ++less;
    }
  }
  s = block_sum_all(s, smd);
  less = block_sum_all(less, smi);
  if (threadIdx.x == 0) density[r] = (float)((s + (double)(m - less) * (double)tau) / (double)n_neighbors);
}

// ---------------------------------------------------------------- C5: Lloyd E step
// one warp per row: direct squared distances to the K centres held in shared memory (K*G*4 bytes may
// exceed smem for large G, so centres are read through L1/L2 instead; they are tiny and hot).
__global__ void __launch_bounds__(256)
kmeans_assign_kernel(const float* __restrict__ S, int R, int G, int ld, const float* __restrict__ C, int K, int ldc,
                     int32_t* __restrict__ labels, float* __restrict__ mind, int* __restrict__ n_changed) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= R) return;
  const float* x = S + (long long)warp * ld;
  float best = 0.f;
  int bl = 0;
  for (int c = 0; c < K; ++c) {
    const float* cc = C + (long long)c * ldc;
    float a = 0.f;
    for (int g = lane; g < G; g += 32) {
      const float d = x[g] - cc[g];
      a = fmaf(d, d, a);
    }
    a = warp_sum(a);
    if (c == 0 || a < best) {   // strict '<': first minimum wins (sklearn _k_means_lloyd.pyx:205-209)
      best = a;
      bl = c;
    }
  }
  if (lane == 0) {
    if (labels[warp] != bl) atomicAdd(n_changed, 1);
    labels[warp] = bl;
    mind[warp] = best;
  }
}

// stable counting sort of row indices by label: thread c lists the members of cluster c in row order
__global__ void members_kernel(const int32_t* __restrict__ labels, int R, int K, int32_t* __restrict__ counts,
                               int32_t* __restrict__ order /* K x R */) {
  const int c = threadIdx.x;
  if (c >= K) return;
  int n = 0;
  for (int i = 0; i < R; ++i)
    if (labels[i] == c) order[(long long)c * R + n++] = i;
  counts[c] = n;
}

// M step: per-cluster column sums in fp64, members visited in row order (deterministic)
__global__ void __launch_bounds__(128)
cluster_sums_kernel(const float* __restrict__ S, int G, int ld, const int32_t* __restrict__ counts,
                    const int32_t* __restrict__ order, int R, double* __restrict__ sums /* K x G */) {
  const int c = blockIdx.y;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const int n = counts[c];
  const int32_t* mem = order + (long long)c * R;
  double a = 0.0;
  for (int i = 0; i < n; ++i) a += (double)S[(long long)mem[i] * ld + g];
  sums[(long long)c * G + g] = a;
}

// M step, second half, on the device: new centre = sums * (1 / count) (sklearn _k_means_common.pyx:274-298),
// squared shift against the current centre, fp32 copy for the next E step.  One block per cluster; a cluster
// without members raises `any_empty` and is left to the host's relocation rule (the caller keeps the old centres).
__global__ void __launch_bounds__(256)
centre_update_kernel(const double* __restrict__ sums, const int32_t* __restrict__ counts, int G,
                     const double* __restrict__ C64_cur, double* __restrict__ C64_new, float* __restrict__ C32_new,
                     double* __restrict__ shift_part, int* __restrict__ any_empty) {
  __shared__ double sm[33];
  const int j = blockIdx.x;
  const int w = counts[j];
  if (w == 0) {
    if (threadIdx.x == 0) {
      atomicExch(any_empty, 1);
      shift_part[j] = 0.0;
    }
    return;
  }
  const double inv = 1.0 / (double)w;
  double acc = 0.0;
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    const double nv = sums[(long long)j * G + g] * inv;
    const double d = nv - C64_cur[(long long)j * G + g];
    acc += d * d;
    C64_new[(long long)j * G + g] = nv;
    C32_new[(long long)j * G + g] = (float)nv;
  }
  acc = block_sum_all(acc, sm);
  if (threadIdx.x == 0) shift_part[j] = acc;
}

__global__ void sum_float_kernel(const float* __restrict__ v, int n, double* __restrict__ out) {
  __shared__ double sm[33];
  double a = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) a += (double)v[i];
  a = block_sum_all(a, sm);
  if (threadIdx.x == 0) *out = a;
}

// ---------------------------------------------------------------- C6: per-(cluster, gene) median by radix select
__device__ __forceinline__ float select_kth(const float* __restrict__ S, int ld, int g, const int32_t* mem, int n, int k) {
  uint32_t prefix = 0;
  for (int bit = 30; bit >= 0; --bit) {
    const uint32_t mask_hi = ~((1u << (bit + 1)) - 1u) & 0x7fffffffu;
    int cnt = 0;
    for (int i = 0; i < n; ++i) {
      const uint32_t u = __float_as_uint(S[(long long)mem[i] * ld + g]);
      cnt += ((u & mask_hi) == prefix) && !((u >> bit) & 1u);
    }
    if (k >= cnt) {
      k -= cnt;
      prefix |= (1u << bit);
    }
  }
  return __uint_as_float(prefix);
}

__global__ void __launch_bounds__(128)
cluster_median_kernel(const float* __restrict__ S, int G, int ld, const int32_t* __restrict__ counts,
                      const int32_t* __restrict__ order, int R, float* __restrict__ M, int ldm) {
  const int c = blockIdx.y;
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const int n = counts[c];
  const int32_t* mem = order + (long long)c * R;
  float med = __int_as_float(0x7fc00000);   // NaN for an empty cluster (pandas drops the group)
  if (n > 0) {
    if (n & 1) {
      med = select_kth(S, ld, g, mem, n, n / 2);
    } else {
      const float v1 = select_kth(S, ld, g, mem, n, n / 2 - 1);
      int le = 0;
      float nxt = __int_as_float(0x7f800000);
      for (int i = 0; i < n; ++i) {
        const float v = S[(long long)mem[i] * ld + g];
        le += (v <= v1);
        if (v > v1) nxt = fminf(nxt, v);
      }
      const float v2 = (le >= n / 2 + 1) ? v1 : nxt;
      med = 0.5f * (v1 + v2);               // pandas: mean of the two middle values
    }
  }
  M[(long long)c * ldm + g] = med;
}

__global__ void row_normalize_sum_kernel(float* __restrict__ M, int G, int ldm) {
  __shared__ double sm[33];
  float* row = M + (long long)blockIdx.x * ldm;
  double s = 0.0;
  for (int g = threadIdx.x; g < G; g += blockDim.x) s += (double)row[g];
  s = block_sum_all(s, sm);
  for (int g = threadIdx.x; g < G; g += blockDim.x) row[g] = (float)((double)row[g] / s);
}

// per-row sums of distances to the members of every cluster (silhouette_score, cnmf.py:923):
// one block per row; per-warp cluster bins in shared memory, folded in warp order (deterministic)
__global__ void __launch_bounds__(256)
cluster_dist_sums_kernel(const float* __restrict__ D, int R, const int32_t* __restrict__ labels, int K,
                         double* __restrict__ out /* R x K */) {
  extern __shared__ double bins[];        // 8 warps x K
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < 8 * K; i += blockDim.x) bins[i] = 0.0;
  __syncthreads();
  const float* row = D + (long long)blockIdx.x * R;
  // each warp owns a contiguous slice of columns and walks it in order, lane by lane
  const int per = (R + 7) / 8;
  const int j0 = warp * per, j1 = min(R, j0 + per);
  for (int jb = j0; jb < j1; jb += 32) {
    const int j = jb + lane;
    const double v = (j < j1) ? (double)row[j] : 0.0;
    const int lab = (j < j1) ? labels[j] : -1;
    for (int l = 0; l < 32; ++l) {        // serialise the lanes: fixed summation order
      const double vl = __shfl_sync(0xffffffffu, v, l);
      const int ll = __shfl_sync(0xffffffffu, lab, l);
      if (lane == 0 && ll >= 0) bins[warp * K + ll] += vl;
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < K; c += blockDim.x) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += bins[w * K + c];
    out[(long long)blockIdx.x * K + c] = s;
  }
}

__global__ void col_stats_dev_kernel(const float* __restrict__ X, int rows, int cols, int ld, double* __restrict__ sum,
                                    double* __restrict__ sq) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  double s = 0.0, q = 0.0;
  for (int r = 0; r < rows; ++r) {           // fixed order: deterministic
    const double v = X[(long long)r * ld + c];
    s += v;
    q += v * v;
  }
  sum[c] = s;
  sq[c] = q;
}

__global__ void gather_rows_idx_kernel(const float* __restrict__ src, int ld_src, const int32_t* __restrict__ idx,
                                       int G, float* __restrict__ dst, int ld_dst) {
  const float* s = src + (long long)idx[blockIdx.x] * ld_src;
  float* d = dst + (long long)blockIdx.x * ld_dst;
  for (int g = threadIdx.x; g < G; g += blockDim.x) d[g] = s[g];
}

}  // namespace

extern "C" {

int cnmf_l2_normalize_rows(cnmf_handle_t h, float* S, int R, int G, int ld, void* stream) {
  CNMF_REQUIRE(h && S && R > 0 && G > 0 && ld >= G, "l2_normalize_rows: bad arguments");
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  l2_normalize_kernel<<<R, 256, 0, as_stream(stream)>>>(S, R, G, ld);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 1;
  return 0;
}

int cnmf_local_density(cnmf_handle_t h, const float* S, int R, int G, int ld, int n_neighbors, float* density_dev,
                       float* D_dev, void* stream) {
  CNMF_REQUIRE(h && S && density_dev && R > 0 && G > 0 && ld >= G, "local_density: bad arguments");
  CNMF_REQUIRE(n_neighbors >= 1 && n_neighbors + 1 <= R, "local_density: need 1 <= n_neighbors < R");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  float* D = D_dev ? D_dev : static_cast<float*>(h->dev_buf("consensus.D", (size_t)R * R * 4));
  if (!D) return -2;
  dim3 grid((R + 63) / 64, (R + 63) / 64);
  pair_dist_kernel<true, true><<<grid, 256, 0, s>>>(S, R, ld, S, R, ld, G, D, R);
  CNMF_CUDA_CHECK(cudaGetLastError());
  knn_density_kernel<<<R, 256, 0, s>>>(D, R, R, n_neighbors + 1, n_neighbors, density_dev);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 2;
  return 0;
}

int cnmf_col_stats_dev(cnmf_handle_t h, const float* S, int R, int G, int ld, double* mean_host, double* var_host,
                       void* stream) {
  CNMF_REQUIRE(h && S && mean_host && var_host && R > 0 && G > 0, "col_stats_dev: bad arguments");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  double* buf = static_cast<double*>(h->dev_buf("consensus.colstats", sizeof(double) * 2 * G));
  if (!buf) return -2;
  col_stats_dev_kernel<<<(G + 127) / 128, 128, 0, s>>>(S, R, G, ld, buf, buf + G);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 1;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(mean_host, buf, sizeof(double) * G, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaMemcpyAsync(var_host, buf + G, sizeof(double) * G, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  for (int c = 0; c < G; ++c) {
    const double m = mean_host[c] / R;
    mean_host[c] = m;
    var_host[c] = std::max(var_host[c] / R - m * m, 0.0);
  }
  return 0;
}

int cnmf_cluster_dist_sums(cnmf_handle_t h, const float* S, int R, int G, int ld, const int32_t* labels_dev, int K,
                           double* sums_host, void* stream) {
  CNMF_REQUIRE(h && S && labels_dev && sums_host && R > 0 && K >= 1 && K <= 512, "cluster_dist_sums: bad arguments");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  float* D = static_cast<float*>(h->dev_buf("consensus.D", (size_t)R * R * 4));
  double* out = static_cast<double*>(h->dev_buf("consensus.dsums", sizeof(double) * (size_t)R * K));
  if (!D || !out) return -2;
  dim3 grid((R + 63) / 64, (R + 63) / 64);
  pair_dist_kernel<true, true><<<grid, 256, 0, s>>>(S, R, ld, S, R, ld, G, D, R);
  cluster_dist_sums_kernel<<<R, 256, sizeof(double) * 8 * K, s>>>(D, R, labels_dev, K, out);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 2;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(sums_host, out, sizeof(double) * (size_t)R * K, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  return 0;
}

int cnmf_gather_rows(cnmf_handle_t h, const float* src_dev, int ld_src, const int32_t* idx_host, int n, int G,
                     float* dst_dev, int ld_dst, void* stream) {
  CNMF_REQUIRE(h && src_dev && idx_host && dst_dev && n > 0 && G > 0, "gather_rows: bad arguments");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  int32_t* d_idx = static_cast<int32_t*>(h->dev_buf("consensus.idx", sizeof(int32_t) * n));
  if (!d_idx) return -2;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(d_idx, idx_host, sizeof(int32_t) * n, cudaMemcpyHostToDevice, s));
  gather_rows_idx_kernel<<<n, 256, 0, s>>>(src_dev, ld_src, d_idx, G, dst_dev, ld_dst);
  CNMF_CUDA_CHECK(cudaGetLastError());
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  h->launches += 1;
  return 0;
}

int cnmf_sq_dists_to_rows(cnmf_handle_t h, const float* S, int R, int G, int ld, const int32_t* idx_host, int n_c,
                          float* out_host, void* stream) {
  CNMF_REQUIRE(h && S && idx_host && out_host && n_c > 0 && R > 0, "sq_dists_to_rows: bad arguments");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  float* C = static_cast<float*>(h->dev_buf("consensus.cand", (size_t)n_c * ld * 4));
  float* out = static_cast<float*>(h->dev_buf("consensus.cand_out", (size_t)n_c * R * 4));
  int32_t* d_idx = static_cast<int32_t*>(h->dev_buf("consensus.idx", sizeof(int32_t) * std::max(n_c, 1)));
  if (!C || !out || !d_idx) return -2;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(d_idx, idx_host, sizeof(int32_t) * n_c, cudaMemcpyHostToDevice, s));
  if (n_c <= 8 && ld % 4 == 0) {
    const int blocks = (R * 32 + 255) / 256;
    if (n_c <= 2) cand_dist_kernel<2><<<blocks, 256, 0, s>>>(S, R, G, ld, d_idx, n_c, out);
    else if (n_c <= 4) cand_dist_kernel<4><<<blocks, 256, 0, s>>>(S, R, G, ld, d_idx, n_c, out);
    else cand_dist_kernel<8><<<blocks, 256, 0, s>>>(S, R, G, ld, d_idx, n_c, out);
  } else {
    gather_rows_idx_kernel<<<n_c, 256, 0, s>>>(S, ld, d_idx, G, C, ld);
    dim3 grid((R + 63) / 64, (n_c + 63) / 64);
    pair_dist_kernel<false, false><<<grid, 256, 0, s>>>(C, n_c, ld, S, R, ld, G, out, R);
  }
  CNMF_CUDA_CHECK(cudaGetLastError());
  CNMF_CUDA_CHECK(cudaMemcpyAsync(out_host, out, (size_t)n_c * R * 4, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  h->launches += 2;
  return 0;
}

int cnmf_kmeans_assign(cnmf_handle_t h, const float* S, int R, int G, int ld, const float* centers_host, int K,
                       int32_t* labels_dev, double* sums_host, int32_t* counts_host, float* mind_dev,
                       int32_t* n_changed_host, double* inertia_host, void* stream) {
  CNMF_REQUIRE(h && S && centers_host && labels_dev && mind_dev && K >= 1 && K <= 1024 && R > 0,
               "kmeans_assign: bad arguments");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  float* C = static_cast<float*>(h->dev_buf("kmeans.C", (size_t)K * G * 4));
  int32_t* cnt = static_cast<int32_t*>(h->dev_buf("kmeans.cnt", sizeof(int32_t) * (K + 2)));
  int32_t* order = static_cast<int32_t*>(h->dev_buf("kmeans.order", sizeof(int32_t) * (size_t)K * R));
  double* sums = static_cast<double*>(h->dev_buf("kmeans.sums", sizeof(double) * ((size_t)K * G + 1)));
  if (!C || !cnt || !order || !sums) return -2;
  int* n_changed = cnt + K;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(C, centers_host, (size_t)K * G * 4, cudaMemcpyHostToDevice, s));
  CNMF_CUDA_CHECK(cudaMemsetAsync(n_changed, 0, sizeof(int), s));
  kmeans_assign_kernel<<<(R * 32 + 255) / 256, 256, 0, s>>>(S, R, G, ld, C, K, G, labels_dev, mind_dev, n_changed);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 1;
  if (sums_host) {
    members_kernel<<<1, 1024, 0, s>>>(labels_dev, R, K, cnt, order);
    dim3 grid((G + 127) / 128, K);
    cluster_sums_kernel<<<grid, 128, 0, s>>>(S, G, ld, cnt, order, R, sums);
    CNMF_CUDA_CHECK(cudaGetLastError());
    h->launches += 2;
    CNMF_CUDA_CHECK(cudaMemcpyAsync(sums_host, sums, sizeof(double) * (size_t)K * G, cudaMemcpyDeviceToHost, s));
    if (counts_host) CNMF_CUDA_CHECK(cudaMemcpyAsync(counts_host, cnt, sizeof(int32_t) * K, cudaMemcpyDeviceToHost, s));
  }
  if (inertia_host) {
    sum_float_kernel<<<1, 1024, 0, s>>>(mind_dev, R, sums + (size_t)K * G);
    CNMF_CUDA_CHECK(cudaGetLastError());
    h->launches += 1;
    CNMF_CUDA_CHECK(cudaMemcpyAsync(inertia_host, sums + (size_t)K * G, sizeof(double), cudaMemcpyDeviceToHost, s));
  }
  if (n_changed_host) CNMF_CUDA_CHECK(cudaMemcpyAsync(n_changed_host, n_changed, sizeof(int), cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  return 0;
}

int cnmf_kmeans_step(cnmf_handle_t h, const float* S, int R, int G, int ld, int K, const float* C32_cur,
                     const double* C64_cur, double* C64_new, float* C32_new, int32_t* labels_dev, float* mind_dev,
                     double* sums_dev, int32_t* counts_dev, int32_t* n_changed_host, int32_t* any_empty_host,
                     double* shift_host, void* stream) {
  CNMF_REQUIRE(h && S && C32_cur && C64_cur && C64_new && C32_new && labels_dev && mind_dev && sums_dev && counts_dev &&
                   n_changed_host && any_empty_host && shift_host && K >= 1 && K <= 1024 && R > 0,
               "kmeans_step: bad arguments");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  int32_t* order = static_cast<int32_t*>(h->dev_buf("kmeans.order", sizeof(int32_t) * (size_t)K * R));
  int32_t* flags = static_cast<int32_t*>(h->dev_buf("kmeans.flags", sizeof(int32_t) * 2));
  double* shift_part = static_cast<double*>(h->dev_buf("kmeans.shift", sizeof(double) * K));
  struct HostOut { int32_t flags[2]; double shift[1024]; };
  HostOut* ho = static_cast<HostOut*>(h->host_buf("kmeans.step_out", sizeof(HostOut)));
  if (!order || !flags || !shift_part || !ho) return -2;
  CNMF_CUDA_CHECK(cudaMemsetAsync(flags, 0, sizeof(int32_t) * 2, s));
  kmeans_assign_kernel<<<(R * 32 + 255) / 256, 256, 0, s>>>(S, R, G, ld, C32_cur, K, G, labels_dev, mind_dev, flags);
  members_kernel<<<1, 1024, 0, s>>>(labels_dev, R, K, counts_dev, order);
  dim3 grid((G + 127) / 128, K);
  cluster_sums_kernel<<<grid, 128, 0, s>>>(S, G, ld, counts_dev, order, R, sums_dev);
  centre_update_kernel<<<K, 256, 0, s>>>(sums_dev, counts_dev, G, C64_cur, C64_new, C32_new, shift_part, flags + 1);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 4;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(ho->flags, flags, sizeof(int32_t) * 2, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaMemcpyAsync(ho->shift, shift_part, sizeof(double) * K, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  *n_changed_host = ho->flags[0];
  *any_empty_host = ho->flags[1];
  double tot = 0.0;
  for (int j = 0; j < K; ++j) tot += ho->shift[j];      // fixed order
  *shift_host = tot;
  return 0;
}

int cnmf_cluster_median(cnmf_handle_t h, const float* S, int R, int G, int ld, const int32_t* labels_dev, int K,
                        float* M_dev, int ldm, void* stream) {
  CNMF_REQUIRE(h && S && labels_dev && M_dev && K >= 1 && K <= 1024 && R > 0 && ldm >= G, "cluster_median: bad arguments");
  cudaStream_t s = as_stream(stream);
  CNMF_CUDA_CHECK(cudaSetDevice(h->device));
  int32_t* cnt = static_cast<int32_t*>(h->dev_buf("kmeans.cnt", sizeof(int32_t) * (K + 2)));
  int32_t* order = static_cast<int32_t*>(h->dev_buf("kmeans.order", sizeof(int32_t) * (size_t)K * R));
  if (!cnt || !order) return -2;
  members_kernel<<<1, 1024, 0, s>>>(labels_dev, R, K, cnt, order);
  dim3 grid((G + 127) / 128, K);
  cluster_median_kernel<<<grid, 128, 0, s>>>(S, G, ld, cnt, order, R, M_dev, ldm);
  row_normalize_sum_kernel<<<K, 256, 0, s>>>(M_dev, G, ldm);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 3;
  return 0;
}

}  // extern "C"
