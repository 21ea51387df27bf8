// Batched multiplicative-update NMF for the generalized Kullback-Leibler (beta = 1) and Itakura-Saito
// (beta = 0) losses -- the `--beta-loss kullback-leibler | itakura-saito` branch behind the same seam
// (cnmf.py:629-631 keeps solver 'mu' for them; sklearn/decomposition/_nmf.py:551-608, 637-694, 726-888).
//
// Unlike the Frobenius path these updates are NOT GEMM-shaped: the numerator
//     num[i, c] = sum_j  X[i, j] * (WH)[i, j]^(beta-2) * H[c, j],      (WH)[i, j] = sum_c W[i, c] H[c, j]
// needs the N x G x K elementwise quotient of every restart, which sklearn materialises (N x G doubles per
// restart per half-iteration).  Here the quotient never exists in memory: a thread owns one or two items
// (cells for the W half, genes for the H half) of one restart, keeps their K factor values and K accumulators in
// registers, and walks the contraction dimension with the other factor staged tile by tile in shared memory
// (one LDS.128 feeds 4 components x CT items).  The data matrix is read in the orientation in which the
// thread's items are contiguous (X^T for the W half, X for the H half): fully coalesced, and with the slot index
// fastest in the grid all restarts of a batch read the same slab together, so X comes from L2, not HBM.
// Bound: FP32 issue (2 K FFMA + one division per (item, j, restart)); see DESIGN.md section 4.4.
//
// Both halves are the same kernel with the roles swapped ("components x items" packing, nmf_kernels.cuh).
// sklearn's asymmetries are kept: KL denominators are the other factor's row sums, where only the H half
// replaces a zero sum by 1 (_nmf.py:669); values below float64 eps are flushed to zero after the H half when
// beta <= 1 and after the W half when beta < 1 (_nmf.py:845-846, 863-865); gamma = 1/(2-beta) for beta < 1.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "engine.h"
#include "nmf_kernels.cuh"

namespace cnmf {

namespace {

constexpr int BT = 128;     // threads per block
constexpr int IPB = 256;    // items per block
constexpr int CC = 128;     // contraction rows staged per shared-memory tile
constexpr int UJ = 4;       // rows per unrolled group (loads of a group are issued together)
constexpr float EPS32 = 1.1920929e-07f;          // sklearn EPSILON = float32 eps (_nmf.py:32)
constexpr float EPS64F = 2.220446049250313e-16f;  // np.finfo(float64).eps, the clipping threshold

struct BetaSide {
  const float* D;        // data, n_contract x ldD, item index contiguous
  long long ldD;
  int n_items, n_contract;
  float* Fown;           // SK x ld_own, updated in place
  int ld_own;
  const float* Foth;     // SK x ld_oth
  int ld_oth;
  const double* oth_sum; // [SK] row sums of Foth (KL denominators)
  float l1, l2;
  int zero_sum_to_one;   // H half of KL: W_sum == 0 -> 1
  int clip;              // flush values < float64 eps to zero after the update
};

// rcp_nr / div_nr (branch-free fp32 reciprocal / quotient) live in common.cuh

template <int KP>
__device__ __forceinline__ void load_row(const float* p, float (&h)[KP]) {
#pragma unroll
  for (int q = 0; q < KP / 4; ++q) {
    const float4 v = *reinterpret_cast<const float4*>(p + 4 * q);
    h[4 * q] = v.x; h[4 * q + 1] = v.y; h[4 * q + 2] = v.z; h[4 * q + 3] = v.w;
  }
}

// stage rows [j0, j0 + CC) of the other factor, transposed: sm[jj * KP + c]; zero beyond k / n_contract
template <int KP>
__device__ __forceinline__ void stage_tile(const BetaSide& sd, int row0, int k, int j0, float* sm) {
  for (int idx = threadIdx.x; idx < KP * CC; idx += BT) {
    const int c = idx / CC, jj = idx - c * CC;
    const int j = j0 + jj;
    float v = 0.0f;
    if (c < k && j < sd.n_contract) v = sd.Foth[(long long)(row0 + c) * sd.ld_oth + j];
    sm[jj * KP + c] = v;
  }
}

template <int KP, int CT, bool IS>
__device__ __forceinline__ void beta_update_body(const BetaSide& sd, int row0, int k, int item_base, float* sm) {
  constexpr int DK = IS ? KP : 1;
  const int tid = threadIdx.x;
  for (int pass = 0; pass < IPB / (BT * CT); ++pass) {
    int item[CT];
    bool valid[CT];
    const float* Dcol[CT];
    float w[CT][KP], acc[CT][KP], dac[CT][DK];
#pragma unroll
    for (int ct = 0; ct < CT; ++ct) {
      item[ct] = item_base + (pass * CT + ct) * BT + tid;
      valid[ct] = item[ct] < sd.n_items;
      const int ic = valid[ct] ? item[ct] : 0;
      Dcol[ct] = sd.D + ic;
#pragma unroll
      for (int c = 0; c < KP; ++c) {
        w[ct][c] = (valid[ct] && c < k) ? sd.Fown[(long long)(row0 + c) * sd.ld_own + ic] : 0.0f;
        acc[ct][c] = 0.0f;
      }
#pragma unroll
      for (int c = 0; c < DK; ++c) dac[ct][c] = 0.0f;
    }
    for (int j0 = 0; j0 < sd.n_contract; j0 += CC) {
      __syncthreads();
      stage_tile<KP>(sd, row0, k, j0, sm);
      __syncthreads();
      const int jn = min(CC, sd.n_contract - j0);
      float part[CT][KP], dpart[CT][DK];       // per-tile partial sums: keeps the fp32 chains short
#pragma unroll
      for (int ct = 0; ct < CT; ++ct) {
#pragma unroll
        for (int c = 0; c < KP; ++c) part[ct][c] = 0.0f;
#pragma unroll
        for (int c = 0; c < DK; ++c) dpart[ct][c] = 0.0f;
      }
      for (int jj = 0; jj < jn; jj += UJ) {
        float x[UJ][CT];
#pragma unroll
        for (int u = 0; u < UJ; ++u) {
          // rows past the end re-read the last row; their staged factor row is zero, so they contribute 0
          const long long row = min(j0 + jj + u, sd.n_contract - 1);
#pragma unroll
          for (int ct = 0; ct < CT; ++ct) x[u][ct] = __ldg(Dcol[ct] + row * sd.ldD);
        }
#pragma unroll
        for (int u = 0; u < UJ; ++u) {
          float h[KP];
          load_row<KP>(sm + (jj + u) * KP, h);
#pragma unroll
          for (int ct = 0; ct < CT; ++ct) {
            float wh = 0.0f;
#pragma unroll
            for (int c = 0; c < KP; ++c) wh = fmaf(w[ct][c], h[c], wh);
            wh = fmaxf(wh, EPS32);                         // _nmf.py:566-567 / :653-654
            if (!IS) {
              const float q = div_nr(x[u][ct], wh);        // X / WH                      (:569-570)
#pragma unroll
              for (int c = 0; c < KP; ++c) part[ct][c] = fmaf(q, h[c], part[ct][c]);
            } else {
              const float inv = rcp_nr(wh);                // WH^-1, then squared, times X (:571-577)
              const float q = x[u][ct] * (inv * inv);
#pragma unroll
              for (int c = 0; c < KP; ++c) {
                part[ct][c] = fmaf(q, h[c], part[ct][c]);
                dpart[ct][c < DK ? c : 0] = fmaf(inv, h[c], dpart[ct][c < DK ? c : 0]);   // (WH^(beta-1)) H^T (:600-602)
              }
            }
          }
        }
      }
#pragma unroll
      for (int ct = 0; ct < CT; ++ct) {
#pragma unroll
        for (int c = 0; c < KP; ++c) acc[ct][c] += part[ct][c];
#pragma unroll
        for (int c = 0; c < DK; ++c) dac[ct][c] += dpart[ct][c];
      }
    }
    // ---- epilogue: denominator, regularisation, zero guard, gamma, clip (_nmf.py:610-624 / :696-721)
#pragma unroll
    for (int ct = 0; ct < CT; ++ct) {
      if (!valid[ct]) continue;
#pragma unroll
      for (int c = 0; c < KP; ++c) {
        if (c >= k) break;
        float den;
        if (!IS) {
          den = (float)sd.oth_sum[row0 + c];
          if (sd.zero_sum_to_one && den == 0.0f) den = 1.0f;
        } else {
          den = dac[ct][c < DK ? c : 0];
        }
        if (sd.l1 > 0.0f) den += sd.l1;
        if (sd.l2 > 0.0f) den += sd.l2 * w[ct][c];
        if (den == 0.0f) den = EPS32;
        float delta = acc[ct][c] / den;
        if (IS) delta = sqrtf(delta);                      // gamma = 1 / (2 - beta) = 1/2
        float v = w[ct][c] * delta;
        if (sd.clip && v < EPS64F) v = 0.0f;
        sd.Fown[(long long)(row0 + c) * sd.ld_own + item[ct]] = v;
      }
    }
  }
}

// Per-restart dispatch on K rounded up to 4.  KPMAX (8 / 16 / 32, from the largest K of the batch) bounds which
// bodies are instantiated, because the kernel's register allocation is the maximum over all of them.
#define CNMF_BETA_SWITCH(FN, CT2, TP, ...)                                          \
  {                                                                                 \
    const int q4 = (k + 3) >> 2;                                                    \
    if (q4 <= 1) FN<4, CT2, TP>(__VA_ARGS__);                                       \
    else if (q4 == 2) FN<8, CT2, TP>(__VA_ARGS__);                                  \
    else if constexpr (KPMAX > 8) {                                                 \
      if (q4 == 3) FN<12, CT2, TP>(__VA_ARGS__);                                    \
      else if (q4 == 4) FN<16, CT2, TP>(__VA_ARGS__);                               \
      else if constexpr (KPMAX > 16) {                                              \
        if (q4 == 5) FN<20, 1, TP>(__VA_ARGS__);                                    \
        else if (q4 == 6) FN<24, 1, TP>(__VA_ARGS__);                               \
        else if (q4 == 7) FN<28, 1, TP>(__VA_ARGS__);                               \
        else FN<32, 1, TP>(__VA_ARGS__);                                            \
      }                                                                             \
    }                                                                               \
  }

template <bool IS, int KPMAX>
__global__ void __launch_bounds__(BT) beta_update_kernel(BetaSide sd, BatchMeta b) {
  __shared__ __align__(16) float sm[CC * KPMAX];
  const int slot = blockIdx.x % b.R, chunk = blockIdx.x / b.R;
  if (b.done[b.rid[slot]]) return;
  const int k = b.k[slot], row0 = b.off[slot];
  CNMF_BETA_SWITCH(beta_update_body, (IS ? 1 : 2), IS, sd, row0, k, chunk * IPB, sm)
}

// ---- divergence (_nmf.py:77-175, dense branch): per block, fp64 partials {sum of terms, sum of X over X > EPS}
// MODE 0: Kullback-Leibler, 1: Itakura-Saito, 2: plain squared residual sum (x - wh)^2 over every entry (the
// Frobenius prediction error the consensus statistics report whatever the fitted loss, cnmf.py:926-930)
enum { ERR_KL = 0, ERR_IS = 1, ERR_FROB = 2 };
template <int KP, int CT, int MODE>
__device__ __forceinline__ void beta_error_body(const BetaSide& sd, int row0, int k, int item_base, float* sm,
                                                double& t_out, double& sx_out) {
  const int tid = threadIdx.x;
  double t_acc = 0.0, sx_acc = 0.0;
  for (int pass = 0; pass < IPB / (BT * CT); ++pass) {
    bool valid[CT];
    const float* Dcol[CT];
    float w[CT][KP];
#pragma unroll
    for (int ct = 0; ct < CT; ++ct) {
      const int item = item_base + (pass * CT + ct) * BT + tid;
      valid[ct] = item < sd.n_items;
      const int ic = valid[ct] ? item : 0;
      Dcol[ct] = sd.D + ic;
#pragma unroll
      for (int c = 0; c < KP; ++c) w[ct][c] = (valid[ct] && c < k) ? sd.Fown[(long long)(row0 + c) * sd.ld_own + ic] : 0.0f;
    }
    for (int j0 = 0; j0 < sd.n_contract; j0 += CC) {
      __syncthreads();
      stage_tile<KP>(sd, row0, k, j0, sm);
      __syncthreads();
      const int jn = min(CC, sd.n_contract - j0);
      float t = 0.0f, sx = 0.0f;
      for (int jj = 0; jj < jn; jj += UJ) {
        float x[UJ][CT];
#pragma unroll
        for (int u = 0; u < UJ; ++u) {
          const bool in = j0 + jj + u < sd.n_contract;
          const long long row = min(j0 + jj + u, sd.n_contract - 1);
#pragma unroll
          for (int ct = 0; ct < CT; ++ct) x[u][ct] = (in && valid[ct]) ? __ldg(Dcol[ct] + row * sd.ldD) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < UJ; ++u) {
          float h[KP];
          load_row<KP>(sm + (jj + u) * KP, h);
#pragma unroll
          for (int ct = 0; ct < CT; ++ct) {
            const float xv = x[u][ct];
            if (MODE == ERR_FROB) {
              float wh = 0.0f;
#pragma unroll
              for (int c = 0; c < KP; ++c) wh = fmaf(w[ct][c], h[c], wh);
              const float d = xv - wh;                     // padded rows / items: x = 0 and w or h = 0 -> d = 0
              t = fmaf(d, d, t);
            } else if (xv > EPS32) {                       // zeros of X are dropped (:140-142)
              float wh = 0.0f;
#pragma unroll
              for (int c = 0; c < KP; ++c) wh = fmaf(w[ct][c], h[c], wh);
              wh = fmaxf(wh, EPS32);                       // :145
              const float div = div_nr(xv, wh);
              if (MODE == ERR_KL) {
                t = fmaf(xv, logf(div), t);                // sum X log(X / WH)          (:152-153)
                sx += xv;
              } else {
                t += div - logf(div);                      // sum div - sum log div      (:160-161)
              }
            }
          }
        }
      }
      t_acc += (double)t;
      sx_acc += (double)sx;
    }
  }
  t_out = t_acc;
  sx_out = sx_acc;
}

template <int MODE, int KPMAX>
__global__ void __launch_bounds__(BT) beta_error_kernel(BetaSide sd, BatchMeta b, double* __restrict__ part, int chunks) {
  __shared__ __align__(16) float sm[CC * KPMAX];
  __shared__ double red[2][BT / 32];
  const int slot = blockIdx.x % b.R, chunk = blockIdx.x / b.R;
  const int rid = b.rid[slot];
  if (b.done[rid]) return;
  const int k = b.k[slot], row0 = b.off[slot];
  double t = 0.0, sx = 0.0;
  CNMF_BETA_SWITCH(beta_error_body, 2, MODE, sd, row0, k, chunk * IPB, sm, t, sx)
  t = warp_sum(t);
  sx = warp_sum(sx);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { red[0][warp] = t; red[1][warp] = sx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, c = 0.0;
    for (int i = 0; i < BT / 32; ++i) { a += red[0][i]; c += red[1][i]; }
    part[((long long)rid * chunks + chunk) * 2] = a;
    part[((long long)rid * chunks + chunk) * 2 + 1] = c;
  }
}

// out[row] = sum_j F[row, j] in fp64, one block per packed row (fixed reduction order)
__global__ void __launch_bounds__(256) row_sum_kernel(const float* __restrict__ F, int n, int ld, double* __restrict__ out) {
  __shared__ double red[8];
  const float* p = F + (long long)blockIdx.x * ld;
  double a = 0.0;
  for (int j = threadIdx.x; j < n; j += 256) a += (double)p[j];
  a = warp_sum(a);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[i];
    out[blockIdx.x] = t;
  }
}

// err = sqrt(2 max(res, 0)) (_nmf.py:170-175); stopping rule of _fit_multiplicative_update (:867-879)
__global__ void beta_check_kernel(ConvState st, const double* __restrict__ part, int chunks, const double* __restrict__ sumR,
                                  const double* __restrict__ sumC, double n_elems, int is, BatchMeta b, int it, double tol,
                                  int max_iter) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= b.R) return;
  const int r = b.rid[slot];
  if (st.done[r]) return;
  double t = 0.0, sx = 0.0;
  for (int c = 0; c < chunks; ++c) {
    t += part[((long long)r * chunks + c) * 2];
    sx += part[((long long)r * chunks + c) * 2 + 1];
  }
  if (is == ERR_FROB) {                                    // ||X - WH||_F, reported only
    st.last[r] = sqrt(fmax(t, 0.0));
    return;
  }
  double res;
  if (is == ERR_KL) {
    double swh = 0.0;                                      // sum(WH) = <sum_i W, sum_j H>          (:150)
    for (int c = 0; c < b.k[slot]; ++c) swh += sumR[b.off[slot] + c] * sumC[b.off[slot] + c];
    res = t + swh - sx;                                    // (:153-155)
  } else {
    res = t - n_elems;                                     // (:161)
  }
  const double err = sqrt(2.0 * fmax(res, 0.0));
  st.last[r] = err;
  if (it == 0) {
    st.err0[r] = err;
    st.prev[r] = err;
    return;
  }
  if ((st.prev[r] - err) / st.err0[r] < tol) {
    st.done[r] = 1;
    st.n_iter[r] = it;
  } else {
    st.prev[r] = err;
    if (it >= max_iter) {
      st.done[r] = 1;
      st.n_iter[r] = it;
    }
  }
}

__global__ void __launch_bounds__(256) matrix_min_kernel(const float* __restrict__ X, int rows, int cols, int ld,
                                                         float* __restrict__ out) {
  float m = INFINITY;
  for (long long r = blockIdx.x; r < rows; r += gridDim.x)
    for (int c = threadIdx.x; c < cols; c += 256) m = fminf(m, X[r * ld + c]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; ++i) m = fminf(m, red[i]);
    out[blockIdx.x] = fminf(m, red[0]);
  }
}

}  // namespace

int matrix_min(cnmf_handle_s* h, const float* X, int rows, int cols, int ld, float* out_host, cudaStream_t s) {
  const int blocks = std::min(rows, 148 * 8);
  float* d = static_cast<float*>(h->dev_buf("beta.min", sizeof(float) * blocks));
  if (!d) return -2;
  matrix_min_kernel<<<blocks, 256, 0, s>>>(X, rows, cols, ld, d);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 1;
  std::vector<float> part(blocks);
  CNMF_CUDA_CHECK(cudaMemcpyAsync(part.data(), d, sizeof(float) * blocks, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  *out_host = *std::min_element(part.begin(), part.end());
  return 0;
}

int solve_batched_beta(cnmf_handle_s* h, const DataView& v, SolveIO& io, const cnmf_nmf_params& p, cudaStream_t s) {
  const int R = io.R;
  CNMF_REQUIRE(R > 0 && (int)io.ks.size() == R, "solve: bad restart list");
  CNMF_REQUIRE(p.solver == CNMF_SOLVER_MU, "beta_loss other than frobenius needs solver 'mu' (sklearn _nmf.py:1195-1199)");
  CNMF_REQUIRE(p.beta_loss == CNMF_LOSS_KULLBACK_LEIBLER || p.beta_loss == CNMF_LOSS_ITAKURA_SAITO, "solve: unknown beta_loss");
  CNMF_REQUIRE(p.max_iter >= 1, "solve: max_iter must be >= 1");
  CNMF_REQUIRE(v.B_rows.full && v.B_cols.full, "solve: the beta-divergence kernels need X and X^T in full fp32");
  const bool is = p.beta_loss == CNMF_LOSS_ITAKURA_SAITO;

  std::vector<int> hm(3 * R);
  int SK = 0, kpmax = 0;
  for (int r = 0; r < R; ++r) {
    kpmax = std::max(kpmax, io.ks[r]);
    CNMF_REQUIRE(io.ks[r] >= 1 && io.ks[r] <= KMAX, "solve: n_components must be in [1, 32] on the CUDA path");
    hm[r] = SK;
    hm[R + r] = io.ks[r];
    hm[2 * R + r] = r;
    SK += io.ks[r];
  }
  const int chunks_r = (v.n_r + IPB - 1) / IPB, chunks_c = (v.n_c + IPB - 1) / IPB;
  int* d_meta = static_cast<int*>(h->dev_buf("solve.meta", sizeof(int) * 8 * R));
  double* d_state = static_cast<double*>(h->dev_buf("solve.state", sizeof(double) * 8 * R));
  double* d_sums = static_cast<double*>(h->dev_buf("beta.sums", sizeof(double) * 2 * SK));
  double* d_part = static_cast<double*>(h->dev_buf("beta.err_part", sizeof(double) * 2 * (size_t)R * chunks_r));
  if (!d_meta || !d_state || !d_sums || !d_part) return -2;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(d_meta, hm.data(), sizeof(int) * 3 * R, cudaMemcpyHostToDevice, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));      // hm is a stack-lifetime vector
  int* d_done = d_meta + 3 * R;
  int* d_niter = d_meta + 4 * R;
  CNMF_CUDA_CHECK(cudaMemsetAsync(d_done, 0, sizeof(int) * 2 * R, s));
  CNMF_CUDA_CHECK(cudaMemsetAsync(d_state, 0, sizeof(double) * 8 * R, s));
  ConvState st{d_state, d_state + R, d_state + 2 * R, d_done, d_niter};
  BatchMeta bm{d_meta, d_meta + R, d_meta + 2 * R, d_done, R, 32};
  double* d_sumR = d_sums;
  double* d_sumC = d_sums + SK;

  // W half: items = rows of the view (cells), contraction over its columns; data read as X^T (n_c x ld_r)
  BetaSide sideR{v.B_cols.full, v.B_cols.ld, v.n_r, v.n_c, io.Fr, v.ld_r, io.Fc, v.ld_c, d_sumC,
                 (float)p.l1_reg_W, (float)p.l2_reg_W, 0, is ? 1 : 0};
  // H half: items = columns (genes), contraction over rows; data read as X (n_r x ld_c)
  BetaSide sideC{v.B_rows.full, v.B_rows.ld, v.n_c, v.n_r, io.Fc, v.ld_c, io.Fr, v.ld_r, d_sumR,
                 (float)p.l1_reg_H, (float)p.l2_reg_H, 1, 1};

  auto row_sums = [&](const float* F, int n, int ld, double* out) -> int {
    row_sum_kernel<<<SK, 256, 0, s>>>(F, n, ld, out);
    CNMF_CUDA_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
  };
  auto update = [&](const BetaSide& sd, int chunks) -> int {
#define CNMF_LAUNCH_UPD(ISV, KPM) beta_update_kernel<ISV, KPM><<<R * chunks, BT, 0, s>>>(sd, bm)
    if (is) { if (kpmax <= 8) CNMF_LAUNCH_UPD(true, 8); else if (kpmax <= 16) CNMF_LAUNCH_UPD(true, 16); else CNMF_LAUNCH_UPD(true, 32); }
    else { if (kpmax <= 8) CNMF_LAUNCH_UPD(false, 8); else if (kpmax <= 16) CNMF_LAUNCH_UPD(false, 16); else CNMF_LAUNCH_UPD(false, 32); }
#undef CNMF_LAUNCH_UPD
    CNMF_CUDA_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
  };
  auto error_pass = [&](int mode, const BatchMeta& m) -> int {
#define CNMF_LAUNCH_ERR(MD, KPM) beta_error_kernel<MD, KPM><<<R * chunks_r, BT, 0, s>>>(sideR, m, d_part, chunks_r)
#define CNMF_LAUNCH_ERR_K(MD) { if (kpmax <= 8) CNMF_LAUNCH_ERR(MD, 8); else if (kpmax <= 16) CNMF_LAUNCH_ERR(MD, 16); else CNMF_LAUNCH_ERR(MD, 32); }
    if (mode == ERR_KL) CNMF_LAUNCH_ERR_K(ERR_KL)
    else if (mode == ERR_IS) CNMF_LAUNCH_ERR_K(ERR_IS)
    else CNMF_LAUNCH_ERR_K(ERR_FROB)
#undef CNMF_LAUNCH_ERR_K
#undef CNMF_LAUNCH_ERR
    CNMF_CUDA_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
  };
  auto check = [&](int it, double tol_eff) -> int {
    if (!is) {
      CNMF_TRY(row_sums(io.Fr, v.n_r, v.ld_r, d_sumR));
      if (it == 0 || !io.update_cols) CNMF_TRY(row_sums(io.Fc, v.n_c, v.ld_c, d_sumC));
    }
    CNMF_TRY(error_pass(is ? ERR_IS : ERR_KL, bm));
    beta_check_kernel<<<(R + 127) / 128, 128, 0, s>>>(st, d_part, chunks_r, d_sumR, d_sumC, (double)v.n_r * (double)v.n_c,
                                                     is ? ERR_IS : ERR_KL, bm, it, tol_eff, p.max_iter);
    CNMF_CUDA_CHECK(cudaGetLastError());
    h->launches += 1;
    return 0;
  };

  CNMF_TRY(check(0, p.tol));                       // error_at_init (:822); also leaves sum(H) rows for the first W half
  std::vector<int> h_done(R, 0);
  for (int it = 1; it <= p.max_iter; ++it) {
    CNMF_TRY(update(sideR, chunks_r));
    if (io.update_cols) {
      if (!is) CNMF_TRY(row_sums(io.Fr, v.n_r, v.ld_r, d_sumR));
      CNMF_TRY(update(sideC, chunks_c));
      if (!is) CNMF_TRY(row_sums(io.Fc, v.n_c, v.ld_c, d_sumC));
    }
    const bool chk = (p.tol > 0 && it % 10 == 0) || it == p.max_iter;
    if (chk) {
      const double tol_eff = (p.tol > 0 && it % 10 == 0) ? p.tol : -1.0;
      CNMF_TRY(check(it, tol_eff));
      CNMF_CUDA_CHECK(cudaMemcpyAsync(h_done.data(), d_done, sizeof(int) * R, cudaMemcpyDeviceToHost, s));
      CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
      bool all = true;
      for (int r = 0; r < R; ++r) all = all && h_done[r];
      if (all) break;
    }
  }
  io.n_iter.assign(R, 0);
  io.last.assign(R, 0.0);
  io.err.assign(R, 0.0);
  CNMF_CUDA_CHECK(cudaMemcpyAsync(io.n_iter.data(), d_niter, sizeof(int) * R, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaMemcpyAsync(io.last.data(), st.last, sizeof(double) * R, cudaMemcpyDeviceToHost, s));   // the fitted divergence
  // err: ||X - W H||_F of the final factors, as for the Frobenius solvers (one more pass, every restart)
  int* d_zero = static_cast<int*>(h->dev_buf("solve.zero", sizeof(int) * 2 * R));
  if (!d_zero) return -2;
  CNMF_CUDA_CHECK(cudaMemsetAsync(d_zero, 0, sizeof(int) * 2 * R, s));
  BatchMeta bm0{d_meta, d_meta + R, d_meta + 2 * R, d_zero, R, 32};
  ConvState st0{d_state + 3 * R, d_state + 4 * R, d_state + 5 * R, d_zero, d_zero + R};
  CNMF_TRY(error_pass(ERR_FROB, bm0));
  beta_check_kernel<<<(R + 127) / 128, 128, 0, s>>>(st0, d_part, chunks_r, d_sumR, d_sumC, 0.0, ERR_FROB, bm0, 0, 0.0, p.max_iter);
  CNMF_CUDA_CHECK(cudaGetLastError());
  h->launches += 1;
  CNMF_CUDA_CHECK(cudaMemcpyAsync(io.err.data(), st0.last, sizeof(double) * R, cudaMemcpyDeviceToHost, s));
  CNMF_CUDA_CHECK(cudaStreamSynchronize(s));
  return 0;
}

}  // namespace cnmf
