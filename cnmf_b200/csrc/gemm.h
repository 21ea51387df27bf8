// Internal GEMM interface: C[z] (M x N) = A[:, Kz] (M x Kd, K-major) * B[:, Kz]^T (N x Kd, K-major).
#pragma once
#include <cuda_runtime.h>

namespace cnmf {

struct GemmArgs {
  const float* A_hi;   // M x Kd, row stride lda   (tf32x3: tf32 "hi" piece; fp32 path: the full matrix)
  const float* A_lo;   // tf32 "lo" piece (unused by the fp32 path)
  const float* B_hi;   // N x Kd, row stride ldb
  const float* B_lo;
  float* C;            // splits_effective x (M x ldc)
  int M, N, Kd;
  int lda, ldb, ldc;
  long long c_split_stride;   // elements between consecutive split-K slices of C
  int splits;                 // requested split-K factor
  int splits_effective;       // gemm_effective_splits(Kd, splits): what the kernel will actually write
  int bn;                     // tf32x3: tile width (UMMA N); 0 = choose from (M, N, Kd, splits)
  int b_exact;                // tf32x3: B_hi holds B exactly (tf32-representable values); B_lo unused -> 2 passes
  const float* out_col_scale; // optional: C[:, n] *= out_col_scale[n] (length >= ldc, 16-byte aligned, zero padded)
  // f16 = 1 (tcgen05 path, b_exact only): A_hi / A_lo / B_hi point to __half arrays (two fp16 pieces of the row-
  // normalised A, the integer matrix B), lda / ldb are in half elements, k-blocks hold 64 elements; kind::f16 MMAs run
  // at twice the kind::tf32 rate and carry the same 11-bit significand per piece
  int f16;
  // f16: the A pieces were divided by a power of two per (row, group of 512 reduction elements); the accumulate warps
  // multiply each drained TMEM chain (128 elements, never straddling a group) by a_tile_scale[m * a_tiles + group]
  const float* a_tile_scale;
  int a_tiles;                // groups per row = ceil(Kd / 512)
};

// number of non-empty split-K slices for a reduction length Kd (k-blocks of 32 fp32 / 64 fp16 elements = 128 B)
int gemm_effective_splits(int Kd, int splits, int f16 = 0);

// split-K factor used by the solver: a function of the reduction length only (slices of 64 k-blocks, <= 16), so that a
// restart's result does not depend on the batch it is solved in
int gemm_fixed_splits(int Kd, int f16 = 0);

// Choice of the split-K factor (gemm_fixed_splits) and the tile width for the tcgen05 kernel: minimises
// (waves of the persistent grid) x (tile cost) x (k-blocks per item + pipeline fill) over the tile widths.
void gemm_plan(int M, int N, int Kd, int sm_count, int* splits, int* bn, int f16 = 0);

// tcgen05 / TMEM / TMA path (gemm_tf32x3.cu)
int gemm_tf32x3(const GemmArgs& g, cudaStream_t stream);

// plain fp32 FFMA path (gemm_simt.cu): A = A_hi, B = B_hi exactly; same split-K contract
int gemm_fp32_simt(const GemmArgs& g, cudaStream_t stream);

struct Operand {     // a K-major matrix as the GEMM sees it
  const float* full;
  const float* hi;     // tf32 hi piece, or the exact integer matrix when `exact`
  const float* lo;
  const void* h16;     // the exact integer matrix as fp16 (f16x2 datasets), else nullptr
  int rows, cols, ld;
};

struct GemmA {       // the M x Kd factor operand (row stride ld)
  const float* full;         // fp32 path
  const float* hi;           // tcgen05 path: tf32 pieces, or two fp16 pieces when B.h16 is set
  const float* lo;
  const float* tile_scale;   // fp16 pieces: scale per (row, group of 512 reduction elements)
  int ld;
};

struct GemmPlan {
  int splits;               // split-K factor, already effective (gemm_effective_splits)
  int bn;                   // tile width for the tcgen05 kernel (0 = let the launcher choose)
  long long split_stride;   // elements between the split-K slices of C
};

// C[z] (M x B.rows) = A (M x B.cols) * B^T.  tc: tcgen05 on the pieces -- b_exact: B.hi holds B exactly (2 passes) and
// C[:, n] *= out_col_scale[n] when that is set; B.h16 set: kind::f16 on the fp16 pieces.  Otherwise FFMA on A.full,
// B.full.  Launches one kernel; counting and profiling it is the caller's.
int gemm_run(bool tc, bool b_exact, const float* out_col_scale, int M, const GemmA& A, const Operand& B, float* C,
             int ldc, const GemmPlan& plan, cudaStream_t s);

}  // namespace cnmf
