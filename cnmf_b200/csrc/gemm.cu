// Front end of the two GEMM kernels (gemm.h): one GemmArgs builder for the solver, the projections and the test hook.
#include "gemm.h"

namespace cnmf {

int gemm_run(bool tc, bool b_exact, const float* out_col_scale, int M, const GemmA& A, const Operand& B, float* C,
             int ldc, const GemmPlan& plan, cudaStream_t s) {
  GemmArgs g{};
  g.M = M; g.N = B.rows; g.Kd = B.cols;
  g.lda = A.ld; g.ldb = B.ld; g.ldc = ldc;
  g.C = C;
  g.c_split_stride = plan.split_stride;
  g.splits = plan.splits;
  g.splits_effective = plan.splits;
  g.bn = plan.bn;
  if (!tc) {
    g.A_hi = A.full; g.B_hi = B.full;
    return gemm_fp32_simt(g, s);
  }
  g.A_hi = A.hi; g.A_lo = A.lo; g.B_hi = B.hi; g.B_lo = B.lo;
  g.b_exact = b_exact ? 1 : 0;
  g.out_col_scale = b_exact ? out_col_scale : nullptr;
  if (B.h16) {       // A.hi / A.lo hold the two fp16 pieces of the row-normalised factor, B its fp16 integer matrix
    g.f16 = 1;
    g.B_hi = static_cast<const float*>(B.h16);
    g.a_tile_scale = A.tile_scale;
    g.a_tiles = (A.ld + 511) / 512;
  }
  return gemm_tf32x3(g, s);
}

}  // namespace cnmf
