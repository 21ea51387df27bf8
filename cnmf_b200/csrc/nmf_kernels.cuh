// Device kernels of the batched NMF engine (declarations; definitions in nmf_kernels.cu).
//
// Layout ("packed factor"): all live restarts are stacked along rows. Restart r owns rows
// [off[r], off[r]+k[r]) of every SK x n factor array (SK = sum of k).  Wt is the transposed
// usage matrix (SK x cells), H the spectra (SK x genes).  Row stride ld = pad_ld(n) floats,
// padding columns stay zero.  Because both factors are stored "components x items", the W half
// and the H half of an iteration are the SAME kernels with the roles of the arrays swapped.
#pragma once
#include <cuda_runtime.h>

#include "common.cuh"

namespace cnmf {

constexpr int UPD_THREADS = 128;
// columns one block of the update kernels covers per pass ("tile"): a thread owns 4 consecutive items (one 16-byte
// access per array and component) when the batch fits the 16-component bodies, 2 otherwise (register budget)
inline int upd_tile_cols(int kp) { return UPD_THREADS * (kp <= 16 ? 4 : 2); }

struct FactorView {
  float* F;        // SK x ld, in/out
  float* F_hi;     // optional tf32 pieces (nullptr in fp32 mode)
  float* F_lo;
  int n;           // valid columns
  int ld;
  const float* piece_scale;   // optional per-column scale folded into the tf32 pieces: hi + lo = F * piece_scale
                              // (exact-count datasets: the per-gene / per-cell scale of X lives in the A operand)
  // f16x2: the Gram-fused update kernels (K <= 16) also emit the fp16 operand pieces of what they write, normalised per
  // (row, 512-column tile): P_hi / P_mid (halves, row stride ld) and tile_scale[row * n_ktiles + tile]; nullptr = off
  void* P_hi;
  void* P_mid;
  float* tile_scale;
  int n_ktiles;    // ceil(ld / 512)
  int cpb;         // columns handled by one block of the update / cross kernels (multiple of upd_tile_cols(kp))
  int gcpb;        // columns handled by one block of the Gram kernel (multiple of 1024)
};

// block granularity: large enough to amortise the per-block prologue, small enough that
// (column chunks) x (restarts) fills the 148 SMs a few times over even for a single refit
inline int pick_cols_per_block(int n, int n_restarts, int max_cols, int min_cols, int min_blocks) {
  int c = max_cols;
  while (c > min_cols && (long long)((n + c - 1) / c) * n_restarts < min_blocks) c /= 2;
  return c;
}

// "slot" = position of a live restart in the packed arrays (changes when converged restarts are
// compacted away); "rid" = its index in the caller's restart list (never changes).  Packed factor
// rows are addressed by slot, every per-restart state array (done, n_iter, Gram, scalars) by rid.
struct BatchMeta {
  const int* off;  // [slots] first packed row of the restart in slot s
  const int* k;    // [slots] its n_components
  const int* rid;  // [slots] its restart id
  const int* done; // [n restarts] 1 = converged, frozen (indexed by rid)
  int R;           // live slots
  int kp;          // 16 or 32: >= max k in the batch (selects the kernel's register budget)
};

inline int col_chunks(const FactorView& f) { return (f.n + f.cpb - 1) / f.cpb; }
inline int gram_chunks(const FactorView& f) { return (f.n + f.gcpb - 1) / f.gcpb; }

// x -> (hi, lo) tf32 pieces, elementwise over rows x ld (padding included)
int launch_split_tf32(const float* src, float* hi, float* lo, long long n_elems, cudaStream_t s);
// (hi, lo) = split(src[r, c] * col_scale[c]) over rows x ld; col_scale may be nullptr (plain split)
int launch_split_scaled(const float* src, float* hi, float* lo, int rows, int ld, const float* col_scale, cudaStream_t s);

// ---- fp16 operand pieces (f16x2 precision, exact-count datasets) ----
// per packed row r and group g of 512 columns: sc = power of two with max(F[r, c] * pscale[c]) / sc in
// [2^14, 2^15) over the group -> tile_scale[r * n_ktiles + g]; hi / mid (fp16, row stride ld halves) = the two pieces of
// F[r, :] * pscale / sc.  Same bits as the update kernels' in-kernel emission
int launch_emit_f16(const float* F, int rows, int n, int ld, const float* pscale, void* hi, void* mid, float* tile_scale,
                    int n_ktiles, cudaStream_t s);
// dst (fp16) = src (fp32), elementwise; used for the exact integer count matrices
int launch_to_half(const float* src, void* dst, long long n_elems, cudaStream_t s);

// ---- exact-count detection (dataset preparation) ----
// col_min[c] / row_min[r] = smallest strictly positive entry of the column / row (+inf if none)
int launch_min_positive(const float* X, int rows, int cols, int ld, float* col_min, float* row_min, cudaStream_t s);
// counts entries that are not (positive-integer <= 2048) * row_scale[r] * col_scale[c] within 5e-7 relative (fp32 rounding of the scaled integer)
// (either scale may be nullptr = 1); *n_bad is accumulated atomically (zero it first)
int launch_check_scaled_int(const float* X, int rows, int cols, int ld, const float* row_scale, const float* col_scale,
                            int* n_bad, cudaStream_t s);
// C[r, c] = rint(X[r, c] / (row_scale[r] * col_scale[c])) as fp32 (exact in tf32 for values <= 2048)
int launch_build_counts(const float* X, int rows, int cols, int ld, const float* row_scale, const float* col_scale,
                        float* C, cudaStream_t s);
// v[i] = isfinite(v[i]) && v[i] > 0 ? v[i] : 1 for i < n, 0 for n <= i < n_pad
int launch_fix_scale(float* v, int n, int n_pad, cudaStream_t s);

// dst (cols x ld_dst) = src (rows x ld_src)^T ; optionally also emits tf32 pieces of dst
int launch_transpose(const float* src, int rows, int cols, int ld_src, float* dst, float* dst_hi, float* dst_lo,
                     int ld_dst, cudaStream_t s);

// out[0] = sum(X), out[1] = sum(X^2) over the valid rows x cols region, fp64
int launch_matrix_sums(const float* X, int rows, int cols, int ld, double* out2, double* scratch, int scratch_len,
                       cudaStream_t s);

// What an update launch can emit besides the updated factor, finalised INSIDE the launch: every block writes its
// fp64 partials, takes a ticket on the restart's counter, and the block that draws the last ticket sums all
// partials of the restart in chunk order (deterministic) -- so neither a Gram pass over the freshly written
// factor nor a finalize launch sits between an update and the GEMM / update that follows it.
struct FusedOut {
  double* gram_part;   // nullptr = no Gram.  [(slot * chunks + chunk) * kp*kp + c*KP + i], KP = K rounded up to 4
  double* gram;        // [rid * KMAX*KMAX + c*KMAX + i]: K x K Gram of the UPDATED factor (kp == 16 batches only)
  double* scal_part;   // nullptr = no scalar.  [slot * chunks + chunk]
  double* scal;        // [rid]: MU <NUM, F_new> (trace-form error), CD sum |projected gradient|
  int* counter;        // [rid] tickets; zero on entry, reset by the last block
};

// Multiplicative update (sklearn _nmf.py:535-549,610-624 / :633-635,696-721):
//   F[c, j] <- F[c, j] * NUM[c, j] / max-style-guard( sum_i gram[c, i] F[i, j] + l1 + l2 F[c, j] )
// NUM = sum over `nsplit` split-K slices (stride num_split_stride elements), summed in slice order.
// gram_in = finalised K x K Gram of the OTHER factor, fp64 [rid * KMAX*KMAX + c*KMAX + i].
int launch_mu_update(const FactorView& f, const float* NUM, int nsplit, long long num_split_stride,
                     const double* gram_in, const BatchMeta& b, float l1, float l2, const FusedOut& out,
                     cudaStream_t s);

// One coordinate-descent sweep over the K coordinates of every column (sklearn _cdnmf_fast.pyx:8-37).
int launch_cd_update(const FactorView& f, const float* NUM, int nsplit, long long num_split_stride,
                     const double* gram_in, const BatchMeta& b, float l1, float l2, const FusedOut& out,
                     cudaStream_t s);

// cross_partial[r*chunks+chunk] = sum_{c,j} NUM[c,j] * F[c,j]   (no update; used for the error at init)
int launch_cross(const FactorView& f, const float* NUM, int nsplit, long long num_split_stride, const BatchMeta& b,
                 double* cross_partial, cudaStream_t s);

// gram_partial[(rid*gram_chunks+chunk)*kp*kp + c*kp + i] = sum_j F[c,j] F[i,j] over the chunk's columns
int launch_gram_partial(const FactorView& f, const BatchMeta& b, double* gram_partial, cudaStream_t s,
                        bool one_warp_blocks = false);

// gram[r][c*KMAX+i] = sum over chunks (fixed order -> deterministic); scal[r] = sum over chunks of scal_partial
int launch_finalize(const double* gram_partial, double* gram, const double* scal_partial, double* scal, int chunks,
                    const BatchMeta& b, cudaStream_t s);

struct ConvState {     // device arrays, one entry per restart
  double* err0;        // MU: error at init            CD: violation of iteration 1
  double* prev;        // MU: error at the last check
  double* last;        // last evaluated error / violation (reported back)
  int* done;
  int* n_iter;
};

// MU: err = sqrt(max(normX2 - 2 cross + <gramA, gramB>, 0)); it==0 initialises err0/prev;
// otherwise stop if (prev - err)/err0 < tol (sklearn _nmf.py:867-879).
int launch_mu_check(const ConvState& st, const double* cross, const double* gramA, const double* gramB, double normX2,
                    const BatchMeta& b, int it, double tol, int max_iter, cudaStream_t s);

// CD: viol = violA (+ violB); it==1 sets viol0; stop if viol0 == 0 or viol/viol0 <= tol (sklearn _nmf.py:504-516)
int launch_cd_check(const ConvState& st, const double* violA, const double* violB, const BatchMeta& b, int it,
                    double tol, int max_iter, cudaStream_t s);

// packed-row gather: dst rows [dst_off[i], +k[i]) <- src rows [src_off[i], +k[i])  for i < R (compaction / output)
int launch_gather_rows(const float* src, const int* src_off, float* dst, const int* dst_off, const int* k, int R,
                       int n_ld, cudaStream_t s);

}  // namespace cnmf
