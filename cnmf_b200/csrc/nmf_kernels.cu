// Elementwise / reduction kernels of the batched NMF engine (see nmf_kernels.cuh for the layout).
// All of these are HBM-bound streaming kernels: coalesced along the item (cell / gene) axis,
// the tiny K x K Gram matrices are broadcast from shared memory, fp64 only for the scalars
// that feed the convergence decisions.
#include "nmf_kernels.cuh"

#include <cuda_fp16.h>

namespace cnmf {

namespace {

constexpr float EPSILON_F32 = 1.1920928955078125e-07f;   // np.finfo(np.float32).eps, sklearn _nmf.py:32

template <typename T>
__device__ __forceinline__ T block_sum(T v, T* smem /* >= 32 entries */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  T r = (threadIdx.x < nw) ? smem[threadIdx.x] : T(0);
  if (warp == 0) r = warp_sum(r);
  return r;   // valid in thread 0
}

// ------------------------------------------------------------------ split / transpose / sums
__global__ void split_tf32_kernel(const float* __restrict__ src, float* __restrict__ hi, float* __restrict__ lo,
                                  long long n4) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    float4 h, l;
    split_tf32(v.x, h.x, l.x);
    split_tf32(v.y, h.y, l.y);
    split_tf32(v.z, h.z, l.z);
    split_tf32(v.w, h.w, l.w);
    reinterpret_cast<float4*>(hi)[i] = h;
    reinterpret_cast<float4*>(lo)[i] = l;
  }
}

__global__ void split_scaled_kernel(const float* __restrict__ src, float* __restrict__ hi, float* __restrict__ lo,
                                    int rows, int ld, const float* __restrict__ col_scale) {
  const int ld4 = ld / 4;
  const long long n4 = (long long)rows * ld4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % ld4);
    float4 v = reinterpret_cast<const float4*>(src)[i];
    if (col_scale) {
      const float4 sc = reinterpret_cast<const float4*>(col_scale)[c4];
      v.x *= sc.x; v.y *= sc.y; v.z *= sc.z; v.w *= sc.w;
    }
    float4 h, l;
    split_tf32(v.x, h.x, l.x);
    split_tf32(v.y, h.y, l.y);
    split_tf32(v.z, h.z, l.z);
    split_tf32(v.w, h.w, l.w);
    reinterpret_cast<float4*>(hi)[i] = h;
    reinterpret_cast<float4*>(lo)[i] = l;
  }
}

// positive floats order like their bit patterns: atomicMin on the int view
__global__ void min_positive_kernel(const float* __restrict__ X, int rows, int cols, int ld, int* __restrict__ col_min,
                                    int* __restrict__ row_min) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int r0 = blockIdx.y * 64;
  int cm = 0x7f800000;
  for (int r = r0; r < min(rows, r0 + 64); ++r) {
    const float v = (c < cols) ? X[(long long)r * ld + c] : 0.f;
    int b = (v > 0.f) ? __float_as_int(v) : 0x7f800000;
    cm = min(cm, b);
    // row minimum: warp reduce then one atomic per warp
    for (int o = 16; o > 0; o >>= 1) b = min(b, __shfl_xor_sync(0xffffffffu, b, o));
    if ((threadIdx.x & 31) == 0 && b != 0x7f800000) atomicMin(&row_min[r], b);
  }
  if (c < cols && cm != 0x7f800000) atomicMin(&col_min[c], cm);
}

__global__ void check_scaled_int_kernel(const float* __restrict__ X, int rows, int cols, int ld,
                                        const float* __restrict__ rs, const float* __restrict__ cs, int* __restrict__ n_bad) {
  int bad = 0;
  const long long total = (long long)rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    const float v = X[(long long)r * ld + c];
    if (v == 0.f) continue;
    const float sc = (rs ? rs[r] : 1.f) * (cs ? cs[c] : 1.f);
    const float q = v / sc;
    const float n = rintf(q);
    // fp32 rounding of a genuinely scaled integer: v, sc and the quotient each carry <= 2^-24 relative error, i.e.
    // |q - n| <= 1.8e-7 n; anything further away (soft-corrected counts, arbitrary matrices) takes the general path
    if (!(v > 0.f) || !(n >= 1.f) || n > 2048.f || fabsf(q - n) > 5e-7f * n) ++bad;
  }
  bad = warp_sum(bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(n_bad, bad);
}

__global__ void build_counts_kernel(const float* __restrict__ X, int rows, int cols, int ld, const float* __restrict__ rs,
                                    const float* __restrict__ cs, float* __restrict__ C) {
  const long long total = (long long)rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    const float v = X[(long long)r * ld + c];
    const float sc = (rs ? rs[r] : 1.f) * (cs ? cs[c] : 1.f);
    C[(long long)r * ld + c] = (v == 0.f) ? 0.f : rintf(v / sc);
  }
}

__global__ void fix_scale_kernel(float* __restrict__ v, int n, int n_pad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pad) return;
  if (i >= n) { v[i] = 0.f; return; }
  const float x = v[i];
  v[i] = (isfinite(x) && x > 0.f && x < 1e30f) ? x : 1.f;   // rows / columns without a positive entry: any scale works
}

__global__ void transpose_kernel(const float* __restrict__ src, int rows, int cols, int ld_src, float* __restrict__ dst,
                                 float* __restrict__ dst_hi, float* __restrict__ dst_lo, int ld_dst) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? src[(long long)r * ld_src + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;      // dst row = c, dst col = r
    if (c < cols && r < rows) {
      const float v = tile[threadIdx.x][i];
      const long long o = (long long)c * ld_dst + r;
      if (dst) dst[o] = v;
      if (dst_hi) {
        float h, l;
        split_tf32(v, h, l);
        dst_hi[o] = h;
        dst_lo[o] = l;
      }
    }
  }
}

__global__ void sums_partial_kernel(const float* __restrict__ X, int rows, int cols, int ld, double* __restrict__ part) {
  __shared__ double sm[32];
  double s = 0, q = 0;
  const long long total = (long long)rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    const double v = X[(long long)r * ld + c];
    s += v;
    q += v * v;
  }
  s = block_sum(s, sm);
  q = block_sum(q, sm);
  if (threadIdx.x == 0) {
    part[2 * blockIdx.x] = s;
    part[2 * blockIdx.x + 1] = q;
  }
}
__global__ void sums_final_kernel(const double* __restrict__ part, int nblocks, double* __restrict__ out2) {
  __shared__ double sm[32];
  double s = 0, q = 0;
  for (int i = threadIdx.x; i < nblocks; i += blockDim.x) {
    s += part[2 * i];
    q += part[2 * i + 1];
  }
  s = block_sum(s, sm);
  q = block_sum(q, sm);
  if (threadIdx.x == 0) {
    out2[0] = s;
    out2[1] = q;
  }
}

// ------------------------------------------------------------------ fp16 operand pieces (f16x2 precision)
// kind::f16 MMAs run at twice the kind::tf32 rate and fp16 carries the same 11-bit significand as tf32; what it
// lacks is exponent range.  So every group of 512 reduction elements of a packed factor row is divided by a power
// of two that puts its largest entry (times the per-column scale of the exact-count path) in [2^14, 2^15) -- far
// above fp16's subnormals -- and split into hi = fp16(x), mid = fp16(x - hi): 22 significant bits like the tf32 pair,
// absolute error <= 2^-39 of the group maximum for entries too small to keep them.  The GEMM multiplies each drained
// 128-element chain by the group's power of two.
// The pieces are a pure function of the factor values: this stand-alone kernel (initial factors, re-packing after a
// compaction, K > 16 batches) and the in-update emission (emit_tile_f16) produce the same bits, so a restart's
// operands do not depend on when the batch around it was compacted.
// One block per row, one warp per group of 512 columns (what the update kernels' tiles emit), a lane owns QUADS = 4
// 16-byte quads of the group.
__global__ void __launch_bounds__(256)
emit_f16_kernel(const float* __restrict__ F, int n, int ld, const float* __restrict__ pscale, __half* __restrict__ hi,
                __half* __restrict__ mid, float* __restrict__ tile_scale, int n_ktiles) {
  constexpr int QUADS = 4;
  const long long row = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float* src = F + row * ld;
  for (int g = warp; g < n_ktiles; g += blockDim.x >> 5) {
    const int t0 = g * (128 * QUADS);
    float4 v[QUADS];
    float m = 0.f;
#pragma unroll
    for (int j = 0; j < QUADS; ++j) {
      const int col = t0 + 4 * lane + 128 * j;
      v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (col < ld) {
        v[j] = *reinterpret_cast<const float4*>(src + col);
        if (pscale) {
          const float4 p = *reinterpret_cast<const float4*>(pscale + col);
          v[j].x *= p.x; v[j].y *= p.y; v[j].z *= p.z; v[j].w *= p.w;
        }
      }
      // |.|: factors are non-negative, but the OLS projection sends signed (centred) rows through the same pieces
      m = fmaxf(fmaxf(m, fmaxf(fabsf(v[j].x), fabsf(v[j].y))), fmaxf(fabsf(v[j].z), fabsf(v[j].w)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    const float sc = f16_group_scale(m);
    const float inv = 1.f / sc;          // power of two: exact
    if (lane == 0) tile_scale[row * n_ktiles + g] = sc;
#pragma unroll
    for (int j = 0; j < QUADS; ++j) {
      const int col = t0 + 4 * lane + 128 * j;
      if (col < ld) {
        const float x0 = v[j].x * inv, x1 = v[j].y * inv, x2 = v[j].z * inv, x3 = v[j].w * inv;
        const __half2 h01 = __floats2half2_rn(x0, x1), h23 = __floats2half2_rn(x2, x3);
        const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
        const __half2 m01 = __floats2half2_rn(x0 - f01.x, x1 - f01.y), m23 = __floats2half2_rn(x2 - f23.x, x3 - f23.y);
        uint2 oh, om;
        oh.x = *reinterpret_cast<const uint32_t*>(&h01); oh.y = *reinterpret_cast<const uint32_t*>(&h23);
        om.x = *reinterpret_cast<const uint32_t*>(&m01); om.y = *reinterpret_cast<const uint32_t*>(&m23);
        *reinterpret_cast<uint2*>(hi + row * ld + col) = oh;
        *reinterpret_cast<uint2*>(mid + row * ld + col) = om;
      }
    }
  }
}

// dst (fp16) = src (fp32, small non-negative integers: exact), elementwise over rows x ld
__global__ void to_half_kernel(const float* __restrict__ src, __half* __restrict__ dst, long long n4) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    const __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
    uint2 o;
    o.x = *reinterpret_cast<const uint32_t*>(&a); o.y = *reinterpret_cast<const uint32_t*>(&b);
    reinterpret_cast<uint2*>(dst)[i] = o;
  }
}

// ------------------------------------------------------------------ update kernels (fused with the Gram)
// Thread = VEC consecutive items (cells / genes) of one restart, held as packed fp32 pairs: every array is
// touched with one 16-byte (VEC = 4) access per component, and the K x K contraction with the Gram of the
// other factor runs on FFMA2 (two items per instruction, the Gram entry a broadcast operand read from shared
// memory as LDS.128 = 4 entries x 2 pairs = 8 packed FMAs per shared-memory instruction).  The quotient is
// the branch-free MUFU.RCP + Newton sequence of common.cuh.  The unrolled body is instantiated per K rounded
// up to 4 and dispatched per restart inside the kernel (block-uniform switch), so a K = 10 restart runs the
// 12 x 12 body even when the batch also holds K = 13 restarts.
//
// The Gram of the UPDATED factor (needed by the next half-iteration's update and by the trace-form error) is
// accumulated in the same launch: the block parks its new values in a shared-memory tile (components x
// tile columns), the warps split the K x K entries by rows and walk the tile with packed FMAs, per-thread
// fp32 sums over at most 16 columns go through shared memory into per-block fp64 sums (fixed order), and the
// last block of a restart adds the per-block partials in chunk order (FusedOut).  The first version -- a scalar
// thread-per-item update (1 052 warp instructions per item at K = 10: 4-byte accesses, 3-register FFMA,
// IEEE division) plus a separate Gram launch re-reading the factor -- spent 168 us per W half at c2 against 107 us
// of DRAM time; see profiles/r1e_ncu_full_summary.txt.
template <int VEC> struct VecIO;
template <> struct VecIO<4> {
  static constexpr int NP = 2;
  static __device__ __forceinline__ void ld(const float* p, float2 (&v)[2]) {
    const float4 q = *reinterpret_cast<const float4*>(p);
    v[0] = make_float2(q.x, q.y);
    v[1] = make_float2(q.z, q.w);
  }
  static __device__ __forceinline__ void st(float* p, const float2 (&v)[2]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0].x, v[0].y, v[1].x, v[1].y);
  }
};
template <> struct VecIO<2> {
  static constexpr int NP = 1;
  static __device__ __forceinline__ void ld(const float* p, float2 (&v)[1]) { v[0] = *reinterpret_cast<const float2*>(p); }
  static __device__ __forceinline__ void st(float* p, const float2 (&v)[1]) { *reinterpret_cast<float2*>(p) = v[0]; }
};

constexpr float FLT_MIN_NORMAL = 1.17549435e-38f;
// KPMAX x TILE is 16 x 512 = 32 x 256 = 8192 floats for both kernel families; the Gram scratch needs
// UPD_THREADS x 68 = 8704 floats (FusedGramCfg<16>::STRIDE)
constexpr int UPD_TILE_N_FLOATS = 8192;
constexpr int UPD_TILE_F_FLOATS = 8192 + 1024;

// finalised Gram of the other factor -> shared memory (KP x KP fp32, zero beyond K), + diag_add on the diagonal
__device__ __forceinline__ void load_gram_smem(float* G, const double* __restrict__ gram_in, int r, int K, int KP,
                                               float diag_add) {
  const double* g = gram_in + (long long)r * KMAX * KMAX;
  for (int idx = threadIdx.x; idx < KP * KP; idx += blockDim.x) {
    const int c = idx / KP, i = idx % KP;
    float v = (c < K && i < K) ? (float)g[c * KMAX + i] : 0.f;
    if (c == i && c < K) v += diag_add;
    G[idx] = v;
  }
}

// A thread's VEC items of one array: base pointer of component 0 plus a 32-bit element offset per component
// (one IMAD.WIDE per access instead of a 64-bit multiply-add chain)
template <int KP, int VEC>
__device__ __forceinline__ void load_items(const float* __restrict__ pF, const float* __restrict__ pN, int nsplit,
                                           long long sstride, int K, unsigned ld, int n_left,
                                           float2 (&fv)[KP][VecIO<VEC>::NP], float2 (&nv)[KP][VecIO<VEC>::NP]) {
  constexpr int NP = VecIO<VEC>::NP;
  // all loads of this item group first (2K independent 16-byte requests in flight per thread)
#pragma unroll
  for (int i = 0; i < KP; ++i) {
    if (i < K) {
      const unsigned off = (unsigned)i * ld;
      VecIO<VEC>::ld(pF + off, fv[i]);
      VecIO<VEC>::ld(pN + off, nv[i]);
    } else {
#pragma unroll
      for (int p = 0; p < NP; ++p) {
        fv[i][p] = make_float2(0.f, 0.f);
        nv[i][p] = make_float2(0.f, 0.f);
      }
    }
  }
  if (nsplit > 1) {                                  // split-K slices, added in slice order
    for (int s = 1; s < nsplit; ++s) {
      const float* pS = pN + s * sstride;
#pragma unroll
      for (int i = 0; i < KP; ++i) {
        if (i < K) {
          float2 t[NP];
          VecIO<VEC>::ld(pS + (unsigned)i * ld, t);
#pragma unroll
          for (int p = 0; p < NP; ++p) nv[i][p] = add2(nv[i][p], t[p]);
        }
      }
    }
  }
  if (n_left < VEC) {                                // ragged tail: product columns >= n are not defined
#pragma unroll
    for (int i = 0; i < KP; ++i)
#pragma unroll
      for (int p = 0; p < NP; ++p) {
        if (2 * p >= n_left) { nv[i][p].x = 0.f; fv[i][p].x = 0.f; }
        if (2 * p + 1 >= n_left) { nv[i][p].y = 0.f; fv[i][p].y = 0.f; }
      }
  }
}

template <int VEC>
__device__ __forceinline__ void store_items(float* pF, float* pH, float* pL, unsigned off,
                                            const float2 (&v)[VecIO<VEC>::NP], const float2 (&pscale)[VecIO<VEC>::NP]) {
  constexpr int NP = VecIO<VEC>::NP;
  VecIO<VEC>::st(pF + off, v);
  if (pH) {
    float2 h[NP], l[NP];
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const float2 sv = mul2(v[p], pscale[p]);
      h[p] = make_float2(to_tf32(sv.x), to_tf32(sv.y));
      const float2 rest = add2(sv, neg2(h[p]));
      l[p] = make_float2(to_tf32(rest.x), to_tf32(rest.y));
    }
    VecIO<VEC>::st(pH + off, h);
    VecIO<VEC>::st(pL + off, l);
  }
}

// per-KP partition of the fused Gram: TPC warps split the K x K entries by rows (RB rows each), the warps
// that share a row block split the tile's column pairs
template <int KP> struct FusedGramCfg {
  static constexpr int WARPS = UPD_THREADS / 32;
  static constexpr int TPC = KP <= 4 ? 1 : (KP <= 8 ? 2 : 4);
  static constexpr int RB = KP / TPC;
  static constexpr int NG = WARPS / TPC;                      // warps per row block
  static constexpr int VALS = RB * KP;                        // sums per thread
  static constexpr int STRIDE = (VALS / 4) % 2 ? VALS : VALS + 4;   // odd number of 16-byte units: conflict-free STS.128
};

// tile: KP x TILE fp32 (new factor values of this pass, zero rows beyond K); gsum[KP*KP] += Gram of the tile.
// `scratch` aliases the tile (it is consumed before it is overwritten).
template <int KP, int TILE>
__device__ __forceinline__ void fused_gram_tile(float* tile, double* gsum) {
  using C = FusedGramCfg<KP>;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rb = warp % C::TPC, grp = warp / C::TPC;
  float2 acc[C::RB][KP];
#pragma unroll
  for (int a = 0; a < C::RB; ++a)
#pragma unroll
    for (int i = 0; i < KP; ++i) acc[a][i] = make_float2(0.f, 0.f);
  const float4* t4 = reinterpret_cast<const float4*>(tile);
  constexpr int QUADS = TILE / 4, ROW4 = TILE / 4;
#pragma unroll 1
  for (int q = grp * 32 + lane; q < QUADS; q += 32 * C::NG) {    // 4 columns = two packed pairs per LDS.128
    float4 v[KP], va[C::RB];
#pragma unroll
    for (int i = 0; i < KP; ++i) v[i] = t4[i * ROW4 + q];
#pragma unroll
    for (int a = 0; a < C::RB; ++a) va[a] = t4[(rb * C::RB + a) * ROW4 + q];
#pragma unroll
    for (int a = 0; a < C::RB; ++a)
#pragma unroll
      for (int i = 0; i < KP; ++i) {
        acc[a][i] = fma2(make_float2(va[a].x, va[a].y), make_float2(v[i].x, v[i].y), acc[a][i]);
        acc[a][i] = fma2(make_float2(va[a].z, va[a].w), make_float2(v[i].z, v[i].w), acc[a][i]);
      }
  }
  __syncthreads();                                            // every warp is done reading the tile
  float* scratch = tile + threadIdx.x * C::STRIDE;
#pragma unroll
  for (int a = 0; a < C::RB; ++a)
#pragma unroll
    for (int i4 = 0; i4 < KP / 4; ++i4) {
      float4 q;
      q.x = acc[a][4 * i4 + 0].x + acc[a][4 * i4 + 0].y;
      q.y = acc[a][4 * i4 + 1].x + acc[a][4 * i4 + 1].y;
      q.z = acc[a][4 * i4 + 2].x + acc[a][4 * i4 + 2].y;
      q.w = acc[a][4 * i4 + 3].x + acc[a][4 * i4 + 3].y;
      *reinterpret_cast<float4*>(scratch + a * KP + 4 * i4) = q;
    }
  __syncthreads();
  for (int e = threadIdx.x; e < KP * KP; e += UPD_THREADS) {  // entry (row, i): fixed-order fp64 sum over its threads
    const int row = e / KP, i = e % KP;
    const int erb = row / C::RB, a = row % C::RB;
    double sum = 0.0;
#pragma unroll
    for (int g = 0; g < C::NG; ++g) {
      const float* src = tile + (size_t)((erb + C::TPC * g) * 32) * C::STRIDE + a * KP + i;
#pragma unroll 8
      for (int l = 0; l < 32; ++l) sum += (double)src[l * C::STRIDE];
    }
    gsum[e] += sum;
  }
  __syncthreads();                                            // scratch (= tile) free again
}

// KP = 12 / 16 (four row blocks of RB = KP / 4 components): the Gram is symmetric, so only the 10 blocks on or above the
// diagonal are accumulated -- 3 + 3 + 3 + 1 blocks over the four warps (27 instead of 36 entries per thread at KP = 12,
// 48 instead of 64 at KP = 16, where the full row block did not fit in 128 registers) -- and the reduction reads an entry
// below the diagonal from its mirror image.  Every entry is still the fixed-order fp64 sum over the 32 lanes of ONE warp
// of per-lane fp32 sums over the same 4 quads in the same order, and a * b = b * a: bit-identical to the full version.
struct SymGramMap {
  // block (bi, bj), bi <= bj  ->  owning warp and its slot in that warp's list
  //   warp 0: (0,0) (0,1) (0,2)   warp 1: (0,3) (1,1) (1,2)   warp 2: (1,3) (2,2) (2,3)   warp 3: (3,3)
  static __device__ __forceinline__ void owner(int bi, int bj, int& warp, int& slot) {
    const int id = bi * 4 + bj - (bi * (bi + 1)) / 2;       // 0..9 in row-major order of the upper triangle
    warp = id / 3;
    slot = id % 3;
  }
};

template <int KP, int TILE, int W>
__device__ __forceinline__ void sym_gram_accumulate(const float* tile, float2 (&acc)[3][KP / 4][KP / 4]) {
  constexpr int RB = KP / 4;
  constexpr int NB = W == 3 ? 1 : 3;
  // blocks of this warp as (bi, bj)
  constexpr int BI[3] = {W == 0 ? 0 : (W == 1 ? 0 : (W == 2 ? 1 : 3)), W == 0 ? 0 : (W == 1 ? 1 : 2), W == 0 ? 0 : (W == 1 ? 1 : 2)};
  constexpr int BJ[3] = {W == 0 ? 0 : (W == 1 ? 3 : (W == 2 ? 3 : 3)), W == 0 ? 1 : (W == 1 ? 1 : 2), W == 0 ? 2 : (W == 1 ? 2 : 3)};
  const int lane = threadIdx.x & 31;
  const float4* t4 = reinterpret_cast<const float4*>(tile);
  constexpr int QUADS = TILE / 4, ROW4 = TILE / 4;
#pragma unroll 1
  for (int q = lane; q < QUADS; q += 32) {
    float4 v[4][RB];                                  // the row blocks this warp touches (unused ones are never loaded)
#pragma unroll
    for (int blk = 0; blk < 4; ++blk) {
      bool used = false;
#pragma unroll
      for (int k = 0; k < NB; ++k) used = used || BI[k] == blk || BJ[k] == blk;
      if (used) {
#pragma unroll
        for (int a = 0; a < RB; ++a) v[blk][a] = t4[(blk * RB + a) * ROW4 + q];
      }
    }
#pragma unroll
    for (int k = 0; k < NB; ++k)
#pragma unroll
      for (int a = 0; a < RB; ++a)
#pragma unroll
        for (int b = 0; b < RB; ++b) {
          const float4 x = v[BI[k]][a], y = v[BJ[k]][b];
          acc[k][a][b] = fma2(make_float2(x.x, x.y), make_float2(y.x, y.y), acc[k][a][b]);
          acc[k][a][b] = fma2(make_float2(x.z, x.w), make_float2(y.z, y.w), acc[k][a][b]);
        }
  }
}

// What a thread adds up in the reduction of fused_gram_tile_sym, fixed for the whole block: entries t = tid, tid + 128
// of the KP (KP + 1) / 2 entries on or above the diagonal (row-major), each read from its owner's scratch slot and added
// to gsum[row][i] and to its mirror image gsum[i][row].
// (Kept in shared memory, 3 words per entry: registers that live across the tile loop would be spilled.)
template <int KP> struct SymGramPlan {
  static constexpr int NUP = KP * (KP + 1) / 2;
  static constexpr int ROUNDS = (NUP + UPD_THREADS - 1) / UPD_THREADS;
};
constexpr int SYM_PLAN_WORDS = 3 * 2 * UPD_THREADS;       // ROUNDS <= 2 for KP <= 16

template <int KP>
__device__ __forceinline__ void sym_gram_plan(int* plan) {    // plan[(r * 3 + {0: src, 1: e1, 2: e2}) * UPD_THREADS + tid]
  constexpr int RB = KP / 4;
  constexpr int STRIDE = 3 * RB * RB + 1;
  static_assert(SymGramPlan<KP>::ROUNDS <= 2, "plan buffer holds two rounds");
#pragma unroll
  for (int r = 0; r < SymGramPlan<KP>::ROUNDS; ++r) {
    const int t = threadIdx.x + r * UPD_THREADS;
    int row = 0, rem = t;
    while (row < KP - 1 && rem >= KP - row) { rem -= KP - row; ++row; }   // t -> (row, i), row <= i, row-major
    const int i = row + rem;
    int src = -1, e1 = 0, e2 = 0;
    if (t < SymGramPlan<KP>::NUP) {
      int w, slot;
      SymGramMap::owner(row / RB, i / RB, w, slot);
      src = (w * 32) * STRIDE + (slot * RB + row % RB) * RB + i % RB;
      e1 = row * KP + i;
      e2 = i * KP + row;
    }
    plan[(r * 3 + 0) * UPD_THREADS + threadIdx.x] = src;
    plan[(r * 3 + 1) * UPD_THREADS + threadIdx.x] = e1;
    plan[(r * 3 + 2) * UPD_THREADS + threadIdx.x] = e2;
  }
}

template <int KP, int TILE>
__device__ __forceinline__ void fused_gram_tile_sym(float* tile, double* gsum, const int* plan) {
  constexpr int RB = KP / 4;
  constexpr int STRIDE = 3 * RB * RB + 1;
  static_assert(UPD_THREADS == 128, "four warps share the ten blocks");
  static_assert(UPD_THREADS * STRIDE <= KP * TILE, "reduction scratch must fit in the tile it aliases");
  const int warp = threadIdx.x >> 5;
  float2 acc[3][RB][RB];
#pragma unroll
  for (int k = 0; k < 3; ++k)
#pragma unroll
    for (int a = 0; a < RB; ++a)
#pragma unroll
      for (int b = 0; b < RB; ++b) acc[k][a][b] = make_float2(0.f, 0.f);
  switch (warp) {                                             // warp-uniform; block lists are compile-time constants
    case 0: sym_gram_accumulate<KP, TILE, 0>(tile, acc); break;
    case 1: sym_gram_accumulate<KP, TILE, 1>(tile, acc); break;
    case 2: sym_gram_accumulate<KP, TILE, 2>(tile, acc); break;
    default: sym_gram_accumulate<KP, TILE, 3>(tile, acc); break;
  }
  __syncthreads();                                            // every warp is done reading the tile
  float* scratch = tile + threadIdx.x * STRIDE;               // odd stride: conflict-free scalar accesses
#pragma unroll
  for (int k = 0; k < 3; ++k)
#pragma unroll
    for (int a = 0; a < RB; ++a)
#pragma unroll
      for (int b = 0; b < RB; ++b) scratch[(k * RB + a) * RB + b] = acc[k][a][b].x + acc[k][a][b].y;
  __syncthreads();
#pragma unroll
  for (int r = 0; r < SymGramPlan<KP>::ROUNDS; ++r) {         // fixed-order fp64 sum over the owner warp's 32 lanes
    const int so = plan[(r * 3 + 0) * UPD_THREADS + threadIdx.x];
    if (so >= 0) {
      const int e1 = plan[(r * 3 + 1) * UPD_THREADS + threadIdx.x], e2 = plan[(r * 3 + 2) * UPD_THREADS + threadIdx.x];
      const float* src = tile + so;
      double sum = 0.0;
#pragma unroll 8
      for (int l = 0; l < 32; ++l) sum += (double)src[l * STRIDE];
      gsum[e1] += sum;
      if (e2 != e1) gsum[e2] += sum;                          // a * b = b * a: the mirror entry is the same sum
    }
  }
  __syncthreads();                                            // scratch (= tile) free again
}

// f16x2: fp16 operand pieces of the tile a block has just written, straight from the shared-memory tile (so the factor
// is not read back from HBM by a separate launch).  Normalisation is per (row, 512-column tile): the warp that owns a
// row takes the tile maximum of F * pscale, picks the power of two that puts it in [2^14, 2^15) and emits
// hi = fp16(x), mid = fp16(x - hi); the GEMM multiplies each drained 128-element chain by the tile's scale.
template <int TILE>
__device__ __forceinline__ void emit_tile_f16(const FactorView& f, const float* tile, int K, int o, int t0) {
  static_assert(TILE == 512, "one lane owns four 16-byte groups of a 512-column tile");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4 ps[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int col = t0 + 4 * lane + 128 * j;
    ps[j] = make_float4(1.f, 1.f, 1.f, 1.f);
    if (f.piece_scale && col < f.ld) ps[j] = *reinterpret_cast<const float4*>(f.piece_scale + col);
  }
  const int group = t0 / TILE;
  for (int c = warp; c < K; c += UPD_THREADS / 32) {
    const float4* src = reinterpret_cast<const float4*>(tile + c * TILE);
    float2 v[4][2];                            // packed pairs: the scalings and the residual run on the 2-wide pipe
    float m = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 q = src[lane + 32 * j];
      v[j][0] = mul2(make_float2(q.x, q.y), make_float2(ps[j].x, ps[j].y));
      v[j][1] = mul2(make_float2(q.z, q.w), make_float2(ps[j].z, ps[j].w));
      m = fmaxf(fmaxf(m, fmaxf(v[j][0].x, v[j][0].y)), fmaxf(v[j][1].x, v[j][1].y));
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, s));
    const float sc = f16_group_scale(m);       // same bits as the stand-alone emit_f16_kernel
    // sc = 2^e with e in [-126, 113] (f16_group_scale): 1 / sc is the same float with the exponent mirrored -- exactly
    // what the division returns, without the division
    const float2 inv = bcast2(__uint_as_float(0x7f000000u - __float_as_uint(sc)));
    const long long rowoff = (long long)(o + c) * f.ld;
    if (lane == 0) f.tile_scale[(long long)(o + c) * f.n_ktiles + group] = sc;
    __half* ph = static_cast<__half*>(f.P_hi) + rowoff + t0 + 4 * lane;
    __half* pm = static_cast<__half*>(f.P_mid) + rowoff + t0 + 4 * lane;
    const int cols_left = f.ld - (t0 + 4 * lane);        // ld is a multiple of 4: a quad is written whole or not at all
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (128 * j < cols_left) {
        const float2 x01 = mul2(v[j][0], inv), x23 = mul2(v[j][1], inv);
        const __half2 h01 = __float22half2_rn(x01), h23 = __float22half2_rn(x23);
        const float2 r01 = add2(x01, neg2(__half22float2(h01))), r23 = add2(x23, neg2(__half22float2(h23)));
        const __half2 m01 = __float22half2_rn(r01), m23 = __float22half2_rn(r23);
        uint2 oh, om;
        oh.x = *reinterpret_cast<const uint32_t*>(&h01); oh.y = *reinterpret_cast<const uint32_t*>(&h23);
        om.x = *reinterpret_cast<const uint32_t*>(&m01); om.y = *reinterpret_cast<const uint32_t*>(&m23);
        *reinterpret_cast<uint2*>(ph + 128 * j) = oh;
        *reinterpret_cast<uint2*>(pm + 128 * j) = om;
      }
    }
  }
}

// 16-byte shared-memory load by 32-bit shared-window address: the Gram rows are addressed from a register that is set up
// once per block (ptxas otherwise rebuilds the window base of the static array inside the component loop)
__device__ __forceinline__ float4 lds128(unsigned addr) {
  float4 v;
  asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

// Component loop of the streamed-product MU update (mu_body, STREAMN): for c = 0..K-1
//   den = Gram[c,:] . F_old[:, items] (component order) + l1 + l2 F_old[c];  F_new[c] = F_old[c] * NUM[c] / den
// with NUM[c + 1] already in flight.  Running pointers (one 64-bit add per array and component), the Gram row by shared
// address, three components per trip (the in-flight registers rotate instead of being copied), and the ragged last
// item group of a row (n % 4 != 0: product columns >= n are undefined) as its own instantiation so that the common
// case carries no selects.  SIMPLE = one product slice and no tf32 pieces to write (the W half of the default f16x2
// path): the slice loop and the piece pointers drop out of the body.  Same arithmetic, same order as the rolled loop
// of round 1.
template <int KP, int VEC, bool GRAM, bool RAGGED, bool SIMPLE>
__device__ __forceinline__ float2 mu_components(float* __restrict__ pFc, float* pH, float* pL, const float* __restrict__ pNc,
                                                int nsplit, long long sstride, unsigned ld, unsigned g_row, int K, float l1,
                                                float l2, int n_left, const float2 (&fv)[KP][VecIO<VEC>::NP],
                                                const float2 (&pscale)[VecIO<VEC>::NP], float* myF) {
  constexpr int NP = VecIO<VEC>::NP;
  constexpr int TILE = UPD_THREADS * VEC;
  float2 sacc = make_float2(0.f, 0.f);
  // products of components c + 1 and c + 2 in flight: one component of lead (~80 instructions) left the quotient
  // waiting on the load (15 % of the kernel's stall samples, profiles/r2s_ncu_update_summary.txt)
  float2 nvn[NP], nvn2[NP];
  VecIO<VEC>::ld(pNc, nvn);
  VecIO<VEC>::ld(pNc + (1 < K ? ld : 0u), nvn2);
#pragma unroll 3
  for (int c = 0; c < K; ++c) {
    float2 den[NP];                                  // summed in component order, like the reference's W @ HHt row
#pragma unroll
    for (int i4 = 0; i4 < KP / 4; ++i4) {
      const float4 gq = lds128(g_row + 16 * i4);
#pragma unroll
      for (int p = 0; p < NP; ++p) {
        den[p] = i4 == 0 ? mul2(bcast2(gq.x), fv[0][p]) : fma2(bcast2(gq.x), fv[4 * i4 + 0][p], den[p]);
        den[p] = fma2(bcast2(gq.y), fv[4 * i4 + 1][p], den[p]);
        den[p] = fma2(bcast2(gq.z), fv[4 * i4 + 2][p], den[p]);
        den[p] = fma2(bcast2(gq.w), fv[4 * i4 + 3][p], den[p]);
      }
    }
    g_row += 4 * KP;
    float2 fvc[NP], nvc[NP], out[NP];
    VecIO<VEC>::ld(myF, fvc);
#pragma unroll
    for (int p = 0; p < NP; ++p) { nvc[p] = nvn[p]; nvn[p] = nvn2[p]; }
    // the last components re-read their own row instead of predicating the load (a predicated load has to preserve its
    // destination registers, which costs the copies the unrolled trip is there to avoid)
    VecIO<VEC>::ld(pNc + ((c + 2 < K) ? 2u * ld : 0u), nvn2);
    if constexpr (!SIMPLE) {
      for (int s = 1; s < nsplit; ++s) {             // split-K slices, added in slice order
        float2 t[NP];
        VecIO<VEC>::ld(pNc + s * sstride, t);
#pragma unroll
        for (int p = 0; p < NP; ++p) nvc[p] = add2(nvc[p], t[p]);
      }
    }
    if constexpr (RAGGED) {
#pragma unroll
      for (int p = 0; p < NP; ++p) {
        if (2 * p >= n_left) nvc[p].x = 0.f;
        if (2 * p + 1 >= n_left) nvc[p].y = 0.f;
      }
    }
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      // regularisation terms unconditionally: adding l1 = 0 and l2 * F = 0 is exact, a uniform branch costs more
      float2 d = fma2(bcast2(l2), fvc[p], add2(den[p], bcast2(l1)));
      // zero denominators -> eps (sklearn _nmf.py:615,701); the Newton quotient needs a normal number
      d.x = (d.x < FLT_MIN_NORMAL) ? EPSILON_F32 : d.x;
      d.y = (d.y < FLT_MIN_NORMAL) ? EPSILON_F32 : d.y;
      out[p] = mul2(fvc[p], div_nr2(nvc[p], d));
      sacc = fma2(nvc[p], out[p], sacc);
    }
    if constexpr (SIMPLE) {
      VecIO<VEC>::st(pFc, out);
    } else {
      store_items<VEC>(pFc, pH, pL, 0u, out, pscale);
      if (pH) { pH += ld; pL += ld; }
    }
    if constexpr (GRAM) VecIO<VEC>::st(myF, out);
    pFc += ld;
    pNc += ld;
    myF += TILE;
  }
  return sacc;
}

// Multiplicative update, rolled over the components: the thread's old values stay in registers for the K x K
// contraction (static indices), while the two values that are addressed by the loop variable -- F[c] and NUM[c] of
// the thread's items -- are read back from the shared-memory tiles the load phase parked them in (tileF doubles as
// the Gram tile: row c is overwritten with the new values once iteration c is done with it).  One compact loop
// body (~80 instructions) instead of K unrolled copies: no per-component predicates for K < KP, and the code
// stays resident in the instruction cache (the unrolled version stalled on instruction fetch, profiles/r1g_*).
// Returns <NUM, F_new> over the thread's items (fp32 within a tile, fp64 across tiles).
template <int KP, int VEC, bool GRAM, bool STREAMN>
__device__ __forceinline__ double mu_body(const FactorView& f, const float* __restrict__ NUM, int nsplit,
                                          long long sstride, const float* G, int K, int o, float l1, float l2,
                                          int col_begin, int col_end, float* tileF, float* tileN, double* gsum) {
  constexpr int NP = VecIO<VEC>::NP;
  constexpr int TILE = UPD_THREADS * VEC;
  const float4* G4 = reinterpret_cast<const float4*>(G);
  const unsigned g_addr = (unsigned)__cvta_generic_to_shared(G);
  const bool simple = nsplit == 1 && f.F_hi == nullptr;        // block-uniform
  const unsigned ld = (unsigned)f.ld;
  float* const myF = tileF + VEC * threadIdx.x;
  float* const myN = tileN + VEC * threadIdx.x;
  double scal = 0.0;
  constexpr bool SYM = GRAM && VEC == 4 && (KP == 12 || KP == 16);
  __shared__ int gplan[SYM ? SYM_PLAN_WORDS : 1];
  if constexpr (SYM) sym_gram_plan<KP>(gplan);                // read after the tile loop's first barrier
#pragma unroll 1
  for (int t0 = col_begin; t0 < col_end; t0 += TILE) {
    const int col = t0 + VEC * threadIdx.x;
    if (col < col_end) {
      const long long e0 = (long long)o * f.ld + col;
      float* const pF = f.F + e0;
      float* const pH = f.F_hi ? f.F_hi + e0 : nullptr;
      float* const pL = f.F_hi ? f.F_lo + e0 : nullptr;
      float2 fv[KP][NP];
      const float* const pN = NUM + e0;
      const int n_left = f.n - col;
      if constexpr (STREAMN) {
#pragma unroll
        for (int i = 0; i < KP; ++i) {
          if (i < K) {
            VecIO<VEC>::ld(pF + (unsigned)i * ld, fv[i]);
          } else {
#pragma unroll
            for (int p = 0; p < NP; ++p) fv[i][p] = make_float2(0.f, 0.f);
          }
        }
        if (n_left < VEC) {                          // ragged tail: columns >= n of the factor count as zeros
#pragma unroll
          for (int i = 0; i < KP; ++i)
#pragma unroll
            for (int p = 0; p < NP; ++p) {
              if (2 * p >= n_left) fv[i][p].x = 0.f;
              if (2 * p + 1 >= n_left) fv[i][p].y = 0.f;
            }
        }
#pragma unroll
        for (int i = 0; i < KP; ++i) VecIO<VEC>::st(myF + i * TILE, fv[i]);
      } else {
        float2 nv[KP][NP];
        load_items<KP, VEC>(pF, pN, nsplit, sstride, K, ld, n_left, fv, nv);
#pragma unroll
        for (int i = 0; i < KP; ++i) {               // rows >= K hold zeros (load_items): the Gram tile needs them
          VecIO<VEC>::st(myF + i * TILE, fv[i]);
          VecIO<VEC>::st(myN + i * TILE, nv[i]);
        }
      }
      float2 pscale[NP];
#pragma unroll
      for (int p = 0; p < NP; ++p) pscale[p] = make_float2(1.f, 1.f);
      if (f.piece_scale) VecIO<VEC>::ld(f.piece_scale + col, pscale);
      float2 sacc = make_float2(0.f, 0.f);
      if constexpr (STREAMN) {
        if (simple) {
          if (n_left >= VEC)
            sacc = mu_components<KP, VEC, GRAM, false, true>(pF, pH, pL, pN, 1, 0, ld, g_addr, K, l1, l2, n_left, fv, pscale, myF);
          else
            sacc = mu_components<KP, VEC, GRAM, true, true>(pF, pH, pL, pN, 1, 0, ld, g_addr, K, l1, l2, n_left, fv, pscale, myF);
        } else {
          if (n_left >= VEC)
            sacc = mu_components<KP, VEC, GRAM, false, false>(pF, pH, pL, pN, nsplit, sstride, ld, g_addr, K, l1, l2, n_left, fv,
                                                              pscale, myF);
          else
            sacc = mu_components<KP, VEC, GRAM, true, false>(pF, pH, pL, pN, nsplit, sstride, ld, g_addr, K, l1, l2, n_left, fv,
                                                             pscale, myF);
        }
      } else {
        unsigned off = 0;
#pragma unroll 1
        for (int c = 0; c < K; ++c, off += ld) {
          float2 den[NP];                            // summed in component order, like the reference's W @ HHt row
#pragma unroll
          for (int i4 = 0; i4 < KP / 4; ++i4) {
            const float4 gq = G4[c * (KP / 4) + i4];
#pragma unroll
            for (int p = 0; p < NP; ++p) {
              den[p] = i4 == 0 ? mul2(bcast2(gq.x), fv[0][p]) : fma2(bcast2(gq.x), fv[4 * i4 + 0][p], den[p]);
              den[p] = fma2(bcast2(gq.y), fv[4 * i4 + 1][p], den[p]);
              den[p] = fma2(bcast2(gq.z), fv[4 * i4 + 2][p], den[p]);
              den[p] = fma2(bcast2(gq.w), fv[4 * i4 + 3][p], den[p]);
            }
          }
          float2 fvc[NP], nvc[NP], out[NP];
          VecIO<VEC>::ld(myF + c * TILE, fvc);
          VecIO<VEC>::ld(myN + c * TILE, nvc);
#pragma unroll
          for (int p = 0; p < NP; ++p) {
            // regularisation terms unconditionally: adding l1 = 0 and l2 * F = 0 is exact, a uniform branch costs more
            const float2 d0 = fma2(bcast2(l2), fvc[p], add2(den[p], bcast2(l1)));
            float2 d = d0;
            // zero denominators -> eps (sklearn _nmf.py:615,701); the Newton quotient needs a normal number
            d.x = (d.x < FLT_MIN_NORMAL) ? EPSILON_F32 : d.x;
            d.y = (d.y < FLT_MIN_NORMAL) ? EPSILON_F32 : d.y;
            out[p] = mul2(fvc[p], div_nr2(nvc[p], d));
            sacc = fma2(nvc[p], out[p], sacc);
          }
          store_items<VEC>(pF, pH, pL, off, out, pscale);
          if constexpr (GRAM) VecIO<VEC>::st(myF + c * TILE, out);
        }
      }
      scal += (double)(sacc.x + sacc.y);
    } else if constexpr (GRAM) {
      float2 z[NP];
#pragma unroll
      for (int p = 0; p < NP; ++p) z[p] = make_float2(0.f, 0.f);
#pragma unroll
      for (int c = 0; c < KP; ++c) VecIO<VEC>::st(myF + c * TILE, z);
    }
    if constexpr (GRAM) {
      __syncthreads();
      if constexpr (VEC == 4) {
        if (f.P_hi) emit_tile_f16<TILE>(f, tileF, K, o, t0);
      }
      if constexpr (SYM) fused_gram_tile_sym<KP, TILE>(tileF, gsum, gplan);
      else fused_gram_tile<KP, TILE>(tileF, gsum);
    }
  }
  return scal;
}

// MU: returns <NUM, F_new> over the thread's items (fp32 within a tile, fp64 across tiles).
// CD: returns sum |projected gradient|.
template <int KP, int VEC, bool CD, bool GRAM>
__device__ __forceinline__ double update_body(const FactorView& f, const float* __restrict__ NUM, int nsplit,
                                              long long sstride, const float* G, int K, int o, float l1, float l2,
                                              int col_begin, int col_end, float* tile, double* gsum) {
  constexpr int NP = VecIO<VEC>::NP;
  constexpr int TILE = UPD_THREADS * VEC;
  const volatile float4* Gv = reinterpret_cast<const volatile float4*>(G);
  const volatile float* Gs = G;
  const unsigned ld = (unsigned)f.ld;
  double scal = 0.0;
  constexpr bool SYM = GRAM && VEC == 4 && (KP == 12 || KP == 16);
  __shared__ int gplan[SYM ? SYM_PLAN_WORDS : 1];
  if constexpr (SYM) sym_gram_plan<KP>(gplan);
#pragma unroll 1
  for (int t0 = col_begin; t0 < col_end; t0 += TILE) {
    const int col = t0 + VEC * threadIdx.x;
    if (col < col_end) {
      const long long e0 = (long long)o * f.ld + col;
      float* const pF = f.F + e0;
      float* const pH = f.F_hi ? f.F_hi + e0 : nullptr;
      float* const pL = f.F_hi ? f.F_lo + e0 : nullptr;
      float2 fv[KP][NP], nv[KP][NP];
      load_items<KP, VEC>(pF, NUM + e0, nsplit, sstride, K, ld, f.n - col, fv, nv);
      float2 pscale[NP];
#pragma unroll
      for (int p = 0; p < NP; ++p) pscale[p] = make_float2(1.f, 1.f);
      if (f.piece_scale) VecIO<VEC>::ld(f.piece_scale + col, pscale);
      float2 sacc = make_float2(0.f, 0.f);
#pragma unroll
      for (int c = 0; c < KP; ++c) {
        float2 out[NP];
        if (c < K) {
          if constexpr (!CD) {
            float2 den[NP];
#pragma unroll
            for (int i4 = 0; i4 < KP / 4; ++i4) {
              const volatile float4& gq = Gv[c * (KP / 4) + i4];
              const float g0 = gq.x, g1 = gq.y, g2 = gq.z, g3 = gq.w;
#pragma unroll
              for (int p = 0; p < NP; ++p) {
                den[p] = i4 == 0 ? mul2(bcast2(g0), fv[0][p]) : fma2(bcast2(g0), fv[4 * i4 + 0][p], den[p]);
                den[p] = fma2(bcast2(g1), fv[4 * i4 + 1][p], den[p]);
                den[p] = fma2(bcast2(g2), fv[4 * i4 + 2][p], den[p]);
                den[p] = fma2(bcast2(g3), fv[4 * i4 + 3][p], den[p]);
              }
            }
#pragma unroll
            for (int p = 0; p < NP; ++p) {
              if (l1 > 0.f) den[p] = add2(den[p], bcast2(l1));
              if (l2 > 0.f) den[p] = fma2(bcast2(l2), fv[c][p], den[p]);
              // zero denominators -> eps (sklearn _nmf.py:615,701); the Newton quotient needs a normal number
              den[p].x = (den[p].x < FLT_MIN_NORMAL) ? EPSILON_F32 : den[p].x;
              den[p].y = (den[p].y < FLT_MIN_NORMAL) ? EPSILON_F32 : den[p].y;
              out[p] = mul2(fv[c][p], div_nr2(nv[c][p], den[p]));
              sacc = fma2(nv[c][p], out[p], sacc);
            }
          } else {
            // -(XHt - l1) + sum_r Gram[t, r] * F[r], summed in the order of the Cython loop (r = 0..K-1)
            float2 g[NP];
#pragma unroll
            for (int p = 0; p < NP; ++p) g[p] = make_float2(l1 - nv[c][p].x, l1 - nv[c][p].y);
#pragma unroll
            for (int i4 = 0; i4 < KP / 4; ++i4) {
              const volatile float4& gq = Gv[c * (KP / 4) + i4];
              const float g0 = gq.x, g1 = gq.y, g2 = gq.z, g3 = gq.w;
#pragma unroll
              for (int p = 0; p < NP; ++p) {
                g[p] = fma2(bcast2(g0), fv[4 * i4 + 0][p], g[p]);
                g[p] = fma2(bcast2(g1), fv[4 * i4 + 1][p], g[p]);
                g[p] = fma2(bcast2(g2), fv[4 * i4 + 2][p], g[p]);
                g[p] = fma2(bcast2(g3), fv[4 * i4 + 3][p], g[p]);
              }
            }
            const float h = Gs[c * KP + c];
            const float hinv = Gs[KP * KP + c];                  // refined 1 / h (0 when h == 0)
#pragma unroll
            for (int p = 0; p < NP; ++p) {
              const float pgx = (fv[c][p].x == 0.f) ? fminf(0.f, g[p].x) : g[p].x;
              const float pgy = (fv[c][p].y == 0.f) ? fminf(0.f, g[p].y) : g[p].y;
              sacc.x += fabsf(pgx);
              sacc.y += fabsf(pgy);
              if (h != 0.f) {                                    // block-uniform
                float2 q = mul2(g[p], bcast2(hinv));             // g / h: quotient + residual correction
                const float2 rem = fma2(bcast2(-h), q, g[p]);
                q = fma2(bcast2(hinv), rem, q);
                fv[c][p].x = fmaxf(fv[c][p].x - q.x, 0.f);
                fv[c][p].y = fmaxf(fv[c][p].y - q.y, 0.f);
              }
              out[p] = fv[c][p];
            }
          }
          store_items<VEC>(pF, pH, pL, (unsigned)c * ld, out, pscale);
        } else {
#pragma unroll
          for (int p = 0; p < NP; ++p) out[p] = make_float2(0.f, 0.f);
        }
        if constexpr (GRAM) VecIO<VEC>::st(tile + c * TILE + VEC * threadIdx.x, out);
      }
      scal += (double)(sacc.x + sacc.y);
    } else if constexpr (GRAM) {
      float2 z[NP];
#pragma unroll
      for (int p = 0; p < NP; ++p) z[p] = make_float2(0.f, 0.f);
#pragma unroll
      for (int c = 0; c < KP; ++c) VecIO<VEC>::st(tile + c * TILE + VEC * threadIdx.x, z);
    }
    if constexpr (GRAM) {
      __syncthreads();
      if constexpr (VEC == 4) {
        if (f.P_hi) emit_tile_f16<TILE>(f, tile, K, o, t0);
      }
      if constexpr (SYM) fused_gram_tile_sym<KP, TILE>(tile, gsum, gplan);
      else fused_gram_tile<KP, TILE>(tile, gsum);
    }
  }
  return scal;
}

#define CNMF_KP_SWITCH(K, KPMAX, CALL)                                            \
  switch (((K) + 3) / 4) {                                                        \
    case 1: { constexpr int KP = 4; CALL; } break;                                \
    case 2: { constexpr int KP = 8; CALL; } break;                                \
    case 3: { constexpr int KP = 12; CALL; } break;                               \
    case 4: { constexpr int KP = 16; CALL; } break;                               \
    case 5: if constexpr (KPMAX >= 20) { constexpr int KP = 20; CALL; } break;    \
    case 6: if constexpr (KPMAX >= 24) { constexpr int KP = 24; CALL; } break;    \
    case 7: if constexpr (KPMAX >= 28) { constexpr int KP = 28; CALL; } break;    \
    default: if constexpr (KPMAX >= 32) { constexpr int KP = 32; CALL; } break;   \
  }

// KPMAX = 16: 4 items per thread, fused Gram available (GRAM).  KPMAX = 32: 2 items per thread, no fused Gram
// (its K x K register tile does not fit beside the update's working set; the engine runs the stand-alone
// Gram kernel for those batches).
template <int KPMAX, bool CD, bool GRAM, int MINB = (KPMAX == 32 ? 2 : 3), bool STREAMN = false>
__global__ void __launch_bounds__(UPD_THREADS, MINB)
update_kernel(FactorView f, const float* __restrict__ NUM, int nsplit, long long sstride,
              const double* __restrict__ gram_in, BatchMeta b, float l1, float l2, FusedOut out) {
  constexpr int VEC = KPMAX == 16 ? 4 : 2;
  const int slot = blockIdx.y;
  const int r = b.rid[slot];
  if (b.done[r]) return;
  const int K = b.k[slot], o = b.off[slot];
  const int KPr = ((K + 3) / 4) * 4;
  __shared__ __align__(16) float G[KPMAX * KPMAX + KPMAX];   // Gram of the other factor (+ CD: 1/diag)
  __shared__ double gsum[GRAM ? KPMAX * KPMAX : 1];
  __shared__ double red[32];
  __shared__ int s_last;
  // dynamic shared memory: [tileF | tileN].  tileF: KP x TILE values of the factor (MU: old, then new; CD + Gram: new)
  // and the Gram reduction scratch; tileN (MU only): KP x TILE products
  extern __shared__ __align__(16) float tile[];
  load_gram_smem(G, gram_in, r, K, KPr, CD ? l2 : 0.f);       // CD: l2 on the diagonal, sklearn _nmf.py:383-385
  if constexpr (GRAM)
    for (int e = threadIdx.x; e < KPr * KPr; e += UPD_THREADS) gsum[e] = 0.0;
  __syncthreads();
  if constexpr (CD) {
    if (threadIdx.x < KPr) {
      const float h = G[threadIdx.x * KPr + threadIdx.x];
      G[KPr * KPr + threadIdx.x] = (h != 0.f) ? rcp_nr(fmaxf(fabsf(h), FLT_MIN_NORMAL)) * (h < 0.f ? -1.f : 1.f) : 0.f;
    }
    __syncthreads();
  }
  const int col_begin = blockIdx.x * f.cpb;
  const int col_end = min(f.n, col_begin + f.cpb);
  const bool want_scal = out.scal_part != nullptr;
  double scal = 0.0;
  if constexpr (CD) {
    CNMF_KP_SWITCH(K, KPMAX, (scal = update_body<KP, VEC, true, GRAM>(f, NUM, nsplit, sstride, G, K, o, l1, 0.f,
                                                                       col_begin, col_end, tile, gsum)));
  } else {
    float* tileN = tile + UPD_TILE_F_FLOATS;
    CNMF_KP_SWITCH(K, KPMAX, (scal = mu_body<KP, VEC, GRAM, STREAMN>(f, NUM, nsplit, sstride, G, K, o, l1, l2, col_begin, col_end,
                                                                      tile, tileN, gsum)));
  }
  const int chunks = gridDim.x;
  if (want_scal) {
    scal = block_sum(scal, red);
    if (threadIdx.x == 0) out.scal_part[(long long)slot * chunks + blockIdx.x] = scal;
  }
  const int stride = b.kp * b.kp;
  if constexpr (GRAM) {
    double* part = out.gram_part + ((long long)slot * chunks + blockIdx.x) * stride;
    for (int e = threadIdx.x; e < KPr * KPr; e += UPD_THREADS) part[e] = gsum[e];
  }
  if (!GRAM && !want_scal) return;
  // ---- last block of the restart: fixed-order sums of the per-block partials
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(&out.counter[r], 1) == chunks - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if constexpr (GRAM) {
    const double* part = out.gram_part + (long long)slot * chunks * stride;
    for (int e = threadIdx.x; e < KPr * KPr; e += UPD_THREADS) {
      double a = 0.0;
#pragma unroll 4
      for (int ch = 0; ch < chunks; ++ch) a += __ldcg(part + (long long)ch * stride + e);
      out.gram[(long long)r * KMAX * KMAX + (e / KPr) * KMAX + (e % KPr)] = a;
    }
  }
  if (want_scal && threadIdx.x < 32) {
    double a = 0.0;
    for (int ch = threadIdx.x; ch < chunks; ch += 32) a += __ldcg(out.scal_part + (long long)slot * chunks + ch);
    a = warp_sum(a);
    if (threadIdx.x == 0) out.scal[r] = a;
  }
  if (threadIdx.x == 0) out.counter[r] = 0;
}

// ------------------------------------------------------------------ <NUM, F> without update
__global__ void __launch_bounds__(UPD_THREADS)
cross_kernel(FactorView f, const float* __restrict__ NUM, int nsplit, long long sstride, BatchMeta b,
             double* __restrict__ cross_partial) {
  const int slot = blockIdx.y;
  const int r = b.rid[slot];
  if (b.done[r]) return;
  const int K = b.k[slot], o = b.off[slot];
  __shared__ double red[32];
  const int col_begin = blockIdx.x * f.cpb;
  const int col_end = min(f.n, col_begin + f.cpb);
  double cross = 0.0;
  for (int col = col_begin + threadIdx.x; col < col_end; col += UPD_THREADS) {
    for (int c = 0; c < K; ++c) {
      const long long e = (long long)(o + c) * f.ld + col;
      float num = NUM[e];
      for (int s = 1; s < nsplit; ++s) num += NUM[s * sstride + e];
      cross += (double)num * (double)f.F[e];
    }
  }
  cross = block_sum(cross, red);
  if (threadIdx.x == 0) cross_partial[(long long)r * gridDim.x + blockIdx.x] = cross;
}

// ------------------------------------------------------------------ K x K Gram partials
// Register-tiled: a thread owns RB rows x KP columns of the K x K Gram and walks over columns of F,
// VEC columns at a time through 8/16-byte loads (KP*VEC values in flight per thread; a first version with
// one 4-byte column per step was latency-bound at ~0.6 TB/s).  TPC threads cooperate on one column group;
// partial sums are fp32 over the thread's columns, then fp64 through shuffles + a fixed-order
// shared-memory reduction (deterministic).  Same per-restart KP dispatch as the update kernels.
template <int KP, int BT>
struct GramCfg {
  static constexpr int TPC = KP <= 8 ? 1 : (KP <= 16 ? 2 : (KP <= 24 ? 4 : 8));   // threads per column group
  static constexpr int RB = (KP + TPC - 1) / TPC;       // rows of the Gram per thread (last block may be partial)
  static constexpr int VEC = KP <= 12 ? 4 : 2;          // consecutive columns per load (register budget)
  static constexpr int COLS_PER_ITER = (BT / TPC) * VEC;
  static constexpr int WARPS = BT / 32;
};

template <int VEC> struct VecLoad;
template <> struct VecLoad<4> {
  static __device__ __forceinline__ void ld(const float* p, float (&v)[4]) {
    const float4 q = *reinterpret_cast<const float4*>(p);
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  }
};
template <> struct VecLoad<2> {
  static __device__ __forceinline__ void ld(const float* p, float (&v)[2]) {
    const float2 q = *reinterpret_cast<const float2*>(p);
    v[0] = q.x; v[1] = q.y;
  }
};

template <int KP, int BT>
__device__ __forceinline__ void gram_body(const FactorView& f, int K, int o, int col_begin, int col_end,
                                          double* part /* smem WARPS x 8 x 32 */, double* __restrict__ out) {
  using C = GramCfg<KP, BT>;
  const int rb = threadIdx.x % C::TPC;                 // which row block of the Gram
  const int cl = threadIdx.x / C::TPC;                 // column-group lane inside the block
  float acc[C::RB][KP];
#pragma unroll
  for (int a = 0; a < C::RB; ++a)
#pragma unroll
    for (int i = 0; i < KP; ++i) acc[a][i] = 0.f;
  const float* __restrict__ Fp = f.F;
  for (int col = col_begin + cl * C::VEC; col < col_end; col += C::COLS_PER_ITER) {   // padding columns hold zeros
    float fv[KP][C::VEC];
#pragma unroll
    for (int i = 0; i < KP; ++i) {
      if (i < K) {
        VecLoad<C::VEC>::ld(Fp + (long long)(o + i) * f.ld + col, fv[i]);
      } else {
#pragma unroll
        for (int u = 0; u < C::VEC; ++u) fv[i][u] = 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < C::VEC; ++u) {
#pragma unroll
      for (int a = 0; a < C::RB; ++a) {
        float fa = 0.f;                                 // fv[rb * RB + a][u] without dynamic register indexing
#pragma unroll
        for (int t = 0; t < C::TPC; ++t)
          if (t == rb && t * C::RB + a < KP) fa = fv[t * C::RB + a < KP ? t * C::RB + a : 0][u];
#pragma unroll
        for (int i = 0; i < KP; ++i) acc[a][i] = fmaf(fa, fv[i][u], acc[a][i]);
      }
    }
  }
  // reduction over the column lanes: xor-shuffles among the lanes that share a row block (lane % TPC),
  // then the 8 warps' partials are summed in fixed order through shared memory -- all in fp64
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < C::RB; ++a) {
    double v[KP];
#pragma unroll
    for (int i = 0; i < KP; ++i) v[i] = (double)acc[a][i];
#pragma unroll
    for (int sh = 16; sh >= C::TPC; sh >>= 1)
#pragma unroll
      for (int i = 0; i < KP; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], sh);
    __syncthreads();
    if (lane < C::TPC) {
#pragma unroll
      for (int i = 0; i < KP; ++i) part[(warp * 8 + lane) * 32 + i] = v[i];
    }
    __syncthreads();
    for (int t = threadIdx.x; t < C::TPC * KP; t += BT) {
      const int rbb = t / KP, i = t % KP;
      const int row = rbb * C::RB + a;
      if (row < KP) {
        double sum = 0.0;
#pragma unroll
        for (int w = 0; w < C::WARPS; ++w) sum += part[(w * 8 + rbb) * 32 + i];
        out[row * KP + i] = sum;
      }
    }
  }
}

// BT = 256: stand-alone launches (one block per SM by registers).  BT = 32: one-warp blocks that fit beside a
// resident GEMM CTA (8 K registers, 2 KB smem), used when the Gram runs on the auxiliary stream under a GEMM.
template <int KPMAX, int BT>
__global__ void __launch_bounds__(BT)
gram_partial_kernel(FactorView f, BatchMeta b, double* __restrict__ gram_partial) {
  const int slot = blockIdx.y;
  const int r = b.rid[slot];
  if (b.done[r]) return;
  const int K = b.k[slot], o = b.off[slot];
  __shared__ double part[(BT / 32) * 8 * 32];
  const int col_begin = blockIdx.x * f.gcpb;
  const int col_end = min(f.n, col_begin + f.gcpb);
  double* out = gram_partial + ((long long)r * gridDim.x + blockIdx.x) * (KPMAX * KPMAX);
  CNMF_KP_SWITCH(K, KPMAX, (gram_body<KP, BT>(f, K, o, col_begin, col_end, part, out)));
}

__global__ void finalize_kernel(const double* __restrict__ gram_partial, double* __restrict__ gram,
                                const double* __restrict__ scal_partial, double* __restrict__ scal, int chunks,
                                BatchMeta b) {
  const int r = b.rid[blockIdx.x];
  if (b.done[r]) return;
  if (gram_partial) {
    const int K = b.k[blockIdx.x];
    const int KP = ((K + 3) / 4) * 4;                   // layout written by gram_body<KP>
    const int stride = b.kp * b.kp;
    for (int e = threadIdx.x; e < KP * KP; e += blockDim.x) {
      double a = 0.0;
      for (int ch = 0; ch < chunks; ++ch) a += gram_partial[((long long)r * chunks + ch) * stride + e];
      const int c = e / KP, i = e % KP;
      gram[(long long)r * KMAX * KMAX + c * KMAX + i] = a;
    }
  }
  if (scal_partial && threadIdx.x == 0) {
    double a = 0.0;
    for (int ch = 0; ch < chunks; ++ch) a += scal_partial[(long long)r * chunks + ch];
    scal[r] = a;
  }
}

// ------------------------------------------------------------------ convergence
__global__ void mu_check_kernel(ConvState st, const double* __restrict__ cross, const double* __restrict__ gramA,
                                const double* __restrict__ gramB, double normX2, BatchMeta b, int it, double tol,
                                int max_iter) {
  // one warp per restart: <gramA, gramB> over K x K entries, lanes stride the entries, fixed-order shuffle tree
  const int slot = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (slot >= b.R) return;
  const int r = b.rid[slot];
  if (st.done[r]) return;
  const int K = b.k[slot];
  double dot = 0.0;
  for (int e = lane; e < K * K; e += 32) {
    const int c = e / K, i = e % K;
    dot += gramA[(long long)r * KMAX * KMAX + c * KMAX + i] * gramB[(long long)r * KMAX * KMAX + c * KMAX + i];
  }
  dot = warp_sum(dot);
  if (lane != 0) return;
  const double err = sqrt(fmax(normX2 - 2.0 * cross[r] + dot, 0.0));
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

__global__ void cd_check_kernel(ConvState st, const double* __restrict__ violA, const double* __restrict__ violB,
                                BatchMeta b, int it, double tol, int max_iter) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= b.R) return;
  const int r = b.rid[slot];
  if (st.done[r]) return;
  const double viol = violA[r] + (violB ? violB[r] : 0.0);
  st.last[r] = viol;
  if (it == 1) st.err0[r] = viol;
  const double v0 = st.err0[r];
  if (v0 == 0.0 || viol / v0 <= tol || it >= max_iter) {
    st.done[r] = 1;
    st.n_iter[r] = it;
  }
}

__global__ void gather_rows_kernel(const float* __restrict__ src, const int* __restrict__ src_off,
                                   float* __restrict__ dst, const int* __restrict__ dst_off,
                                   const int* __restrict__ k, int ld) {
  const int r = blockIdx.x / KMAX, c = blockIdx.x % KMAX;
  if (c >= k[r]) return;
  const float4* s = reinterpret_cast<const float4*>(src + (long long)(src_off[r] + c) * ld);
  float4* d = reinterpret_cast<float4*>(dst + (long long)(dst_off[r] + c) * ld);
  for (int i = threadIdx.x; i < ld / 4; i += blockDim.x) d[i] = s[i];
}

}  // namespace

// ============================================================================ launchers
int launch_split_tf32(const float* src, float* hi, float* lo, long long n_elems, cudaStream_t s) {
  CNMF_REQUIRE(n_elems % 4 == 0, "split_tf32: element count must be a multiple of 4");
  const long long n4 = n_elems / 4;
  if (n4 == 0) return 0;
  const int blocks = (int)((n4 + 255) / 256 < 148 * 16 ? (n4 + 255) / 256 : 148 * 16);
  split_tf32_kernel<<<blocks, 256, 0, s>>>(src, hi, lo, n4);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_split_scaled(const float* src, float* hi, float* lo, int rows, int ld, const float* col_scale, cudaStream_t s) {
  CNMF_REQUIRE(ld % 4 == 0, "split_scaled: ld must be a multiple of 4");
  const long long n4 = (long long)rows * (ld / 4);
  if (n4 == 0) return 0;
  const int blocks = (int)((n4 + 255) / 256 < 148 * 16 ? (n4 + 255) / 256 : 148 * 16);
  split_scaled_kernel<<<blocks, 256, 0, s>>>(src, hi, lo, rows, ld, col_scale);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_emit_f16(const float* F, int rows, int n, int ld, const float* pscale, void* hi, void* mid, float* tile_scale,
                    int n_ktiles, cudaStream_t s) {
  CNMF_REQUIRE(ld % 8 == 0 && (long long)n_ktiles * 512 >= ld, "emit_f16: bad ld / n_ktiles");
  if (rows <= 0) return 0;
  emit_f16_kernel<<<rows, 256, 0, s>>>(F, n, ld, pscale, static_cast<__half*>(hi), static_cast<__half*>(mid), tile_scale,
                                       n_ktiles);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_to_half(const float* src, void* dst, long long n_elems, cudaStream_t s) {
  CNMF_REQUIRE(n_elems % 4 == 0, "to_half: element count must be a multiple of 4");
  const long long n4 = n_elems / 4;
  if (n4 == 0) return 0;
  const int blocks = (int)((n4 + 255) / 256 < 148 * 16 ? (n4 + 255) / 256 : 148 * 16);
  to_half_kernel<<<blocks, 256, 0, s>>>(src, static_cast<__half*>(dst), n4);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_min_positive(const float* X, int rows, int cols, int ld, float* col_min, float* row_min, cudaStream_t s) {
  CNMF_CUDA_CHECK(cudaMemsetAsync(col_min, 0x7f, sizeof(float) * cols, s));   // 0x7f7f7f7f: a huge finite float
  CNMF_CUDA_CHECK(cudaMemsetAsync(row_min, 0x7f, sizeof(float) * rows, s));
  dim3 grid((cols + 255) / 256, (rows + 63) / 64);
  CNMF_REQUIRE(grid.y <= 65535, "min_positive: too many rows for one launch");
  min_positive_kernel<<<grid, 256, 0, s>>>(X, rows, cols, ld, reinterpret_cast<int*>(col_min), reinterpret_cast<int*>(row_min));
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_check_scaled_int(const float* X, int rows, int cols, int ld, const float* row_scale, const float* col_scale,
                            int* n_bad, cudaStream_t s) {
  check_scaled_int_kernel<<<148 * 8, 256, 0, s>>>(X, rows, cols, ld, row_scale, col_scale, n_bad);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_build_counts(const float* X, int rows, int cols, int ld, const float* row_scale, const float* col_scale,
                        float* C, cudaStream_t s) {
  build_counts_kernel<<<148 * 8, 256, 0, s>>>(X, rows, cols, ld, row_scale, col_scale, C);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_fix_scale(float* v, int n, int n_pad, cudaStream_t s) {
  fix_scale_kernel<<<(n_pad + 255) / 256, 256, 0, s>>>(v, n, n_pad);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_transpose(const float* src, int rows, int cols, int ld_src, float* dst, float* dst_hi, float* dst_lo,
                     int ld_dst, cudaStream_t s) {
  dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 8);
  CNMF_REQUIRE(grid.y <= 65535, "transpose: too many rows for one launch");
  transpose_kernel<<<grid, block, 0, s>>>(src, rows, cols, ld_src, dst, dst_hi, dst_lo, ld_dst);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_matrix_sums(const float* X, int rows, int cols, int ld, double* out2, double* scratch, int scratch_len,
                       cudaStream_t s) {
  int blocks = 148 * 8;
  if (2 * blocks > scratch_len) blocks = scratch_len / 2;
  CNMF_REQUIRE(blocks >= 1, "matrix_sums: scratch too small");
  sums_partial_kernel<<<blocks, 256, 0, s>>>(X, rows, cols, ld, scratch);
  sums_final_kernel<<<1, 256, 0, s>>>(scratch, blocks, out2);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

#define CNMF_DISPATCH_KPMAX(kp, CALL)                               \
  switch (kp) {                                                      \
    case 16: { constexpr int KPMAX = 16; CALL; } break;              \
    case 32: { constexpr int KPMAX = 32; CALL; } break;              \
    default: set_last_error("kp must be 16 or 32"); return -1;       \
  }

// MU with the fused Gram at kp == 16 streams the products from global memory one component ahead of their use (no
// product tile in shared memory) at 4 blocks per SM (128 registers); every other form stages what it needs in shared
// memory at 3 (kp 16) or 2 (kp 32) blocks per SM.  The streamed form was the fastest of the layouts and occupancies
// measured on c3 (profiles/r2m_update_variants.log); the kernel is bound by its instruction count, not by occupancy.
template <int KPMAX, bool CD, bool GRAM>
static int launch_update_inst(dim3 grid, const FactorView& f, const float* NUM, int nsplit, long long sstride,
                              const double* gram_in, const BatchMeta& b, float l1, float l2, const FusedOut& out,
                              cudaStream_t s) {
  constexpr bool STREAMN = KPMAX == 16 && !CD && GRAM;
  constexpr int MINB = STREAMN ? 4 : (KPMAX == 32 ? 2 : 3);
  // MU stages the thread's factor values (and, unless the products are streamed, the products) in shared memory
  // (rolled component loop); CD only needs the tile when it also emits the Gram
  const size_t smem = sizeof(float) * (CD ? (GRAM ? (size_t)UPD_TILE_F_FLOATS : 0)
                                          : (size_t)UPD_TILE_F_FLOATS + (STREAMN ? 0 : UPD_TILE_N_FLOATS));
  static bool attr_set[64] = {};               // per device: the attribute belongs to the device's copy of the function
  int dev = 0;
  CNMF_CUDA_CHECK(cudaGetDevice(&dev));
  if (smem > 0 && (dev < 0 || dev >= 64 || !attr_set[dev])) {
    CNMF_CUDA_CHECK(cudaFuncSetAttribute(update_kernel<KPMAX, CD, GRAM, MINB, STREAMN>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  update_kernel<KPMAX, CD, GRAM, MINB, STREAMN><<<grid, UPD_THREADS, smem, s>>>(f, NUM, nsplit, sstride, gram_in, b, l1, l2, out);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

template <bool CD>
static int launch_update(const FactorView& f, const float* NUM, int nsplit, long long sstride, const double* gram_in,
                         const BatchMeta& b, float l1, float l2, const FusedOut& out, cudaStream_t s) {
  CNMF_REQUIRE(f.cpb % upd_tile_cols(b.kp) == 0, "update: cpb must be a multiple of the update tile");
  CNMF_REQUIRE(f.ld % 4 == 0, "update: ld must be a multiple of 4");
  static_assert(16 * UPD_THREADS * 4 == UPD_TILE_N_FLOATS && 32 * UPD_THREADS * 2 == UPD_TILE_N_FLOATS, "tile sizes");
  dim3 grid(col_chunks(f), b.R);
  if (b.kp == 16) {
    if (out.gram_part) return launch_update_inst<16, CD, true>(grid, f, NUM, nsplit, sstride, gram_in, b, l1, l2, out, s);
    return launch_update_inst<16, CD, false>(grid, f, NUM, nsplit, sstride, gram_in, b, l1, l2, out, s);
  }
  if (b.kp == 32) {
    CNMF_REQUIRE(out.gram_part == nullptr, "update: the fused Gram exists for kp == 16 batches only");
    return launch_update_inst<32, CD, false>(grid, f, NUM, nsplit, sstride, gram_in, b, l1, l2, out, s);
  }
  set_last_error("kp must be 16 or 32");
  return -1;
}

int launch_mu_update(const FactorView& f, const float* NUM, int nsplit, long long sstride, const double* gram_in,
                     const BatchMeta& b, float l1, float l2, const FusedOut& out, cudaStream_t s) {
  return launch_update<false>(f, NUM, nsplit, sstride, gram_in, b, l1, l2, out, s);
}

int launch_cd_update(const FactorView& f, const float* NUM, int nsplit, long long sstride, const double* gram_in,
                     const BatchMeta& b, float l1, float l2, const FusedOut& out, cudaStream_t s) {
  return launch_update<true>(f, NUM, nsplit, sstride, gram_in, b, l1, l2, out, s);
}

int launch_cross(const FactorView& f, const float* NUM, int nsplit, long long sstride, const BatchMeta& b,
                 double* cross_partial, cudaStream_t s) {
  dim3 grid(col_chunks(f), b.R);
  cross_kernel<<<grid, UPD_THREADS, 0, s>>>(f, NUM, nsplit, sstride, b, cross_partial);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_gram_partial(const FactorView& f, const BatchMeta& b, double* gram_partial, cudaStream_t s, bool one_warp_blocks) {
  dim3 grid(gram_chunks(f), b.R);
  if (one_warp_blocks) {
    CNMF_DISPATCH_KPMAX(b.kp, (gram_partial_kernel<KPMAX, 32><<<grid, 32, 0, s>>>(f, b, gram_partial)));
  } else {
    CNMF_DISPATCH_KPMAX(b.kp, (gram_partial_kernel<KPMAX, 256><<<grid, 256, 0, s>>>(f, b, gram_partial)));
  }
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_finalize(const double* gram_partial, double* gram, const double* scal_partial, double* scal, int chunks,
                    const BatchMeta& b, cudaStream_t s) {
  finalize_kernel<<<b.R, 256, 0, s>>>(gram_partial, gram, scal_partial, scal, chunks, b);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_mu_check(const ConvState& st, const double* cross, const double* gramA, const double* gramB, double normX2,
                    const BatchMeta& b, int it, double tol, int max_iter, cudaStream_t s) {
  mu_check_kernel<<<(b.R + 3) / 4, 128, 0, s>>>(st, cross, gramA, gramB, normX2, b, it, tol, max_iter);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_cd_check(const ConvState& st, const double* violA, const double* violB, const BatchMeta& b, int it,
                    double tol, int max_iter, cudaStream_t s) {
  cd_check_kernel<<<(b.R + 127) / 128, 128, 0, s>>>(st, violA, violB, b, it, tol, max_iter);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int launch_gather_rows(const float* src, const int* src_off, float* dst, const int* dst_off, const int* k, int R,
                       int ld, cudaStream_t s) {
  if (R == 0) return 0;
  gather_rows_kernel<<<R * KMAX, 128, 0, s>>>(src, src_off, dst, dst_off, k, ld);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace cnmf
