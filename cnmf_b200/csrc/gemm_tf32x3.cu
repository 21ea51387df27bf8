// 3xTF32 tensor-core GEMM for sm_100a (tcgen05 + TMEM + TMA), hand-written PTX.
//
//   C[z] (M x N, row-major, ldc) = A[:, Kz] * B[:, Kz]^T          z = split-K slice
//
// A (M x Kd) and B (N x Kd) are both K-major (row-major with the reduction index contiguous),
// each given as two tf32-representable pieces  A = A_hi + A_lo,  B = B_hi + B_lo  and the
// product is accumulated in fp32 in tensor memory as  A_hi*B_hi + A_lo*B_hi + A_hi*B_lo
// (the dropped A_lo*B_lo term is <= 2^-22 relative): fp32-class accuracy from kind::tf32 MMAs.
//
// This is the shape of both big products of an NMF multiplicative-update / coordinate-descent
// iteration once the restarts are batched (SURVEY.md section 8a rows A2/A3):
//   M = sum of K over live restarts (rows of H_batch or W^T_batch),  N = cells or genes.
//   X H^T   (sklearn _nmf.py:538, :380)  ->  A = H_batch (SK x G),   B = X   (cells x G)
//   W^T X   (sklearn _nmf.py:634, :380)  ->  A = W^T_batch (SK x N), B = X^T (G x cells), split-K
//
// Structure (one CTA per SM, persistent over a static tile schedule, 320 threads):
//   warp 0     TMA producer: cp.async.bulk.tensor 2D, 128B-swizzled tiles, mbarrier full/empty ring
//   warp 1     TMEM allocator + single-thread tcgen05.mma issuer (UMMA 128 x BN x 8, kind::tf32)
//   warps 2-9  accumulate/epilogue: tcgen05.ld 32x32b -> fp32 register accumulators -> float4 stores
//
// Accumulation accuracy.  The tensor core adds each MMA result into the TMEM accumulator with
// truncation: measured on B200, a chain of n MMAs on non-negative data is biased low by about
// n * 3e-8 relative (2.3e-5 at K = 2048), which is far outside the 1e-4 parity budget of an NMF
// run.  So TMEM only ever holds SHORT chains (`chain_kb` k-blocks, at most 16 MMAs: 1 k-block of 12 MMAs
// in the general 3-pass form, 2 k-blocks of 8 MMAs in the exact-B 2-pass form):
// the MMA warp ping-pongs between two TMEM buffers, and the eight accumulate warps drain each
// finished chain into round-to-nearest fp32 register accumulators (128 per thread) while the next
// chain is being issued.  Result: ~4e-7 relative, the same class as an FFMA fp32 GEMM.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <algorithm>
#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"
#include "gemm.h"

namespace cnmf {

namespace {

constexpr int BM = 128;          // UMMA M (rows of A per tile) -- one TMEM lane per row
constexpr int BK = 32;           // fp32 elements per k-block = 128 B = one swizzle row
constexpr int UMMA_K = 8;        // kind::tf32: 32 B of K per instruction
constexpr int NUM_EPI_WARPS = 8;                         // two per TMEM lane quadrant (column halves)
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;      // 320
constexpr long long WAIT_TIMEOUT_CYCLES = 4000000000LL;   // ~2 s: a dead pipeline traps instead of hanging

// BEXACT: the B operand is exactly representable in tf32 (e.g. integer counts), so it needs no "lo" piece:
// 2 MMAs per k-step instead of 3, 64 KB stages (3 of them) instead of 96 KB (2).
template <int BN, int STAGES, bool BEXACT>
struct SmemLayout {
  static constexpr int A_BYTES = BM * BK * 4;              // 16 KB
  static constexpr int B_BYTES = BN * BK * 4;
  static constexpr int STAGE_BYTES = 2 * A_BYTES + (BEXACT ? 1 : 2) * B_BYTES;
  static constexpr int TILE_BYTES = STAGES * STAGE_BYTES;
  static constexpr int BAR_OFFSET = TILE_BYTES;            // full[STAGES], empty[STAGES], tfull[2], tempty[2]
  static constexpr int TMEM_PTR_OFFSET = BAR_OFFSET + (2 * STAGES + 4) * 8;
  static constexpr int EPI_OFFSET = TMEM_PTR_OFFSET + 16;   // per accumulate warp: 32 x 20-float transpose patch
  static constexpr int EPI_BYTES = NUM_EPI_WARPS * 32 * 20 * 4;
  static constexpr int TOTAL = EPI_OFFSET + EPI_BYTES;
  static constexpr int DYN_BYTES = TOTAL + 1024;           // slack for manual 1024 B alignment
};

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int who) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > WAIT_TIMEOUT_CYCLES) {
      printf("cnmf gemm_tf32x3: mbarrier wait timed out (block %d, role %d, parity %u)\n", blockIdx.x, who, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// K-major, 128B-swizzled operand tile: rows of 128 B, 8-row groups 1024 B apart
// (cute::UMMA::SmemDescriptor, canonical layout Swizzle<3,4,3> o ((8,m),(T,2)):((8T,SBO),(1,T))).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);   // start address   bits [0,14)
  d |= static_cast<uint64_t>(1) << 16;                        // LBO (unused for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;                // SBO = 1024 B    bits [32,46)
  d |= static_cast<uint64_t>(1) << 46;                        // descriptor version 1 (sm_100)
  d |= static_cast<uint64_t>(2) << 61;                        // SWIZZLE_128B
  return d;
}

template <bool F16>
__device__ __forceinline__ uint32_t make_idesc(int bn) {
  // cute::UMMA::InstrDescriptor: c=F32 (1<<4), a/b format @7/@10 (TF32 = 2, F16 = 0), K-major A and B, N>>3 @17, M>>4 @24
  const uint32_t fmt = F16 ? 0u : 2u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (static_cast<uint32_t>(bn >> 3) << 17) |
         (static_cast<uint32_t>(BM >> 4) << 24);
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------ the kernel
// F16 (with BEXACT): operands are fp16 (two pieces of A, one exact B); a k-block is still 128 B per row = 64 elements,
// a k-step still 32 B = 16 elements (UMMA_K of kind::f16), so the smem / TMA / descriptor byte geometry is unchanged.
//
// 320 threads = 10 warps, allocated as 12 (granularity 4): at most 65536 / (12 * 32) = 170 registers per thread --
// __launch_bounds__ makes ptxas pick 168; a higher __maxnreg__ compiles but cannot launch
template <int BN, int STAGES, bool BEXACT, bool F16>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                   const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                   float* __restrict__ C, int M, int N, int ldc, long long c_split_stride,
                   int m_tiles, int n_tiles, int splits, int total_kb, int kb_per_split, int chain_kb, int bn,
                   const float* __restrict__ out_scale, const float* __restrict__ a_tile_scale, int a_tiles, int a_gshift) {
  static_assert(!F16 || BEXACT, "the fp16 path exists for exact integer B operands only");
  constexpr int BKE = F16 ? 2 * BK : BK;                        // elements per k-block
  using L = SmemLayout<BN, STAGES, BEXACT>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;     // SWIZZLE_128B needs 1024 B alignment
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  const uint32_t bar_base = smem_base + L::BAR_OFFSET;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem_gen + L::TMEM_PTR_OFFSET);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr uint32_t TMEM_COLS = 2 * BN;                      // two accumulators (power of two: 256 or 512)
  const int worker = static_cast<int>(blockIdx.x);
  const int n_workers = static_cast<int>(gridDim.x);

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), NUM_EPI_WARPS);               // one arrival per accumulate warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_base + L::TMEM_PTR_OFFSET), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  const int items = m_tiles * n_tiles * splits;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int w = worker; w < items; w += n_workers) {
        const int mt = w % m_tiles;
        const int nt = (w / m_tiles) % n_tiles;
        const int z = w / (m_tiles * n_tiles);
        const int kb0 = z * kb_per_split;
        const int kb1 = min(total_kb, kb0 + kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u, 0);
          const uint32_t st = smem_base + stage * L::STAGE_BYTES;
          const uint32_t stage_tx = 2u * L::A_BYTES + (BEXACT ? 1u : 2u) * static_cast<uint32_t>(bn) * BK * 4u;
          mbar_arrive_expect_tx(full_bar(stage), stage_tx);
          tma_load_2d(st, &tmA_hi, full_bar(stage), kb * BKE, mt * BM);
          tma_load_2d(st + L::A_BYTES, &tmA_lo, full_bar(stage), kb * BKE, mt * BM);
          tma_load_2d(st + 2 * L::A_BYTES, &tmB_hi, full_bar(stage), kb * BKE, nt * bn);
          if constexpr (!BEXACT) tma_load_2d(st + 2 * L::A_BYTES + L::B_BYTES, &tmB_lo, full_bar(stage), kb * BKE, nt * bn);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one thread) =====================
    if (lane == 0) {
      const uint32_t idesc = make_idesc<F16>(bn);               // UMMA N = bn (multiple of 16, <= BN)
      int stage = 0;
      uint32_t phase = 0;
      int buf = 0;
      uint32_t buf_phase = 0;
      for (int w = worker; w < items; w += n_workers) {
        const int z = w / (m_tiles * n_tiles);
        const int kb0 = z * kb_per_split;
        const int kb1 = min(total_kb, kb0 + kb_per_split);
        for (int c0 = kb0; c0 < kb1; c0 += chain_kb) {          // one short accumulation chain per TMEM buffer
          const int c1 = min(kb1, c0 + chain_kb);
          mbar_wait(tempty_bar(buf), buf_phase ^ 1u, 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(buf * BN);
          for (int kb = c0; kb < c1; ++kb) {
            mbar_wait(full_bar(stage), phase, 2);
            tc_fence_after();
            const uint32_t st = smem_base + stage * L::STAGE_BYTES;
            const uint64_t a_hi = make_smem_desc(st);
            const uint64_t a_lo = make_smem_desc(st + L::A_BYTES);
            const uint64_t b_hi = make_smem_desc(st + 2 * L::A_BYTES);
            const uint64_t b_lo = make_smem_desc(st + 2 * L::A_BYTES + L::B_BYTES);
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint64_t koff = static_cast<uint64_t>((k * UMMA_K * 4) >> 4);   // +32 B per k-step inside the swizzle row
              const uint32_t acc0 = (kb > c0 || k > 0) ? 1u : 0u;
              if constexpr (F16) {
                umma_f16(tmem_d, a_lo + koff, b_hi + koff, idesc, acc0);    // small terms first
                umma_f16(tmem_d, a_hi + koff, b_hi + koff, idesc, 1u);
              } else {
                umma_tf32(tmem_d, a_lo + koff, b_hi + koff, idesc, acc0);   // small terms first
                if constexpr (!BEXACT) umma_tf32(tmem_d, a_hi + koff, b_lo + koff, idesc, 1u);
                umma_tf32(tmem_d, a_hi + koff, b_hi + koff, idesc, 1u);
              }
            }
            umma_commit(empty_bar(stage));                       // smem slot is free once these MMAs have read it
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
          umma_commit(tfull_bar(buf));                           // chain complete -> accumulate warps
          if (++buf == 2) { buf = 0; buf_phase ^= 1u; }
        }
      }
    }
  } else {
    // ===================== accumulate + epilogue (8 warps) =====================
    // tcgen05.ld: warp w may touch TMEM lanes 32*(w%4) .. +31.  Warps 2-5 own columns [0, BN/2),
    // warps 6-9 own [BN/2, BN) of their lane quadrant.
    constexpr int HALF = BN / 2;
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    int buf = 0;
    uint32_t buf_phase = 0;
    for (int w = worker; w < items; w += n_workers) {
      const int mt = w % m_tiles;
      const int nt = (w / m_tiles) % n_tiles;
      const int z = w / (m_tiles * n_tiles);
      const int kb0 = z * kb_per_split;
      const int kb1 = min(total_kb, kb0 + kb_per_split);
      float acc[HALF];
#pragma unroll
      for (int i = 0; i < HALF; ++i) acc[i] = 0.f;
      // f16: power-of-two scale of this thread's A row for the 512-element group a chain belongs to (8 k-blocks)
      const int arow = mt * BM + q * 32 + lane;
      const float* sc_row = (F16 && a_tile_scale && arow < M) ? a_tile_scale + static_cast<long long>(arow) * a_tiles : nullptr;
      for (int c0 = kb0; c0 < kb1; c0 += chain_kb) {
        float sc = 1.f;
        if (F16 && sc_row) sc = sc_row[c0 >> a_gshift];
        mbar_wait(tfull_bar(buf), buf_phase, 3);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                               static_cast<uint32_t>(buf * BN + half * HALF);
#pragma unroll
        for (int c = 0; c < HALF; c += 32) {
          if (half * HALF + c < bn) {                  // warp-uniform: columns >= bn were not computed
            uint32_t r[32];
            tmem_ld32(taddr + c, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              if constexpr (F16) acc[c + i] = fmaf(__uint_as_float(r[i]), sc, acc[c + i]);   // exact scaling, one rounding
              else acc[c + i] += __uint_as_float(r[i]);   // round-to-nearest fp32
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(buf));    // one arrival per warp
        if (++buf == 2) { buf = 0; buf_phase ^= 1u; }
      }
      // Epilogue.  A thread owns one output row, so a direct store touches 32 rows x 16 B per instruction (32 cache
      // lines: the LSU, not the tensor pipe, then paces short tiles -- the 720-tile W half ran at 0.76 of the MMA rate
      // against 0.92 for the long-K H half).  Each warp transposes 16-column chunks through a private 32 x 20-float
      // shared-memory patch instead, so that one store instruction writes 8 rows x 64 B.
      {
        float* patch = reinterpret_cast<float*>(smem_gen + L::EPI_OFFSET) + (warp - 2) * (32 * 20);
        const int row0 = mt * BM + q * 32;
        const int col0 = nt * bn + half * HALF;
        const int sub_r = lane >> 2, sub_c = (lane & 3) * 4;
        float* cbase = C + static_cast<long long>(z) * c_split_stride;
#pragma unroll
        for (int c = 0; c < HALF; c += 16) {
          if (half * HALF + c < bn) {                     // warp-uniform (bn is a multiple of 16)
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              float4 v = make_float4(acc[c + i], acc[c + i + 1], acc[c + i + 2], acc[c + i + 3]);
              if (out_scale && col0 + c + i + 3 < ldc) {  // per-output-column scale (length >= ldc, zero padded)
                const float4 sc = *reinterpret_cast<const float4*>(out_scale + col0 + c + i);
                v.x *= sc.x; v.y *= sc.y; v.z *= sc.z; v.w *= sc.w;
              }
              *reinterpret_cast<float4*>(patch + lane * 20 + i) = v;
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int r = sub_r + 8 * j;
              const float4 v = *reinterpret_cast<const float4*>(patch + r * 20 + sub_c);
              const int grow = row0 + r, gcol = col0 + c + sub_c;
              if (grow < M && gcol + 3 < ldc) *reinterpret_cast<float4*>(cbase + static_cast<long long>(grow) * ldc + gcol) = v;
            }
            __syncwarp();
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  });
  return fn;
}

// 2D fp32 tensor (rows x cols, row stride ld elements), box = 32 cols x box_rows rows, 128B swizzle, zero OOB fill.
// Encoded maps are cached by (pointer, shape, box): the solver relaunches the same few operand views a thousand
// times per solve, and the driver call costs more than the launch itself.
struct MapKey {
  const void* ptr; int rows, cols, ld, box_rows, f16;
  bool operator<(const MapKey& o) const {
    return std::tie(ptr, rows, cols, ld, box_rows, f16) < std::tie(o.ptr, o.rows, o.cols, o.ld, o.box_rows, o.f16);
  }
};

int make_map(CUtensorMap* map, const float* ptr, int rows, int cols, int ld, int box_rows, bool f16 = false) {
  static std::mutex mu;
  static std::map<MapKey, CUtensorMap> cache;
  const MapKey key{ptr, rows, cols, ld, box_rows, f16 ? 1 : 0};
  {
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find(key);
    if (it != cache.end()) { *map = it->second; return 0; }
  }
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) { set_last_error("cuTensorMapEncodeTiled entry point not available"); return -2; }
  const int esize = f16 ? 2 : 4;                      // a box row is always 128 B: 32 fp32 or 64 fp16 elements
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * esize};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(128 / esize), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)));
    return -2;
  }
  std::lock_guard<std::mutex> lock(mu);
  if (cache.size() >= 512) cache.clear();             // views are few; a runaway caller just re-encodes
  cache.emplace(key, *map);
  return 0;
}

template <int BN, int STAGES, bool BEXACT, bool F16>
int launch(const GemmArgs& g, cudaStream_t stream) {
  using L = SmemLayout<BN, STAGES, BEXACT>;
  constexpr int BKE = F16 ? 2 * BK : BK;
  CUtensorMap mAh, mAl, mBh, mBl;
  int rc;
  if ((rc = make_map(&mAh, g.A_hi, g.M, g.Kd, g.lda, BM, F16))) return rc;
  if ((rc = make_map(&mAl, g.A_lo, g.M, g.Kd, g.lda, BM, F16))) return rc;
  int dev = 0, sms = 0;
  CNMF_CUDA_CHECK(cudaGetDevice(&dev));
  CNMF_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int m_tiles = (g.M + BM - 1) / BM;
  // Tile width: the UMMA N is a runtime value (multiple of 16, <= BN), normally supplied by gemm_plan().
  int bn = g.bn;
  if (bn <= 0 || bn > BN || bn % 16 != 0) {
    const int sp = gemm_effective_splits(g.Kd, g.splits, F16 ? 1 : 0);
    if (g.N <= BN) {
      bn = ((g.N + 15) / 16) * 16;
    } else {
      long long best = -1;
      bn = BN;
      for (int cand = BN; cand >= 192; cand -= 16) {
        const long long tiles = (long long)m_tiles * ((g.N + cand - 1) / cand) * sp;
        const long long cost = ((tiles + sms - 1) / sms) * (cand + 64);
        if (best < 0 || cost < best) { best = cost; bn = cand; }
      }
    }
  }
  if ((rc = make_map(&mBh, g.B_hi, g.N, g.Kd, g.ldb, bn, F16))) return rc;
  if ((rc = make_map(&mBl, BEXACT ? g.B_hi : g.B_lo, g.N, g.Kd, g.ldb, bn, F16))) return rc;

  const int n_tiles = (g.N + bn - 1) / bn;
  const int total_kb = (g.Kd + BKE - 1) / BKE;
  int splits = g.splits < 1 ? 1 : g.splits;
  if (splits > total_kb) splits = total_kb;
  int kb_per_split = (total_kb + splits - 1) / splits;
  if (F16 && (kb_per_split & 1)) ++kb_per_split;             // chains (2 k-blocks) must not straddle a 512-element scale group
  splits = (total_kb + kb_per_split - 1) / kb_per_split;      // no empty slices
  if (splits != g.splits_effective) { set_last_error("gemm: splits_effective mismatch (use gemm_effective_splits)"); return -1; }

  auto kern = gemm_tf32x3_kernel<BN, STAGES, BEXACT, F16>;
  static bool attr_set[64] = {};              // per device: a second GPU in the same process needs its own call
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    CNMF_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::DYN_BYTES));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  const int items = m_tiles * n_tiles * splits;
  const int grid = items < sms ? items : sms;
  // k-blocks per TMEM accumulation chain: at most 16 MMAs between drains (general: 1 k-block = 12 MMAs,
  // exact-B and f16: 2 k-blocks = 16 MMAs; with 8 MMAs per chain the drain, not the tensor pipe, paced the kernel).
  // f16 scale groups of 512 elements = 8 k-blocks (a_gshift = 3): chains of 2 never straddle one.
  const int chain_kb = BEXACT ? 2 : 1;
  kern<<<grid, NUM_THREADS, L::DYN_BYTES, stream>>>(mAh, mAl, mBh, mBl, g.C, g.M, g.N, g.ldc, g.c_split_stride,
                                                    m_tiles, n_tiles, splits, total_kb, kb_per_split,
                                                    chain_kb, bn, g.out_col_scale, g.a_tile_scale, g.a_tiles, 3);
  CNMF_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

// Split-K factor as a function of the reduction length ONLY: slices of 64 k-blocks (4 096 fp16 / 2 048 fp32
// elements), at most 16 of them.  The partition of a restart's reduction -- and with it every rounding of its
// products -- is then the same whatever else shares the batch and however far the batch has been compacted:
// a (k, seed) restart gives the same spectra alone, in a worker's shard or in the full K-sweep, which is the
// reference's semantics (independent sklearn calls, cnmf.py:735-745).
int gemm_fixed_splits(int Kd, int f16) {
  const int bke = f16 ? 2 * BK : BK;
  const int total_kb = (Kd + bke - 1) / bke;
  const int s = std::max(1, std::min(16, (total_kb + 63) / 64));
  return gemm_effective_splits(Kd, s, f16);
}

void gemm_plan(int M, int N, int Kd, int sm_count, int* splits_out, int* bn_out, int f16) {
  const int m_tiles = (M + BM - 1) / BM;
  const int bke = f16 ? 2 * BK : BK;
  const int total_kb = (Kd + bke - 1) / bke;
  const int s = gemm_fixed_splits(Kd, f16);
  const int kbps = (total_kb + s - 1) / s;
  double best = -1.0;
  int best_bn = 256;
  // the tile width only groups output columns (no effect on any sum): narrow tiles (down to 128 columns; below
  // that the accumulate warps, not the MMA chain, pace a tile) pay off when a compacted batch leaves less than
  // one wave of 256-wide tiles
  const int bn_lo = N <= 256 ? ((N + 15) / 16) * 16 : 128;
  const int bn_hi = N <= 256 ? bn_lo : 256;
  for (int bn = bn_hi; bn >= bn_lo; bn -= 16) {
    const long long items = (long long)m_tiles * ((N + bn - 1) / bn) * s;
    const long long waves = (items + sm_count - 1) / sm_count;
    // tile cost bn + 64: per-tile A traffic / fill that does not shrink with bn; + 6 k-blocks of pipeline
    // fill and epilogue per item
    const double cost = (double)waves * (bn + 64) * (kbps + 6);
    if (best < 0 || cost < best) { best = cost; best_bn = bn; }
  }
  *splits_out = s;
  *bn_out = best_bn;
}

int gemm_effective_splits(int Kd, int splits, int f16) {
  const int bke = f16 ? 2 * BK : BK;
  const int total_kb = (Kd + bke - 1) / bke;
  if (splits < 1) splits = 1;
  if (splits > total_kb) splits = total_kb;
  int kb_per_split = (total_kb + splits - 1) / splits;
  if (f16 && (kb_per_split & 1)) ++kb_per_split;   // same rule as the launcher: slices start on even k-blocks
  return (total_kb + kb_per_split - 1) / kb_per_split;
}

int gemm_tf32x3(const GemmArgs& g, cudaStream_t stream) {
  CNMF_REQUIRE(g.M > 0 && g.N > 0 && g.Kd > 0, "gemm: empty problem");
  CNMF_REQUIRE(g.lda % 4 == 0 && g.ldb % 4 == 0 && g.ldc % 4 == 0, "gemm: leading dimensions must be multiples of 4 floats");
  CNMF_REQUIRE((reinterpret_cast<uintptr_t>(g.A_hi) | reinterpret_cast<uintptr_t>(g.A_lo) |
                reinterpret_cast<uintptr_t>(g.B_hi) | reinterpret_cast<uintptr_t>(g.B_lo) |
                reinterpret_cast<uintptr_t>(g.C) | reinterpret_cast<uintptr_t>(g.out_col_scale)) % 16 == 0,
               "gemm: pointers must be 16-byte aligned");
  if (g.f16) {
    CNMF_REQUIRE(g.b_exact, "gemm: the fp16 path needs an exact B operand");
    CNMF_REQUIRE(g.lda % 8 == 0 && g.ldb % 8 == 0, "gemm: fp16 leading dimensions must be multiples of 8 halves");
    CNMF_REQUIRE(!g.a_tile_scale || g.a_tiles * 512 >= g.Kd, "gemm: a_tiles does not cover the reduction length");
    return launch<256, 3, true, true>(g, stream);
  }
  if (g.b_exact) {
    return launch<256, 3, true, false>(g, stream);
  }
  return launch<256, 2, false, false>(g, stream);
}

}  // namespace cnmf
