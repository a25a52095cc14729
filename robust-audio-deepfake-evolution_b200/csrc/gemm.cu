// C[M, N] = A[M, K] . B[N, K]^T (+ bias) on the 5th-generation tensor cores.  sm_100a only.
//
// Reference: the nn.Linear projections of the Bi-Mamba block - in_proj (mamba_block.py:22,48),
// x_proj (:33,73), out_proj (:39,62) - and the data-gradient GEMMs of their autograd, plus the two
// Linear layers of the encoder's feed-forward (DualStreamSEMamba.py:460-464).  All of them are
// "NT" products of row-major (K-major) bf16/fp16 operands with fp32 accumulation.
//
// Structure (one 128 x BLOCK_N output tile per CTA, 4 warps):
//   * warp 0, one elected lane: TMA producer.  `cp.async.bulk.tensor.2d` (UTMALDG) loads 128 x 64
//     and BLOCK_N x 64 boxes of A and B into a ring of shared-memory stages in the 128-byte
//     swizzled K-major layout the tensor core reads; rows / columns beyond M, N, K are zero-filled by
//     the TMA unit, so ragged shapes (K = 144, N = 48, M = B*L) need no padding copies.
//   * warp 1, one elected lane: MMA issuer.  `tcgen05.mma.cta_group::1.kind::f16` (UTCHMMA),
//     M = 128, N = BLOCK_N, K = 16 per instruction, accumulating in TMEM; `tcgen05.commit` releases
//     each stage back to the producer and finally signals the epilogue.
//   * all 4 warps: epilogue.  `tcgen05.ld` (LDTM) moves the accumulator rows (one TMEM lane per
//     thread) to registers 16 columns at a time; bias add, conversion and 16/32-byte global stores.
// Stages, full/empty mbarriers and the TMEM allocation follow the usual sm_100 pipeline.
#include <cuda.h>

#include <cstdlib>
#include <type_traits>

#include "common.cuh"

namespace bimamba {

constexpr int kGM = 128;       // tile rows (UMMA M)
constexpr int kGK = 64;        // K per stage: 64 x 2 B = one 128-byte swizzle row
constexpr int kGStagesMax = 4;
constexpr int kGThreads = 128;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}

// 16 fp32 accumulators (+ bias) -> 16 outputs in a padded shared-memory row
template <typename TOut>
__device__ __forceinline__ void stage16(TOut* dst, const uint32_t* r, const float* bias, int n, int N) {
  float v[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    v[j] = __uint_as_float(r[j]);
    if (bias != nullptr && n + j < N) v[j] += __ldg(bias + n + j);
  }
  if constexpr (sizeof(TOut) == 2) {
    uint32_t pk[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if constexpr (std::is_same<TOut, __nv_bfloat16>::value) {
        const __nv_bfloat162 h2 = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
        pk[j] = *reinterpret_cast<const uint32_t*>(&h2);
      } else {
        const __half2 h2 = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
        pk[j] = *reinterpret_cast<const uint32_t*>(&h2);
      }
    }
    reinterpret_cast<uint4*>(dst)[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    reinterpret_cast<uint4*>(dst)[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      reinterpret_cast<float4*>(dst)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  }
}

// K-major, 128-byte swizzle: 8-row atoms of 1024 bytes; LBO = 1 (unused), SBO = 1024 B, version 1.
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}

template <typename TOut>
__global__ void __launch_bounds__(kGThreads)
gemm_nt_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               TOut* __restrict__ C, const float* __restrict__ bias, const TOut* __restrict__ addend, int M, int N,
               int K, int64_t ldc, int block_n,
               int stages, uint32_t idesc, uint32_t tmem_cols, int staged) {
  pdl_prologue();
  extern __shared__ __align__(1024) unsigned char gsm[];
  __shared__ __align__(8) uint64_t full_bar[kGStagesMax], empty_bar[kGStagesMax], accum_bar;
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * kGM, n0 = blockIdx.y * block_n;
  const int nkb = (K + kGK - 1) / kGK;
  const uint32_t a_bytes = kGM * kGK * 2, b_bytes = (uint32_t)block_n * kGK * 2;
  const uint32_t stage_bytes = a_bytes + ((b_bytes + 1023u) & ~1023u);  // keep every operand 1024-byte aligned
  // 1024-byte aligned start of the stages; derived by offset (not by integer casts) so that the compiler keeps
  // the shared address space and the epilogue's tile accesses are STS / LDS, not generic stores
  unsigned char* base = gsm + ((1024u - (smem_u32(gsm) & 1023u)) & 1023u);

  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&accum_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_b)) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0 && lane == 0) {
    // ---- TMA producer
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % stages;
      if (kb >= stages) mbar_wait(&empty_bar[s], ((kb / stages) - 1) & 1);
      unsigned char* sa = base + (size_t)s * stage_bytes;
      mbar_expect_tx(&full_bar[s], a_bytes + b_bytes);
      tma_load_2d(sa, &map_a, &full_bar[s], kb * kGK, m0);
      tma_load_2d(sa + a_bytes, &map_b, &full_bar[s], kb * kGK, n0);
    }
  } else if (warp == 1 && lane == 0) {
    // ---- MMA issuer
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % stages;
      mbar_wait(&full_bar[s], (kb / stages) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t sa = smem_u32(base + (size_t)s * stage_bytes);
      const uint64_t da = make_kmajor_sw128_desc(sa), db = make_kmajor_sw128_desc(sa + a_bytes);
#pragma unroll
      for (int k = 0; k < kGK / 16; ++k) {
        // advance 16 elements (32 bytes) along K inside the swizzle row: +2 in 16-byte units
        umma_f16(tmem_base, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
      }
      umma_commit(&empty_bar[s]);  // frees this stage when the MMAs above have read it
    }
    umma_commit(&accum_bar);       // accumulator complete
  }
  __syncwarp();  // lanes 1..31 of the two role warps park here instead of spinning next to their leader

  // ---- epilogue: all warps; thread = one accumulator row (TMEM lane)
  mbar_wait(&accum_bar, 0);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  __syncwarp();
  const int row = warp * 32 + lane;
  const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
  if (staged) {
    // TMEM -> registers -> padded shared tile (the pipeline stages are free: every MMA has completed),
    // then row-contiguous 16-byte global stores (and addend loads) by consecutive threads.
    const int row_bytes = block_n * (int)sizeof(TOut) + 16;  // +16: consecutive rows start 4 banks apart
    unsigned char* tile = base;
    unsigned char* my_row = tile + (size_t)row * row_bytes;
    int c = 0;
    for (; c + 32 <= block_n; c += 32) {
      uint32_t r[32];
      tmem_ld32(trow + (uint32_t)c, r);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      stage16<TOut>(reinterpret_cast<TOut*>(my_row) + c, r, bias, n0 + c, N);
      stage16<TOut>(reinterpret_cast<TOut*>(my_row) + c + 16, r + 16, bias, n0 + c + 16, N);
    }
    if (c < block_n) {
      uint32_t r[16];
      tmem_ld16(trow + (uint32_t)c, r);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      stage16<TOut>(reinterpret_cast<TOut*>(my_row) + c, r, bias, n0 + c, N);
    }
    __syncthreads();
    constexpr int EV = 16 / sizeof(TOut);          // elements per 16-byte vector
    const int vpr = block_n / EV;                  // vectors per tile row (block_n is a multiple of 16)
    const int drr = kGThreads / vpr, dvv = kGThreads % vpr;
    int rr = (int)threadIdx.x / vpr, vv = (int)threadIdx.x % vpr;
    const int total = kGM * vpr;
#pragma unroll 4
    for (int idx = threadIdx.x; idx < total; idx += kGThreads) {
      const int m = m0 + rr, n = n0 + vv * EV;
      if (m < M && n < N) {   // N is a multiple of EV on this path
        uint4 val = *reinterpret_cast<const uint4*>(tile + (size_t)rr * row_bytes + (size_t)vv * 16);
        TOut* dst = C + (int64_t)m * ldc + n;
        if (addend != nullptr) {
          const uint4 ad = *reinterpret_cast<const uint4*>(addend + (int64_t)m * ldc + n);
          TOut* pv = reinterpret_cast<TOut*>(&val);
          const TOut* pa = reinterpret_cast<const TOut*>(&ad);
#pragma unroll
          for (int j = 0; j < EV; ++j) pv[j] = from_f<TOut>(to_f(pv[j]) + to_f(pa[j]));
        }
        *reinterpret_cast<uint4*>(dst) = val;
      }
      rr += drr;
      vv += dvv;
      if (vv >= vpr) {
        vv -= vpr;
        ++rr;
      }
    }
  } else {
    const int m = m0 + row;
    for (int c = 0; c < block_n; c += 16) {
      uint32_t r[16];
      tmem_ld16(trow + (uint32_t)c, r);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      const int n = n0 + c;
      if (m < M && n < N) {
        TOut* dst = C + (int64_t)m * ldc + n;
        const TOut* src = addend != nullptr ? addend + (int64_t)m * ldc + n : nullptr;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          if (n + j < N) {
            float v = __uint_as_float(r[j]);
            if (bias != nullptr) v += __ldg(bias + n + j);
            // round the Linear output to TOut before the addend, as the staged epilogue does: same bits on both paths
            if (src != nullptr) v = to_f(from_f<TOut>(v)) + to_f(src[j]);
            dst[j] = from_f<TOut>(v);
          }
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

// ---- persistent, warp-specialised variant --------------------------------------------------------------
// One CTA per SM walks the (M tile, N tile) list with a static stride.  Roles: warp 0 = TMA producer over a
// 4-stage shared-memory ring that runs ahead across tiles; warp 1 = MMA issuer alternating between TWO TMEM
// accumulators; warps 2-5 = epilogue (each owns the TMEM lane quarter warp % 4): they drain accumulator j
// (TMEM -> registers -> padded shared tile -> row-contiguous global stores) while the MMAs of tile j+1 run, so
// load, tensor-core and store phases of consecutive tiles overlap inside one CTA.
constexpr int kPStages = 4;
constexpr int kPEpiWarps = 8;                       // two warps per TMEM lane quarter, each takes half of the columns
constexpr int kPThreads = 64 + 32 * kPEpiWarps;

template <typename TOut>
__global__ void __launch_bounds__(kPThreads, 1)
gemm_nt_persist_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                       TOut* __restrict__ C, const float* __restrict__ bias, const TOut* __restrict__ addend, int M,
                       int N, int K, int64_t ldc, int block_n, uint32_t idesc, uint32_t tmem_cols, uint32_t acc_stride) {
  pdl_prologue();
  extern __shared__ __align__(1024) unsigned char gsm[];
  __shared__ __align__(8) uint64_t full_bar[kPStages], empty_bar[kPStages], acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = (K + kGK - 1) / kGK;
  const int ntm = (M + kGM - 1) / kGM, ntn = (N + block_n - 1) / block_n;
  const int ntiles = ntm * ntn;
  const uint32_t a_bytes = kGM * kGK * 2, b_bytes = (uint32_t)block_n * kGK * 2;
  const uint32_t stage_bytes = a_bytes + ((b_bytes + 1023u) & ~1023u);
  unsigned char* base = gsm + ((1024u - (smem_u32(gsm) & 1023u)) & 1023u);
  unsigned char* tile = base + (size_t)kPStages * stage_bytes;   // epilogue staging tile (after the ring)

  if (threadIdx.x == 0) {
    for (int s = 0; s < kPStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int j = 0; j < 2; ++j) {
      mbar_init(&acc_full[j], 1);
      mbar_init(&acc_empty[j], kPEpiWarps);   // one arrival per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_b)) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    if (lane == 0) {  // ---- TMA producer
      uint32_t it = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int m0 = (t / ntn) * kGM, n0 = (t % ntn) * block_n;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const uint32_t s = it % kPStages, ph = (it / kPStages) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          unsigned char* sa = base + (size_t)s * stage_bytes;
          mbar_expect_tx(&full_bar[s], a_bytes + b_bytes);
          tma_load_2d(sa, &map_a, &full_bar[s], kb * kGK, m0);
          tma_load_2d(sa + a_bytes, &map_b, &full_bar[s], kb * kGK, n0);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {  // ---- MMA issuer
      uint32_t it = 0, lt = 0;
      for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++lt) {
        const uint32_t ab = lt & 1;
        mbar_wait(&acc_empty[ab], ((lt >> 1) & 1) ^ 1);   // epilogue has drained this accumulator
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t tacc = tmem_base + ab * acc_stride;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const uint32_t s = it % kPStages, ph = (it / kPStages) & 1;
          mbar_wait(&full_bar[s], ph);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t sa = smem_u32(base + (size_t)s * stage_bytes);
          const uint64_t da = make_kmajor_sw128_desc(sa), db = make_kmajor_sw128_desc(sa + a_bytes);
#pragma unroll
          for (int k = 0; k < kGK / 16; ++k)
            umma_f16(tacc, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty_bar[s]);
        }
        umma_commit(&acc_full[ab]);
      }
    }
  } else {
    // ---- epilogue warps 2..9: TMEM lane quarter q = warp % 4 (rows q*32 .. q*32+31), column half hcol
    const int q = warp & 3;
    const int hcol = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const int et = threadIdx.x - 64;               // 0..255 within the epilogue group
    constexpr int kET = 32 * kPEpiWarps;
    const int row_bytes = block_n * (int)sizeof(TOut) + 16;
    constexpr int EV = 16 / sizeof(TOut);
    const int vpr = block_n / EV;
    const int drr = kET / vpr, dvv = kET % vpr;
    // this warp's 16-column chunks: [c_lo, c_hi) in units of 16 columns
    const int nch = block_n / 16;
    const int c_lo = hcol == 0 ? 0 : (nch + 1) / 2, c_hi = hcol == 0 ? (nch + 1) / 2 : nch;
    uint32_t lt = 0;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++lt) {
      const int m0 = (t / ntn) * kGM, n0 = (t % ntn) * block_n;
      const uint32_t ab = lt & 1;
      mbar_wait(&acc_full[ab], (lt >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t trow = tmem_base + ab * acc_stride + ((uint32_t)(q * 32) << 16);
      unsigned char* my_row = tile + (size_t)row * row_bytes;
      // all TMEM loads of this warp's columns are issued before the single wait (<= 6 chunks of 16 columns)
      uint32_t r[6][16];
#pragma unroll
      for (int j = 0; j < 6; ++j)
        if (c_lo + j < c_hi) tmem_ld16(trow + (uint32_t)((c_lo + j) * 16), r[j]);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      // the accumulator can go back to the MMA warp as soon as every epilogue warp has its registers
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&acc_empty[ab])) : "memory");
#pragma unroll
      for (int j = 0; j < 6; ++j)
        if (c_lo + j < c_hi)
          stage16<TOut>(reinterpret_cast<TOut*>(my_row) + (c_lo + j) * 16, r[j], bias, n0 + (c_lo + j) * 16, N);
      asm volatile("bar.sync 1, %0;" ::"n"(kET) : "memory");   // staged tile complete (epilogue warps only)
      int rr = et / vpr, vv = et % vpr;
      const int total = kGM * vpr;
#pragma unroll 4
      for (int idx = et; idx < total; idx += kET) {
        const int m = m0 + rr, n = n0 + vv * EV;
        if (m < M && n < N) {
          uint4 val = *reinterpret_cast<const uint4*>(tile + (size_t)rr * row_bytes + (size_t)vv * 16);
          TOut* dst = C + (int64_t)m * ldc + n;
          if (addend != nullptr) {
            const uint4 ad = *reinterpret_cast<const uint4*>(addend + (int64_t)m * ldc + n);
            TOut* pv = reinterpret_cast<TOut*>(&val);
            const TOut* pa = reinterpret_cast<const TOut*>(&ad);
#pragma unroll
            for (int j = 0; j < EV; ++j) pv[j] = from_f<TOut>(to_f(pv[j]) + to_f(pa[j]));
          }
          *reinterpret_cast<uint4*>(dst) = val;
        }
        rr += drr;
        vv += dvv;
        if (vv >= vpr) {
          vv -= vpr;
          ++rr;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kET) : "memory");   // tile may be overwritten by the next tile's staging
    }
  }
  __syncwarp();
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

// ---- weight-gradient product: C[N1, N2] = A[M, N1]^T . B[M, N2]  (contraction over the rows) ------------------
// Both operands are read as they lie in memory (row-major activations), i.e. as MN-major UMMA operands: TMA loads
// 64-feature x 64-row boxes with the 128-byte swizzle; a 64 x 8 sub-block is one 1024-byte swizzle atom, atoms of
// the same 64 features follow each other along the contraction (SBO = 1024 B), 64-feature groups are 8 KB apart
// (LBO).  One operand ("P") takes the 128 TMEM lanes of the tile, the other ("Q") its columns.  The long contraction
// (M = B*L*ndir rows) is split over blockIdx.z so that the grid is one wave; every CTA writes an fp32 partial tile
// part[z][q][p] (lanes run along p: 128-byte coalesced stores) and tn_reduce_kernel sums the splits in fixed order
// (deterministic, unlike an atomic split-K), transposing on the way out when P is the row index of C.
constexpr int kTNStages = 3;
constexpr int kTNBox = 64 * 64 * 2;   // bytes of one 64-feature x 64-row box

__device__ __forceinline__ uint64_t make_mnmajor_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)(kTNBox >> 4) << 16;   // LBO: next 64-feature group
  d |= (uint64_t)(1024 >> 4) << 32;     // SBO: next 8 rows of the contraction
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;               // SWIZZLE_128B
  return d;
}

__global__ void __launch_bounds__(kGThreads)
gemm_tn_kernel(const __grid_constant__ CUtensorMap map_p, const __grid_constant__ CUtensorMap map_q,
               float* __restrict__ part, int M, int NP, int NQ, int block_q, int kb_per_split, uint32_t idesc,
               uint32_t tmem_cols) {
  pdl_prologue();
  extern __shared__ __align__(1024) unsigned char gsm[];
  __shared__ __align__(8) uint64_t full_bar[kTNStages], empty_bar[kTNStages], accum_bar;
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p0 = blockIdx.x * kGM, q0 = blockIdx.y * block_q;
  const int nkb_all = (M + 63) / 64;
  const int kb0 = blockIdx.z * kb_per_split;
  const int nkb = min(kb_per_split, nkb_all - kb0);
  const int nbq = (block_q + 63) / 64;
  const uint32_t p_bytes = 2 * kTNBox, q_bytes = (uint32_t)nbq * kTNBox;
  const uint32_t stage_bytes = p_bytes + q_bytes;
  unsigned char* base = gsm + ((1024u - (smem_u32(gsm) & 1023u)) & 1023u);

  if (threadIdx.x == 0) {
    for (int s = 0; s < kTNStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&accum_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < nkb; ++i) {
      const int s = i % kTNStages;
      if (i >= kTNStages) mbar_wait(&empty_bar[s], ((i / kTNStages) - 1) & 1);
      unsigned char* sp = base + (size_t)s * stage_bytes;
      const int m0 = (kb0 + i) * 64;
      mbar_expect_tx(&full_bar[s], p_bytes + q_bytes);
      tma_load_2d(sp, &map_p, &full_bar[s], p0, m0);
      tma_load_2d(sp + kTNBox, &map_p, &full_bar[s], p0 + 64, m0);
      for (int gb = 0; gb < nbq; ++gb) tma_load_2d(sp + p_bytes + gb * kTNBox, &map_q, &full_bar[s], q0 + 64 * gb, m0);
    }
  } else if (warp == 1 && lane == 0) {
    for (int i = 0; i < nkb; ++i) {
      const int s = i % kTNStages;
      mbar_wait(&full_bar[s], (i / kTNStages) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t sp = smem_u32(base + (size_t)s * stage_bytes);
      const uint64_t dp = make_mnmajor_sw128_desc(sp), dq = make_mnmajor_sw128_desc(sp + p_bytes);
#pragma unroll
      for (int k = 0; k < 4; ++k)   // 16 rows of the contraction per instruction = two 8-row atoms = 2048 bytes
        umma_f16(tmem_base, dp + (uint64_t)(k * (2048 >> 4)), dq + (uint64_t)(k * (2048 >> 4)), idesc, (i | k) != 0 ? 1u : 0u);
      umma_commit(&empty_bar[s]);
    }
    umma_commit(&accum_bar);
  }
  __syncwarp();
  if (nkb > 0) {
    mbar_wait(&accum_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  }
  __syncwarp();
  const int pi = p0 + warp * 32 + lane;      // this thread's P feature (TMEM lane)
  const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
  float* dst = part + ((int64_t)blockIdx.z * NQ + q0) * NP + pi;
  for (int c = 0; c < block_q; c += 16) {
    uint32_t r[16];
    if (nkb > 0) {
      tmem_ld16(trow + (uint32_t)c, r);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) r[j] = 0u;
    }
    if (pi < NP) {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (q0 + c + j < NQ) dst[(int64_t)(c + j) * NP] = __uint_as_float(r[j]);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

// out = sum over the splits of part[z][q][p], in split order; p_is_row: out is (NP, NQ) row-major, else (NQ, NP).
__global__ void __launch_bounds__(256)
tn_reduce_kernel(const float* __restrict__ part, float* __restrict__ out, int nsplit, int NP, int NQ, int p_is_row) {
  pdl_prologue();
  const int idx = blockIdx.x * 256 + threadIdx.x;
  const int total = NP * NQ;
  if (idx >= total) return;
  float acc = 0.f;
  for (int z = 0; z < nsplit; ++z) acc += part[(int64_t)z * total + idx];
  const int q = idx / NP, p = idx - q * NP;
  out[p_is_row ? (int64_t)p * NQ + q : (int64_t)idx] = acc;
}

// ---- host side -------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

static int make_map(CUtensorMap* map, const void* ptr, int dtype, int64_t rows, int64_t cols, int64_t ld, int box_rows,
                    int box_cols = kGK) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_err("cuTensorMapEncodeTiled is not available from the driver"); return -20; }
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = dtype == BIMAMBA_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = enc(map, dt, 2, const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_err("cuTensorMapEncodeTiled failed (operand must be 16-byte aligned with a row stride that is a multiple of 8 elements)"); return -21; }
  return 0;
}

}  // namespace bimamba

using namespace bimamba;

// These projections are short-K, bandwidth/latency-bound products: what pays is many co-resident CTAs per SM
// whose load / MMA / epilogue phases overlap each other, i.e. a small shared-memory and TMEM footprint:
// two stages and tiles of at most 128 accumulator columns when N allows it (measured, tools/bench_gemm.py).
static int gemm_stages(int block_n, int K) {
  const int nkb = (K + kGK - 1) / kGK;
  (void)block_n;
  return nkb < 2 ? 1 : 2;
}

extern "C" int bimamba_gemm_nt_block_n_k(int N, int K) {
  (void)K;
  if (N <= 0) return 0;
  int best = 0;
  long best_cost = 1L << 60;
  for (int bn = 256; bn >= 16; bn -= 16) {
    const int tiles = (N + bn - 1) / bn;
    const long waste = (long)tiles * bn - N;
    const long cost = waste * 8 + tiles * 32 + (bn > 128 ? 200 : 0);
    if (cost < best_cost) { best_cost = cost; best = bn; }
  }
  return best;
}
extern "C" int bimamba_gemm_nt_block_n(int N) { return bimamba_gemm_nt_block_n_k(N, 0); }

// Tile width of the persistent variant: these products are bound by L2 traffic (A is re-read once per N tile, B
// once per M tile), so it takes the widest tile (<= 192 columns: two accumulators fit the 512 TMEM columns) that
// splits N evenly.
static int persist_block_n(int N) {
  int best = 0;
  long best_cost = 1L << 60;
  for (int bn = 192; bn >= 16; bn -= 16) {
    const int tiles = (N + bn - 1) / bn;
    const long cost = ((long)tiles * bn - N) * 8 + tiles * 64;
    if (cost < best_cost) { best_cost = cost; best = bn; }
  }
  return best;
}

extern "C" int bimamba_gemm_nt(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc,
                               const float* bias, const void* addend, int64_t M, int N, int K, int in_dtype,
                               int out_dtype, bimamba_stream_t stream) {
  if (M == 0 || N == 0) return 0;
  if (!A || !B || !C) { set_err("gemm: null operand"); return -1; }
  if (M < 0 || N < 0 || K < 1) { set_err("gemm: bad sizes"); return -3; }
  if (in_dtype != BIMAMBA_BF16 && in_dtype != BIMAMBA_F16) { set_err("gemm: operands must be bf16 or fp16 (fp32 products stay on the fp32 library path)"); return -6; }
  if (out_dtype < 0 || out_dtype > 2 || (out_dtype != BIMAMBA_F32 && out_dtype != in_dtype)) { set_err("gemm: output must be fp32 or the operand dtype"); return -6; }
  if ((lda & 7) || (ldb & 7) || (reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(B) & 15)) {
    set_err("gemm: operands must be 16-byte aligned with row strides that are multiples of 8 elements");
    return -7;
  }
  if (M > (int64_t)kGM * 2147483647LL / 2) { set_err("gemm: M too large"); return -3; }
  int block_n = bimamba_gemm_nt_block_n_k(N, K);
  int max_stages = kGStagesMax;
  // persistent warp-specialised variant when there is more than one tile per SM (and rows are 16-byte friendly)
  const int kv = g_tune[BIMAMBA_TUNE_GEMM_KERNEL];   // tuning experiments / variant tests only: 1 = tile, 2 = persistent
  const int osz = out_dtype == BIMAMBA_F32 ? 4 : 2;
  const bool can_stage = (N % (16 / osz) == 0) && (ldc % (16 / osz) == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0) &&
                         (!addend || (reinterpret_cast<uintptr_t>(addend) & 15) == 0);
  bool persist = false;
  {
    const int bnp = persist_block_n(N);
    const int64_t nt = ((M + kGM - 1) / kGM) * ((N + bnp - 1) / bnp);
    persist = can_stage && nt >= 4 * 148;   // measured: below ~4 tiles per SM the one-tile-per-CTA kernel wins
    if (kv) persist = can_stage && kv == 2;
    if (persist) block_n = bnp;
  }
  // Measured choices for the Phase-6 projection shapes at the benchmark's row counts (tools/sweep_gemm.py on a B200, eight
  // back-to-back launches on rotating operands; profiles/r2_gemm_table.md): what decides is whether the tiles fit ONE wave
  // at the TMEM / shared-memory occupancy of the configuration, and - for the long contractions - the persistent kernel's
  // 4-stage ring and 8 epilogue warps even at one tile per CTA.
  int tuned_stages = 0;
  if (!kv && M >= 8192 && M <= 32768) {
    struct Tuned { int N, K, persist, bn, stages; };
    static const Tuned kTuned[] = {
        {576, 144, 0, 128, 1},   // in_proj, FFN up, FFN-down data gradient: 14.2 -> 11.8 us (one stage = 4 CTAs / SM = one wave)
        {144, 576, 1, 144, 0},   // out_proj, FFN down, in_proj / FFN-up data gradients: 11.9 -> 10.5 us
        {288, 48, 0, 64, 1},     // x_proj data gradient: 11.8 -> 10.9 us
        {48, 288, 0, 32, 2},     // x_proj: 9.7 -> 9.3 us
    };
    for (const Tuned& t : kTuned) {
      if (t.N == N && t.K == K && (!t.persist || can_stage)) {
        persist = t.persist != 0;
        block_n = t.bn;
        tuned_stages = t.stages;
      }
    }
  }
  if (g_tune[BIMAMBA_TUNE_GEMM_BN]) block_n = g_tune[BIMAMBA_TUNE_GEMM_BN];            // tuning experiments only
  if (g_tune[BIMAMBA_TUNE_GEMM_STAGES]) max_stages = g_tune[BIMAMBA_TUNE_GEMM_STAGES];  // tuning experiments only
  CUtensorMap map_a, map_b;
  int rc = make_map(&map_a, A, in_dtype, M, K, lda, kGM);
  if (rc) return rc;
  rc = make_map(&map_b, B, in_dtype, N, K, ldb, block_n);
  if (rc) return rc;
  const uint32_t stage_bytes = kGM * kGK * 2 + (((uint32_t)block_n * kGK * 2 + 1023u) & ~1023u);
  int stages = tuned_stages ? tuned_stages : gemm_stages(block_n, K);
  if (stages > max_stages) stages = max_stages;
  size_t smem = (size_t)stages * stage_bytes + 1024;
  // staged epilogue: 16-byte aligned output rows and a tile that fits next to (in place of) the stages
  const int osize = out_dtype == BIMAMBA_F32 ? 4 : 2;
  const size_t tile_bytes = (size_t)kGM * ((size_t)block_n * osize + 16);
  int staged = (N % (16 / osize) == 0) && (ldc % (16 / osize) == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0) &&
               (!addend || (reinterpret_cast<uintptr_t>(addend) & 15) == 0) && tile_bytes <= 110 * 1024;
  if (staged && tile_bytes + 1024 > smem) smem = tile_bytes + 1024;
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < block_n) tmem_cols <<= 1;
  // instruction descriptor: D fp32, A/B bf16|fp16, both K-major, N >> 3, M >> 4
  const uint32_t fmt = in_dtype == BIMAMBA_BF16 ? 1u : 0u;
  const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(block_n >> 3) << 17) | ((uint32_t)(kGM >> 4) << 24);
  dim3 grid((unsigned)((M + kGM - 1) / kGM), (unsigned)((N + block_n - 1) / block_n));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t ntiles = (int64_t)grid.x * grid.y;
  if (persist && staged) {
    const uint32_t acc_stride = (uint32_t)((block_n + 31) / 32 * 32);
    uint32_t pcols = 32;
    while (pcols < 2 * acc_stride) pcols <<= 1;
    const size_t psmem = (size_t)kPStages * stage_bytes + tile_bytes + 1024;
    int sms = 148, cur_dev = 0;
    cudaGetDevice(&cur_dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cur_dev);
    const unsigned pgrid = (unsigned)(ntiles < sms ? ntiles : sms);
#define GEMM_PLAUNCH(TOUT)                                                                                         \
  do {                                                                                                             \
    cudaFuncSetAttribute(gemm_nt_persist_kernel<TOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem);   \
    launch_k(gemm_nt_persist_kernel<TOUT>, pgrid, kPThreads, psmem, st, map_a, map_b, reinterpret_cast<TOUT*>(C), bias,   \
                                                                  reinterpret_cast<const TOUT*>(addend), (int)M, N, K, \
                                                                  ldc, block_n, idesc, pcols, acc_stride);         \
  } while (0)
    if (psmem <= 220 * 1024) {
      if (out_dtype == BIMAMBA_F32) GEMM_PLAUNCH(float);
      else if (out_dtype == BIMAMBA_BF16) GEMM_PLAUNCH(__nv_bfloat16);
      else GEMM_PLAUNCH(__half);
#undef GEMM_PLAUNCH
      cudaError_t pe = cudaGetLastError();
      if (pe != cudaSuccess) { set_err(cudaGetErrorString(pe)); return (int)pe; }
      return 0;
    }
  }
#define GEMM_LAUNCH(TOUT)                                                                                          \
  do {                                                                                                             \
    cudaFuncSetAttribute(gemm_nt_kernel<TOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);            \
    launch_k(gemm_nt_kernel<TOUT>, grid, kGThreads, smem, st, map_a, map_b, reinterpret_cast<TOUT*>(C), bias,             \
                                                         reinterpret_cast<const TOUT*>(addend), (int)M, N, K, ldc, \
                                                         block_n, stages, idesc, tmem_cols, staged);               \
  } while (0)
  if (out_dtype == BIMAMBA_F32) GEMM_LAUNCH(float);
  else if (out_dtype == BIMAMBA_BF16) GEMM_LAUNCH(__nv_bfloat16);
  else GEMM_LAUNCH(__half);
#undef GEMM_LAUNCH
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}

namespace {
struct TnPlan { int p_is_a, NP, NQ, block_q, nsplit, per; };
inline int64_t tn_padded(int np, int nq, int* bq_out) {
  const int nblk = (nq + 255) / 256;
  const int bq = ((nq + nblk - 1) / nblk + 15) / 16 * 16;
  if (bq_out) *bq_out = bq;
  return (int64_t)((np + kGM - 1) / kGM) * kGM * ((nq + bq - 1) / bq) * bq;
}
inline TnPlan tn_plan(int64_t M, int N1, int N2) {
  TnPlan pl;
  int bq_a, bq_b;
  const int64_t cost_a = tn_padded(N1, N2, &bq_a);   // A's features on the TMEM lanes
  const int64_t cost_b = tn_padded(N2, N1, &bq_b);
  pl.p_is_a = cost_a < cost_b;                        // tie: B on the lanes, no transpose on the way out
  pl.NP = pl.p_is_a ? N1 : N2;
  pl.NQ = pl.p_is_a ? N2 : N1;
  pl.block_q = pl.p_is_a ? bq_a : bq_b;
  const int64_t tiles = (int64_t)((pl.NP + kGM - 1) / kGM) * ((pl.NQ + pl.block_q - 1) / pl.block_q);
  const int64_t nkb = (M + 63) / 64;
  int64_t want = 148 / tiles;                         // one wave, one CTA per SM
  if (want > nkb) want = nkb;
  if (want < 1) want = 1;
  pl.per = (int)((nkb + want - 1) / want);
  pl.nsplit = (int)((nkb + pl.per - 1) / pl.per);
  return pl;
}
}  // namespace

extern "C" int bimamba_gemm_tn_splits(int64_t M, int N1, int N2) {
  if (M <= 0 || N1 <= 0 || N2 <= 0) return 1;
  return tn_plan(M, N1, N2).nsplit;
}

extern "C" int bimamba_gemm_tn(const void* A, int64_t lda, const void* B, int64_t ldb, float* C, float* part, int64_t M,
                               int N1, int N2, int in_dtype, bimamba_stream_t stream) {
  if (M == 0 || N1 == 0 || N2 == 0) return 0;
  if (!A || !B || !C || !part) { set_err("gemm_tn: null operand"); return -1; }
  if (M < 0 || N1 < 0 || N2 < 0) { set_err("gemm_tn: bad sizes"); return -3; }
  if (in_dtype != BIMAMBA_BF16 && in_dtype != BIMAMBA_F16) { set_err("gemm_tn: operands must be bf16 or fp16"); return -6; }
  if ((lda & 7) || (ldb & 7) || (reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(B) & 15)) {
    set_err("gemm_tn: operands must be 16-byte aligned with row strides that are multiples of 8 elements");
    return -7;
  }
  const TnPlan pl = tn_plan(M, N1, N2);
  CUtensorMap map_p, map_q;
  int rc = make_map(&map_p, pl.p_is_a ? A : B, in_dtype, M, pl.NP, pl.p_is_a ? lda : ldb, 64, 64);
  if (rc) return rc;
  rc = make_map(&map_q, pl.p_is_a ? B : A, in_dtype, M, pl.NQ, pl.p_is_a ? ldb : lda, 64, 64);
  if (rc) return rc;
  const int nbq = (pl.block_q + 63) / 64;
  const size_t smem = (size_t)kTNStages * (2 + nbq) * kTNBox + 1024;
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < pl.block_q) tmem_cols <<= 1;
  const uint32_t fmt = in_dtype == BIMAMBA_BF16 ? 1u : 0u;
  const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (1u << 15) | (1u << 16) |
                         ((uint32_t)(pl.block_q >> 3) << 17) | ((uint32_t)(kGM >> 4) << 24);
  dim3 grid((unsigned)((pl.NP + kGM - 1) / kGM), (unsigned)((pl.NQ + pl.block_q - 1) / pl.block_q), (unsigned)pl.nsplit);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // per device / context attribute: set on every launch (a process-wide flag would miss the second device)
  cudaFuncSetAttribute(gemm_tn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * 6 * kTNBox + 1024);
  launch_k(gemm_tn_kernel, grid, kGThreads, smem, st, map_p, map_q, part, (int)M, pl.NP, pl.NQ, pl.block_q, pl.per, idesc, tmem_cols);
  launch_k(tn_reduce_kernel, (unsigned)(((int64_t)N1 * N2 + 255) / 256), 256, 0, st, part, C, pl.nsplit, pl.NP, pl.NQ, pl.p_is_a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_err(cudaGetErrorString(e)); return (int)e; }
  return 0;
}
