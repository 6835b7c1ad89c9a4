// Tensor-core Linear for sm_100a: out[M,N] = A[M,K] * W[N,K]^T (+bias) (+residual)
//
//   * W is bf16 [N,K] (K contiguous) exactly as nn.Linear stores it -> UMMA "B" operand, K-major.
//   * A is fp32 in the model; it arrives here split into two bf16 planes, A = A_hi + A_lo
//     (A_hi = bf16(A), A_lo = bf16(A - A_hi)), and the kernel accumulates A_hi*W^T + A_lo*W^T into the same
//     fp32 TMEM accumulator. bf16 x bf16 products are exact in fp32, so the result carries ~16 mantissa bits
//     of the activations (vs 8 for a plain bf16 cast) — what keeps hidden states within 1e-3 and action
//     tokens bit-exact against the fp32 oracle while still running on tcgen05.
//   * One CTA computes a 128 x BLOCK_N tile: warp 0 = TMA producer (cp.async.bulk.tensor, 128B swizzle),
//     warp 1 = TMEM allocator + single-thread tcgen05.mma issuer, warps 2..5 = epilogue
//     (tcgen05.ld -> registers -> bias/residual -> global). kStages-deep smem ring with mbarriers.
//
// Descriptor formats follow CUTLASS cute/arch/mma_sm100_desc.hpp (SmemDescriptor / InstrDescriptor).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "xl_common.cuh"
#include "xl_internal.h"

namespace xl {

namespace tc {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;   // 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;
constexpr int kThreads = 192;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// multicast forms (thread-block cluster of column-tile CTAs sharing one A tile)
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                               uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster "
      "[%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void tcgen05_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, 128B-swizzled operand tile: rows of 128 B, 8-row atoms of 1024 B (SBO = 1024 B), LBO unused (=1),
// descriptor version 1 (Blackwell), layout type 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);   // start address, bits [0,14)
  d |= (uint64_t)1 << 16;                        // leading byte offset (ignored for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;                        // version = 1
  d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
  return d;
}

// kind::f16 instruction descriptor: D = F32, A = B = BF16, both K-major, M = 128, N = BLOCK_N.
__host__ __device__ constexpr uint32_t make_idesc(int n, int m = BLOCK_M) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// kBM = rows of the MMA tile: 128, or 64 for skinny batches (M <= 192 rows leave a quarter of a second 128-row tile
// empty, and — what matters at these sizes — a 64-row tile halves the A bytes per k-block, so the ring holds twice as
// many k-blocks in flight: the K loop of these GEMMs is bound by (k-blocks / ring depth) L2 round trips).
template <int BLOCK_N, int kStages, int kBM = BLOCK_M>
struct Smem {
  static constexpr int kABytes = kBM * BLOCK_K * 2;
  static constexpr int kBBytes = BLOCK_N * BLOCK_K * 2;
  static constexpr int kStageBytes = 2 * kABytes + kBBytes;
  static constexpr int kTotal = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

// kCX > 1: the kCX column-tile CTAs of a thread-block cluster (consecutive blockIdx.x) share their A tile. CTA r
// loads rows [r, r+1) * kBM/kCX of the hi and lo planes and MULTICASTS them into every CTA of the cluster (one L2 read
// instead of kCX); each CTA's full barrier counts the bytes of all slices + its own W tile, and a stage is released to
// every producer of the cluster (tcgen05.commit multicast on the empty barriers, which expect kCX arrivals).
template <int BLOCK_N, int kStages, int kBM, int kCX>
__global__ void __launch_bounds__(kThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
               const __grid_constant__ CUtensorMap map_w, const float* __restrict__ bias,
               const float* __restrict__ residual, float* __restrict__ out, int M, int N, int K,
               long long split_stride, int m64_rows_contiguous) {
  using S = Smem<BLOCK_N, kStages, kBM>;
  constexpr uint16_t kMask = (uint16_t)((1u << kCX) - 1u);
  constexpr int kSliceRows = kBM / kCX;
  constexpr int kSliceBytes = kSliceRows * BLOCK_K * 2;
  const uint32_t crank = kCX > 1 ? cluster_ctarank() : 0u;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + kStages * S::kStageBytes;     // full[kStages], empty[kStages], tmem_full
  const uint32_t tmem_slot = bar_base + 8 * (2 * kStages + 1);
  auto full_bar = [&](int s) { return bar_base + 8 * s; };
  auto empty_bar = [&](int s) { return bar_base + 8 * (kStages + s); };
  const uint32_t tmem_full_bar = bar_base + 8 * (2 * kStages);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BLOCK_N, m0 = blockIdx.y * kBM;
  // split-K: blockIdx.z owns k-blocks [kb0, kb0 + num_kb) and writes its raw partial tile to the plane
  // out + blockIdx.z * split_stride; the CONSUMER kernels (LayerNorm, conv/qkv, finalize) add the planes in
  // plane order, so there is no reduction step, no atomics and no inter-CTA synchronisation here.
  const int splits = gridDim.z;
  const int kb_total = K / BLOCK_K;
  const int kb_per = (kb_total + splits - 1) / splits;
  const int kb0 = blockIdx.z * kb_per;
  const int num_kb = max(0, min(kb_total, kb0 + kb_per) - kb0);

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_hi) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_lo) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), kCX);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    // allocate BLOCK_N (power of two >= 32) TMEM columns; address is written to shared memory
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(BLOCK_N)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  // The weight tiles of the first ring round are requested BEFORE the dependency wait (weights are never
  // written by a kernel): they stream in while the kernel that produces the activations is still running.
  const int pre_kb = num_kb < kStages ? num_kb : kStages;
  if (warp == 0 && lane == 0) {
    for (int kb = 0; kb < pre_kb; ++kb) {
      mbar_expect_tx(full_bar(kb), S::kStageBytes);
      tma_load_2d(base + kb * S::kStageBytes + 2 * S::kABytes, &map_w, full_bar(kb), (kb0 + kb) * BLOCK_K, n0);
    }
  }
  pdl_wait();
  pdl_trigger();
  // peers multicast into this CTA's ring and arrive on its barriers: those must be initialised cluster-wide first
  if (kCX > 1) cluster_sync_all();

  // A tile of one stage: the whole tile (kCX == 1) or this CTA's row slice, multicast to the cluster
  auto load_a = [&](uint32_t st, uint32_t bar, int kcol) {
    if (kCX == 1) {
      tma_load_2d(st, &map_a_hi, bar, kcol, m0);
      tma_load_2d(st + S::kABytes, &map_a_lo, bar, kcol, m0);
    } else {
      const int r0 = m0 + (int)crank * kSliceRows;
      tma_load_2d_mc(st + crank * kSliceBytes, &map_a_hi, bar, kcol, r0, kMask);
      tma_load_2d_mc(st + S::kABytes + crank * kSliceBytes, &map_a_lo, bar, kcol, r0, kMask);
    }
  };
  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      for (int kb = 0; kb < pre_kb; ++kb) load_a(base + kb * S::kStageBytes, full_bar(kb), (kb0 + kb) * BLOCK_K);
      for (int kb = pre_kb; kb < num_kb; ++kb) {
        const int s = kb % kStages;
        const uint32_t ph = (kb / kStages) & 1;
        mbar_wait(empty_bar(s), ph ^ 1);              // every CTA of the cluster has consumed this stage
        const uint32_t st = base + s * S::kStageBytes;
        mbar_expect_tx(full_bar(s), S::kStageBytes);
        load_a(st, full_bar(s), (kb0 + kb) * BLOCK_K);
        tma_load_2d(st + 2 * S::kABytes, &map_w, full_bar(s), (kb0 + kb) * BLOCK_K, n0);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread) =====
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(BLOCK_N, kBM);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % kStages;
        const uint32_t ph = (kb / kStages) & 1;
        mbar_wait(full_bar(s), ph);
        tcgen05_fence_after();
        const uint32_t st = base + s * S::kStageBytes;
        const uint64_t a_hi = make_smem_desc(st);
        const uint64_t a_lo = make_smem_desc(st + S::kABytes);
        const uint64_t bw = make_smem_desc(st + 2 * S::kABytes);
#pragma unroll
        for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
          const uint64_t kofs = (uint64_t)((k * UMMA_K * 2) >> 4);   // advance inside the 128-B swizzle row
          umma_bf16(tmem_base, a_hi + kofs, bw + kofs, idesc, (kb | k) != 0);
          umma_bf16(tmem_base, a_lo + kofs, bw + kofs, idesc, 1u);
        }
        // frees the smem stage when these MMAs retire — in every CTA of the cluster that multicasts into it
        if (kCX == 1) tcgen05_commit(empty_bar(s));
        else tcgen05_commit_mc(empty_bar(s), kMask);
      }
      tcgen05_commit(tmem_full_bar);             // accumulator complete
    }
  }

  // ===== epilogue: warps 2..5; a warp may only touch TMEM lanes 32*(warp%4) .. +31 =====================
  // TMEM -> registers -> (bias, residual: only when splits == 1, host-enforced) -> global, 32 columns at a time.
  const bool is_epi = warp >= 2;
  const int q = warp & 3;
  // M = 128: accumulator row r lives in TMEM lane r. M = 64 (cta_group::1): the 64 rows occupy lanes 0-15 of each
  // 32-lane quarter (row r -> lane 32*(r/16) + r%16), so each epilogue warp owns 16 rows in its lanes 0..15.
  // (m64_rows_contiguous = 1 selects the alternative reading, rows = lanes 0..63; kept as a probe, see the unit test.)
  int lrow = q * 32 + lane;
  bool row_ok = true;
  if (kBM == 64) {
    if (m64_rows_contiguous) { row_ok = q < 2; }
    else { lrow = q * 16 + lane; row_ok = lane < 16; }
  }
  const int row = m0 + lrow;
  out += (long long)blockIdx.z * split_stride;

  auto store_chunk = [&](const float (&v)[32], int c) {       // bias + residual + store of 32 columns
    if (row >= M || !row_ok) return;
    const int col0 = n0 + c;
    float* orow = out + (int64_t)row * N + col0;
    const float* rrow = residual ? residual + (int64_t)row * N + col0 : nullptr;
    if (col0 + 32 <= N && (N & 3) == 0) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        float4 o = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        if (bias) {
          const float4 b4 = *reinterpret_cast<const float4*>(bias + col0 + j);
          o.x += b4.x; o.y += b4.y; o.z += b4.z; o.w += b4.w;
        }
        if (rrow) {
          const float4 r4 = *reinterpret_cast<const float4*>(rrow + j);
          o.x += r4.x; o.y += r4.y; o.z += r4.z; o.w += r4.w;
        }
        *reinterpret_cast<float4*>(orow + j) = o;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        if (col0 + j < N) {
          float o = v[j];
          if (bias) o += bias[col0 + j];
          if (rrow) o += rrow[j];
          orow[j] = o;
        }
      }
    }
  };
  auto tmem_load_chunk = [&](float (&v)[32], int c) {
    uint32_t r[32];
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c;
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]),
          "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
          "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  };

  if (is_epi) {
    mbar_wait(tmem_full_bar, 0);
    tcgen05_fence_after();
    if (num_kb > 0) {
#pragma unroll
      for (int c = 0; c < BLOCK_N; c += 32) {
        float v[32];
        tmem_load_chunk(v, c);
        store_chunk(v, c);
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(BLOCK_N) : "memory");
  }
  // peers' stage releases still arrive on this CTA's empty barriers: nobody leaves before everybody is done
  if (kCX > 1) cluster_sync_all();
}


// ------------------------------------------------------------------------------------------------------------------
// 2-SM variant for GEMM-sized M (context prefill): a CTA PAIR (cluster of 2 along M) computes one 256 x 256 tile with
// tcgen05.mma.cta_group::2. Each CTA stages its own 128 rows of the A planes and only HALF of the W tile (128 of its
// 256 rows): 48 KB of operands per k-block and SM for a 128 x 256 output slice instead of 64 KB -- these GEMMs are bound
// by operand delivery (L2 -> SM), not by the tensor pipe. Protocol (CUTLASS sm100 2-SM mainloop): both CTAs' TMA loads
// (cp.async.bulk.tensor ... .cta_group::2) complete on the LEADER's full barrier, which expects the bytes of both; the
// leader issues the MMAs (it reads the peer's shared memory at the same offsets) and releases a stage / publishes the
// accumulator in both CTAs with tcgen05.commit.cta_group::2 ... multicast::cluster; each CTA's epilogue reads its own 128
// accumulator rows from its own TMEM.
// ------------------------------------------------------------------------------------------------------------------
namespace two {

constexpr int BN2 = 256;
constexpr int kABytes = BLOCK_M * BLOCK_K * 2;        // one A plane of this CTA's 128 rows
constexpr int kWBytes = 128 * BLOCK_K * 2;            // this CTA's half of the W tile
constexpr int kStageBytes = 2 * kABytes + kWBytes;    // 48 KB
constexpr int kStages = 4;
constexpr int kTotal = kStages * kStageBytes + 1024 + 256;

__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// TMA load of this CTA's tile into its own shared memory; completion bytes go to `bar` (an address in the cluster window:
// the leader's full barrier)
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void commit2_mc(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(mask) : "memory");
}

__global__ void __launch_bounds__(kThreads, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                const __grid_constant__ CUtensorMap map_w, const float* __restrict__ bias,
                const float* __restrict__ residual, float* __restrict__ out, int M, int N, int K) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + kStages * kStageBytes;     // full[kStages], empty[kStages], tmem_full, slot
  const uint32_t tmem_slot = bar_base + 8 * (2 * kStages + 1);
  auto full_bar = [&](int s) { return bar_base + 8 * s; };
  auto empty_bar = [&](int s) { return bar_base + 8 * (kStages + s); };
  const uint32_t tmem_full_bar = bar_base + 8 * (2 * kStages);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int n0 = blockIdx.y * BN2;
  const int m0 = ((int)blockIdx.x >> 1) * 2 * BLOCK_M + (int)crank * BLOCK_M;      // the pair = consecutive blockIdx.x
  const int num_kb = K / BLOCK_K;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_hi) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_lo) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {     // the same warp of BOTH CTAs allocates the pair's accumulator columns
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(BN2) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");
  pdl_wait();
  pdl_trigger();
  cluster_sync_all();        // the peer signals this CTA's barriers: they must be initialised cluster-wide first

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % kStages;
        if (kb >= kStages) mbar_wait(empty_bar(s), ((kb / kStages) & 1) ^ 1);
        const uint32_t st = base + s * kStageBytes;
        if (leader) mbar_expect_tx(full_bar(s), 2 * kStageBytes);          // the bytes of both CTAs
        const uint32_t lbar = mapa_u32(full_bar(s), 0u);
        tma_load_2d_pair(st, &map_a_hi, lbar, kb * BLOCK_K, m0);
        tma_load_2d_pair(st + kABytes, &map_a_lo, lbar, kb * BLOCK_K, m0);
        tma_load_2d_pair(st + 2 * kABytes, &map_w, lbar, kb * BLOCK_K, n0 + (int)crank * 128);
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc(BN2, 2 * BLOCK_M);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % kStages;
        mbar_wait(full_bar(s), (kb / kStages) & 1);
        tcgen05_fence_after();
        const uint32_t st = base + s * kStageBytes;
        const uint64_t a_hi = make_smem_desc(st);
        const uint64_t a_lo = make_smem_desc(st + kABytes);
        const uint64_t bw = make_smem_desc(st + 2 * kABytes);
#pragma unroll
        for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
          const uint64_t kofs = (uint64_t)((k * UMMA_K * 2) >> 4);
          umma2_bf16(tmem_base, a_hi + kofs, bw + kofs, idesc, (kb | k) != 0);
          umma2_bf16(tmem_base, a_lo + kofs, bw + kofs, idesc, 1u);
        }
        commit2_mc(empty_bar(s), (uint16_t)3);       // the stage is free in both CTAs once these MMAs retire
      }
      commit2_mc(tmem_full_bar, (uint16_t)3);
    }
  } else {
    const int q = warp & 3;
    const int row = m0 + q * 32 + lane;
    mbar_wait(tmem_full_bar, 0);
    tcgen05_fence_after();
#pragma unroll 1
    for (int c = 0; c < BN2; c += 32) {
      uint32_t r[32];
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c;
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
          "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
          : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
            "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
            "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]),
            "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
            "=r"(r[30]), "=r"(r[31])
          : "r"(taddr)
          : "memory");
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      const int col0 = n0 + c;
      if (row < M && col0 < N) {
        float* orow = out + (int64_t)row * N + col0;
        const float* rrow = residual ? residual + (int64_t)row * N + col0 : nullptr;
        if (col0 + 32 <= N && (N & 3) == 0) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 o = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]),
                                   __uint_as_float(r[j + 3]));
            if (bias) {
              const float4 b4 = *reinterpret_cast<const float4*>(bias + col0 + j);
              o.x += b4.x; o.y += b4.y; o.z += b4.z; o.w += b4.w;
            }
            if (rrow) {
              const float4 r4 = *reinterpret_cast<const float4*>(rrow + j);
              o.x += r4.x; o.y += r4.y; o.z += r4.z; o.w += r4.w;
            }
            *reinterpret_cast<float4*>(orow + j) = o;
          }
        } else {
          for (int j = 0; j < 32; ++j) {
            if (col0 + j < N) {
              float o = __uint_as_float(r[j]);
              if (bias) o += bias[col0 + j];
              if (rrow) o += rrow[j];
              orow[j] = o;
            }
          }
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();        // nobody frees TMEM or leaves while the pair's MMAs / barrier signals may still be in flight
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(BN2) : "memory");
  }
}

// Persistent form of the same 2-SM kernel: one CTA pair per SM pair walks the 256 x 256 tiles p, p + P, ... The
// accumulator is double-buffered in TMEM (2 x 256 columns): the MMAs of tile j+1 run while both CTAs' epilogue warps drain
// tile j (tcgen05.ld -> bias / residual -> global) and hand the buffer back by arriving -- the peer CTA remotely -- on the
// leader's tmem-empty barrier. The operand ring simply continues across tiles.
constexpr int kStagesP = 4;
constexpr int kTotalP = kStagesP * kStageBytes + 1024 + 256;

__global__ void __launch_bounds__(kThreads, 1)
gemm_tc2p_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                 const __grid_constant__ CUtensorMap map_w, const float* __restrict__ bias,
                 const float* __restrict__ residual, float* __restrict__ out, int M, int N, int K) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + kStagesP * kStageBytes;   // full[S], empty[S], tfull[2], tempty[2], slot
  auto full_bar = [&](int s) { return bar_base + 8 * s; };
  auto empty_bar = [&](int s) { return bar_base + 8 * (kStagesP + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8 * (2 * kStagesP + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8 * (2 * kStagesP + 2 + b); };
  const uint32_t tmem_slot = bar_base + 8 * (2 * kStagesP + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int num_kb = K / BLOCK_K;
  const int ntiles_n = (N + BN2 - 1) / BN2, ntiles_m = (M + 2 * BLOCK_M - 1) / (2 * BLOCK_M);
  const int ntiles = ntiles_n * ntiles_m;
  const int pair = (int)blockIdx.x >> 1, npairs = (int)gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_hi) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_lo) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    for (int s = 0; s < kStagesP; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), 8);          // 4 epilogue warps of each CTA of the pair (used in the leader only)
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(2 * BN2) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");
  pdl_wait();
  pdl_trigger();
  cluster_sync_all();

  if (warp == 0) {
    if (lane == 0) {
      int it = 0;
      for (int t = pair; t < ntiles; t += npairs) {
        const int mt = t / ntiles_n, nt = t - mt * ntiles_n;
        const int m0 = mt * 2 * BLOCK_M + (int)crank * BLOCK_M, n0 = nt * BN2;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % kStagesP;
          if (it >= kStagesP) mbar_wait(empty_bar(s), ((it / kStagesP) & 1) ^ 1);
          const uint32_t st = base + s * kStageBytes;
          if (leader) mbar_expect_tx(full_bar(s), 2 * kStageBytes);
          const uint32_t lbar = mapa_u32(full_bar(s), 0u);
          tma_load_2d_pair(st, &map_a_hi, lbar, kb * BLOCK_K, m0);
          tma_load_2d_pair(st + kABytes, &map_a_lo, lbar, kb * BLOCK_K, m0);
          tma_load_2d_pair(st + 2 * kABytes, &map_w, lbar, kb * BLOCK_K, n0 + (int)crank * 128);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc(BN2, 2 * BLOCK_M);
      int it = 0, j = 0;
      for (int t = pair; t < ntiles; t += npairs, ++j) {
        const int b = j & 1, use = j >> 1;
        if (use > 0) {                      // both CTAs' epilogues have drained this accumulator
          mbar_wait(tempty_bar(b), (use - 1) & 1);
          tcgen05_fence_after();
        }
        const uint32_t tacc = tmem_base + (uint32_t)(b * BN2);
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % kStagesP;
          mbar_wait(full_bar(s), (it / kStagesP) & 1);
          tcgen05_fence_after();
          const uint32_t st = base + s * kStageBytes;
          const uint64_t a_hi = make_smem_desc(st);
          const uint64_t a_lo = make_smem_desc(st + kABytes);
          const uint64_t bw = make_smem_desc(st + 2 * kABytes);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t kofs = (uint64_t)((k * UMMA_K * 2) >> 4);
            umma2_bf16(tacc, a_hi + kofs, bw + kofs, idesc, (kb | k) != 0);
            umma2_bf16(tacc, a_lo + kofs, bw + kofs, idesc, 1u);
          }
          commit2_mc(empty_bar(s), (uint16_t)3);
        }
        commit2_mc(tfull_bar(b), (uint16_t)3);
      }
    }
  } else {
    const int q = warp & 3;
    const uint32_t lead_tempty0 = mapa_u32(tempty_bar(0), 0u), lead_tempty1 = mapa_u32(tempty_bar(1), 0u);
    int j = 0;
    for (int t = pair; t < ntiles; t += npairs, ++j) {
      const int b = j & 1, use = j >> 1;
      const int mt = t / ntiles_n, nt = t - mt * ntiles_n;
      const int m0 = mt * 2 * BLOCK_M + (int)crank * BLOCK_M, n0 = nt * BN2;
      const int row = m0 + q * 32 + lane;
      mbar_wait(tfull_bar(b), use & 1);
      tcgen05_fence_after();
#pragma unroll 1
      for (int c = 0; c < BN2; c += 32) {
        uint32_t r[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * BN2 + c);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
              "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
              "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]),
              "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
              "=r"(r[30]), "=r"(r[31])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        const int col0 = n0 + c;
        if (row < M && col0 < N) {
          float* orow = out + (int64_t)row * N + col0;
          const float* rrow = residual ? residual + (int64_t)row * N + col0 : nullptr;
          if (col0 + 32 <= N && (N & 3) == 0) {
            float4 rv[8];
            if (rrow) {
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) rv[jj] = *reinterpret_cast<const float4*>(rrow + 4 * jj);   // all in flight
            }
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              float4 o = make_float4(__uint_as_float(r[4 * jj]), __uint_as_float(r[4 * jj + 1]),
                                     __uint_as_float(r[4 * jj + 2]), __uint_as_float(r[4 * jj + 3]));
              if (bias) {
                const float4 b4 = *reinterpret_cast<const float4*>(bias + col0 + 4 * jj);
                o.x += b4.x; o.y += b4.y; o.z += b4.z; o.w += b4.w;
              }
              if (rrow) { o.x += rv[jj].x; o.y += rv[jj].y; o.z += rv[jj].z; o.w += rv[jj].w; }
              *reinterpret_cast<float4*>(orow + 4 * jj) = o;
            }
          } else {
            for (int jj = 0; jj < 32; ++jj) {
              if (col0 + jj < N) {
                float o = __uint_as_float(r[jj]);
                if (bias) o += bias[col0 + jj];
                if (rrow) o += rrow[jj];
                orow[jj] = o;
              }
            }
          }
        }
      }
      // this warp is done with accumulator b: tell the leader's MMA thread (remote arrive from the peer CTA)
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0)
        asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(b ? lead_tempty1 : lead_tempty0)
                     : "memory");
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(2 * BN2) : "memory");
  }
}

}  // namespace two

// ------------------------------------------------------------------------------------------------------------------
// Up-projection with the pre-cell epilogue (fused 3-token step): u = LN(x) W_up^T as above, but the x_m half of u
// never reaches global memory — CausalConv1d.step + SiLU + headwise q/k/v + gate partials ([ext-xlstm]
// mLSTMLayer.step; what conv_qkv_gates_kernel does, same arithmetic in the same order) run on the accumulator tile
// while it is on chip. One dependent launch and one round trip of x_m less per block.
//   * row tiles hold whole envs: 42 envs x 3 tokens = 126 of the 128 MMA rows (the TMA box still loads 128 rows);
//   * x_m tiles are 32 channels wide (8 four-channel blocks), z tiles 64: inner/32 + inner/64 column tiles, e.g.
//     72 x 2 = 144 CTAs at 48M x 64 envs -> one wave, and the pre-cell work is spread over 2/3 of them;
//   * 12 epilogue warps: TMEM -> shared (x_m) or TMEM -> global (z); then thread = (env, 4-channel block): the conv
//     window lives in registers across the 3 tokens, weights come from shared memory (fetched before the dependency
//     wait together with the envs' conv windows), gate partials of the tile's 8 blocks meet through a shuffle
//     reduce-scatter in a fixed order (deterministic) and leave as chunk blockIdx.x of gate_part [M, inner/32, 2*NH].
// ------------------------------------------------------------------------------------------------------------------
namespace upc {

constexpr int kT = 3;                       // tokens per env step
constexpr int kEnvs = BLOCK_M / kT;         // 42 envs per row tile
constexpr int kRows = kEnvs * kT;           // 126 rows owned by a tile
constexpr int kXW = 32;                     // x_m tile width (channels)
constexpr int kZW = 64;                     // z tile width
constexpr int kStages = 4;
constexpr int kEpiWarps = 12;            // 384 threads >= 42 envs x 8 blocks: one (env, block) item per thread
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kThreadsUp = 64 + kEpiThreads;
constexpr int kXS = kXW + 1;                // padded row stride of the staged x_m tile
constexpr int kABytes = BLOCK_M * BLOCK_K * 2;
constexpr int kWBoxBytes = kXW * BLOCK_K * 2;          // one 32-row box of W
constexpr int kStageBytes = 2 * kABytes + 2 * kWBoxBytes;
constexpr int kXsFloats = BLOCK_M * kXS;
constexpr int kWinFloats = kEnvs * 3 * kXW;            // rows 1..3 of each env's conv window
// per-tile weights in shared memory (floats): conv_w [32][4], conv_b [32], wq/wk/wv [8][16] each,
// gate weights [gate 2][head 4][part 3][32]
constexpr int kWConv = 0, kWBias = 128, kWQ = 160, kWK = 288, kWV = 416, kWG = 544, kWFloats = 544 + 768;
constexpr int kEpiOff = kStages * kStageBytes + 256;
constexpr int kSmemTotal = kEpiOff + (kXsFloats + kWinFloats + kWFloats) * 4 + 1024;

__global__ void __launch_bounds__(kThreadsUp, 1)
gemm_up_conv_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                    const __grid_constant__ CUtensorMap map_w, float* __restrict__ u, int M, int K, UpEpiParams ep) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = base + kStages * kStageBytes;        // full[kStages], empty[kStages], tmem_full, slot, win
  const uint32_t tmem_slot = bar_base + 8 * (2 * kStages + 1);
  const uint32_t win_bar = bar_base + 8 * (2 * kStages + 2);
  auto full_bar = [&](int s) { return bar_base + 8 * s; };
  auto empty_bar = [&](int s) { return bar_base + 8 * (kStages + s); };
  const uint32_t tmem_full_bar = bar_base + 8 * (2 * kStages);
  float* epi = reinterpret_cast<float*>(smem_raw + (base + kEpiOff - smem_u32(smem_raw)));
  float* xs = epi;                          // [128][33]  staged x_m tile
  float* cwin = xs + kXsFloats;             // [42][3][32] conv windows (rows 1..3)
  float* wsm = cwin + kWinFloats;           // per-tile weights

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inner = ep.inner, N = 2 * inner;
  const int NX = inner / kXW;                                    // x_m column tiles come first
  const bool xm_tile = (int)blockIdx.x < NX;
  const int n0 = xm_tile ? blockIdx.x * kXW : inner + ((int)blockIdx.x - NX) * kZW;
  const int nboxes = xm_tile ? 1 : 2;
  const int m0 = blockIdx.y * kRows;
  const int env0 = blockIdx.y * kEnvs;
  const int envs_here = min(kEnvs, ep.B - env0);
  const int num_kb = K / BLOCK_K;
  const uint32_t stage_tx = (uint32_t)(2 * kABytes + nboxes * kWBoxBytes);

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_hi) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a_lo) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    mbar_init(win_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(kZW) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

  // ---- before the dependency wait: weight tiles of the first ring round (never written by a kernel), and for x_m
  // tiles the conv windows of the tile's envs (only this kernel writes them, one env step ago) and the tile's
  // pre-cell weights
  const int pre_kb = num_kb < kStages ? num_kb : kStages;
  if (warp == 0 && lane == 0) {
    for (int kb = 0; kb < pre_kb; ++kb) {
      mbar_expect_tx(full_bar(kb), stage_tx);
      for (int bx = 0; bx < nboxes; ++bx)
        tma_load_2d(base + kb * kStageBytes + 2 * kABytes + bx * kWBoxBytes, &map_w, full_bar(kb), kb * BLOCK_K,
                    n0 + bx * kXW);
    }
  }
  const int et = (int)threadIdx.x - 64;                          // epilogue thread 0..511
  if (xm_tile && et >= 0) {
    if (et == 0) mbar_expect_tx(win_bar, (uint32_t)(envs_here * 3 * kXW * 4));
    asm volatile("bar.sync 2, %0;" ::"n"(kEpiThreads) : "memory");
    if (et < envs_here * 3) {
      const int e = et / 3, r = et - e * 3;
      const float* src = ep.conv_state + ((int64_t)(env0 + e) * 4 + 1 + r) * inner + n0;
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(smem_u32(cwin + et * kXW)), "l"(src), "r"((uint32_t)(kXW * 4)), "r"(win_bar)
                   : "memory");
    }
    for (int i = et; i < kWFloats; i += kEpiThreads) {
      float w;
      if (i < kWBias) w = ep.conv_w[(int64_t)n0 * 4 + i];                       // [ch][4], contiguous for the tile
      else if (i < kWQ) w = ep.conv_b[n0 + (i - kWBias)];
      else if (i < kWK) w = ep.wq[(int64_t)(n0 >> 2) * 16 + (i - kWQ)];          // [block][4][4]
      else if (i < kWV) w = ep.wk[(int64_t)(n0 >> 2) * 16 + (i - kWK)];
      else if (i < kWG) w = ep.wv[(int64_t)(n0 >> 2) * 16 + (i - kWV)];
      else {
        const int g = i - kWG, gate = g / 384, rem = g - gate * 384, h = rem / 96, rem2 = rem - h * 96;
        const int part = rem2 >> 5, ch = rem2 & 31;
        w = (gate ? ep.wf : ep.wi)[((int64_t)h * 3 + part) * inner + n0 + ch];
      }
      wsm[i] = w;
    }
  }
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      for (int kb = 0; kb < pre_kb; ++kb) {
        const uint32_t st = base + kb * kStageBytes;
        tma_load_2d(st, &map_a_hi, full_bar(kb), kb * BLOCK_K, m0);
        tma_load_2d(st + kABytes, &map_a_lo, full_bar(kb), kb * BLOCK_K, m0);
      }
      for (int kb = pre_kb; kb < num_kb; ++kb) {
        const int s = kb % kStages;
        const uint32_t ph = (kb / kStages) & 1;
        mbar_wait(empty_bar(s), ph ^ 1);
        const uint32_t st = base + s * kStageBytes;
        mbar_expect_tx(full_bar(s), stage_tx);
        tma_load_2d(st, &map_a_hi, full_bar(s), kb * BLOCK_K, m0);
        tma_load_2d(st + kABytes, &map_a_lo, full_bar(s), kb * BLOCK_K, m0);
        for (int bx = 0; bx < nboxes; ++bx)
          tma_load_2d(st + 2 * kABytes + bx * kWBoxBytes, &map_w, full_bar(s), kb * BLOCK_K, n0 + bx * kXW);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread): N = 32 (x_m tile) or 64 (z tile; the two 32-row W boxes are contiguous) =====
    if (lane == 0) {
      const uint32_t idesc = make_idesc(xm_tile ? kXW : kZW);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % kStages;
        const uint32_t ph = (kb / kStages) & 1;
        mbar_wait(full_bar(s), ph);
        tcgen05_fence_after();
        const uint32_t st = base + s * kStageBytes;
        const uint64_t a_hi = make_smem_desc(st);
        const uint64_t a_lo = make_smem_desc(st + kABytes);
        const uint64_t bw = make_smem_desc(st + 2 * kABytes);
#pragma unroll
        for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
          const uint64_t kofs = (uint64_t)((k * UMMA_K * 2) >> 4);
          umma_bf16(tmem_base, a_hi + kofs, bw + kofs, idesc, (kb | k) != 0);
          umma_bf16(tmem_base, a_lo + kofs, bw + kofs, idesc, 1u);
        }
        tcgen05_commit(empty_bar(s));
      }
      tcgen05_commit(tmem_full_bar);
    }
  } else {
    // ===== epilogue: 12 warps. TMEM lane quarter = warp % 4; two of the three warps of a quarter read the columns =====
    const int q = warp & 3, cg = (warp - 2) >> 2;                  // cg 0..2
    const int lrow = q * 32 + lane;                                // row inside the tile
    const int row = m0 + lrow;
    mbar_wait(tmem_full_bar, 0);
    tcgen05_fence_after();
    auto tmem_ld16 = [&](float (&v)[16], int c0) {
      uint32_t r[16];
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
          : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
            "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
          : "r"(taddr)
          : "memory");
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
    };
    if (!xm_tile) {
      // z tile: 32 columns per reading warp (two x16 loads), straight to u[:, inner + ...]
      if (cg < 2) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          float v[16];
          const int c0 = cg * 32 + half * 16;
          tmem_ld16(v, c0);
          if (lrow < kRows && row < M) {
            float* orow = u + (int64_t)row * N + n0 + c0;
#pragma unroll
            for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(orow + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          }
        }
      }
    } else {
      // x_m tile, phase 1: 16 columns per reading warp -> shared memory
      if (cg < 2) {
        float v[16];
        tmem_ld16(v, cg * 16);
#pragma unroll
        for (int j = 0; j < 16; ++j) xs[lrow * kXS + cg * 16 + j] = v[j];
      }
      asm volatile("bar.sync 2, %0;" ::"n"(kEpiThreads) : "memory");
      mbar_wait(win_bar, 0);
      // phase 2: thread = (env e, 4-channel block jb); the 8 blocks of an env are 8 consecutive lanes. Threads
      // without an env (e >= envs_here) run on env 0's data so that every lane takes part in the shuffles, and
      // store nothing. The token loop is NOT unrolled: weights are re-read from shared memory per token instead of
      // being hoisted into ~160 registers.
      const int jb = et & 7, e_raw = et >> 3;
      const bool valid = e_raw < envs_here;
      const int e = valid ? e_raw : 0;
      const int b = env0 + e;
      const int c = n0 + 4 * jb;
      float win[4][4];
#pragma unroll
      for (int rr = 0; rr < 3; ++rr) {
        const float4 w4 = *reinterpret_cast<const float4*>(cwin + (e * 3 + rr) * kXW + 4 * jb);
        win[rr + 1][0] = w4.x; win[rr + 1][1] = w4.y; win[rr + 1][2] = w4.z; win[rr + 1][3] = w4.w;
      }
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) win[0][ch] = 0.f;
      const float* cwp = wsm + kWConv + jb * 16;                 // [ch][4]
      const float* wqp = wsm + kWQ + jb * 16;
      const float* wkp = wsm + kWK + jb * 16;
      const float* wvp = wsm + kWV + jb * 16;
      // after the reduce-scatter (xor 4, 2, 1) lane jb holds the complete sum of gate value vi
      const int vi = ((jb & 4) ? 4 : 0) + ((jb & 2) ? 2 : 0) + (jb & 1);
#pragma unroll 1
      for (int t = 0; t < kT; ++t) {
        const int64_t grow = (int64_t)b * kT + t;
        float xm[4];
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) xm[ch] = xs[(e * kT + t) * kXS + 4 * jb + ch];
#pragma unroll
        for (int rr = 0; rr < 3; ++rr)
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) win[rr][ch] = win[rr + 1][ch];
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) win[3][ch] = xm[ch];
        float a[4];
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          float acc = 0.f;
#pragma unroll
          for (int rr = 0; rr < 4; ++rr) acc = fmaf(win[rr][ch], cwp[ch * 4 + rr], acc);
          a[ch] = silu(acc + wsm[kWBias + 4 * jb + ch]);
        }
        float qv[4], kv[4], vv[4];
#pragma unroll
        for (int o = 0; o < 4; ++o) {
          float sq = 0.f, sk = 0.f, sv = 0.f;
#pragma unroll
          for (int dd = 0; dd < 4; ++dd) {
            sq = fmaf(a[dd], wqp[4 * o + dd], sq);
            sk = fmaf(a[dd], wkp[4 * o + dd], sk);
            sv = fmaf(xm[dd], wvp[4 * o + dd], sv);
          }
          qv[o] = sq; kv[o] = sk; vv[o] = sv;
        }
        if (valid) {
          float* qk = ep.qk + (grow * inner + c) * 2;
          *reinterpret_cast<float4*>(qk) = make_float4(qv[0], kv[0], qv[1], kv[1]);
          *reinterpret_cast<float4*>(qk + 4) = make_float4(qv[2], kv[2], qv[3], kv[3]);
          *reinterpret_cast<float4*>(ep.v + grow * inner + c) = make_float4(vv[0], vv[1], vv[2], vv[3]);
          *reinterpret_cast<float4*>(ep.act + grow * inner + c) = make_float4(a[0], a[1], a[2], a[3]);
        }
        float gp[8];                                             // [gate][head]
#pragma unroll
        for (int gate = 0; gate < 2; ++gate)
#pragma unroll
          for (int h = 0; h < 4; ++h) {
            const float* gw = wsm + kWG + (gate * 4 + h) * 96 + 4 * jb;      // [part][32]
            const float4 wq4 = *reinterpret_cast<const float4*>(gw);
            const float4 wk4 = *reinterpret_cast<const float4*>(gw + 32);
            const float4 wv4 = *reinterpret_cast<const float4*>(gw + 64);
            float sg = qv[0] * wq4.x + qv[1] * wq4.y + qv[2] * wq4.z + qv[3] * wq4.w;
            sg += kv[0] * wk4.x + kv[1] * wk4.y + kv[2] * wk4.z + kv[3] * wk4.w;
            sg += vv[0] * wv4.x + vv[1] * wv4.y + vv[2] * wv4.z + vv[3] * wv4.w;
            gp[gate * 4 + h] = sg;
          }
        // gate partials of the tile's 32 channels: reduce-scatter over the env's 8 lanes, always
        // (lower lane's value) + (upper lane's value): a fixed order, so the sums are reproducible
        float w4v[4], w2v[2], w1v;
        {
          const bool hi = (jb & 4) != 0;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float send = hi ? gp[i] : gp[i + 4];
            const float keep = hi ? gp[i + 4] : gp[i];
            const float recv = __shfl_xor_sync(0xffffffffu, send, 4);
            w4v[i] = hi ? recv + keep : keep + recv;
          }
        }
        {
          const bool hi = (jb & 2) != 0;
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const float send = hi ? w4v[i] : w4v[i + 2];
            const float keep = hi ? w4v[i + 2] : w4v[i];
            const float recv = __shfl_xor_sync(0xffffffffu, send, 2);
            w2v[i] = hi ? recv + keep : keep + recv;
          }
        }
        {
          const bool hi = (jb & 1) != 0;
          const float send = hi ? w2v[0] : w2v[1];
          const float keep = hi ? w2v[1] : w2v[0];
          const float recv = __shfl_xor_sync(0xffffffffu, send, 1);
          w1v = hi ? recv + keep : keep + recv;
        }
        if (valid) ep.gate_part[((grow * ep.NCH) + blockIdx.x) * 8 + vi] = w1v;
      }
      if (valid) {
        // the window after the step: the last 4 inputs, oldest first (reference conv_state layout)
        float* cs = ep.conv_state + (int64_t)b * 4 * inner + c;
#pragma unroll
        for (int rr = 0; rr < 4; ++rr)
          *reinterpret_cast<float4*>(cs + (int64_t)rr * inner) = make_float4(win[rr][0], win[rr][1], win[rr][2], win[rr][3]);
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kZW) : "memory");
  }
}

}  // namespace upc

// fp32 rows -> bf16 hi/lo planes (dense [rows, K])
__global__ void __launch_bounds__(256) split_bf16_kernel(const float* __restrict__ in, int64_t in_stride,
                                                         __nv_bfloat16* __restrict__ hi,
                                                         __nv_bfloat16* __restrict__ lo, int rows, int K) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  pdl_wait();
  pdl_trigger();
  if (i >= (int64_t)rows * K) return;
  const int r = (int)(i / K), c = (int)(i - (int64_t)r * K);
  const float4 v = *reinterpret_cast<const float4*>(in + (int64_t)r * in_stride + c);
  const float x[4] = {v.x, v.y, v.z, v.w};
  __nv_bfloat16 h[4], l[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    h[j] = __float2bfloat16_rn(x[j]);
    l[j] = __float2bfloat16_rn(x[j] - __bfloat162float(h[j]));
  }
  *reinterpret_cast<uint2*>(hi + i) = *reinterpret_cast<uint2*>(h);
  *reinterpret_cast<uint2*>(lo + i) = *reinterpret_cast<uint2*>(l);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  // function-local static: initialised once, thread-safe (C++11); the driver entry point is process-wide
  static const EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      return (EncodeTiledFn)p;
    return (EncodeTiledFn) nullptr;
  }();
  return fn;
}

// bf16 row-major [rows, K] -> 2D map, box = {BLOCK_K, box_rows}, 128B swizzle, OOB reads give zeros
static bool make_map(CUtensorMap* m, const void* ptr, int rows, int K, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int g_m64_rows_contiguous = 0;     // xl_set_option("gemm_m64_layout"): probe of the M = 64 accumulator layout

template <int BLOCK_N, int kStages, int kBM = BLOCK_M, int kCX = 1>
static cudaError_t launch(const CUtensorMap& ma, const CUtensorMap& ml, const CUtensorMap& mw, const float* bias,
                          const float* residual, float* out, int M, int N, int K, int splits, long long split_stride,
                          cudaStream_t s) {
  using S = Smem<BLOCK_N, kStages, kBM>;
  if (cudaError_t e = ensure_dyn_smem<&gemm_tc_kernel<BLOCK_N, kStages, kBM, kCX>>(S::kTotal); e != cudaSuccess)
    return e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((N + BLOCK_N - 1) / BLOCK_N, (M + kBM - 1) / kBM, splits);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = S::kTotal;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (g_use_pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  if (kCX > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = kCX;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BLOCK_N, kStages, kBM, kCX>, ma, ml, mw, bias, residual, out, M, N, K,
                            split_stride, g_m64_rows_contiguous);
}

}  // namespace tc

// xl_set_option("gemm_2cta"): the 2-SM (cta_group::2) Linear with 256 x 256 tiles per CTA pair. -1 (default) = the
// persistent form for M >= 2048 rows (context prefill; measured -7 % on the 206M prefill), 0 = never, 1 / 2 = the
// one-tile-per-pair / persistent form whenever M >= 512
int g_gemm_2cta = -1;
int g_gemm_cluster = 1;   // xl_set_option("gemm_cluster"): 1 = off, 2 / 4 = A-tile TMA multicast across that many column tiles
int g_gemm_bm = 0;     // xl_set_option("gemm_bm"): 64 = 64-row MMA tiles where the shape allows, 0 / 128 = 128-row tiles
void gemm_tc_set_m64_layout(int contiguous) { tc::g_m64_rows_contiguous = contiguous ? 1 : 0; }

bool gemm_tc_supported(int M, int N, int K) { return K % tc::BLOCK_K == 0 && K >= tc::BLOCK_K && M >= 1 && N >= 8; }

void launch_split_bf16(const float* in, int64_t in_stride, void* hi, void* lo, int rows, int K, cudaStream_t s) {
  const int64_t n4 = (int64_t)rows * K / 4;
  launch_k(tc::split_bf16_kernel, dim3((unsigned)((n4 + 255) / 256)), dim3(256), 0, s, in, in_stride,
           (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, rows, K);
}

// Tile width and split-K factor from a small cost model. These skinny GEMMs (M = envs x tokens, a few hundred
// rows) are bound by the rate at which ONE SM can pull operand tiles out of L2 (~80 GB/s per SM through TMA,
// ~6.3 KB/clk chip-wide), not by the tensor pipe and not by L2 bandwidth: every CTA re-reads the A planes of
// its row tile. So the goal is to put ~one CTA on every SM with as few operand bytes per CTA as possible:
// wide tiles (fewer A re-reads) x split-K (more CTAs). A split-K CTA writes its partial tile to its own
// plane; the consumer kernels add the planes (costed below at L2 speed).
void gemm_tc_plan(int M, int N, int K, int num_sms, int max_splits, int* bn_out, int* splits_out) {
  const int m_tiles = (M + tc::BLOCK_M - 1) / tc::BLOCK_M;
  const int kb = K / tc::BLOCK_K;
  double best = 1e30;
  int best_bn = 64, best_sp = 1;
  const int bns[3] = {128, 64, 32};
  for (int bi = 0; bi < 3; ++bi) {
    const int bn = bns[bi];
    const int n_tiles = (N + bn - 1) / bn;
    for (int sp = 1; sp <= (max_splits < 1 ? 1 : max_splits); ++sp) {
      if (kb % sp) continue;
      const int kbp = kb / sp;
      const int ctas = m_tiles * n_tiles * sp;
      const int waves = (ctas + num_sms - 1) / num_sms;
      const double fill_kb = kbp * (2.0 * 16.0 + bn * 0.125);                // operand KB through TMA per CTA
      const double store_kb = 128.0 * bn * 4.0 / 1024.0;                     // output tile written per CTA
      double t = waves * (2.5 + fill_kb / 80.0 + store_kb / 80.0);           // us
      // consumers re-read sp planes; they are latency-bound kernels, so the extra loads cost as if at ~1.5 TB/s
      // (fitted to the B200 sweep in profiles/r01_gemm_splitk.md)
      if (sp > 1) t += 0.6 + (double)(sp - 1) * M * N * 4.0 / 1.5e6;
      if (t < best) { best = t; best_bn = bn; best_sp = sp; }
    }
  }
  *bn_out = best_bn;
  *splits_out = best_sp;
}

bool gemm_up_conv_supported(int T, int KS, int NH, int inner, int d) {
  return T == tc::upc::kT && KS == 4 && NH == 4 && inner % 64 == 0 && d % tc::BLOCK_K == 0 && d >= tc::BLOCK_K;
}
int gemm_up_conv_chunks(int inner) { return inner / tc::upc::kXW; }

// proj_up with the pre-cell epilogue: `u` [M, 2*inner] receives only its z half (columns >= inner)
cudaError_t launch_gemm_up_conv(const void* a_hi, const void* a_lo, const __nv_bfloat16* W, float* u, int M, int d,
                                const UpEpiParams& ep, cudaStream_t s) {
  namespace U = tc::upc;
  if (!gemm_up_conv_supported(ep.T, 4, 4, ep.inner, d) || M != ep.B * ep.T || ep.NCH != ep.inner / U::kXW)
    return cudaErrorInvalidValue;
  const int N = 2 * ep.inner;
  CUtensorMap ma, ml, mw;
  if (!tc::make_map(&ma, a_hi, M, d, tc::BLOCK_M) || !tc::make_map(&ml, a_lo, M, d, tc::BLOCK_M) ||
      !tc::make_map(&mw, W, N, d, U::kXW))
    return cudaErrorUnknown;
  if (cudaError_t e = ensure_dyn_smem<&U::gemm_up_conv_kernel>(U::kSmemTotal); e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(ep.inner / U::kXW + ep.inner / U::kZW, (ep.B + U::kEnvs - 1) / U::kEnvs, 1);
  cfg.blockDim = dim3(U::kThreadsUp);
  cfg.dynamicSmemBytes = U::kSmemTotal;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_use_pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, U::gemm_up_conv_kernel, ma, ml, mw, u, M, d, ep);
}

// bn: 128 / 64 / 32 (0 = plan it, without split-K). splits > 1: raw partial tiles go to out + z * split_stride
// (bias and residual must be null; the consumer adds the planes).
cudaError_t launch_gemm_tc(const void* a_hi, const void* a_lo, const __nv_bfloat16* W, const float* bias,
                           const float* residual, float* out, int M, int N, int K, int num_sms, int bn, int splits,
                           long long split_stride, cudaStream_t s) {
  if (!gemm_tc_supported(M, N, K)) return cudaErrorInvalidValue;
  if (splits < 1) splits = 1;
  if (splits > 1 && (bias || residual || (K / tc::BLOCK_K) % splits)) return cudaErrorInvalidValue;
  if (bn != 256 && bn != 128 && bn != 64 && bn != 32) {
    int sp;
    gemm_tc_plan(M, N, K, num_sms, 1, &bn, &sp);
  }
  const int two_sm = g_gemm_2cta < 0 ? (M >= 2048 ? 2 : 0) : (M >= 512 ? g_gemm_2cta : 0);
  if (two_sm && splits == 1 && N >= 256 && (bn == 256 || bn == 128)) {
    CUtensorMap ma2, ml2, mw2;
    if (!tc::make_map(&ma2, a_hi, M, K, tc::BLOCK_M) || !tc::make_map(&ml2, a_lo, M, K, tc::BLOCK_M) ||
        !tc::make_map(&mw2, W, N, K, 128))
      return cudaErrorUnknown;
    const bool persistent = two_sm == 2;
    if (cudaError_t e = persistent ? ensure_dyn_smem<&tc::two::gemm_tc2p_kernel>(tc::two::kTotalP)
                                   : ensure_dyn_smem<&tc::two::gemm_tc2_kernel>(tc::two::kTotal);
        e != cudaSuccess)
      return e;
    cudaLaunchConfig_t cfg = {};
    const int tiles = ((M + 255) / 256) * ((N + 255) / 256);
    const int pairs = tiles < num_sms / 2 ? tiles : num_sms / 2;
    cfg.gridDim = persistent ? dim3(2 * pairs, 1, 1) : dim3(2 * ((M + 255) / 256), (N + 255) / 256, 1);
    cfg.blockDim = dim3(tc::kThreads);
    cfg.dynamicSmemBytes = persistent ? tc::two::kTotalP : tc::two::kTotal;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g_use_pdl ? 2 : 1;
    if (persistent) return cudaLaunchKernelEx(&cfg, tc::two::gemm_tc2p_kernel, ma2, ml2, mw2, bias, residual, out, M, N, K);
    return cudaLaunchKernelEx(&cfg, tc::two::gemm_tc2_kernel, ma2, ml2, mw2, bias, residual, out, M, N, K);
  }
  if (bn == 256 && N % 256 != 0) bn = 128;
  // 64-row MMA tiles (option "gemm_bm" = 64): half the A bytes per k-block and a ring twice as deep (9 stages), no
  // empty quarter tile at M = 192. Bit-identical results; measured 1.2 % SLOWER on the 48M x 64 step (3 row tiles read
  // W three times: 42 MB instead of 38 MB of L2 -> SM traffic for proj_up, and these GEMMs sit at the aggregate L2
  // read rate), equal elsewhere (profiles/r02_chain_fusion.md) -> not the default.
  const bool bm64 = g_gemm_bm == 64 && bn == 64 && M > 16;
  // A-tile multicast across a cluster of 2 or 4 column-tile CTAs (option "gemm_cluster"; 128-row, 64-wide tiles only)
  const int n_tiles = (N + bn - 1) / bn;
  int cx = (!bm64 && (bn == 64 || bn == 128) && N % bn == 0) ? g_gemm_cluster : 1;
  while (cx > 1 && n_tiles % cx) cx >>= 1;
  CUtensorMap ma, ml, mw;
  const int box_m = bm64 ? 64 : tc::BLOCK_M / (cx > 1 ? cx : 1);
  if (!tc::make_map(&ma, a_hi, M, K, box_m) || !tc::make_map(&ml, a_lo, M, K, box_m) ||
      !tc::make_map(&mw, W, N, K, bn))
    return cudaErrorUnknown;
  if (bm64) return tc::launch<64, 9, 64>(ma, ml, mw, bias, residual, out, M, N, K, splits, split_stride, s);
  if (cx == 2 && bn == 64) return tc::launch<64, 4, tc::BLOCK_M, 2>(ma, ml, mw, bias, residual, out, M, N, K, splits, split_stride, s);
  if (cx == 4 && bn == 64) return tc::launch<64, 4, tc::BLOCK_M, 4>(ma, ml, mw, bias, residual, out, M, N, K, splits, split_stride, s);
  if (cx == 2) return tc::launch<128, 4, tc::BLOCK_M, 2>(ma, ml, mw, bias, residual, out, M, N, K, splits, split_stride, s);
  if (cx == 4) return tc::launch<128, 4, tc::BLOCK_M, 4>(ma, ml, mw, bias, residual, out, M, N, K, splits, split_stride, s);
  switch (bn) {
    // 128 x 256 tiles (GEMM-sized M, e.g. the context prefill): 2/3 of the operand bytes per flop of a 128 x 128 tile
    case 256: return tc::launch<256, 3>(ma, ml, mw, bias, residual, out, M, N, K, splits, split_stride, s);
    case 128: return tc::launch<128, 4>(ma, ml, mw, bias, residual, out, M, N, K, splits, split_stride, s);
    case 64: return tc::launch<64, 4>(ma, ml, mw, bias, residual, out, M, N, K, splits, split_stride, s);
    default: return tc::launch<32, 6>(ma, ml, mw, bias, residual, out, M, N, K, splits, split_stride, s);
  }
}

}  // namespace xl
