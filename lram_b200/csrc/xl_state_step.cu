// mLSTM recurrent state step — the HBM-bound kernel of the path.
//
// Replaces, per block and per env step, what the reference runs as ~17 ATen kernels per token
// ([ext-xlstm] mLSTMCell.step -> recurrent_step_stabilized_simple + MultiHeadLayerNorm, reached from
// src/algos/models/decision_xlstm.py:163) plus the output gating of mLSTMLayer.step:
//
//   for t in 0..T-1 (the T tokens of one env step, in order):
//     lf = logsigmoid(f~_t);  m' = max(lf + m, i~_t);  f = exp(lf + m - m');  i = exp(i~_t - m')
//     C  = f*C + i*(k_t/sqrt(DH)) (x) v_t          C[dk, dv], fp32, resident in HBM
//     n  = f*n + i*(k_t/sqrt(DH))
//     h_t = (q_t^T C) / (max(|q_t^T n|, exp(-m')) + eps)
//     out_t = (GroupNorm_head(h_t)*(1+w) + skip*a_t) * silu(z_t)
//
// Kernel 1 (stream): touches every C element exactly once (one 128-bit read, T fused multiply-adds + T
// dot-product FMAs in registers, one 128-bit write): algorithmic bytes = 8*NH*DH^2 per env regardless of T.
//   CTA = (env b, head h, row chunk rs, column slab cs). A thread owns 4 consecutive columns (dv) and walks
//   rows (dk); the q^T C reduction over rows is thread-local in the loop, crosses warps once through shared
//   memory, and leaves the CTA as a partial numerator [T, slab]. Nothing else: no atomics, no fences, so a CTA
//   retires while its stores are still draining.
//     impl 1 (default): a producer warp keeps a ring of [32 rows x 128 cols] fp32 tiles of C in flight with
//       TMA (cp.async.bulk.tensor.2d + mbarrier, L2 evict-first) and bulk-copies the step's (q,k) pairs;
//       8 consumer warps pull their rows from shared memory into registers, release the slot at once, do the
//       FMAs and write C back with streaming 128-bit stores.
//     impl 0: plain 128-bit global loads with register batching (comparison baseline).
// Kernel 2 (finalize): one CTA per (env, head): sums the row-chunk partials in fixed order (deterministic),
//   updates n and m, divides by the stabilised denominator, applies the multi-head GroupNorm, the learnable
//   skip and the output gate, and emits the bf16 hi/lo planes the proj_down tensor-core GEMM consumes.
#include <cuda.h>
#include <cuda_bf16.h>

#include "xl_common.cuh"
#include "xl_internal.h"

namespace xl {

constexpr int kThreads = 256;        // consumer threads
constexpr int kUnroll = 8;
constexpr int kMaxNCH = 128;

// stream-K partition of N stage tiles over G CTAs (impl 2): CTA c owns [sk_start(c), sk_start(c+1))
__host__ __device__ __forceinline__ int sk_start(const StateStepParams& p, int c) {
  return c * p.sk_q + (c < p.sk_r ? c : p.sk_r);
}
__host__ __device__ __forceinline__ int sk_cta_of(const StateStepParams& p, int tile) {
  const int big = p.sk_r * (p.sk_q + 1);
  return tile < big ? tile / (p.sk_q + 1) : p.sk_r + (tile - big) / p.sk_q;
}

// Gate pre-activation (token t, gate g in {i, f}) of head hd = sum of the NCH chunk partials + bias, for the warp's
// lanes 4*(2t+g). Four lanes per sum: lane `sub` adds chunks sub, sub+4, ... (independent loads: one round trip
// whatever NCH is), then the four sub-sums are added in a fixed order -> the same bits wherever this is evaluated
// (stream, finalize, fused and persistent variants). Must be called by a full warp.
template <int T>
__device__ __forceinline__ float gate_preact(const StateStepParams& p, int b, int hd, int lane) {
  const int NH = p.NH;
  const int pair = lane >> 2, sub = lane & 3;
  const int t = pair >> 1, is_f = pair & 1;
  float s = 0.f;
  if (pair < 2 * T) {
    const float* gp = p.gate_part + ((int64_t)b * T + t) * p.NCH * 2 * NH + (is_f ? NH : 0) + hd;
    for (int c = sub; c < p.NCH; c += 4) s += gp[c * 2 * NH];
  }
  const float s1 = __shfl_down_sync(0xffffffffu, s, 1);
  const float s01 = s + s1;                                   // valid in sub 0 and sub 2
  const float s23 = __shfl_down_sync(0xffffffffu, s01, 2);
  float tot = s01 + s23;
  if (pair < 2 * T && sub == 0) {
    const float* bias = is_f ? p.fgate_b : p.igate_b;
    if (bias) tot += bias[hd];
  }
  return tot;
}

// Gate recurrence of one (env, head) for the T tokens of the step. Called by one full warp; results in shared
// memory. Streaming CTAs and the finalize CTA run this same code on the same inputs -> identical f, i, m.
template <int T>
__device__ __forceinline__ void compute_gates(const StateStepParams& p, int b, int hd, int bh, float* s_f,
                                              float* s_i, float* s_m, float* s_pre) {
  const int lane = threadIdx.x & 31;
  const int NH = p.NH;
  {
    const float pre = gate_preact<T>(p, b, hd, lane);
    if ((lane & 3) == 0 && (lane >> 2) < 2 * T) s_pre[lane >> 2] = pre;
  }
  __syncwarp();
  if (lane == 0) {
    float mprev = p.m[bh];
    s_m[0] = mprev;
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const float ig = s_pre[2 * t], fg = s_pre[2 * t + 1];
      const float lf = log_sigmoid(fg);
      const float mnew = fmaxf(lf + mprev, ig);
      s_f[t] = expf(lf + mprev - mnew);
      s_i[t] = expf(ig - mnew);
      s_m[t + 1] = mnew;
      mprev = mnew;
    }
  }
  __syncwarp();
}

// One row of 4 columns through the T tokens: c <- f_t*c + k_t[r] * vi_t ; acc_t += q_t[r] * c
// with vi_t = v_t * i_t / sqrt(DH) pre-scaled per thread. qk = (q,k) pair of token 0 for this row; token t's
// pair is tstride floats further.
template <int T>
__device__ __forceinline__ void row_update(float (&c)[4], const float* __restrict__ qk, int tstride,
                                           const float (&f)[T], const float (&vi)[T][4], float (&acc)[T][4]) {
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const float2 q2 = *reinterpret_cast<const float2*>(qk + t * tstride);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      c[j] = fmaf(f[t], c[j], q2.y * vi[t][j]);
      acc[t][j] = fmaf(q2.x, c[j], acc[t][j]);
    }
  }
}

// C is stored SLAB-MAJOR in HBM: [B, NH, DH/Wc, DH (dk rows), Wc (dv cols)] with Wc = 128 when DH % 128 == 0
// (else Wc = DH, i.e. plain row-major): every [32 rows x 128 cols] tile is 16 contiguous KB, and the slabs of
// an (env, head) follow each other. Logical element C[bh][r][c] lives at
//   C + ((bh * (DH/Wc) + c / Wc) * DH + r) * Wc + c % Wc.
__host__ __device__ __forceinline__ int slab_width(int DH) { return (DH % 128 == 0) ? 128 : DH; }

struct TileCoord {
  int bh, b, hd, rs, cs, r0, nrows, c0, rows_per;
  int wc, slab_row0, cin;      // slab width, first row of the tile in the [B*NH*CSl*DH, Wc] view, column inside the slab
};
__device__ __forceinline__ TileCoord tile_coord(const StateStepParams& p) {
  TileCoord tc;
  const int CS = p.DH / p.cols_per_cta;
  const int tiles_per_head = CS * p.rows_split;
  tc.bh = blockIdx.x / tiles_per_head;
  const int tile = blockIdx.x - tc.bh * tiles_per_head;
  tc.rs = tile / CS;
  tc.cs = tile - tc.rs * CS;
  tc.b = tc.bh / p.NH;
  tc.hd = tc.bh - tc.b * p.NH;
  tc.rows_per = (p.DH + p.rows_split - 1) / p.rows_split;
  tc.r0 = tc.rs * tc.rows_per;
  tc.nrows = max(0, min(p.DH, tc.r0 + tc.rows_per) - tc.r0);
  tc.c0 = tc.cs * p.cols_per_cta;
  tc.wc = slab_width(p.DH);
  const int slab = tc.c0 / tc.wc;
  tc.cin = tc.c0 - slab * tc.wc;
  tc.slab_row0 = (tc.bh * (p.DH / tc.wc) + slab) * p.DH + tc.r0;
  return tc;
}

// cross-row-lane reduction of the per-thread numerators -> partial[bh][rs][t][c0 + c]
template <int T>
__device__ __forceinline__ void write_partials(const StateStepParams& p, const TileCoord& tc, float* sacc,
                                               const float (&acc)[T][4], int tx, int ty, int TX, int TY,
                                               int tid) {
#pragma unroll
  for (int t = 0; t < T; ++t)
    *reinterpret_cast<float4*>(sacc + ((ty * T + t) * TX + tx) * 4) =
        make_float4(acc[t][0], acc[t][1], acc[t][2], acc[t][3]);
  asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");
  const int W = p.cols_per_cta;
  for (int idx = tid; idx < T * W; idx += kThreads) {
    const int t = idx / W, c = idx - t * W;
    float s = 0.f;
    for (int y = 0; y < TY; ++y) s += sacc[(y * T + t) * W + c];
    p.partial[(((int64_t)tc.bh * p.rows_split + tc.rs) * T + t) * p.DH + tc.c0 + c] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// impl 0: register-batched global loads
// ------------------------------------------------------------------------------------------------
template <int T>
__global__ void __launch_bounds__(kThreads, 3) mlstm_state_stream_ldg_kernel(StateStepParams p) {
  extern __shared__ __align__(16) float smem[];
  __shared__ float s_f[T], s_i[T], s_m[T + 1], s_pre[2 * T];
  const TileCoord tc = tile_coord(p);
  const int DH = p.DH;
  const int TX = p.cols_per_cta >> 2, TY = kThreads / TX;
  const int tid = threadIdx.x, tx = tid % TX, ty = tid / TX;
  const int tstride = 2 * tc.rows_per;
  float* sqk = smem;                         // [T][rows_per][2]
  float* sacc = smem + T * tstride;          // [TY][T][cols_per_cta]

  pdl_wait();
  pdl_trigger();
  if (tid < 32) compute_gates<T>(p, tc.b, tc.hd, tc.bh, s_f, s_i, s_m, s_pre);
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const float2* src = reinterpret_cast<const float2*>(p.qk) + (((int64_t)tc.b * T + t) * p.NH + tc.hd) * DH + tc.r0;
    for (int r = tid; r < tc.nrows; r += kThreads) reinterpret_cast<float2*>(sqk + t * tstride)[r] = src[r];
  }
  float vi[T][4];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const float4 vv = *reinterpret_cast<const float4*>(p.v + ((int64_t)tc.b * T + t) * p.inner + tc.hd * DH +
                                                       tc.c0 + 4 * tx);
    vi[t][0] = vv.x; vi[t][1] = vv.y; vi[t][2] = vv.z; vi[t][3] = vv.w;
  }
  __syncthreads();
  const float kscale = rsqrtf((float)DH);
  float f[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    f[t] = s_f[t];
    const float it = s_i[t] * kscale;
#pragma unroll
    for (int j = 0; j < 4; ++j) vi[t][j] *= it;
  }
  float acc[T][4];
#pragma unroll
  for (int t = 0; t < T; ++t) acc[t][0] = acc[t][1] = acc[t][2] = acc[t][3] = 0.f;

  float4* Cp = reinterpret_cast<float4*>(p.C + (int64_t)tc.slab_row0 * tc.wc + tc.cin) + tx;
  const int64_t rs4 = tc.wc >> 2;            // row stride in float4 (slab-major C)
  int rbase = ty;
  for (; rbase + (kUnroll - 1) * TY < tc.nrows; rbase += TY * kUnroll) {   // full batches: no predicates
    float4 cv[kUnroll];
    float4* rp = Cp + (int64_t)rbase * rs4;
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) cv[u] = ld_stream(rp + (int64_t)u * TY * rs4);
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      float c[4] = {cv[u].x, cv[u].y, cv[u].z, cv[u].w};
      row_update<T>(c, sqk + 2 * (rbase + u * TY), tstride, f, vi, acc);
      st_stream(rp + (int64_t)u * TY * rs4, make_float4(c[0], c[1], c[2], c[3]));
    }
  }
  for (; rbase < tc.nrows; rbase += TY) {
    float4* rp = Cp + (int64_t)rbase * rs4;
    const float4 cv = ld_stream(rp);
    float c[4] = {cv.x, cv.y, cv.z, cv.w};
    row_update<T>(c, sqk + 2 * rbase, tstride, f, vi, acc);
    st_stream(rp, make_float4(c[0], c[1], c[2], c[3]));
  }
  write_partials<T>(p, tc, sacc, acc, tx, ty, TX, TY, tid);
}

// ------------------------------------------------------------------------------------------------
// impl 1: TMA-fed ring
// ------------------------------------------------------------------------------------------------
namespace tma {

constexpr int kStageRows = 32;
constexpr int kStages = 3;
constexpr int kConsumerWarps = kThreads / 32;
constexpr int kBlock = kThreads + 32;   // + producer warp

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
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
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// ---- fused finalize (kFused): the CS = DH/128 column-slab CTAs of one (env, head) form a thread-block CLUSTER.
// Each CTA ends the stream holding the complete numerators q^T C of its 128 columns (rows are not split), computes
// q.n for the whole head redundantly (DH FMAs per token), normalises its columns, and the GroupNorm statistics of
// the head meet over distributed shared memory: every CTA posts (sum, M2) of its 128 columns into every peer's
// shared memory with st.async, which completes the peer's mbarrier by byte count -- no global ticket, no memory
// fence on the streaming stores, no cluster barrier on the critical path (Chan's parallel-variance combination of
// the CS partial statistics, in rank order, identical in every CTA). Rank 0 writes n and m back after it has
// received every peer's statistics (which depend on the old n, m: all reads of them are done by then).
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_async_f32(uint32_t raddr, float v, uint32_t rbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
               ::"r"(raddr), "r"(__float_as_uint(v)), "r"(rbar) : "memory");
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire;" ::: "memory"); }

constexpr int kNRowsMax = 4;          // n rows per consumer thread: DH <= 4 * 256
constexpr int kMaxCluster = 8;
constexpr int kMaxClusterOptIn = 16;   // non-portable cluster size (per-kernel opt-in)

// sum of T values over the first `nwarps` consumer warps (fixed order); every consumer thread calls it
template <int T>
__device__ __forceinline__ void consumer_sum(float (&v)[T], float* red /* [T][8] */, int warp, int lane, int nwarps) {
#pragma unroll
  for (int t = 0; t < T; ++t) v[t] = warp_sum(v[t]);
  asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");      // protect `red` from its previous use
  if (lane == 0 && warp < nwarps) {
#pragma unroll
    for (int t = 0; t < T; ++t) red[t * 8 + warp] = v[t];
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");
#pragma unroll
  for (int t = 0; t < T; ++t) {
    float s = 0.f;
    for (int w = 0; w < nwarps; ++w) s += red[t * 8 + w];
    v[t] = s;
  }
}

template <int T>
__device__ __forceinline__ void fused_finalize(const StateStepParams& p, const TileCoord& tc, const float* sacc,
                                               const float* sqk, const float* sn, int tstride, const float* s_f,
                                               const float* s_i, const float* s_m, float* s_red, float* s_x,
                                               uint32_t xbar, int tid) {
  constexpr int W = 128;
  const int DH = p.DH, inner = p.inner, CS = DH / W;
  const int warp = tid >> 5, lane = tid & 31;
  const bool col = tid < W;                               // threads 0..127 own one output column each
  const int ch = tc.hd * DH + tc.c0 + (col ? tid : 0);
  // tail operands: issued first, consumed last (a and z were written two kernels back, weights never)
  float wn = 0.f, wskip = 0.f, act[T], zz[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int64_t row = (int64_t)tc.b * T + t;
    act[t] = (col && p.skip) ? p.act[row * inner + ch] : 0.f;
    zz[t] = (col && p.skip) ? p.u[row * 2 * inner + inner + ch] : 0.f;
    if (col && p.skip)
      for (int z = 1; z < p.u_splits; ++z) zz[t] += p.u[z * p.u_stride + row * 2 * inner + inner + ch];
  }
  if (col) {
    wn = p.outnorm_w[ch];
    wskip = p.skip ? p.skip[ch] : 0.f;
  }
  // numerators of this CTA's columns: sum over the 8 row lanes, fixed order
  float num[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    float s = 0.f;
    if (col)
      for (int y = 0; y < 8; ++y) s += sacc[(y * T + t) * W + tid];
    num[t] = s;
  }
  // n recurrence and q.n over the whole head (every CTA of the cluster computes the same numbers)
  const float kscale = rsqrtf((float)DH);
  float qn[T], nreg[kNRowsMax];
#pragma unroll
  for (int t = 0; t < T; ++t) qn[t] = 0.f;
#pragma unroll
  for (int j = 0; j < kNRowsMax; ++j) {
    const int r = tid + j * kThreads;
    nreg[j] = 0.f;
    if (r < DH) {
      float nv = sn[r];
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const float2 q2 = *reinterpret_cast<const float2*>(sqk + t * tstride + 2 * r);
        nv = fmaf(s_f[t], nv, s_i[t] * kscale * q2.y);
        qn[t] = fmaf(q2.x, nv, qn[t]);
      }
      nreg[j] = nv;
    }
  }
  consumer_sum<T>(qn, s_red, warp, lane, 8);
  // h and the statistics of this CTA's 128 columns: sum, then M2 about the local mean
  float hs[T], m2[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const float den = fmaxf(fabsf(qn[t]), expf(-s_m[t + 1])) + p.cell_eps;
    num[t] = num[t] / den;
    hs[t] = col ? num[t] : 0.f;
  }
  consumer_sum<T>(hs, s_red, warp, lane, 4);
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const float dlt = col ? num[t] - hs[t] * (1.f / W) : 0.f;
    m2[t] = dlt * dlt;
  }
  consumer_sum<T>(m2, s_red, warp, lane, 4);
  // post (sum, M2) into slot [rank] of every CTA of the cluster (own included)
  if (tid < 2 * T) {
    const float val = tid < T ? hs[tid] : m2[tid - T];
    const uint32_t slot = smem_u32(s_x + tc.cs * 8 + tid);
    for (int r = 0; r < CS; ++r) st_async_f32(mapa_u32(slot, (uint32_t)r), val, mapa_u32(xbar, (uint32_t)r));
  }
  mbar_wait(xbar, 0);
  float mean[T], rstd[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    float tot = 0.f;
    for (int k = 0; k < CS; ++k) tot += s_x[k * 8 + t];
    const float mu = tot / (float)DH;
    float M2 = 0.f;
    for (int k = 0; k < CS; ++k) {
      const float dk = s_x[k * 8 + t] * (1.f / W) - mu;
      M2 += s_x[k * 8 + T + t] + (float)W * dk * dk;
    }
    mean[t] = mu;
    rstd[t] = rsqrtf(M2 / (float)DH + p.ln_eps);
  }
  if (col) {
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int64_t row = (int64_t)tc.b * T + t;
      float o = (num[t] - mean[t]) * rstd[t] * (1.f + wn);
      if (p.h_raw) p.h_raw[row * inner + ch] = num[t];
      if (p.skip) o = (o + wskip * act[t]) * silu_fast(zz[t]);
      if (p.out) p.out[row * inner + ch] = o;
      if (p.out_hi) {
        const __nv_bfloat16 hi = __float2bfloat16_rn(o);
        reinterpret_cast<__nv_bfloat16*>(p.out_hi)[row * inner + ch] = hi;
        reinterpret_cast<__nv_bfloat16*>(p.out_lo)[row * inner + ch] = __float2bfloat16_rn(o - __bfloat162float(hi));
      }
    }
  }
  if (tc.cs == 0) {        // every peer's statistics are in: nobody still needs the old n, m
#pragma unroll
    for (int j = 0; j < kNRowsMax; ++j) {
      const int r = tid + j * kThreads;
      if (r < DH) p.n[(int64_t)tc.bh * DH + r] = nreg[j];
    }
    if (tid == 0) p.m[tc.bh] = s_m[T];
  }
}

// Leader variant (fuse_finalize == 2): every CTA of the cluster pushes the numerators of its [rows chunk x 128 columns]
// tile into rank 0's shared memory (st.async, counted by rank 0's mbarrier) and retires at once -- a fire-and-forget
// store from registers; only rank 0 stays, waits for the CS*RS contributions and finalizes the whole head.
// One tail per (env, head) instead of one per CTA. Rows may be split (RS > 1, the few-env tilings): the cluster is
// then the CS*RS tiles of the head and rank 0 adds the RS row-chunk numerators in chunk order.
// The sums are the finalize kernel's, in its order: value j of thread tid stands for that kernel's thread tid + 256*j,
// and leader_sum() reproduces its block_sum_n() tree (warp sums, then one warp sum over the warp totals). n, m and the
// numerators come out bit-identical to the two-kernel step; h differs in the last ulp (the compiler folds the
// division by the per-token denominator differently in the two kernels), 1e-7 relative on the hidden states.
template <int T>
__device__ __forceinline__ void leader_sum(float (&v)[kNRowsMax][T], float (&out)[T], float* red /* [T][32] */,
                                           int warp, int lane, int nw) {
#pragma unroll
  for (int j = 0; j < kNRowsMax; ++j)
#pragma unroll
    for (int t = 0; t < T; ++t) v[j][t] = warp_sum(v[j][t]);
  asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");      // protect `red` from its previous use
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < kNRowsMax; ++j)
      if (warp + 8 * j < nw) {
#pragma unroll
        for (int t = 0; t < T; ++t) red[t * 32 + warp + 8 * j] = v[j][t];
      }
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");
#pragma unroll
  for (int t = 0; t < T; ++t) out[t] = warp_sum(lane < nw ? red[t * 32 + lane] : 0.f);
}

template <int T>
__device__ __forceinline__ void leader_finalize(const StateStepParams& p, const TileCoord& tc, const float* sacc,
                                                const float* sqk, const float* sqkh, const float* sn, float* snum,
                                                int tstride, const float* s_f, const float* s_i, const float* s_m,
                                                float* s_red, uint32_t xbar, int tid) {
  constexpr int W = 128;
  const int DH = p.DH, inner = p.inner, CS = DH / W, RS = p.rows_split;
  const int warp = tid >> 5, lane = tid & 31;
  const int tile = tc.rs * CS + tc.cs;                   // == rank of this CTA in the cluster
  if (tid < W) {
    const uint32_t rbase = mapa_u32(smem_u32(snum + (tile * T) * W + tid), 0u);
    const uint32_t rbar = mapa_u32(xbar, 0u);
#pragma unroll
    for (int t = 0; t < T; ++t) {
      float s = 0.f;
      for (int y = 0; y < 8; ++y) s += sacc[(y * T + t) * W + tid];      // fixed order over the 8 row lanes
      st_async_f32(rbase + (uint32_t)(t * W * sizeof(float)), s, rbar);
    }
  }
  if (tile != 0) return;
  // ---- rank 0: the whole head. Thread tid owns channels (and n rows) tid + j*256
  const float* qkh = RS > 1 ? sqkh : sqk;                // (q,k) of every row of the head
  const int hstride = RS > 1 ? 2 * DH : tstride;
  const int nw = (DH + 31) >> 5;
  const float kscale = rsqrtf((float)DH);
  float nreg[kNRowsMax], v[kNRowsMax][T], qn[T];
#pragma unroll
  for (int j = 0; j < kNRowsMax; ++j) {
    const int r = tid + j * kThreads;
    float nv = r < DH ? sn[r] : 0.f;
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const float2 q2 = r < DH ? *reinterpret_cast<const float2*>(qkh + t * hstride + 2 * r) : make_float2(0.f, 0.f);
      nv = fmaf(s_f[t], nv, s_i[t] * kscale * q2.y);
      v[j][t] = q2.x * nv;
    }
    nreg[j] = nv;
  }
  leader_sum<T>(v, qn, s_red, warp, lane, nw);
  float den[T];
#pragma unroll
  for (int t = 0; t < T; ++t) den[t] = fmaxf(fabsf(qn[t]), expf(-s_m[t + 1])) + p.cell_eps;
  mbar_wait(xbar, 0);                                    // every tile's numerators have landed
  float hh[kNRowsMax][T], mean[T], var[T];
#pragma unroll
  for (int j = 0; j < kNRowsMax; ++j) {
    const int c = tid + j * kThreads;
#pragma unroll
    for (int t = 0; t < T; ++t) {
      float s = 0.f;
      if (c < DH)
        for (int r = 0; r < RS; ++r) s += snum[((r * CS + (c >> 7)) * T + t) * W + (c & 127)];   // chunk order
      hh[j][t] = s / den[t];
      v[j][t] = hh[j][t];
    }
  }
  leader_sum<T>(v, mean, s_red, warp, lane, nw);
#pragma unroll
  for (int t = 0; t < T; ++t) mean[t] /= (float)DH;
#pragma unroll
  for (int j = 0; j < kNRowsMax; ++j) {
    const int c = tid + j * kThreads;
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const float dlt = c < DH ? hh[j][t] - mean[t] : 0.f;
      v[j][t] = dlt * dlt;
    }
  }
  leader_sum<T>(v, var, s_red, warp, lane, nw);
#pragma unroll
  for (int j = 0; j < kNRowsMax; ++j) {
    const int c = tid + j * kThreads;
    if (c < DH) {
      const int ch = tc.hd * DH + c;
      const float wn = p.outnorm_w[ch];
      const float wskip = p.skip ? p.skip[ch] : 0.f;
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const int64_t row = (int64_t)tc.b * T + t;
        const float rstd = rsqrtf(var[t] / (float)DH + p.ln_eps);
        float o = (hh[j][t] - mean[t]) * rstd * (1.f + wn);
        if (p.h_raw) p.h_raw[row * inner + ch] = hh[j][t];
        if (p.skip) {
          float z = p.u[row * 2 * inner + inner + ch];
          for (int zz = 1; zz < p.u_splits; ++zz) z += p.u[zz * p.u_stride + row * 2 * inner + inner + ch];
          o = (o + wskip * p.act[row * inner + ch]) * silu_fast(z);
        }
        if (p.out) p.out[row * inner + ch] = o;
        if (p.out_hi) {
          const __nv_bfloat16 hi = __float2bfloat16_rn(o);
          reinterpret_cast<__nv_bfloat16*>(p.out_hi)[row * inner + ch] = hi;
          reinterpret_cast<__nv_bfloat16*>(p.out_lo)[row * inner + ch] = __float2bfloat16_rn(o - __bfloat162float(hi));
        }
      }
      p.n[(int64_t)tc.bh * DH + c] = nreg[j];
    }
  }
  if (tid == 0) p.m[tc.bh] = s_m[T];
}

template <int T, bool kStream, bool kFused>
__global__ void __launch_bounds__(kBlock, 3)
mlstm_state_stream_tma_kernel(const __grid_constant__ CUtensorMap mapC, StateStepParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ float s_f[T], s_i[T], s_m[T + 1], s_pre[2 * T];
  __shared__ __align__(8) uint64_t s_bar[2 * kStages + 2];
  __shared__ float s_red[4 * 32], s_x[kMaxCluster * 8];

  const TileCoord tc = tile_coord(p);
  const int DH = p.DH;
  const int W = p.cols_per_cta;
  const bool leader = kFused && p.fuse_finalize == 2 && tc.rs == 0 && tc.cs == 0;
  const bool head_qk = leader && p.rows_split > 1;       // rank 0 of a row-split cluster needs every (q,k) of the head
  const int TX = W >> 2, TY = kThreads / TX;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tstride = 2 * tc.rows_per;
  const int nblk = (tc.nrows + kStageRows - 1) / kStageRows;
  const uint32_t stage_bytes = (uint32_t)(kStageRows * W * sizeof(float));

  // dynamic smem: [ring: kStages x (32 x W) fp32 | 128-B aligned] [sqk: T x rows_per x 2]; the reduction
  // scratch aliases the ring once the loop is over
  const uint32_t sbase = (smem_u32(smem_raw) + 127u) & ~127u;
  float* stage0 = reinterpret_cast<float*>(smem_raw + (sbase - smem_u32(smem_raw)));
  float* sqk = stage0 + (size_t)kStages * kStageRows * W;
  float* sn = sqk + (size_t)T * tstride;      // kFused: n of the whole head [DH]
  float* snum = sn + DH;                      // kFused, leader variant: numerators of the head [RS*CS][T][128] (rank 0)
  float* sqkh = snum + (size_t)p.rows_split * T * DH;   // leader of a row-split cluster: (q,k) of the head [T][DH][2]
  float* sacc = stage0;
  const uint32_t bar0 = smem_u32(s_bar);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kStages + s); };
  const uint32_t qk_bar = bar0 + 8u * (2 * kStages);
  const uint32_t xbar = bar0 + 8u * (2 * kStages + 1);

  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), kConsumerWarps);
    }
    mbar_init(qk_bar, 1);
    if (kFused) {
      // the exchange barrier completes when the 2T statistics of each of the CS CTAs have landed (bytes)
      mbar_init(xbar, 1);
      if (p.fuse_finalize == 2) {
        if (leader) mbar_expect_tx(xbar, (uint32_t)(p.rows_split * DH * T * sizeof(float)));   // the head's numerators
      } else {
        mbar_expect_tx(xbar, (uint32_t)((DH / 128) * 2 * T * sizeof(float)));
      }
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  // peers may only target this CTA's exchange barrier once it is initialised: arrive now, wait after the
  // dependency wait (by then every CTA of the cluster has long arrived)
  if (kFused) cluster_arrive();

  if (warp == kConsumerWarps) {
    // ===== producer warp =====
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapC) : "memory");
      uint64_t policy = 0;
      if (kStream) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
      const int grow0 = tc.slab_row0;
      auto issue = [&](int i) {
        const int s = i % kStages;
        mbar_wait(empty_bar(s), ((i / kStages) & 1) ^ 1);
        mbar_expect_tx(full_bar(s), stage_bytes);
        const uint32_t dst = sbase + s * stage_bytes;
        if (kStream) {
          asm volatile(
              "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
              "[%0], [%1, {%3, %4}], [%2], %5;"
              ::"r"(dst), "l"(&mapC), "r"(full_bar(s)), "r"(tc.cin), "r"(grow0 + i * kStageRows), "l"(policy)
              : "memory");
        } else {
          asm volatile(
              "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
              ::"r"(dst), "l"(&mapC), "r"(full_bar(s)), "r"(tc.cin), "r"(grow0 + i * kStageRows)
              : "memory");
        }
      };
      // C was last written by the previous env step: the ring is filled before the dependency wait
      const int pre = nblk < kStages ? nblk : kStages;
      for (int i = 0; i < pre; ++i) issue(i);
      pdl_wait();
      pdl_trigger();
      if (kFused) cluster_wait();
      // the step's (q, k) pairs of this row chunk: T contiguous runs of nrows*8 bytes (+ n of the head when fused)
      mbar_expect_tx(qk_bar, (uint32_t)(T * tc.nrows * 8 + (kFused ? DH * 4 : 0) + (head_qk ? T * DH * 8 : 0)));
      if (kFused) bulk_copy_g2s(smem_u32(sn), p.n + (int64_t)tc.bh * DH, (uint32_t)(DH * 4), qk_bar);
      if (head_qk) {
#pragma unroll
        for (int t = 0; t < T; ++t)
          bulk_copy_g2s(smem_u32(sqkh + t * 2 * DH), p.qk + ((((int64_t)tc.b * T + t) * p.NH + tc.hd) * DH) * 2,
                        (uint32_t)(DH * 8), qk_bar);
      }
#pragma unroll
      for (int t = 0; t < T; ++t)
        bulk_copy_g2s(smem_u32(sqk + t * tstride),
                      p.qk + ((((int64_t)tc.b * T + t) * p.NH + tc.hd) * DH + tc.r0) * 2,
                      (uint32_t)(tc.nrows * 8), qk_bar);
      for (int i = pre; i < nblk; ++i) issue(i);
    } else {
      pdl_wait();
      pdl_trigger();
      if (kFused) cluster_wait();
    }
    return;   // consumers only use the named barrier 1 from here on
  }

  // ===== consumers =====
  const int tx = tid % TX, ty = tid / TX;
  pdl_wait();
  pdl_trigger();
  if (kFused) cluster_wait();
  if (warp == 0) compute_gates<T>(p, tc.b, tc.hd, tc.bh, s_f, s_i, s_m, s_pre);
  float vi[T][4];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const float4 vv = *reinterpret_cast<const float4*>(p.v + ((int64_t)tc.b * T + t) * p.inner + tc.hd * DH +
                                                       tc.c0 + 4 * tx);
    vi[t][0] = vv.x; vi[t][1] = vv.y; vi[t][2] = vv.z; vi[t][3] = vv.w;
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");
  const float kscale = rsqrtf((float)DH);
  float f[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    f[t] = s_f[t];
    const float it = s_i[t] * kscale;
#pragma unroll
    for (int j = 0; j < 4; ++j) vi[t][j] *= it;
  }
  float acc[T][4];
#pragma unroll
  for (int t = 0; t < T; ++t) acc[t][0] = acc[t][1] = acc[t][2] = acc[t][3] = 0.f;

  float4* Cp = reinterpret_cast<float4*>(p.C + (int64_t)tc.slab_row0 * tc.wc + tc.cin) + tx;
  const int64_t rs4 = tc.wc >> 2;
  constexpr int kRowsPerThread = 4;                 // fast path: TY == 8 -> 32 rows / 8 row lanes
  const bool fast = (TY * kRowsPerThread == kStageRows);
  mbar_wait(qk_bar, 0);
  for (int i = 0; i < nblk; ++i) {
    const int s = i % kStages;
    const float* st = stage0 + (size_t)s * kStageRows * W;
    const int rblk = i * kStageRows;
    const int rcur = min(kStageRows, tc.nrows - rblk);
    mbar_wait(full_bar(s), (i / kStages) & 1);
    if (fast && rcur == kStageRows) {
      float4 cv[kRowsPerThread];
#pragma unroll
      for (int j = 0; j < kRowsPerThread; ++j)
        cv[j] = *reinterpret_cast<const float4*>(st + (ty + j * 8) * W + 4 * tx);
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_bar(s));     // the slot is free as soon as it sits in registers
      float4* rp = Cp + (int64_t)(rblk + ty) * rs4;
#pragma unroll
      for (int j = 0; j < kRowsPerThread; ++j) {
        float c[4] = {cv[j].x, cv[j].y, cv[j].z, cv[j].w};
        row_update<T>(c, sqk + 2 * (rblk + ty + j * 8), tstride, f, vi, acc);
        const float4 o = make_float4(c[0], c[1], c[2], c[3]);
        if (kStream) st_stream(rp + (int64_t)j * 8 * rs4, o);
        else rp[(int64_t)j * 8 * rs4] = o;
      }
    } else {
      // generic path (small heads / ragged last tile)
      for (int r = ty; r < rcur; r += TY) {
        const float4 cv = *reinterpret_cast<const float4*>(st + r * W + 4 * tx);
        float c[4] = {cv.x, cv.y, cv.z, cv.w};
        row_update<T>(c, sqk + 2 * (rblk + r), tstride, f, vi, acc);
        Cp[(int64_t)(rblk + r) * rs4] = make_float4(c[0], c[1], c[2], c[3]);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_bar(s));
    }
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");   // every warp is done with the ring
  if (kFused) {
    // stage the per-row-lane numerators (TX == 32, TY == 8) and finish the (env, head) inside the cluster
#pragma unroll
    for (int t = 0; t < T; ++t)
      *reinterpret_cast<float4*>(sacc + ((ty * T + t) * TX + tx) * 4) =
          make_float4(acc[t][0], acc[t][1], acc[t][2], acc[t][3]);
    asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");
    if (p.fuse_finalize == 2)
      leader_finalize<T>(p, tc, sacc, sqk, sqkh, sn, snum, tstride, s_f, s_i, s_m, s_red, xbar, tid);
    else
      fused_finalize<T>(p, tc, sacc, sqk, sn, tstride, s_f, s_i, s_m, s_red, s_x, xbar, tid);
    return;
  }
  write_partials<T>(p, tc, sacc, acc, tx, ty, TX, TY, tid);
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

template <int T, bool kStream, bool kFused>
static cudaError_t launch(const StateStepParams& p, cudaStream_t s) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return cudaErrorUnknown;
  CUtensorMap map;
  const int wc = slab_width(p.DH);
  cuuint64_t gdim[2] = {(cuuint64_t)wc, (cuuint64_t)p.B * p.NH * (p.DH / wc) * p.DH};
  cuuint64_t gstride[1] = {(cuuint64_t)wc * sizeof(float)};
  cuuint32_t box[2] = {(cuuint32_t)p.cols_per_cta, (cuuint32_t)kStageRows};
  cuuint32_t estr[2] = {1, 1};
  if (enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, p.C, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) !=
      CUDA_SUCCESS)
    return cudaErrorInvalidValue;
  const int rows_per = (p.DH + p.rows_split - 1) / p.rows_split;
  const size_t ring = sizeof(float) * (size_t)kStages * kStageRows * p.cols_per_cta;
  const int TY = kThreads / (p.cols_per_cta / 4);
  const size_t red = sizeof(float) * (size_t)TY * T * p.cols_per_cta;       // aliases the ring
  const size_t smem = 128 + (ring > red ? ring : red) +
                      sizeof(float) * ((size_t)2 * T * rows_per +
                                       (kFused ? (size_t)p.DH * (1 + T * p.rows_split + (p.rows_split > 1 ? 2 * T : 0)) : 0));
  if (cudaError_t e = ensure_dyn_smem<&mlstm_state_stream_tma_kernel<T, kStream, kFused>>(smem); e != cudaSuccess)
    return e;
  const int CS = p.DH / p.cols_per_cta;
  const int64_t grid = (int64_t)p.B * p.NH * CS * p.rows_split;
  if (!kFused && p.fuse_finalize != 3)
    return launch_k(mlstm_state_stream_tma_kernel<T, kStream, false>, dim3((unsigned)grid), dim3(kBlock), smem, s, map,
                    p);
  // one cluster per (env, head): its CS column-slab (x RS row-chunk) CTAs
  const int csize = CS * p.rows_split;
  if (csize > 8) {      // > 8 CTAs per cluster is a per-kernel opt-in
    static std::atomic<bool> allowed[kMaxDevices];
    int dev = 0;
    if (cudaError_t e = cudaGetDevice(&dev); e != cudaSuccess) return e;
    const bool tracked = dev >= 0 && dev < kMaxDevices;
    if (!tracked || !allowed[dev].load(std::memory_order_acquire)) {
      if (cudaError_t e = cudaFuncSetAttribute(mlstm_state_stream_tma_kernel<T, kStream, kFused>,
                                               cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
          e != cudaSuccess)
        return e;
      if (tracked) allowed[dev].store(true, std::memory_order_release);
    }
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kBlock);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)csize;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_use_pdl ? 2 : 1;
  // (fuse_finalize == 3 is a measurement aid: the UNFUSED kernel under the same cluster shape)
  return cudaLaunchKernelEx(&cfg, mlstm_state_stream_tma_kernel<T, kStream, kFused>, map, p);
}

}  // namespace tma

// ------------------------------------------------------------------------------------------------
// impl 2: persistent TMA-fed ring with a stream-K partition of the state.
// The state of the launch is a list of N = B*NH*(DH/128)*(DH/32) stage tiles ([32 rows x 128 cols] fp32,
// 16 KB), ordered (env*head, column slab, row block). CTA c of G (one per SM) owns the contiguous run
// [c*q + min(c,r), ...) of q or q+1 tiles (q = N/G, r = N%G): every CTA moves the same number of bytes
// (+-16 KB), the ring of C tiles never drains between items, and there is neither wave quantisation nor a
// slow tail. A run crosses item = (env*head, column slab) boundaries; each (item, CTA) segment leaves one
// partial numerator [T, 128] in slot (c - first CTA of the item), and the finalize kernel adds an item's
// slots in slot order (deterministic; the same integer arithmetic on both sides).
//   warp 8  (1 thread): C-tile producer — cp.async.bulk.tensor.2d into a `stages`-deep ring, evict-first
//   warp 9            : segment-metadata producer — bulk copies of the segment's (q,k) pairs and v slab and
//                       the gate recurrence of its (env, head) into a small ring, ahead of the consumers
//   warps 0..7        : consumers — 128-bit shared loads, T x (2 FMA + 1 FMA) per element in registers,
//                       128-bit streaming stores back to C, one cross-warp reduction of q^T C per segment
// A 1-CTA/SM launch leaves shared memory and ~1700 thread slots per SM for the kernels that run beside it: the L2
// warm-up of the next block's C on the step's side stream, and the next kernel of the chain once programmatic
// dependent launch lets it start.
// ------------------------------------------------------------------------------------------------
namespace pers {

using tma::bulk_copy_g2s;
using tma::mbar_arrive;
using tma::mbar_expect_tx;
using tma::mbar_init;
using tma::mbar_wait;
using tma::smem_u32;

constexpr int kStageRows = 32;
constexpr int kW = 128;                       // column slab
constexpr int kMaxStages = 8;
constexpr int kMaxMetaSlots = 4;
constexpr int kMetaSlots = 3;                 // depth of the segment-metadata ring the launcher uses
constexpr int kConsumerWarps = kThreads / 32;
constexpr int kBlock = kThreads + 64;         // + C-tile producer warp + metadata producer warp
constexpr int kStageFloats = kStageRows * kW;

__device__ __forceinline__ void mbar_expect_tx_only(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

__host__ __device__ inline int meta_floats(int T, int DH) { return T * DH * 2 + T * kW + 16; }

template <int T, bool kStream>
__global__ void __launch_bounds__(kBlock, 2)
mlstm_state_stream_persistent_kernel(const __grid_constant__ CUtensorMap mapC, StateStepParams p, int stages,
                                     int meta_slots) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t s_bar[2 * kMaxStages + 2 * kMaxMetaSlots];

  const int DH = p.DH, CS = DH / kW, NH = p.NH;
  const int nblk = DH / kStageRows;                 // stage tiles per item
  const int mfl = meta_floats(T, DH);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cta = blockIdx.x;
  const int tile_begin = sk_start(p, cta), tile_end = sk_start(p, cta + 1);

  // dynamic smem: [ring: stages x 32 x 128 fp32 | 128-B aligned][meta ring][red: 2 x 8 x T x 128]
  const uint32_t sbase = (smem_u32(smem_raw) + 127u) & ~127u;
  float* ring = reinterpret_cast<float*>(smem_raw + (sbase - smem_u32(smem_raw)));
  float* meta = ring + (size_t)stages * kStageFloats;
  float* red = meta + (size_t)meta_slots * mfl;
  const uint32_t bar0 = smem_u32(s_bar);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kMaxStages + s); };
  auto meta_full = [&](int s) { return bar0 + 8u * (2 * kMaxStages + s); };
  auto meta_empty = [&](int s) { return bar0 + 8u * (2 * kMaxStages + kMaxMetaSlots + s); };

  if (tid == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), kConsumerWarps);
    }
    for (int s = 0; s < meta_slots; ++s) {
      mbar_init(meta_full(s), 1);
      mbar_init(meta_empty(s), kConsumerWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == kConsumerWarps) {
    // ===== C-tile producer: one TMA per stage tile, straight through the CTA's run =====
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapC) : "memory");
      uint64_t policy = 0;
      if (kStream) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
      int s = 0;
      uint32_t ph = 0;
      int item = tile_begin / nblk;
      int i = tile_begin - item * nblk;
      // C was last written by the previous env step: the first `stages` tiles are in flight before the
      // dependency wait, i.e. while the kernel that produces this step's q/k/v/gates is still running
      bool waited = false;
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        if (!waited && tile - tile_begin == stages) {
          pdl_wait();
          pdl_trigger();
          waited = true;
        }
        mbar_wait(empty_bar(s), ph ^ 1);
        mbar_expect_tx(full_bar(s), (uint32_t)(kStageFloats * sizeof(float)));
        const uint32_t dst = sbase + (uint32_t)(s * kStageFloats * sizeof(float));
        // slab-major C: tile t of the launch is the 16 KB at C + t * 16 KB
        const int c0 = 0, r0 = tile * kStageRows;
        if (kStream) {
          asm volatile(
              "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
              "[%0], [%1, {%3, %4}], [%2], %5;"
              ::"r"(dst), "l"(&mapC), "r"(full_bar(s)), "r"(c0), "r"(r0), "l"(policy)
              : "memory");
        } else {
          asm volatile(
              "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
              ::"r"(dst), "l"(&mapC), "r"(full_bar(s)), "r"(c0), "r"(r0)
              : "memory");
        }
        if (++s == stages) { s = 0; ph ^= 1; }
        if (++i == nblk) { i = 0; ++item; }
      }
      if (!waited) {
        pdl_wait();
        pdl_trigger();
      }
    } else {
      pdl_wait();
      pdl_trigger();
    }
    return;
  }

  if (warp == kConsumerWarps + 1) {
    // ===== segment-metadata producer =====
    pdl_wait();
    pdl_trigger();
    int slot = 0;
    uint32_t ph = 0;
    for (int tile = tile_begin; tile < tile_end;) {
      const int item = tile / nblk, i0 = tile - item * nblk;
      const int cnt = min(nblk - i0, tile_end - tile);
      const int bh = item / CS, cs = item - bh * CS;
      const int b = bh / NH, hd = bh - b * NH;
      const int r0 = i0 * kStageRows, rows = cnt * kStageRows;
      float* ms = meta + (size_t)slot * mfl;
      float* s_gate = ms + T * DH * 2 + T * kW;                 // f[0..T) at +0, i[0..T) at +4
      // gate pre-activations: loads issued before anything waits
      const float pre = gate_preact<T>(p, b, hd, lane);          // the same sums, in the same order, as compute_gates()
      float mprev = p.m[bh];
      if (lane == 0) {
        mbar_wait(meta_empty(slot), ph ^ 1);                     // consumers released this slot
        mbar_expect_tx_only(meta_full(slot), (uint32_t)(T * rows * 8 + T * kW * 4));
#pragma unroll
        for (int t = 0; t < T; ++t) {
          bulk_copy_g2s(smem_u32(ms + t * DH * 2),
                        p.qk + ((((int64_t)b * T + t) * NH + hd) * DH + r0) * 2, (uint32_t)(rows * 8),
                        meta_full(slot));
          bulk_copy_g2s(smem_u32(ms + T * DH * 2 + t * kW),
                        p.v + ((int64_t)b * T + t) * p.inner + hd * DH + cs * kW, (uint32_t)(kW * 4),
                        meta_full(slot));
        }
      }
      // same arithmetic, same order as compute_gates() (the finalize kernel) -> identical f, i
      float fv[T], iv[T];
#pragma unroll
      for (int t = 0; t < T; ++t) {
        const float ig = __shfl_sync(0xffffffffu, pre, 8 * t);
        const float fg = __shfl_sync(0xffffffffu, pre, 8 * t + 4);
        const float lf = log_sigmoid(fg);
        const float mnew = fmaxf(lf + mprev, ig);
        fv[t] = expf(lf + mprev - mnew);
        iv[t] = expf(ig - mnew);
        mprev = mnew;
      }
      if (lane == 0) {
#pragma unroll
        for (int t = 0; t < T; ++t) {
          s_gate[t] = fv[t];
          s_gate[4 + t] = iv[t];
        }
        mbar_arrive(meta_full(slot));                            // release: gates visible with the phase
      }
      __syncwarp();
      if (++slot == meta_slots) { slot = 0; ph ^= 1; }
      tile += cnt;
    }
    return;
  }

  // ===== consumers: warp w owns rows w, w+8, w+16, w+24 of every 32-row tile; lane owns 4 columns =====
  const int tx = lane, ty = warp;
  const float kscale = rsqrtf((float)DH);
  const int64_t rs4 = kW >> 2;
  const int tstride = 2 * DH;
  pdl_wait();
  pdl_trigger();
  int s = 0, slot = 0, seg = 0;
  uint32_t ph = 0, mph = 0;
  for (int tile = tile_begin; tile < tile_end; ++seg) {
    const int item = tile / nblk, i0 = tile - item * nblk;
    const int cnt = min(nblk - i0, tile_end - tile);
    const int bh = item / CS, cs = item - bh * CS;
    const float* ms = meta + (size_t)slot * mfl;
    const float* sqk = ms;                                       // [T][rows of this segment][2]
    const float* sv = ms + T * DH * 2;
    const float* s_gate = sv + T * kW;
    mbar_wait(meta_full(slot), mph);
    float f[T], vi[T][4], acc[T][4];
#pragma unroll
    for (int t = 0; t < T; ++t) {
      f[t] = s_gate[t];
      const float it_ = s_gate[4 + t] * kscale;
      const float4 vv = *reinterpret_cast<const float4*>(sv + t * kW + 4 * tx);
      vi[t][0] = vv.x * it_; vi[t][1] = vv.y * it_; vi[t][2] = vv.z * it_; vi[t][3] = vv.w * it_;
      acc[t][0] = acc[t][1] = acc[t][2] = acc[t][3] = 0.f;
    }
    float4* Cp = reinterpret_cast<float4*>(p.C + (int64_t)tile * kStageFloats) + tx;   // slab-major C
    for (int i = 0; i < cnt; ++i) {
      const float* st = ring + (size_t)s * kStageFloats;
      const int rblk = i * kStageRows;
      mbar_wait(full_bar(s), ph);
      float4 cv[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) cv[r] = *reinterpret_cast<const float4*>(st + (ty + r * 8) * kW + 4 * tx);
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_bar(s));       // the slot is free as soon as it sits in registers
      if (++s == stages) { s = 0; ph ^= 1; }
      float4* rp = Cp + (int64_t)(rblk + ty) * rs4;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        float c[4] = {cv[r].x, cv[r].y, cv[r].z, cv[r].w};
        row_update<T>(c, sqk + 2 * (rblk + ty + r * 8), tstride, f, vi, acc);
        const float4 o = make_float4(c[0], c[1], c[2], c[3]);
        if (kStream) st_stream(rp + (int64_t)r * 8 * rs4, o);
        else rp[(int64_t)r * 8 * rs4] = o;
      }
    }
    // q^T C of this segment: cross-warp reduction in a double-buffered scratch (one named barrier per segment)
    float* rb = red + (seg & 1) * (kConsumerWarps * T * kW);
#pragma unroll
    for (int t = 0; t < T; ++t)
      *reinterpret_cast<float4*>(rb + (ty * T + t) * kW + 4 * tx) =
          make_float4(acc[t][0], acc[t][1], acc[t][2], acc[t][3]);
    __syncwarp();
    if (lane == 0) mbar_arrive(meta_empty(slot));     // (q,k), v, gates of this slot are no longer needed
    if (++slot == meta_slots) { slot = 0; mph ^= 1; }
    asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");
    const int pslot = cta - sk_cta_of(p, item * nblk);
    float* dst = p.partial + (((int64_t)item * p.sk_smax + pslot) * T) * kW;
    for (int idx = tid; idx < T * kW; idx += kThreads) {
      float sum = 0.f;
      const int t = idx / kW, c = idx - t * kW;
#pragma unroll
      for (int y = 0; y < kConsumerWarps; ++y) sum += rb[(y * T + t) * kW + c];
      dst[idx] = sum;
    }
    tile += cnt;
  }
}

static size_t smem_bytes(int T, int DH, int stages, int meta_slots) {
  return 128 + sizeof(float) * ((size_t)stages * kStageFloats + (size_t)meta_slots * meta_floats(T, DH) +
                                2 * (size_t)kConsumerWarps * T * kW);
}

template <int T, bool kStream>
static cudaError_t launch(const StateStepParams& p, cudaStream_t s) {
  tma::EncodeTiledFn enc = tma::get_encode();
  if (!enc) return cudaErrorUnknown;
  CUtensorMap map;
  cuuint64_t gdim[2] = {(cuuint64_t)kW, (cuuint64_t)p.B * p.NH * p.DH * (p.DH / kW)};
  cuuint64_t gstride[1] = {(cuuint64_t)kW * sizeof(float)};
  cuuint32_t box[2] = {(cuuint32_t)kW, (cuuint32_t)kStageRows};
  cuuint32_t estr[2] = {1, 1};
  if (enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, p.C, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) !=
      CUDA_SUCCESS)
    return cudaErrorInvalidValue;
  int stages = p.stages > 0 ? p.stages : 6;
  if (stages > kMaxStages) stages = kMaxStages;
  if (stages < 2) stages = 2;
  const size_t smem = smem_bytes(T, p.DH, stages, kMetaSlots);
  if (cudaError_t e = ensure_dyn_smem<&mlstm_state_stream_persistent_kernel<T, kStream>>(smem); e != cudaSuccess)
    return e;
  return launch_k(mlstm_state_stream_persistent_kernel<T, kStream>, dim3((unsigned)p.sk_grid), dim3(kBlock), smem,
                  s, map, p, stages, kMetaSlots);
}

}  // namespace pers

// ------------------------------------------------------------------------------------------------
// kernel 2: finalize one (env, head)
// Latency-bound (a few KB per CTA), so: every global load is issued up front, and the T tokens share each
// block reduction (3 reductions in total: q.n, mean, variance) instead of doing 3 per token.
// ------------------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void block_sum_n(float (&v)[N], float* red /* [N][32] */) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int k = 0; k < N; ++k) v[k] = warp_sum(v[k]);
  __syncthreads();                     // protect `red` from the previous use
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < N; ++k) red[k * 32 + wid] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < N; ++k) {
    float r = (lane < nw) ? red[k * 32 + lane] : 0.f;
    v[k] = warp_sum(r);
  }
}

// blockDim = DH rounded up to a warp multiple (<= 1024): one head channel per thread, all T tokens. Straight
// and short on purpose: every CTA runs this code once, so its size is what the instruction cache sees.
template <int T>
__global__ void __launch_bounds__(1024) mlstm_state_finalize_kernel(StateStepParams p) {
  __shared__ float s_f[T], s_i[T], s_m[T + 1], s_pre[2 * T];
  __shared__ float s_red[T * 32];
  const int bh = blockIdx.x;
  const int b = bh / p.NH, hd = bh - b * p.NH;
  const int DH = p.DH, inner = p.inner, RS = p.rows_split;
  const int a = threadIdx.x;
  const bool ok = a < DH;
  const int ch = hd * DH + (ok ? a : 0);

  // ---- all global loads first ---------------------------------------------------------------------
  float nreg = ok ? p.n[(int64_t)bh * DH + a] : 0.f;
  const float wn = ok ? p.outnorm_w[ch] : 0.f;
  const float wskip = (ok && p.skip) ? p.skip[ch] : 0.f;
  // Only the partial numerators come from the kernel right before this one (the state stream); n, m, the gate
  // partials, (q,k), a and z were written at least two kernels back, so they are loaded, and the gate
  // recurrence is computed, BEFORE the dependency wait — i.e. while the state stream is still running.
  float2 qk[T];
  float num[T], act[T], zz[T];
  int sk_item = 0, sk_nseg = 0;
  if (p.sk_grid > 0 && ok) {
    const int nblk = DH >> 5;
    sk_item = bh * (DH >> 7) + (a >> 7);
    sk_nseg = sk_cta_of(p, (sk_item + 1) * nblk - 1) - sk_cta_of(p, sk_item * nblk) + 1;
  }
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int64_t row = (int64_t)b * T + t;
    qk[t] = ok ? reinterpret_cast<const float2*>(p.qk)[(row * p.NH + hd) * DH + a] : make_float2(0.f, 0.f);
    act[t] = (ok && p.skip) ? p.act[row * inner + ch] : 0.f;
    zz[t] = (ok && p.skip) ? p.u[row * 2 * inner + inner + ch] : 0.f;
    if (ok && p.skip)
      for (int z = 1; z < p.u_splits; ++z) zz[t] += p.u[z * p.u_stride + row * 2 * inner + inner + ch];
  }
  if (threadIdx.x < 32) compute_gates<T>(p, b, hd, bh, s_f, s_i, s_m, s_pre);
  __syncthreads();
  // ---- n recurrence, q.n and the denominators for the T tokens: nothing here depends on the state stream either, so
  // this block reduction also runs before the dependency wait ------------------------------------------------------
  const float kscale = rsqrtf((float)DH);
  float qn[T], den[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    nreg = fmaf(s_f[t], nreg, s_i[t] * kscale * qk[t].y);
    qn[t] = qk[t].x * nreg;
  }
  block_sum_n<T>(qn, s_red);
#pragma unroll
  for (int t = 0; t < T; ++t) den[t] = fmaxf(fabsf(qn[t]), expf(-s_m[t + 1])) + p.cell_eps;
  pdl_wait();
  pdl_trigger();
#pragma unroll
  for (int t = 0; t < T; ++t) {
    float s = 0.f;
    if (ok) {
      if (p.sk_grid > 0) {     // stream-K slots of item (bh, column slab), in slot order
        const float* pp = p.partial + ((int64_t)sk_item * p.sk_smax * T + t) * 128 + (a & 127);
        for (int r = 0; r < sk_nseg; ++r) s += pp[(int64_t)r * T * 128];
      } else {
        // row-chunk partials in fixed order; the first 8 are requested as one batch (a plain loop is scheduled as
        // load -> add -> load: one L2 round trip per row chunk on the critical path of the few-env tilings)
        const float* pp = p.partial + ((int64_t)bh * RS * T + t) * DH + a;
        if (RS == 1) {
          s += pp[0];
        } else {
          float pr[8];
#pragma unroll
          for (int r = 0; r < 8; ++r) pr[r] = pp[(int64_t)(r < RS ? r : 0) * T * DH];
#pragma unroll
          for (int r = 0; r < 8; ++r)
            if (r < RS) s += pr[r];
          for (int r = 8; r < RS; ++r) s += pp[(int64_t)r * T * DH];
        }
      }
    }
    num[t] = s;
  }
  if (ok) p.n[(int64_t)bh * DH + a] = nreg;
  // ---- h = num / den, GroupNorm over the head, skip + output gate -----------------------------------
  float mean[T], var[T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    num[t] = num[t] / den[t];                // h (zero for the padded threads)
    mean[t] = num[t];
  }
  block_sum_n<T>(mean, s_red);
#pragma unroll
  for (int t = 0; t < T; ++t) {
    mean[t] /= (float)DH;
    const float dlt = ok ? num[t] - mean[t] : 0.f;
    var[t] = dlt * dlt;
  }
  block_sum_n<T>(var, s_red);
  if (ok) {
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const float rstd = rsqrtf(var[t] / (float)DH + p.ln_eps);
      const int64_t row = (int64_t)b * T + t;
      float o = (num[t] - mean[t]) * rstd * (1.f + wn);
      if (p.h_raw) p.h_raw[row * inner + ch] = num[t];
      if (p.skip) o = (o + wskip * act[t]) * silu_fast(zz[t]);
      if (p.out) p.out[row * inner + ch] = o;
      if (p.out_hi) {
        // A = hi + lo with hi = bf16(A), lo = bf16(A - hi): operand planes of the tcgen05 proj_down
        const __nv_bfloat16 hi = __float2bfloat16_rn(o);
        reinterpret_cast<__nv_bfloat16*>(p.out_hi)[row * inner + ch] = hi;
        reinterpret_cast<__nv_bfloat16*>(p.out_lo)[row * inner + ch] = __float2bfloat16_rn(o - __bfloat162float(hi));
      }
    }
  }
  if (threadIdx.x == 0) p.m[bh] = s_m[T];
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
void state_step_auto_tiling(int B, int NH, int DH, int num_sms, int* rows_split, int* cols_per_cta) {
  // column slab: widest of {128, 64, 32, 16, 8, 4} that divides DH (a warp then reads 512 contiguous B)
  int cols = 128;
  while (cols > 4 && (DH % cols) != 0) cols >>= 1;
  if (cols > DH) cols = DH;
  const int CS = DH / cols;
  // split rows (in multiples of the 32-row TMA tile) until there are enough CTAs to fill the machine
  const int64_t target = (int64_t)num_sms * 3;
  int rs = 1;
  while ((int64_t)B * NH * CS * rs < target && (DH % (rs * 2 * 32)) == 0 && rs < 32) rs *= 2;
  *rows_split = rs;
  *cols_per_cta = cols;
}

static bool persistent_ok(const StateStepParams& p) {
  return p.impl == 2 && p.DH % pers::kW == 0 && p.DH >= pers::kW && p.rows_split <= 0 &&
         (p.cols_per_cta <= 0 || p.cols_per_cta == pers::kW);
}

template <int T>
static cudaError_t launch_T(const StateStepParams& p, cudaStream_t s) {
  // stream (evict-first) when the stack's C does not fit comfortably in L2; keep it cached when it does
  const size_t c_bytes = sizeof(float) * (size_t)p.B * p.NH * p.DH * p.DH;
  const bool stream = c_bytes * (size_t)(p.num_layers > 0 ? p.num_layers : 1) > ((size_t)64 << 20);
  if (p.sk_grid > 0) return stream ? pers::launch<T, true>(p, s) : pers::launch<T, false>(p, s);
  const int rows_per = (p.DH + p.rows_split - 1) / p.rows_split;
  cudaError_t e;
  if (p.impl >= 1 && rows_per % 4 == 0) {
    if (p.fuse_finalize == 1 || p.fuse_finalize == 2)
      e = stream ? tma::launch<T, true, true>(p, s) : tma::launch<T, false, true>(p, s);
    else
      e = stream ? tma::launch<T, true, false>(p, s) : tma::launch<T, false, false>(p, s);
  } else {
    const int TX = p.cols_per_cta / 4, TY = kThreads / TX;
    const size_t smem = sizeof(float) * ((size_t)2 * T * rows_per + (size_t)TY * T * p.cols_per_cta);
    e = ensure_dyn_smem<&mlstm_state_stream_ldg_kernel<T>>(smem);
    if (e != cudaSuccess) return e;
    const int CS = p.DH / p.cols_per_cta;
    const int64_t grid = (int64_t)p.B * p.NH * CS * p.rows_split;
    e = launch_k(mlstm_state_stream_ldg_kernel<T>, dim3((unsigned)grid), dim3(kThreads), smem, s, p);
  }
  return e;
}

// Both kernels of the step resolve the tiling with this function, from the same inputs.
// rows_split / cols_per_cta given explicitly (> 0) select the rows_split layout of impl 0/1.
static void resolve_tiling(StateStepParams& p, int num_sms) {
  p.sk_grid = 0;
  if (persistent_ok(p)) {
    const int64_t N = (int64_t)p.B * p.NH * (p.DH / pers::kW) * (p.DH / pers::kStageRows);
    const int64_t cap = (int64_t)num_sms * (p.ctas_per_sm > 0 ? p.ctas_per_sm : 1);
    const int G = (int)(N < cap ? N : cap);
    const int nblk = p.DH / pers::kStageRows;
    p.sk_grid = G;
    p.sk_q = (int)(N / G);
    p.sk_r = (int)(N % G);
    const int by_q = (nblk + p.sk_q - 1) / p.sk_q + 1;
    p.sk_smax = by_q < nblk ? by_q : nblk;
    p.cols_per_cta = pers::kW;
    p.rows_split = 1;
    return;
  }
  if (p.rows_split <= 0 || p.cols_per_cta <= 0) {
    int rs, cols;
    state_step_auto_tiling(p.B, p.NH, p.DH, num_sms, &rs, &cols);
    // leader-fused finalize: the CS*RS tiles of a head are one thread-block cluster (<= 16 CTAs)
    if (p.fuse_finalize == 2 && cols == 128) {
      const int cap = (p.max_cluster > 0 && p.max_cluster < tma::kMaxClusterOptIn) ? p.max_cluster : tma::kMaxClusterOptIn;
      while (rs > 1 && (p.DH / 128) * rs > cap) rs >>= 1;
    }
    if (p.rows_split <= 0) p.rows_split = rs;
    if (p.cols_per_cta <= 0) p.cols_per_cta = cols;
  }
}

// True when launch_state_step(p) will also finalize (n/m update, normalise, gate) inside the stream kernel: the
// one-shot TMA kernel, 128-column slabs, DH <= 1024, and the tiles of a head fit one cluster -- rows not split and
// <= 8 slabs for the symmetric variant (1); <= 16 tiles (slabs x row chunks) for the leader variant (2).
bool state_step_fuses_finalize(StateStepParams p, int num_sms) {
  if (p.fuse_finalize != 1 && p.fuse_finalize != 2) return false;
  if (p.impl != 1) return false;
  resolve_tiling(p, num_sms);
  if (p.sk_grid != 0 || p.cols_per_cta != 128 || p.DH % 128 != 0 || p.DH > tma::kNRowsMax * kThreads || p.T > 4)
    return false;
  const int CS = p.DH / 128;
  if (p.fuse_finalize == 1) return p.rows_split == 1 && CS <= tma::kMaxCluster;
  return p.DH % (p.rows_split * 4) == 0 && CS * p.rows_split <= tma::kMaxClusterOptIn &&
         (p.rows_split == 1 ? CS <= tma::kMaxCluster : true);
}

// The separate finalize kernel and the stream kernel must resolve the same tiling: a fuse request the stream kernel
// cannot honour is dropped before the tiling is resolved (the leader variant caps the row split).
static void drop_unfusable(StateStepParams& p, int num_sms) {
  if (!state_step_fuses_finalize(p, num_sms)) {
    // the cluster probe (3) keeps its value only where the fused kernel would have run
    StateStepParams q = p;
    q.fuse_finalize = 1;
    p.fuse_finalize = (p.fuse_finalize == 3 && state_step_fuses_finalize(q, num_sms)) ? 3 : 0;
  }
}

// kernel 2; p must carry the same rows_split the stream kernel ran with (resolved here the same way)
cudaError_t launch_state_finalize(StateStepParams p, int num_sms, cudaStream_t s) {
  drop_unfusable(p, num_sms);
  resolve_tiling(p, num_sms);
  const int thr = ((p.DH + 31) / 32) * 32;
  switch (p.T) {
    case 1: return launch_k(mlstm_state_finalize_kernel<1>, dim3(p.B * p.NH), dim3(thr), 0, s, p);
    case 2: return launch_k(mlstm_state_finalize_kernel<2>, dim3(p.B * p.NH), dim3(thr), 0, s, p);
    case 3: return launch_k(mlstm_state_finalize_kernel<3>, dim3(p.B * p.NH), dim3(thr), 0, s, p);
    case 4: return launch_k(mlstm_state_finalize_kernel<4>, dim3(p.B * p.NH), dim3(thr), 0, s, p);
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

// kernel 1
cudaError_t launch_state_step(StateStepParams p, int num_sms, cudaStream_t s) {
  drop_unfusable(p, num_sms);
  resolve_tiling(p, num_sms);
  if (p.cols_per_cta % 4 || p.DH % p.cols_per_cta || slab_width(p.DH) % p.cols_per_cta ||
      kThreads % (p.cols_per_cta / 4) || p.DH > 1024 || p.NCH > kMaxNCH || p.rows_split > p.DH)
    return cudaErrorInvalidValue;
  switch (p.T) {
    case 1: return launch_T<1>(p, s);
    case 2: return launch_T<2>(p, s);
    case 3: return launch_T<3>(p, s);
    case 4: return launch_T<4>(p, s);
    default: return cudaErrorInvalidValue;
  }
}

// [M, 3, inner] (q | k | v) -> qk [M, NH, DH, 2] interleaved + v [M, inner]   (unit-test entry point only)
__global__ void repack_qkv_kernel(const float* __restrict__ qkv, float* __restrict__ qk, float* __restrict__ v,
                                  int M, int inner) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_trigger();
  if (i >= (int64_t)M * inner) return;
  const int64_t m = i / inner;
  const int c = (int)(i - m * inner);
  const float* row = qkv + m * 3 * inner;
  reinterpret_cast<float2*>(qk)[i] = make_float2(row[c], row[inner + c]);
  v[i] = row[2 * inner + c];
}
void launch_repack_qkv(const float* qkv, float* qk, float* v, int M, int inner, cudaStream_t s) {
  const int64_t n = (int64_t)M * inner;
  launch_k(repack_qkv_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, qkv, qk, v, M, inner);
}

}  // namespace xl
