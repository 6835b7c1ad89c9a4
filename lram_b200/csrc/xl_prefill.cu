// Context prefill: the encoder over S tokens per env, layer by layer, leaving exactly the recurrent state that
// S calls of xLSTMBlockStack.step would leave (the reference reaches long contexts only by stepping:
// src/algos/models/decision_xlstm.py:161-165; its `chunkwise_step` hook :158-159 calls layers.step with S > 1,
// which pip xlstm 1.0.x does not implement). SURVEY.md §8 row a11 / BASELINE.json configs[3].
//
// Because every token of the context is known up front, the stack runs LAYER-major over chunks of tokens:
//   LayerNorm rows -> proj_up as ONE tcgen05 GEMM over all rows of the chunk -> sequence conv/qkv/gates ->
//   gate scan (m, f, i per token) -> sequence cell -> sequence finalize -> proj_down GEMM (+ residual).
// The projections are real GEMMs here (M = envs x chunk tokens rows) and run on the tensor cores. The cell
// keeps the matrix memory ON CHIP for the whole chunk: a CTA owns 16 columns (dv) of one (env, head) C in
// registers, streams the chunk's (q,k) pairs / v / gates through a TMA-fed shared-memory ring, and touches HBM
// for C once per chunk instead of once per token. The arithmetic per element is the recurrent step's
// (c <- f c + k v i, num += q c), in token order, so the state it leaves is the stepping state to rounding.
// The normaliser n rides along as one more column slab whose "v" is the unit vector e0 (n = f n + i k is the
// same recurrence), which also yields q.n per token.
#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>

#include "xl_common.cuh"
#include "xl_internal.h"

namespace xl {

namespace pf {

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

// ------------------------------------------------------------------------------------------------
// Sequence pre-cell kernel: CausalConv1d over the chunk (window seeded from conv_state) + SiLU + headwise
// q/k/v + partial gate pre-activations. Same arithmetic as conv_qkv_gates_kernel (xl_elementwise.cu), token by
// token. grid = (NCH channel chunks, B envs, token runs); a thread owns one 4-channel block for a run of
// tokens and keeps the conv window in registers; gate partials are reduced 4 tokens at a time.
// ------------------------------------------------------------------------------------------------
constexpr int kConvRuns = 4;       // token runs per CTA (threadIdx.y): they share the gate weights in shared memory
template <int KS, int NH>
__global__ void __launch_bounds__(64 * kConvRuns, 2) conv_qkv_gates_seq_kernel(ConvQkvParams p, int S, int run) {
  constexpr int TG = 4;                                  // tokens per gate-reduction group
  __shared__ float red[kConvRuns][2 * NH * TG * 4];
  // gate weights of the chunk's channels, [gate][head][q|k|v][channel]: kept out of the registers (hoisted there, the 96
  // loop-invariant values per thread cut the occupancy to 8 warps per SM)
  extern __shared__ __align__(16) float s_gw[];
  const int b = blockIdx.y, chunk = blockIdx.x;
  const int sub = threadIdx.y;
  const int nruns = blockDim.y;
  const int s_begin = min(S, ((int)blockIdx.z * nruns + sub) * run);
  const int s_end = min(S, s_begin + run);
  const int s_cta_end = min(S, (int)blockIdx.z * nruns * run + run);   // longest run of the CTA (sub 0): loop bound
  const int inner = p.inner;
  const int nblk = inner >> 2;
  const int blk_per_chunk = (nblk + p.NCH - 1) / p.NCH;
  const int j = chunk * blk_per_chunk + threadIdx.x;
  const bool active = threadIdx.x < blk_per_chunk && j < nblk;
  const int c = 4 * (active ? j : 0);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nw = (blockDim.x + 31) >> 5;
  const int cw = 4 * blockDim.x;                          // channels covered by the CTA's threads
  {
    const int c_base = 4 * chunk * blk_per_chunk;
    const int flat = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
    for (int i = flat; i < 2 * NH * 3 * cw; i += nthr) {
      const int ch = i % cw, row = i / cw;                // row = (gate * NH + head) * 3 + part
      const int gate = row / (NH * 3), hp = row - gate * NH * 3;
      const int gc = c_base + ch;
      s_gw[i] = gc < inner ? (gate ? p.wf : p.wi)[(int64_t)hp * inner + gc] : 0.f;
    }
  }

  float win[KS][4];
  float cw4[4][KS];
  float cbv[4] = {0.f, 0.f, 0.f, 0.f};
  float wq[16], wk[16], wv[16];
  if (active) {
#pragma unroll
    for (int ch = 0; ch < 4; ++ch)
#pragma unroll
      for (int r = 0; r < KS; ++r) cw4[ch][r] = p.conv_w[(int64_t)(c + ch) * KS + r];
    const float4 cb = *reinterpret_cast<const float4*>(p.conv_b + c);
    cbv[0] = cb.x; cbv[1] = cb.y; cbv[2] = cb.z; cbv[3] = cb.w;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 a4 = reinterpret_cast<const float4*>(p.wq + (int64_t)j * 16)[i];
      const float4 k4 = reinterpret_cast<const float4*>(p.wk + (int64_t)j * 16)[i];
      const float4 v4 = reinterpret_cast<const float4*>(p.wv + (int64_t)j * 16)[i];
      wq[4 * i] = a4.x; wq[4 * i + 1] = a4.y; wq[4 * i + 2] = a4.z; wq[4 * i + 3] = a4.w;
      wk[4 * i] = k4.x; wk[4 * i + 1] = k4.y; wk[4 * i + 2] = k4.z; wk[4 * i + 3] = k4.w;
      wv[4 * i] = v4.x; wv[4 * i + 1] = v4.y; wv[4 * i + 2] = v4.z; wv[4 * i + 3] = v4.w;
    }
  }
  pdl_wait();
  pdl_trigger();
  __syncthreads();                                        // s_gw
  if (active && s_begin < s_end) {
    // window rows 1..KS-1 = the KS-1 inputs before token s_begin: earlier rows of this chunk, or the carried
    // conv_state (rows = last KS inputs, oldest first) for tokens before the chunk
#pragma unroll
    for (int r = 1; r < KS; ++r) {
      const int s = s_begin - (KS - r);
      float4 w4;
      if (s >= 0) w4 = *reinterpret_cast<const float4*>(p.u + ((int64_t)b * S + s) * 2 * inner + c);
      else w4 = *reinterpret_cast<const float4*>(p.conv_state + ((int64_t)b * KS + (KS + s)) * inner + c);
      win[r][0] = w4.x; win[r][1] = w4.y; win[r][2] = w4.z; win[r][3] = w4.w;
    }
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) win[0][ch] = 0.f;
  }
  const int nsteps = (s_cta_end - (int)blockIdx.z * nruns * run + TG - 1) / TG;   // same for every thread of the CTA
  for (int st = 0; st < nsteps; ++st) {
    const int s0 = s_begin + st * TG;
    float gi[NH][TG], gf[NH][TG];
#pragma unroll
    for (int h = 0; h < NH; ++h)
#pragma unroll
      for (int t = 0; t < TG; ++t) gi[h][t] = gf[h][t] = 0.f;
    if (active) {
      // the group's inputs are requested together (the stores below would otherwise order the loads token by token)
      float4 xg[TG];
#pragma unroll
      for (int t = 0; t < TG; ++t)
        xg[t] = s0 + t < s_end ? *reinterpret_cast<const float4*>(p.u + ((int64_t)b * S + s0 + t) * 2 * inner + c)
                               : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int t = 0; t < TG; ++t) {
        const int s = s0 + t;
        if (s < s_end) {
          const int64_t row = (int64_t)b * S + s;
          const float4 x4 = xg[t];
          const float xm[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
          for (int r = 0; r < KS - 1; ++r)
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) win[r][ch] = win[r + 1][ch];
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) win[KS - 1][ch] = xm[ch];
          float a[4];
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) {
            float acc = 0.f;
#pragma unroll
            for (int r = 0; r < KS; ++r) acc = fmaf(win[r][ch], cw4[ch][r], acc);
            a[ch] = silu(acc + cbv[ch]);
          }
          float q[4], k[4], v[4];
#pragma unroll
          for (int o = 0; o < 4; ++o) {
            float sq = 0.f, sk = 0.f, sv = 0.f;
#pragma unroll
            for (int dd = 0; dd < 4; ++dd) {
              sq = fmaf(a[dd], wq[4 * o + dd], sq);
              sk = fmaf(a[dd], wk[4 * o + dd], sk);
              sv = fmaf(xm[dd], wv[4 * o + dd], sv);
            }
            q[o] = sq; k[o] = sk; v[o] = sv;
          }
          // prefill layout: q plane then k plane ([M, inner] each) instead of the step path's interleaved pairs
          *reinterpret_cast<float4*>(p.qk + row * inner + c) = make_float4(q[0], q[1], q[2], q[3]);
          *reinterpret_cast<float4*>(p.qk + ((int64_t)p.B * S + row) * inner + c) = make_float4(k[0], k[1], k[2], k[3]);
          *reinterpret_cast<float4*>(p.v + row * inner + c) = make_float4(v[0], v[1], v[2], v[3]);
          *reinterpret_cast<float4*>(p.act + row * inner + c) = make_float4(a[0], a[1], a[2], a[3]);
#pragma unroll
          for (int h = 0; h < NH; ++h) {
            const float* wi = s_gw + (h * 3) * cw + 4 * threadIdx.x;
            const float* wf = s_gw + ((NH + h) * 3) * cw + 4 * threadIdx.x;
            const float4 iq = *reinterpret_cast<const float4*>(wi);
            const float4 ik = *reinterpret_cast<const float4*>(wi + cw);
            const float4 iv = *reinterpret_cast<const float4*>(wi + 2 * cw);
            const float4 fq = *reinterpret_cast<const float4*>(wf);
            const float4 fk = *reinterpret_cast<const float4*>(wf + cw);
            const float4 fv = *reinterpret_cast<const float4*>(wf + 2 * cw);
            float si = q[0] * iq.x + q[1] * iq.y + q[2] * iq.z + q[3] * iq.w;
            si += k[0] * ik.x + k[1] * ik.y + k[2] * ik.z + k[3] * ik.w;
            si += v[0] * iv.x + v[1] * iv.y + v[2] * iv.z + v[3] * iv.w;
            float sf = q[0] * fq.x + q[1] * fq.y + q[2] * fq.z + q[3] * fq.w;
            sf += k[0] * fk.x + k[1] * fk.y + k[2] * fk.z + k[3] * fk.w;
            sf += v[0] * fv.x + v[1] * fv.y + v[2] * fv.z + v[3] * fv.w;
            gi[h][t] = si;
            gf[h][t] = sf;
          }
        }
      }
    }
    // chunk-level partial sums of the 4 tokens: warp tree, then fixed-order sum over the (<= 4) warps of the run
    if constexpr (NH * 2 * TG == 32) {
      // 32 values x 32 lanes: a transposing butterfly (each xor step halves the values a lane carries) needs 31 shuffles
      // instead of 160 and forms exactly the pairwise sums of warp_sum(); lane l ends with the warp total of value l
      float vals[32];
#pragma unroll
      for (int h = 0; h < NH; ++h)
#pragma unroll
        for (int t = 0; t < TG; ++t) {
          vals[(h * 2 + 0) * TG + t] = gi[h][t];
          vals[(h * 2 + 1) * TG + t] = gf[h][t];
        }
#pragma unroll
      for (int m = 16; m > 0; m >>= 1) {
        const bool up = (lane & m) != 0;
#pragma unroll
        for (int i = 0; i < m; ++i) {
          const float keep = up ? vals[i + m] : vals[i];
          const float send = up ? vals[i] : vals[i + m];
          vals[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
        }
      }
      red[sub][lane * 4 + wid] = vals[0];
    } else {
#pragma unroll
      for (int h = 0; h < NH; ++h)
#pragma unroll
        for (int t = 0; t < TG; ++t) {
          const float si = warp_sum(gi[h][t]);
          const float sf = warp_sum(gf[h][t]);
          if (lane == 0) {
            red[sub][((h * 2 + 0) * TG + t) * 4 + wid] = si;
            red[sub][((h * 2 + 1) * TG + t) * 4 + wid] = sf;
          }
        }
    }
    __syncthreads();
    if ((int)threadIdx.x < NH * 2 * TG) {
      const int h = threadIdx.x / (2 * TG);
      const int rem = threadIdx.x - h * 2 * TG;
      const int g = rem / TG, t = rem - g * TG;
      if (s0 + t < s_end) {
        float s = 0.f;
        for (int w = 0; w < nw; ++w) s += red[sub][((h * 2 + g) * TG + t) * 4 + w];
        p.gate_part[(((int64_t)b * S + s0 + t) * p.NCH + chunk) * 2 * NH + g * NH + h] = s;
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// The same kernel on packed fp32 pairs (default; xl_set_option("prefill_conv", 0) selects the scalar one above).
// The scalar kernel is bound by instruction issue: ~550 instructions per token and 4-channel block, half of them
// FP32, behind 16 warps per SM. sm_100 has FFMA2 / FMUL2 / FADD2 (fma.rn.f32x2 ...: two IEEE fp32 results per
// instruction and lane, an operand may be one register broadcast to both halves), so
//   conv       : channel pairs (c0,c1), (c2,c3)                           8 FFMA2 per token instead of 16 FFMA
//   q / k / v  : output pairs (o0,o1), (o2,o3), a[dd] broadcast          24 instead of 48
//   gates      : the (igate, fgate) pair of a head, q/k/v[o] broadcast   14 per head instead of 28
// with every chain in the order the scalar kernel's SASS has (mul of term 1, fma of terms 0, 2, 3; q-, k-, v-sums added
// in that order), i.e. q, k, v, a and the gate partials are BIT-IDENTICAL to the scalar kernel (tested). Around that:
//   * the gate weights sit in shared memory as (i, f) pairs and are read once per TWO tokens (an LDS.128 of distinct
//     addresses costs 4 shared-memory cycles per warp; at one read per token they alone were 111 us per launch);
//   * the headwise q/k/v blocks live in shared memory as well (the 4 token runs of a CTA share them), which keeps the
//     kernel under 128 registers without spills;
//   * a token run synchronises on its own named barrier (one per 2-token group, double-buffered partial sums) instead
//     of two CTA-wide barriers, and the next group's input rows are in flight while a group computes;
//   * row pointers advance by constant strides (no 64-bit index arithmetic per store).
// ------------------------------------------------------------------------------------------------
// shared-memory read the compiler may neither hoist nor merge with an earlier one of the same address (the weights are
// loop-invariant: merged, they would occupy > 100 registers)
__device__ __forceinline__ float4 lds_v4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

template <int NH, bool FAST_SILU>
__global__ void __launch_bounds__(64 * kConvRuns, 2) conv_qkv_gates_seq2_kernel(ConvQkvParams p, int S, int run) {
  constexpr int KS = 4, TG = 2, NV = NH * 2 * TG;         // NV gate values per token group
  __shared__ float red[kConvRuns][2][NV * 4];
  // per thread (channel block) kRows float4 of weights, thread-major with a stride of kRows + 1 float4 (an odd multiple of
  // 16 B: the 8 lanes of a quarter warp hit all 32 banks, and every read below is [thread base + immediate]):
  //   rows [0, 6 NH)      : (head * 3 + q|k|v) * 2 + half -> (i, f) gate weights of channels (2*half, 2*half + 1)
  //   rows [6 NH, 6 NH+12): (q|k|v) * 4 + dd -> column dd of the 4 x 4 headwise block (outputs o = 0..3)
  constexpr int kGateRows = NH * 3 * 2, kRows = kGateRows + 12, kStride = kRows + 1;
  extern __shared__ __align__(16) float4 s_dyn[];
  const int nx = blockDim.x;
  const int chunk = blockIdx.x;
  const int sub = threadIdx.y, nruns = blockDim.y, tx = threadIdx.x;
  const int inner = p.inner;
  const int nblk = inner >> 2;
  const int blk_per_chunk = (nblk + p.NCH - 1) / p.NCH;
  const int j = chunk * blk_per_chunk + tx;
  const bool active = tx < blk_per_chunk && j < nblk;
  const int c = 4 * (active ? j : 0);
  const int lane = tx & 31, wid = tx >> 5;
  const int nw = (nx + 31) >> 5;
  {
    const int flat = sub * nx + tx, nthr = nx * nruns;
    for (int i = flat; i < kGateRows * nx; i += nthr) {
      const int t = i % nx, row = i / nx;                 // row = (head * 3 + part) * 2 + half
      const int half = row & 1, hp = row >> 1;
      const int jb = chunk * blk_per_chunk + t;
      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t < blk_per_chunk && jb < nblk) {
        const int64_t o = (int64_t)hp * inner + 4 * jb + 2 * half;
        w = make_float4(p.wi[o], p.wf[o], p.wi[o + 1], p.wf[o + 1]);
      }
      s_dyn[t * kStride + row] = w;
    }
    for (int i = flat; i < 3 * 4 * nx; i += nthr) {
      const int t = i % nx, row = i / nx;                 // row = part * 4 + dd
      const int dd = row & 3, part = row >> 2;
      const int jb = chunk * blk_per_chunk + t;
      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t < blk_per_chunk && jb < nblk) {
        const float* hw = (part == 0 ? p.wq : part == 1 ? p.wk : p.wv) + (int64_t)jb * 16 + dd;
        w = make_float4(hw[0], hw[4], hw[8], hw[12]);
      }
      s_dyn[t * kStride + kGateRows + row] = w;
    }
  }
  f32x2 cwp[KS][2];                                        // conv taps of channel pairs
  f32x2 cbp[2];
  {
    float4 w4[4];
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) w4[ch] = *reinterpret_cast<const float4*>(p.conv_w + (int64_t)(c + ch) * KS);
    cwp[0][0] = pk2(w4[0].x, w4[1].x); cwp[0][1] = pk2(w4[2].x, w4[3].x);
    cwp[1][0] = pk2(w4[0].y, w4[1].y); cwp[1][1] = pk2(w4[2].y, w4[3].y);
    cwp[2][0] = pk2(w4[0].z, w4[1].z); cwp[2][1] = pk2(w4[2].z, w4[3].z);
    cwp[3][0] = pk2(w4[0].w, w4[1].w); cwp[3][1] = pk2(w4[2].w, w4[3].w);
    const float4 cb = *reinterpret_cast<const float4*>(p.conv_b + c);
    cbp[0] = pk2(cb.x, cb.y);
    cbp[1] = pk2(cb.z, cb.w);
  }
  pdl_wait();
  pdl_trigger();
  __syncthreads();                                        // s_gw, s_hw
  const uint32_t bar_id = 1 + sub, bar_threads = nw * 32;
  const uint32_t gw = smem_u32(s_dyn + tx * kStride), hw = gw + 16u * kGateRows;
  const int u_step = 2 * inner, g_step = p.NCH * 2 * NH;
  uint32_t group = 0;                                     // groups this run has reduced so far: parity of its buffer
  // PERSISTENT over the (env, run block) items of its channel chunk: the weights above are staged once per CTA (at 16
  // tokens per run the staging was a quarter of a CTA's life). gridDim.y == 1: CTA z walks the flattened item list
  // z, z + gridDim.z, ...; gridDim.y == B: one env per CTA row, items = its run blocks.
  const int nzb = (S + run * nruns - 1) / (run * nruns);
  const int nitems = gridDim.y == 1 ? p.B * nzb : nzb;
#pragma unroll 1
  for (int item = blockIdx.z; item < nitems; item += gridDim.z) {
    const int b = gridDim.y == 1 ? item / nzb : (int)blockIdx.y;
    const int zb = gridDim.y == 1 ? item - b * nzb : item;
    const int s_begin = min(S, (zb * nruns + sub) * run);
    const int s_end = min(S, s_begin + run);
    if (s_begin >= s_end) continue;                         // (a run past the end of this env's tokens)

    // the KS-1 inputs before token s_begin: earlier rows of this chunk, or the carried conv_state (rows = last KS
    // inputs, oldest first) for tokens before the chunk
    f32x2 win[KS - 1][2];
#pragma unroll
    for (int r = 0; r < KS - 1; ++r) {
      const int s = s_begin - (KS - 1 - r);
      float4 w4;
      if (s >= 0) w4 = *reinterpret_cast<const float4*>(p.u + ((int64_t)b * S + s) * 2 * inner + c);
      else w4 = *reinterpret_cast<const float4*>(p.conv_state + ((int64_t)b * KS + (KS + s)) * inner + c);
      win[r][0] = pk2(w4.x, w4.y);
      win[r][1] = pk2(w4.z, w4.w);
    }
    const int64_t row_begin = (int64_t)b * S + s_begin;
    const float* up = p.u + row_begin * 2 * inner + c;
    float* qp = p.qk + row_begin * inner + c;
    float* kp = qp + (int64_t)p.B * S * inner;
    float* vp = p.v + row_begin * inner + c;
    float* ap = p.act + row_begin * inner + c;
    float* gp = p.gate_part + (row_begin * p.NCH + chunk) * 2 * NH;

    const int ntok = s_end - s_begin;
    const int nsteps = (ntok + TG - 1) / TG;
    float4 xc[TG];
#pragma unroll
    for (int t = 0; t < TG; ++t)
      xc[t] = (active && t < ntok) ? *reinterpret_cast<const float4*>(up + t * u_step) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int st = 0; st < nsteps; ++st) {
      const int nleft = ntok - st * TG;                     // tokens of this group that exist (>= 1)
      float4 xn[TG];                                        // next group's inputs: in flight while this group computes
#pragma unroll
      for (int t = 0; t < TG; ++t)
        xn[t] = (active && TG + t < nleft) ? *reinterpret_cast<const float4*>(up + (TG + t) * u_step)
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
      float a[TG][4];
#pragma unroll
      for (int t = 0; t < TG; ++t) {
        const f32x2 x01 = pk2(xc[t].x, xc[t].y), x23 = pk2(xc[t].z, xc[t].w);
        // conv over (win[0], win[1], win[2], x), oldest first; fma(w, c, 0) == w * c
        f32x2 a01 = fma2(win[0][0], cwp[0][0], 0ull), a23 = fma2(win[0][1], cwp[0][1], 0ull);
        a01 = fma2(win[1][0], cwp[1][0], a01); a23 = fma2(win[1][1], cwp[1][1], a23);
        a01 = fma2(win[2][0], cwp[2][0], a01); a23 = fma2(win[2][1], cwp[2][1], a23);
        a01 = fma2(x01, cwp[3][0], a01);       a23 = fma2(x23, cwp[3][1], a23);
        a01 = add2(a01, cbp[0]);               a23 = add2(a23, cbp[1]);
        win[0][0] = win[1][0]; win[0][1] = win[1][1];
        win[1][0] = win[2][0]; win[1][1] = win[2][1];
        win[2][0] = x01;       win[2][1] = x23;
        unpk2(a01, a[t][0], a[t][1]);
        unpk2(a23, a[t][2], a[t][3]);
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) a[t][ch] = FAST_SILU ? silu_fast(a[t][ch]) : silu(a[t][ch]);
      }
      // headwise 4 x 4 blocks: out[o] = sum_dd in[dd] * W[o][dd], dd ascending from 0; one read of a column per group
      f32x2 qq[TG][2], kk[TG][2], vv[TG][2];
#pragma unroll
      for (int t = 0; t < TG; ++t) qq[t][0] = qq[t][1] = kk[t][0] = kk[t][1] = vv[t][0] = vv[t][1] = 0ull;
#pragma unroll
      for (int dd = 0; dd < 4; ++dd) {
        const float4 wq = lds_v4(hw + 16 * (0 * 4 + dd)), wk = lds_v4(hw + 16 * (1 * 4 + dd)), wv = lds_v4(hw + 16 * (2 * 4 + dd));
#pragma unroll
        for (int t = 0; t < TG; ++t) {
          const float xm = dd == 0 ? xc[t].x : dd == 1 ? xc[t].y : dd == 2 ? xc[t].z : xc[t].w;
          qq[t][0] = fma2(bc2(a[t][dd]), pk2(wq.x, wq.y), qq[t][0]);
          qq[t][1] = fma2(bc2(a[t][dd]), pk2(wq.z, wq.w), qq[t][1]);
          kk[t][0] = fma2(bc2(a[t][dd]), pk2(wk.x, wk.y), kk[t][0]);
          kk[t][1] = fma2(bc2(a[t][dd]), pk2(wk.z, wk.w), kk[t][1]);
          vv[t][0] = fma2(bc2(xm), pk2(wv.x, wv.y), vv[t][0]);
          vv[t][1] = fma2(bc2(xm), pk2(wv.z, wv.w), vv[t][1]);
        }
      }
      float q[TG][4], k[TG][4], v[TG][4];
#pragma unroll
      for (int t = 0; t < TG; ++t) {
        unpk2(qq[t][0], q[t][0], q[t][1]); unpk2(qq[t][1], q[t][2], q[t][3]);
        unpk2(kk[t][0], k[t][0], k[t][1]); unpk2(kk[t][1], k[t][2], k[t][3]);
        unpk2(vv[t][0], v[t][0], v[t][1]); unpk2(vv[t][1], v[t][2], v[t][3]);
        if (active && t < nleft) {
          // prefill layout: q plane then k plane ([M, inner] each) instead of the step path's interleaved pairs
          *reinterpret_cast<float4*>(qp + t * inner) = make_float4(q[t][0], q[t][1], q[t][2], q[t][3]);
          *reinterpret_cast<float4*>(kp + t * inner) = make_float4(k[t][0], k[t][1], k[t][2], k[t][3]);
          *reinterpret_cast<float4*>(vp + t * inner) = make_float4(v[t][0], v[t][1], v[t][2], v[t][3]);
          *reinterpret_cast<float4*>(ap + t * inner) = make_float4(a[t][0], a[t][1], a[t][2], a[t][3]);
        }
      }
      // gate partials: (igate, fgate) of head h for the group's tokens against one read of the head's weights
      f32x2 G[NH][TG];
#pragma unroll
      for (int h = 0; h < NH; ++h) {
        const uint32_t g = gw + 16 * (h * 3) * 2;
        {
          const float4 w0 = lds_v4(g), w1 = lds_v4(g + 16);
#pragma unroll
          for (int t = 0; t < TG; ++t) G[h][t] = dot4_bc(q[t], w0, w1);
        }
        {
          const float4 w0 = lds_v4(g + 32), w1 = lds_v4(g + 48);
#pragma unroll
          for (int t = 0; t < TG; ++t) G[h][t] = add2(G[h][t], dot4_bc(k[t], w0, w1));
        }
        {
          const float4 w0 = lds_v4(g + 64), w1 = lds_v4(g + 80);
#pragma unroll
          for (int t = 0; t < TG; ++t) G[h][t] = add2(G[h][t], dot4_bc(v[t], w0, w1));
        }
        if (!active) {
#pragma unroll
          for (int t = 0; t < TG; ++t) G[h][t] = 0ull;
        }
      }
      // sums of the group's NV values over the run's channels: warp tree (xor 16, 8, 4, 2, 1: the pairwise sums of
      // warp_sum()), then a fixed-order sum over the run's (<= 4) warps
      float* rbuf = red[sub][group & 1];
      ++group;
      float vals[NV];
#pragma unroll
      for (int h = 0; h < NH; ++h)
#pragma unroll
        for (int t = 0; t < TG; ++t) unpk2(G[h][t], vals[(h * 2 + 0) * TG + t], vals[(h * 2 + 1) * TG + t]);
      if constexpr (NV == 32 || NV == 16) {
        // transposing butterfly: every xor step halves the values a lane carries, NV - 1 (+ 1) shuffles instead of 5 * NV
        constexpr int M0 = NV == 32 ? 16 : 8;               // values kept after the first (xor 16) step
#pragma unroll
        for (int m = 16, nv = M0; m > 0; m >>= 1, nv >>= 1) {
          const bool upper = (lane & m) != 0;
          if (nv >= 1) {
#pragma unroll
            for (int i = 0; i < nv; ++i) {
              const float keep = upper ? vals[i + nv] : vals[i];
              const float send = upper ? vals[i] : vals[i + nv];
              vals[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
            }
          } else {
            vals[0] += __shfl_xor_sync(0xffffffffu, vals[0], m);   // NV == 16: one value left, lanes l and l^1 share it
          }
        }
        // lane l holds the warp total of value l (NV == 32) or l >> 1 (NV == 16)
        if (NV == 32 || (lane & 1) == 0) rbuf[(NV == 32 ? lane : lane >> 1) * 4 + wid] = vals[0];
      } else {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const float sum = warp_sum(vals[i]);
          if (lane == 0) rbuf[i * 4 + wid] = sum;
        }
      }
      asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(bar_threads) : "memory");
      if (tx < NV) {
        const int h = tx / (2 * TG);
        const int rem = tx - h * 2 * TG;
        const int g = rem / TG, t = rem - g * TG;
        if (t < nleft) {
          float s = 0.f;
          for (int w = 0; w < nw; ++w) s += rbuf[tx * 4 + w];
          gp[t * g_step + g * NH + h] = s;
        }
      }
#pragma unroll
      for (int t = 0; t < TG; ++t) xc[t] = xn[t];
      up += TG * u_step;
      qp += TG * inner; kp += TG * inner; vp += TG * inner; ap += TG * inner;
      gp += TG * g_step;
    }
  }
}

// new conv_state = the last KS x_m rows of the chunk (S >= KS): separate kernel, because the first token run of
// the conv kernel still reads the old window while its last run would overwrite it.
// Ragged (len != nullptr): one thread per (env, 4-channel group) takes the last KS rows of (old window ++ the env's n_b
// valid rows) -- old rows still count when n_b < KS -- and reads all of them before it writes.
__global__ void __launch_bounds__(256) conv_state_seq_kernel(const float* __restrict__ u, float* __restrict__ conv_state,
                                                             int B, int S, int KS, int inner,
                                                             const int32_t* __restrict__ len, int pos) {
  pdl_wait();
  pdl_trigger();
  if (len) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)B * (inner >> 2)) return;
    const int c4 = (int)(i % (inner >> 2));
    const int b = (int)(i / (inner >> 2));
    const int nb = min(max(len[b] - pos, 0), S);
    float4 w[4];                                           // KS <= 4
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      if (r >= KS) break;
      const int idx = nb - KS + r;                         // chunk row, or (< 0) row KS + idx of the old window
      w[r] = idx >= 0 ? reinterpret_cast<const float4*>(u + ((int64_t)b * S + idx) * 2 * inner)[c4]
                      : reinterpret_cast<const float4*>(conv_state + ((int64_t)b * KS + KS + idx) * inner)[c4];
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      if (r >= KS) break;
      reinterpret_cast<float4*>(conv_state + ((int64_t)b * KS + r) * inner)[c4] = w[r];
    }
    return;
  }
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n4 = (int64_t)B * KS * (inner >> 2);
  if (i >= n4) return;
  const int c4 = (int)(i % (inner >> 2));
  const int r = (int)((i / (inner >> 2)) % KS);
  const int b = (int)(i / ((int64_t)KS * (inner >> 2)));
  const float4 v = reinterpret_cast<const float4*>(u + ((int64_t)b * S + (S - KS + r)) * 2 * inner)[c4];
  reinterpret_cast<float4*>(conv_state + ((int64_t)b * KS + r) * inner)[c4] = v;
}

// ------------------------------------------------------------------------------------------------
// Gate scan: per (env, head) the stabiliser recurrence over the chunk's tokens,
//   lf = logsigmoid(f~);  m' = max(lf + m, i~);  f = exp(lf + m - m');  i = exp(i~ - m')
// A token is the map m -> max(m + lf, i~); maps compose as (A1, B1) then (A2, B2) = (A1 + A2, max(B1 + A2, B2)), so the
// chain is a scan. Two kernels over a grid of (env*head, super-chunks of 2048 tokens), 1024 threads:
//   gate_pre_seq_kernel : pre-activations of the super-chunk's tokens summed (fixed order, as compute_gates() of
//                         xl_state_step.cu) and log-sigmoided in parallel -> lf, i~ (parked in fseq / iseq) and the
//                         composed map of the whole super-chunk;
//   gate_scan_seq_kernel: m at the start of the super-chunk from the carried m and the maps of the super-chunks before it,
//                         then warp 0 scans the 32 segment maps of its super-chunk with shuffles and every lane replays
//                         its segment from its true start value; f, i, m of all tokens again in parallel.
// m differs from token-by-token stepping only by the association of the lf sums between resets (~1 ulp of m; the
// stabiliser cancels in h). Outputs are [B*NH][S]: a head's tokens are contiguous. scratch: [B*NH] carried m, then
// [B*NH][nsuper][2] maps.
// ------------------------------------------------------------------------------------------------
constexpr int kScanThreads = 1024;
constexpr int kSuper = 2048;                     // tokens per super-chunk (2 per thread)

// fold of this lane's segment [lo, hi) and the inclusive scan of the 32 segment maps (full warp)
__device__ __forceinline__ void segment_scan(const float* s_lf, const float* s_ig, int lo, int hi, int lane, float& Ai,
                                             float& Bi) {
  float A = 0.f, Bv = -INFINITY;
  for (int u = lo; u < hi; ++u) {
    A += s_lf[u];
    Bv = fmaxf(Bv + s_lf[u], s_ig[u]);
  }
  Ai = A;
  Bi = Bv;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float Ap = __shfl_up_sync(0xffffffffu, Ai, o);
    const float Bp = __shfl_up_sync(0xffffffffu, Bi, o);
    if (lane >= o) {
      Bi = fmaxf(Bp + Ai, Bi);
      Ai = Ap + Ai;
    }
  }
}

__global__ void __launch_bounds__(kScanThreads) gate_pre_seq_kernel(const float* __restrict__ gate_part,
                                                                    const float* __restrict__ igate_b,
                                                                    const float* __restrict__ fgate_b,
                                                                    const float* __restrict__ m_state,
                                                                    float* __restrict__ fseq, float* __restrict__ iseq,
                                                                    float* __restrict__ scratch, int B, int S, int NH,
                                                                    int NCH, const int32_t* __restrict__ len, int pos) {
  __shared__ float s_ig[kSuper + 32], s_lf[kSuper + 32];
  pdl_wait();
  pdl_trigger();
  const int bh = blockIdx.x, sp = blockIdx.y, nsuper = gridDim.y;
  const int b = bh / NH, hd = bh - b * NH;
  const int tid = threadIdx.x, lane = tid & 31;
  const float bi = igate_b ? igate_b[hd] : 0.f, bf = fgate_b ? fgate_b[hd] : 0.f;
  const int s0 = sp * kSuper;
  const int cnt = min(kSuper, S - s0);
  const int nreal = len ? len[b] - pos - s0 : cnt;   // tokens u >= nreal of the super-chunk are identity pads
  for (int u = tid; u < cnt; u += kScanThreads) {
    const float* gp = gate_part + ((int64_t)b * S + s0 + u) * NCH * 2 * NH + hd;
    float si = 0.f, sf = 0.f;
    for (int c = 0; c < NCH; ++c) {            // fixed order, as compute_gates()
      si += gp[c * 2 * NH];
      sf += gp[c * 2 * NH + NH];
    }
    float ig = si + bi, lf = log_sigmoid(sf + bf);
    if (u >= nreal) {                           // m' = max(m, -inf) = m, f = exp(0) = 1, i = exp(-inf) = 0 exactly
      ig = -INFINITY;
      lf = 0.f;
    }
    s_ig[u] = ig;
    s_lf[u] = lf;
    const int64_t o = (int64_t)bh * S + s0 + u;
    iseq[o] = ig;
    fseq[o] = lf;
  }
  __syncthreads();
  if (tid < 32) {
    const int seg = ((cnt + 31) / 32) | 1;               // odd stride: conflict-free shared-memory walks
    const int lo = min(cnt, lane * seg), hi = min(cnt, lo + seg);
    float Ai, Bi;
    segment_scan(s_lf, s_ig, lo, hi, lane, Ai, Bi);
    if (lane == 31) {
      float* comp = scratch + (int64_t)B * NH + ((int64_t)bh * nsuper + sp) * 2;
      comp[0] = Ai;
      comp[1] = Bi;
    }
    if (sp == 0 && lane == 0) scratch[bh] = m_state[bh];
  }
}

__global__ void __launch_bounds__(kScanThreads) gate_scan_seq_kernel(float* __restrict__ m_state, float* __restrict__ fseq,
                                                                     float* __restrict__ iseq, float* __restrict__ mseq,
                                                                     const float* __restrict__ scratch, int B, int S,
                                                                     int NH) {
  __shared__ float s_ig[kSuper + 32], s_lf[kSuper + 32], s_mp[kSuper], s_mn[kSuper];
  pdl_wait();
  pdl_trigger();
  const int bh = blockIdx.x, sp = blockIdx.y, nsuper = gridDim.y;
  const int tid = threadIdx.x, lane = tid & 31;
  const int s0 = sp * kSuper;
  const int cnt = min(kSuper, S - s0);
  for (int u = tid; u < cnt; u += kScanThreads) {
    const int64_t o = (int64_t)bh * S + s0 + u;
    s_ig[u] = iseq[o];
    s_lf[u] = fseq[o];
  }
  __syncthreads();
  if (tid < 32) {
    // m at the start of this super-chunk: the carried m through the maps of the super-chunks before it
    float m = scratch[bh];
    const float* comp = scratch + (int64_t)B * NH + (int64_t)bh * nsuper * 2;
    for (int k = 0; k < sp; ++k) m = fmaxf(m + comp[2 * k], comp[2 * k + 1]);
    const int seg = ((cnt + 31) / 32) | 1;
    const int lo = min(cnt, lane * seg), hi = min(cnt, lo + seg);
    float Ai, Bi;
    segment_scan(s_lf, s_ig, lo, hi, lane, Ai, Bi);
    const float Aex = __shfl_up_sync(0xffffffffu, Ai, 1), Bex = __shfl_up_sync(0xffffffffu, Bi, 1);
    float mm = lane == 0 ? m : fmaxf(m + Aex, Bex);      // m at the start of this lane's segment
    for (int u = lo; u < hi; ++u) {
      const float mn = fmaxf(s_lf[u] + mm, s_ig[u]);
      s_mp[u] = mm;
      s_mn[u] = mn;
      mm = mn;
    }
    // NOTE the maps of the super-chunks (pre kernel) and this replay agree to rounding; the carried m is the replay's
    if (sp == nsuper - 1) {
      const float mlast = __shfl_sync(0xffffffffu, mm, (cnt - 1) / seg);
      if (lane == 0) m_state[bh] = mlast;
    }
  }
  __syncthreads();
  for (int u = tid; u < cnt; u += kScanThreads) {
    const float mp = s_mp[u], mn = s_mn[u];
    const int64_t o = (int64_t)bh * S + s0 + u;
    fseq[o] = expf(s_lf[u] + mp - mn);
    iseq[o] = expf(s_ig[u] - mn);
    mseq[o] = mn;
  }
}

// ------------------------------------------------------------------------------------------------
// Sequence cell: CTA = (env*head, w-column slab of C, or the extra "n slab"); the C slab [DH x w] lives in
// registers for the whole chunk. w = DH/32 for the shipped presets, so that one env is 4 heads x 32 slabs + 4
// n slabs = 132 CTAs: one CTA per SM, one wave, and 16 consumer warps keep the fp32 pipe busy on their own.
// Thread = (row lane rl, column group cg in 0..3): rows rl + RL r (r < R), columns CPT cg .. CPT cg + CPT - 1
// (CPT = w / 4). A warp holds 8 row lanes x 4 column groups, so q/k shared loads are 8-address broadcasts and the
// row reduction needs 3 shuffle steps. A producer warp streams the chunk's tokens through a 3-deep ring of
// 8-token stages (q and k of the whole head, the slab's v, f and i) with bulk copies + mbarriers.
// The fp32 pipe is the bound (3-register FFMA issues every 2nd cycle per SM sub-partition), so the per-element
// work per token is cut from 3 to 2 operations by deferring the forget gate inside a stage:
//   with F_t = f_1 ... f_t (stage-local), c^ = c / F_t obeys  c^ <- c^ + k (v i / F_t),  num_t = F_t (q . c^),
//   and c = F_8 c^ once per stage. When F_8 is too small for that to be safe (a forget gate near 0, i.e. an
//   input-gate spike) the stage runs the plain recurrence  c <- f c + k v i  instead (CTA-uniform branch).
// ------------------------------------------------------------------------------------------------
constexpr int kTB = 8;          // tokens per stage
constexpr int kStages = 3;
constexpr float kMinDecay = 1e-12f;

struct CellSeqParams {
  float* C;               // [B, NH, DH/Wc, DH, Wc] slab-major state
  float* n;               // [B, NH, DH]
  const float* q;         // [B*S, inner]   (prefill layout: separate q / k planes)
  const float* k;         // [B*S, inner]
  const float* v;         // [B*S, inner]
  const float* fseq;      // [B*NH, S]
  const float* iseq;      // [B*NH, S]
  float* num;             // [B*S, inner]   q^T C per token (un-normalised)
  float* qn;              // [B*S, NH]      q . n per token
  int B, S, NH, DH, inner;
  int nw;                 // consumer warps (row lanes RL = 8 * nw, R = DH / RL)
};

__host__ __device__ inline int cell_stage_floats(int DH, int w) { return kTB * (2 * DH + w + 2); }

template <int R, int CPT, int NW>
__global__ void __launch_bounds__((NW + 1) * 32, 1) mlstm_cell_seq_kernel(CellSeqParams p) {
  constexpr int W = 4 * CPT;
  constexpr int RL = 8 * NW;                                    // row lanes
  constexpr int DH = RL * R;                                    // compile-time: shared-memory offsets are immediates
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t s_bar[2 * kStages];
  const int NH = p.NH, S = p.S;
  constexpr int nsl = DH / W;
  const int bh = blockIdx.x / (nsl + 1);
  const int slab = blockIdx.x - bh * (nsl + 1);
  const bool n_slab = slab == nsl;
  const int b = bh / NH, hd = bh - b * NH;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int sfl = kTB * (2 * DH + W + 2);
  const uint32_t sbase = (smem_u32(smem_raw) + 127u) & ~127u;
  float* stage0 = reinterpret_cast<float*>(smem_raw + (sbase - smem_u32(smem_raw)));
  float* red = stage0 + (size_t)kStages * sfl;                  // 2 x [NW][kTB][W]
  const uint32_t bar0 = smem_u32(s_bar);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kStages + s); };
  const int nbatch = S / kTB;                                   // S % kTB == 0 (host-checked)

  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), NW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_wait();
  pdl_trigger();

  if (warp == NW) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int bt = 0; bt < nbatch; ++bt) {
        mbar_wait(empty_bar(s), ph ^ 1);
        float* st = stage0 + (size_t)s * sfl;
        const uint32_t bytes = (uint32_t)(kTB * DH * 8 + (n_slab ? 0 : kTB * W * 4) + 2 * kTB * 4);
        mbar_expect_tx(full_bar(s), bytes);
        const int64_t row0 = (int64_t)b * S + (int64_t)bt * kTB;
#pragma unroll
        for (int t = 0; t < kTB; ++t) {
          bulk_copy_g2s(smem_u32(st + t * DH), p.q + (row0 + t) * p.inner + hd * DH, (uint32_t)(DH * 4), full_bar(s));
          bulk_copy_g2s(smem_u32(st + (kTB + t) * DH), p.k + (row0 + t) * p.inner + hd * DH, (uint32_t)(DH * 4),
                        full_bar(s));
          if (!n_slab)
            bulk_copy_g2s(smem_u32(st + kTB * DH * 2 + t * W), p.v + (row0 + t) * p.inner + hd * DH + slab * W,
                          (uint32_t)(W * 4), full_bar(s));
        }
        bulk_copy_g2s(smem_u32(st + kTB * (2 * DH + W)), p.fseq + (int64_t)bh * S + (int64_t)bt * kTB,
                      (uint32_t)(kTB * 4), full_bar(s));
        bulk_copy_g2s(smem_u32(st + kTB * (2 * DH + W) + kTB), p.iseq + (int64_t)bh * S + (int64_t)bt * kTB,
                      (uint32_t)(kTB * 4), full_bar(s));
        if (++s == kStages) { s = 0; ph ^= 1; }
      }
    }
    return;
  }

  // ===== consumers =====
  const int cg = lane & 3;                      // columns CPT cg .. CPT cg + CPT - 1 of the slab
  const int rl = (warp << 3) + (lane >> 2);     // row lane 0 .. RL - 1
  constexpr int wc = (DH % 128 == 0) ? 128 : DH;    // slab width of the state layout in HBM
  constexpr int CSl = DH / wc;
  const float kscale = rsqrtf((float)DH);
  // C[bh][row][col] of the slab-major layout
  auto c_ptr = [&](int row, int col) {
    const int hs = col / wc;
    return p.C + ((int64_t)(bh * CSl + hs) * DH + row) * wc + (col - hs * wc);
  };
  float c[R][CPT];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int row = rl + RL * r;
#pragma unroll
    for (int j = 0; j < CPT; ++j) {
      if (!n_slab) c[r][j] = *c_ptr(row, slab * W + CPT * cg + j);
      else c[r][j] = (cg == 0 && j == 0) ? p.n[(int64_t)bh * DH + row] : 0.f;   // the n slab: n in column 0
    }
  }
  int s = 0;
  uint32_t ph = 0;
  for (int bt = 0; bt < nbatch; ++bt) {
    const float* st = stage0 + (size_t)s * sfl;
    const float* sq = st + rl;
    const float* sk = st + kTB * DH + rl;
    const float* sv = st + kTB * DH * 2 + CPT * cg;
    const float* sf = st + kTB * (2 * DH + W);
    const float* si = sf + kTB;
    mbar_wait(full_bar(s), ph);
    float F[kTB];                               // stage-local cumulative decay
    {
      float a = 1.f;
#pragma unroll
      for (int t = 0; t < kTB; ++t) {
        a *= sf[t];
        F[t] = a;
      }
    }
    const bool deferred = F[kTB - 1] >= kMinDecay;              // CTA-uniform
    float* rb = red + (bt & 1) * (NW * kTB * W);
    // two half-stages of 4 tokens: 4 x CPT accumulators live at a time
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      float acc[4][CPT];
#pragma unroll
      for (int tt = 0; tt < 4; ++tt) {
        const int t = half * 4 + tt;
        const float it = si[t] * kscale;
        float vi[CPT];
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
          if (!n_slab) vi[j] = sv[t * W + j] * it;
          else vi[j] = (cg == 0 && j == 0) ? it : 0.f;
          acc[tt][j] = 0.f;
        }
        if (deferred) {
          const float inv = __frcp_rn(F[t]);
#pragma unroll
          for (int j = 0; j < CPT; ++j) vi[j] *= inv;
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const float qv = sq[t * DH + RL * r], kv = sk[t * DH + RL * r];
#pragma unroll
            for (int j = 0; j < CPT; ++j) {
              c[r][j] = fmaf(kv, vi[j], c[r][j]);
              acc[tt][j] = fmaf(qv, c[r][j], acc[tt][j]);
            }
          }
#pragma unroll
          for (int j = 0; j < CPT; ++j) acc[tt][j] *= F[t];
        } else {
          const float f = sf[t];
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const float qv = sq[t * DH + RL * r], kv = sk[t * DH + RL * r];
#pragma unroll
            for (int j = 0; j < CPT; ++j) {
              c[r][j] = fmaf(f, c[r][j], kv * vi[j]);
              acc[tt][j] = fmaf(qv, c[r][j], acc[tt][j]);
            }
          }
        }
      }
      // reduce over the 8 row lanes of the warp (lane bits 2..4); the warps meet in shared memory
#pragma unroll
      for (int tt = 0; tt < 4; ++tt)
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
          float v = acc[tt][j];
          v += __shfl_xor_sync(0xffffffffu, v, 4);
          v += __shfl_xor_sync(0xffffffffu, v, 8);
          v += __shfl_xor_sync(0xffffffffu, v, 16);
          acc[tt][j] = v;
        }
      if (lane < 4) {
#pragma unroll
        for (int tt = 0; tt < 4; ++tt)
#pragma unroll
          for (int j = 0; j < CPT; ++j) rb[(warp * kTB + half * 4 + tt) * W + CPT * cg + j] = acc[tt][j];
      }
    }
    if (deferred) {
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int j = 0; j < CPT; ++j) c[r][j] *= F[kTB - 1];
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty_bar(s));
    if (++s == kStages) { s = 0; ph ^= 1; }
    asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");
    if (tid < kTB * W) {
      const int t = tid / W, col = tid - t * W;
      float sum = 0.f;
#pragma unroll
      for (int y = 0; y < NW; ++y) sum += rb[(y * kTB + t) * W + col];      // fixed order
      const int64_t row = (int64_t)b * S + (int64_t)bt * kTB + t;
      if (!n_slab) p.num[row * p.inner + hd * DH + slab * W + col] = sum;
      else if (col == 0) p.qn[row * NH + hd] = sum;
    }
  }
  // write the slab back
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int row = rl + RL * r;
#pragma unroll
    for (int j = 0; j < CPT; ++j) {
      if (!n_slab) *c_ptr(row, slab * W + CPT * cg + j) = c[r][j];
      else if (cg == 0 && j == 0) p.n[(int64_t)bh * DH + row] = c[r][0];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Sequence finalize (token-parallel): h = num / (max(|q.n|, exp(-m)) + eps), MultiHeadLayerNorm over the head,
// learnable skip and output gate; emits the bf16 hi/lo planes of proj_down's A operand (or fp32).
// One warp per (row, head).
// ------------------------------------------------------------------------------------------------
struct FinalizeSeqParams {
  const float* num;       // [M, inner]
  const float* qn;        // [M, NH]
  const float* mseq;      // [B*NH, S]
  const float* outnorm_w; // [inner]
  const float* skip;      // [inner]
  const float* act;       // [M, inner]
  const float* u;         // [M, 2*inner]
  float* out;             // [M, inner] or nullptr
  __nv_bfloat16 *out_hi, *out_lo;
  int B, S, NH, DH, inner;
  float ln_eps, cell_eps;
};

// one warp per (row, head): shuffle reductions only, no block barriers. A lane owns groups of 4 consecutive channels
// (128-bit loads of num / a / z, 64-bit stores of the bf16 planes); DH % 4 == 0, DH <= 1024.
// E = float4 groups per lane (DH <= 128 E): sized to the head so that the three operand rows fit in fewer registers
// (E = 5 at DH = 640: 3 CTAs per SM instead of 2 -- the kernel is a pure HBM stream).
template <int E>
__global__ void __launch_bounds__(256, E <= 5 ? 3 : 2) mlstm_finalize_seq_kernel(FinalizeSeqParams p) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  if (w >= (int64_t)p.B * p.S * p.NH) return;
  const int64_t row = w / p.NH;
  const int hd = (int)(w - row * p.NH);
  const int DH = p.DH, inner = p.inner;
  const int b = (int)(row / p.S), s = (int)(row - (int64_t)b * p.S);
  const float qn = p.qn[row * p.NH + hd];
  const float m = p.mseq[((int64_t)b * p.NH + hd) * p.S + s];
  const float den = fmaxf(fabsf(qn), expf(-m)) + p.cell_eps;
  const float4* num = reinterpret_cast<const float4*>(p.num + row * inner + hd * DH);
  const float4* act = reinterpret_cast<const float4*>(p.act + row * inner + hd * DH);
  const float4* zz = reinterpret_cast<const float4*>(p.u + row * 2 * inner + inner + hd * DH);
  const int ng = DH >> 2;
  float4 hv[E], av[E], zv[E];
  // every global load is issued up front
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int g = lane + 32 * e;
    hv[e] = av[e] = zv[e] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (g < ng) {
      hv[e] = num[g];
      av[e] = act[g];
      zv[e] = zz[g];
    }
  }
  float sum = 0.f;
#pragma unroll
  for (int e = 0; e < E; ++e) {
    if (lane + 32 * e < ng) {
      hv[e].x /= den; hv[e].y /= den; hv[e].z /= den; hv[e].w /= den;
      sum += (hv[e].x + hv[e].y) + (hv[e].z + hv[e].w);
    }
  }
  const float mean = warp_sum(sum) / (float)DH;
  float sq = 0.f;
#pragma unroll
  for (int e = 0; e < E; ++e) {
    if (lane + 32 * e < ng) {
      const float d0 = hv[e].x - mean, d1 = hv[e].y - mean, d2 = hv[e].z - mean, d3 = hv[e].w - mean;
      sq += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)DH + p.ln_eps);
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int g = lane + 32 * e;
    if (g < ng) {
      const int ch = hd * DH + 4 * g;
      const float4 wn = *reinterpret_cast<const float4*>(p.outnorm_w + ch);
      const float4 sk = *reinterpret_cast<const float4*>(p.skip + ch);
      float o[4];
      o[0] = ((hv[e].x - mean) * rstd * (1.f + wn.x) + sk.x * av[e].x) * silu_fast(zv[e].x);
      o[1] = ((hv[e].y - mean) * rstd * (1.f + wn.y) + sk.y * av[e].y) * silu_fast(zv[e].y);
      o[2] = ((hv[e].z - mean) * rstd * (1.f + wn.z) + sk.z * av[e].z) * silu_fast(zv[e].z);
      o[3] = ((hv[e].w - mean) * rstd * (1.f + wn.w) + sk.w * av[e].w) * silu_fast(zv[e].w);
      if (p.out) *reinterpret_cast<float4*>(p.out + row * inner + ch) = make_float4(o[0], o[1], o[2], o[3]);
      if (p.out_hi) {
        __nv_bfloat16 h4[4], l4[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          h4[j] = __float2bfloat16_rn(o[j]);
          l4[j] = __float2bfloat16_rn(o[j] - __bfloat162float(h4[j]));
        }
        *reinterpret_cast<uint2*>(p.out_hi + row * inner + ch) = *reinterpret_cast<uint2*>(h4);
        *reinterpret_cast<uint2*>(p.out_lo + row * inner + ch) = *reinterpret_cast<uint2*>(l4);
      }
    }
  }
}

}  // namespace pf

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
// (R, CPT, NW) instantiations: head dims 640 / 512 / 384 / 256 (the presets: 32 slabs per head -> 132 CTAs per env
// at NH = 4), 768 and 1024, and the small test heads 128 / 64 / 32
#define XL_CELL_CASES(X) X(5, 5, 16) X(4, 4, 16) X(3, 3, 16) X(2, 2, 16) X(6, 6, 16) X(8, 8, 16) X(1, 1, 16) X(1, 4, 8) X(1, 4, 4)

static bool cell_plan(int DH, int* R, int* CPT, int* NW) {
#define XL_CELL_MATCH(r, c, n) \
  if (DH == 8 * n * r && DH % (4 * c) == 0) { *R = r; *CPT = c; *NW = n; return true; }
  XL_CELL_CASES(XL_CELL_MATCH)
#undef XL_CELL_MATCH
  return false;
}

bool prefill_cell_supported(int DH) {
  int R, CPT, NW;
  return cell_plan(DH, &R, &CPT, &NW);
}

int g_prefill_conv_run = 16;   // xl_set_option("prefill_conv_run")
int g_prefill_conv_impl = 2;   // xl_set_option("prefill_conv"): 0 = scalar kernel, 1 = packed fp32 pairs, 2 = + SFU SiLU (default)
int g_prefill_conv_persist = 1;   // xl_set_option("prefill_conv_persist"): packed kernel walks the run blocks (1) or one block per CTA (0)

template <int NH>
static bool launch_conv_seq2(const ConvQkvParams& p, int S, int run, dim3 grid, dim3 block, cudaStream_t s) {
  // persistent over the run blocks: 2 CTAs per SM in total (128 registers x 256 threads), each staging its weights once
  static const int sms = [] {
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n > 0 ? n : 148;
  }();
  if (g_prefill_conv_persist) {
    // 2 CTAs per SM in total: each channel chunk gets 2 * sms / NCH CTAs that walk its (env, run block) items
    const unsigned items = grid.y * grid.z;
    const unsigned per = (unsigned)std::max(1, 2 * sms / (int)grid.x);
    grid.y = 1;
    grid.z = std::min(items, per);
  }
  const size_t smem = sizeof(float4) * (size_t)(NH * 3 * 2 + 3 * 4 + 1) * block.x;
  if (g_prefill_conv_impl == 2) {
    if (ensure_dyn_smem<&pf::conv_qkv_gates_seq2_kernel<NH, true>>(smem) != cudaSuccess) return false;
    return launch_k(pf::conv_qkv_gates_seq2_kernel<NH, true>, grid, block, smem, s, p, S, run) == cudaSuccess;
  }
  if (ensure_dyn_smem<&pf::conv_qkv_gates_seq2_kernel<NH, false>>(smem) != cudaSuccess) return false;
  return launch_k(pf::conv_qkv_gates_seq2_kernel<NH, false>, grid, block, smem, s, p, S, run) == cudaSuccess;
}

bool launch_conv_qkv_gates_seq(const ConvQkvParams& p, int S, cudaStream_t s, const int32_t* len, int pos) {
  const int nblk = p.inner / 4;
  const int per_chunk = (nblk + p.NCH - 1) / p.NCH;
  const int threads = ((per_chunk + 31) / 32) * 32;
  const int run = g_prefill_conv_run;                   // tokens per run (multiple of 4); kConvRuns runs per CTA
  if (threads > 128) return false;
  const int nruns = threads > 64 ? pf::kConvRuns / 2 : pf::kConvRuns;   // <= 256 threads per CTA
  dim3 grid(p.NCH, p.B, (S + run * nruns - 1) / (run * nruns));
  const dim3 block(threads, nruns);
  const size_t smem = sizeof(float) * 2 * p.NH * 3 * 4 * threads;
  if (g_prefill_conv_impl != 0 && p.KS == 4 && (p.NH == 4 || p.NH == 8 || p.NH == 2 || p.NH == 1)) {
    const bool ok = p.NH == 4   ? launch_conv_seq2<4>(p, S, run, grid, block, s)
                    : p.NH == 8 ? launch_conv_seq2<8>(p, S, run, grid, block, s)
                    : p.NH == 2 ? launch_conv_seq2<2>(p, S, run, grid, block, s)
                                : launch_conv_seq2<1>(p, S, run, grid, block, s);
    if (!ok) return false;
  } else if (p.KS == 4 && p.NH == 4) {
    launch_k(pf::conv_qkv_gates_seq_kernel<4, 4>, grid, block, smem, s, p, S, run);
  } else if (p.KS == 4 && p.NH == 8) {
    launch_k(pf::conv_qkv_gates_seq_kernel<4, 8>, grid, block, smem, s, p, S, run);
  } else if (p.KS == 4 && p.NH == 2) {
    launch_k(pf::conv_qkv_gates_seq_kernel<4, 2>, grid, block, smem, s, p, S, run);
  } else if (p.KS == 4 && p.NH == 1) {
    launch_k(pf::conv_qkv_gates_seq_kernel<4, 1>, grid, block, smem, s, p, S, run);
  } else {
    return false;
  }
  const int64_t n4 = (int64_t)p.B * (len ? 1 : p.KS) * (p.inner / 4);
  launch_k(pf::conv_state_seq_kernel, dim3((unsigned)((n4 + 255) / 256)), dim3(256), 0, s, p.u, p.conv_state, p.B, S,
           p.KS, p.inner, len, pos);
  return true;
}

size_t gate_scan_seq_scratch_floats(int B, int S, int NH) {
  return (size_t)B * NH * (1 + 2 * (size_t)((S + pf::kSuper - 1) / pf::kSuper));
}

void launch_gate_scan_seq(const float* gate_part, const float* igate_b, const float* fgate_b, float* m_state,
                          float* fseq, float* iseq, float* mseq, float* scratch, int B, int S, int NH, int NCH,
                          cudaStream_t s, const int32_t* len, int pos) {
  const dim3 grid(B * NH, (S + pf::kSuper - 1) / pf::kSuper);
  launch_k(pf::gate_pre_seq_kernel, grid, dim3(pf::kScanThreads), 0, s, gate_part, igate_b, fgate_b,
           (const float*)m_state, fseq, iseq, scratch, B, S, NH, NCH, len, pos);
  launch_k(pf::gate_scan_seq_kernel, grid, dim3(pf::kScanThreads), 0, s, m_state, fseq, iseq, mseq,
           (const float*)scratch, B, S, NH);
}

template <int R, int CPT, int NW>
static cudaError_t launch_cell_RC(const pf::CellSeqParams& p, cudaStream_t s) {
  const int w = 4 * CPT;
  const size_t smem = 128 + sizeof(float) * ((size_t)pf::kStages * pf::cell_stage_floats(p.DH, w) +
                                             2 * (size_t)NW * pf::kTB * w);
  if (cudaError_t e = ensure_dyn_smem<&pf::mlstm_cell_seq_kernel<R, CPT, NW>>(smem); e != cudaSuccess) return e;
  const int grid = p.B * p.NH * (p.DH / w + 1);
  return launch_k(pf::mlstm_cell_seq_kernel<R, CPT, NW>, dim3(grid), dim3((NW + 1) * 32), smem, s, p);
}

cudaError_t launch_cell_seq(float* C, float* n, const float* q, const float* k, const float* v, const float* fseq,
                            const float* iseq, float* num, float* qn, int B, int S, int NH, int DH, int inner,
                            cudaStream_t s) {
  int R, CPT, NW;
  if (!cell_plan(DH, &R, &CPT, &NW) || S % pf::kTB != 0) return cudaErrorInvalidValue;
  pf::CellSeqParams p;
  p.C = C; p.n = n; p.q = q; p.k = k; p.v = v; p.fseq = fseq; p.iseq = iseq; p.num = num; p.qn = qn;
  p.B = B; p.S = S; p.NH = NH; p.DH = DH; p.inner = inner; p.nw = NW;
#define XL_CELL_LAUNCH(r, c, n) \
  if (R == r && CPT == c && NW == n) return launch_cell_RC<r, c, n>(p, s);
  XL_CELL_CASES(XL_CELL_LAUNCH)
#undef XL_CELL_LAUNCH
  return cudaErrorInvalidValue;
}

cudaError_t launch_finalize_seq(const float* num, const float* qn, const float* mseq, const float* outnorm_w,
                                const float* skip, const float* act, const float* u, float* out, void* out_hi,
                                void* out_lo, int B, int S, int NH, int DH, int inner, float ln_eps, float cell_eps,
                                cudaStream_t s) {
  pf::FinalizeSeqParams p;
  p.num = num; p.qn = qn; p.mseq = mseq; p.outnorm_w = outnorm_w; p.skip = skip; p.act = act; p.u = u; p.out = out;
  p.out_hi = (__nv_bfloat16*)out_hi; p.out_lo = (__nv_bfloat16*)out_lo;
  p.B = B; p.S = S; p.NH = NH; p.DH = DH; p.inner = inner; p.ln_eps = ln_eps; p.cell_eps = cell_eps;
  const int64_t warps = (int64_t)B * S * NH;
  const dim3 grid((unsigned)((warps + 7) / 8));
  if (DH <= 256) return launch_k(pf::mlstm_finalize_seq_kernel<2>, grid, dim3(256), 0, s, p);
  if (DH <= 384) return launch_k(pf::mlstm_finalize_seq_kernel<3>, grid, dim3(256), 0, s, p);
  if (DH <= 512) return launch_k(pf::mlstm_finalize_seq_kernel<4>, grid, dim3(256), 0, s, p);
  if (DH <= 640) return launch_k(pf::mlstm_finalize_seq_kernel<5>, grid, dim3(256), 0, s, p);
  return launch_k(pf::mlstm_finalize_seq_kernel<8>, grid, dim3(256), 0, s, p);
}

}  // namespace xl
