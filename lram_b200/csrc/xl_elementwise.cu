// Small fused kernels around the GEMMs and the state step: LayerNorms, token embedding, the pre-cell
// conv / SiLU / headwise-qkv / gate pre-activation kernel, argmax + inv_tokenize, state reset.
// Reference arithmetic: SURVEY.md Appendix A (xlstm v1.0.x mLSTMLayer.step) and the LRAM files cited at
// each kernel.
#include <cuda_bf16.h>

#include <algorithm>

#include "xl_common.cuh"
#include "xl_internal.h"

namespace xl {

int g_use_pdl = 1;

// ------------------------------------------------------------------------------------------------
// LayerNorm rows: one warp per row, three passes over an L1-resident row (two-pass variance like ATen).
// xlstm LayerNorm: F.layer_norm(x, weight = 1 + w, bias = None, eps)  (residual_weight = 1)
// HF embed_ln:     nn.LayerNorm(d) affine                              (residual_weight = 0, bias)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ln_rows_kernel(const float* __restrict__ in, int64_t in_stride,
                                                      float* __restrict__ out, int64_t out_stride,
                                                      const float* __restrict__ w,
                                                      const float* __restrict__ bias, int residual_weight,
                                                      float eps, int rows, int d,
                                                      __nv_bfloat16* __restrict__ a_hi,
                                                      __nv_bfloat16* __restrict__ a_lo) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  if (warp >= rows) return;
  const float* x = in + (int64_t)warp * in_stride;
  const int d4 = d >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  float s = 0.f;
  for (int i = lane; i < d4; i += 32) {
    float4 v = x4[i];
    s += (v.x + v.y) + (v.z + v.w);
  }
  s = warp_sum(s);
  const float mean = s / (float)d;
  float q = 0.f;
  for (int i = lane; i < d4; i += 32) {
    float4 v = x4[i];
    float a = v.x - mean, b = v.y - mean, c = v.z - mean, e = v.w - mean;
    q += (a * a + b * b) + (c * c + e * e);
  }
  q = warp_sum(q);
  const float rstd = rsqrtf(q / (float)d + eps);
  float* o = out ? out + (int64_t)warp * out_stride : nullptr;
  const float4* w4 = reinterpret_cast<const float4*>(w);
  const float4* b4 = reinterpret_cast<const float4*>(bias);
  const float wofs = residual_weight ? 1.f : 0.f;
  for (int i = lane; i < d4; i += 32) {
    float4 v = x4[i];
    float4 g = w4[i];
    float4 r;
    r.x = (v.x - mean) * rstd * (g.x + wofs);
    r.y = (v.y - mean) * rstd * (g.y + wofs);
    r.z = (v.z - mean) * rstd * (g.z + wofs);
    r.w = (v.w - mean) * rstd * (g.w + wofs);
    if (bias) {
      float4 bb = b4[i];
      r.x += bb.x; r.y += bb.y; r.z += bb.z; r.w += bb.w;
    }
    if (o) reinterpret_cast<float4*>(o)[i] = r;
    if (a_hi) {
      // x = hi + lo with hi = bf16(x), lo = bf16(x - hi): two bf16 tensor-core passes recover ~16 bits
      float rr[4] = {r.x, r.y, r.z, r.w};
      __nv_bfloat16 hi[4], lo[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        hi[j] = __float2bfloat16_rn(rr[j]);
        lo[j] = __float2bfloat16_rn(rr[j] - __bfloat162float(hi[j]));
      }
      const int64_t base = (int64_t)warp * d + 4 * i;
      *reinterpret_cast<uint2*>(a_hi + base) = *reinterpret_cast<uint2*>(hi);
      *reinterpret_cast<uint2*>(a_lo + base) = *reinterpret_cast<uint2*>(lo);
    }
  }
}

// One CTA per row, one float4 per thread held in registers: a single global read, two block reductions.
// kPlanes: the residual stream first takes the split-K planes of proj_down (the plain instantiation stays at ~32
// registers: the prefill runs it over 16 k rows, where occupancy matters).
template <bool kPlanes>
__global__ void __launch_bounds__(1024) ln_rows_cta_kernel(const float* __restrict__ in, int64_t in_stride,
                                                           float* __restrict__ out, int64_t out_stride,
                                                           const float* __restrict__ w,
                                                           const float* __restrict__ bias, int residual_weight,
                                                           float eps, int d, __nv_bfloat16* __restrict__ a_hi,
                                                           __nv_bfloat16* __restrict__ a_lo,
                                                           const float* __restrict__ part, int splits,
                                                           int64_t part_stride, float* __restrict__ x_out,
                                                           int src_row_mul, int src_row_off) {
  __shared__ float red[32];
  const int row = blockIdx.x;                             // output row
  const int srow = row * src_row_mul + src_row_off;       // input row (gather: e.g. the action-token row of each env)
  const int i = threadIdx.x;
  const bool ok = i < (d >> 2);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 g = v, bb = v;
  if (ok) {                                // weights: before the dependency wait
    g = reinterpret_cast<const float4*>(w)[i];
    if (bias) bb = reinterpret_cast<const float4*>(bias)[i];
  }
  pdl_wait();
  pdl_trigger();
  if (ok) {
    v = reinterpret_cast<const float4*>(in + (int64_t)srow * in_stride)[i];
    if (kPlanes && part) {
      // residual stream += split-K planes of proj_down, in plane order (deterministic); written back in place
      const float4* pp = reinterpret_cast<const float4*>(part + (int64_t)srow * d) + i;
      // the first 8 planes are requested together (a plain loop gets scheduled as load -> add -> load: one L2 round
      // trip per plane on the critical path of the block), then added in plane order
      float4 pl[8];
#pragma unroll
      for (int z = 0; z < 8; ++z) pl[z] = pp[((z < splits ? z : 0) * part_stride) >> 2];   // (unpredicated: one batch)
#pragma unroll
      for (int z = 0; z < 8; ++z)
        if (z < splits) { v.x += pl[z].x; v.y += pl[z].y; v.z += pl[z].z; v.w += pl[z].w; }
      for (int z = 8; z < splits; ++z) {
        const float4 a4 = pp[(z * part_stride) >> 2];
        v.x += a4.x; v.y += a4.y; v.z += a4.z; v.w += a4.w;
      }
      if (x_out) reinterpret_cast<float4*>(x_out + (int64_t)srow * in_stride)[i] = v;
    }
  }
  const float mean = block_sum((v.x + v.y) + (v.z + v.w), red) / (float)d;
  const float a = v.x - mean, b = v.y - mean, c = v.z - mean, e = v.w - mean;
  const float q = ok ? (a * a + b * b) + (c * c + e * e) : 0.f;
  const float rstd = rsqrtf(block_sum(q, red) / (float)d + eps);
  if (!ok) return;
  const float wofs = residual_weight ? 1.f : 0.f;
  float4 r;
  r.x = a * rstd * (g.x + wofs) + bb.x;
  r.y = b * rstd * (g.y + wofs) + bb.y;
  r.z = c * rstd * (g.z + wofs) + bb.z;
  r.w = e * rstd * (g.w + wofs) + bb.w;
  if (out) reinterpret_cast<float4*>(out + (int64_t)row * out_stride)[i] = r;
  if (a_hi) {
    const float rr[4] = {r.x, r.y, r.z, r.w};
    __nv_bfloat16 hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      hi[j] = __float2bfloat16_rn(rr[j]);
      lo[j] = __float2bfloat16_rn(rr[j] - __bfloat162float(hi[j]));
    }
    const int64_t base = (int64_t)row * d + 4 * i;
    *reinterpret_cast<uint2*>(a_hi + base) = *reinterpret_cast<uint2*>(hi);
    *reinterpret_cast<uint2*>(a_lo + base) = *reinterpret_cast<uint2*>(lo);
  }
}

void launch_ln_rows(const float* in, int64_t in_stride, float* out, int64_t out_stride, const float* w,
                    const float* bias, int residual_weight, float eps, int rows, int d, void* a_hi,
                    void* a_lo, cudaStream_t s) {
  if (rows <= 0) return;
  if (d <= 4096) {
    const int threads = (((d >> 2) + 31) / 32) * 32;
    launch_k(ln_rows_cta_kernel<false>, dim3(rows), dim3(threads), 0, s, in, in_stride, out, out_stride, w, bias,
             residual_weight, eps, d, (__nv_bfloat16*)a_hi, (__nv_bfloat16*)a_lo, (const float*)nullptr, 0,
             (int64_t)0, (float*)nullptr, 1, 0);
    return;
  }
  const int warps_per_block = 8;
  dim3 grid((rows + warps_per_block - 1) / warps_per_block);
  launch_k(ln_rows_kernel, grid, dim3(warps_per_block * 32), 0, s, in, in_stride, out, out_stride, w, bias,
           residual_weight, eps, rows, d, (__nv_bfloat16*)a_hi, (__nv_bfloat16*)a_lo);
}

void launch_ln_rows_reduce(float* x, const float* part, int splits, int64_t part_stride, float* out,
                           int64_t out_stride, const float* w, float eps, int rows, int d, void* a_hi, void* a_lo,
                           cudaStream_t s) {
  if (rows <= 0) return;
  const int threads = (((d >> 2) + 31) / 32) * 32;     // d <= 4096 (checked where the split is planned)
  launch_k(ln_rows_cta_kernel<true>, dim3(rows), dim3(threads), 0, s, (const float*)x, (int64_t)d, out, out_stride, w,
           (const float*)nullptr, 1, eps, d, (__nv_bfloat16*)a_hi, (__nv_bfloat16*)a_lo, part, splits, part_stride,
           x, 1, 0);
}

// post_blocks_norm of ONE token row per env (the action-token row: x row b*row_mul + row_off, plus the pending
// split-K planes of the last proj_down) -> dense [rows, d] bf16 hi/lo operand planes of the action head. Replaces
// norm-all-rows + row gather + split when the caller does not ask for the hidden states.
void launch_ln_rows_gather(const float* x, const float* part, int splits, int64_t part_stride, const float* w,
                           float eps, int rows, int d, int row_mul, int row_off, void* a_hi, void* a_lo,
                           cudaStream_t s) {
  if (rows <= 0) return;
  const int threads = (((d >> 2) + 31) / 32) * 32;
  launch_k(ln_rows_cta_kernel<true>, dim3(rows), dim3(threads), 0, s, x, (int64_t)d, (float*)nullptr, (int64_t)0, w,
           (const float*)nullptr, 1, eps, d, (__nv_bfloat16*)a_hi, (__nv_bfloat16*)a_lo, splits > 1 ? part : nullptr,
           splits, part_stride, (float*)nullptr, row_mul, row_off);
}

// ------------------------------------------------------------------------------------------------
// Token embedding: embed_inputs + stack (s, rtg, r) + embed_ln
// (online_decision_transformer_model.py:522-530,588-612; discrete_decision_transformer_model.py:266-275)
// The per-row arithmetic lives in embed_token_row_warp / embed_token_row_cta, shared by the step's embed kernels and the
// sequence embed kernels below, so that a timestep's tokens get the same bits on either path.
// ------------------------------------------------------------------------------------------------

// One token row, one warp: o[0, d) = embed_ln(tok == 0 ? s_row : scal * wv + bv). kPads: s_row == nullptr is a zero
// state embedding (the step always has one; its instantiation is free of the check).
template <bool kPads>
__device__ __forceinline__ void embed_token_row_warp(int tok, int lane, const float* __restrict__ s_row, float scal,
                                                     const float* __restrict__ wv, const float* __restrict__ bv,
                                                     const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                                                     float eps, float* __restrict__ o, int d) {
  auto val = [&](int i) -> float {
    return tok == 0 ? ((!kPads || s_row) ? s_row[i] : 0.f) : fmaf(scal, wv[i], bv[i]);
  };
  float s = 0.f;
  for (int i = lane; i < d; i += 32) s += val(i);
  s = warp_sum(s);
  const float mean = s / (float)d;
  float q = 0.f;
  for (int i = lane; i < d; i += 32) {
    float a = val(i) - mean;
    q += a * a;
  }
  q = warp_sum(q);
  const float rstd = rsqrtf(q / (float)d + eps);
  for (int i = lane; i < d; i += 32) o[i] = (val(i) - mean) * rstd * ln_w[i] + ln_b[i];
}

// one warp per (b, tok) row
__global__ void __launch_bounds__(256) embed_tokens_kernel(
    const float* __restrict__ s_emb, const float* __restrict__ rtg, const float* __restrict__ rew,
    const float* __restrict__ w_ret, const float* __restrict__ b_ret, const float* __restrict__ w_rew,
    const float* __restrict__ b_rew, const float* __restrict__ ln_w, const float* __restrict__ ln_b,
    float eps, float* __restrict__ x, int B, int d, unsigned* __restrict__ step_counter,
    unsigned* __restrict__ sample_counter,
    const float* __restrict__ ln0_w, float ln0_eps, float* __restrict__ xn0, __nv_bfloat16* __restrict__ a_hi,
    __nv_bfloat16* __restrict__ a_lo) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  pdl_wait();
  // token ring (xl_set_token_ring): this is the first kernel of an env step that every step runs -> it advances the
  // step counter the argmax kernel at the end of the step derives its ring slot from
  if (step_counter && blockIdx.x == 0 && threadIdx.x == 0) *step_counter = *step_counter + 1;
  // the sampler's step (xl_set_sampling) advances here for the same reason
  if (sample_counter && blockIdx.x == 0 && threadIdx.x == 0) *sample_counter = *sample_counter + 1;
  pdl_trigger();
  if (row >= 3 * B) return;
  const int b = row / 3, tok = row - 3 * b;
  const float scal = (tok == 1) ? rtg[b] : ((tok == 2 && rew) ? rew[b] : 0.f);
  float* o = x + (int64_t)row * d;
  embed_token_row_warp<false>(tok, lane, s_emb + (int64_t)b * d, scal, tok == 1 ? w_ret : w_rew, tok == 1 ? b_ret : b_rew,
                       ln_w, ln_b, eps, o, d);
  if (!ln0_w) return;
  // the first block's pre-norm (xlstm LayerNorm, gamma = 1 + w) on the row this warp just produced: the block stack's
  // first LayerNorm launch disappears. Each lane re-reads only what it wrote itself.
  float s2 = 0.f;
  for (int i = lane; i < d; i += 32) s2 += o[i];
  s2 = warp_sum(s2);
  const float mean2 = s2 / (float)d;
  float q2 = 0.f;
  for (int i = lane; i < d; i += 32) {
    const float a = o[i] - mean2;
    q2 += a * a;
  }
  q2 = warp_sum(q2);
  const float rstd2 = rsqrtf(q2 / (float)d + ln0_eps);
  for (int i = lane; i < d; i += 32) {
    const float r = (o[i] - mean2) * rstd2 * (1.f + ln0_w[i]);
    if (xn0) xn0[(int64_t)row * d + i] = r;
    if (a_hi) {
      const __nv_bfloat16 hi = __float2bfloat16_rn(r);
      a_hi[(int64_t)row * d + i] = hi;
      a_lo[(int64_t)row * d + i] = __float2bfloat16_rn(r - __bfloat162float(hi));
    }
  }
}

// CTA-per-row form (d <= 4096): thread i holds channels 4i..4i+3 (ok: 4i < d) in registers, block reductions.
// The weights of token `tok`, loaded before the dependency wait.
__device__ __forceinline__ void embed_token_weights_cta(int tok, int i, bool ok, const float* __restrict__ w_ret,
                                                        const float* __restrict__ b_ret, const float* __restrict__ w_rew,
                                                        const float* __restrict__ b_rew, const float* __restrict__ ln_w,
                                                        const float* __restrict__ ln_b, float4& g, float4& bb,
                                                        float4& wv, float4& bv) {
  g = bb = wv = bv = make_float4(0.f, 0.f, 0.f, 0.f);
  if (!ok) return;
  g = reinterpret_cast<const float4*>(ln_w)[i];
  bb = reinterpret_cast<const float4*>(ln_b)[i];
  if (tok != 0) {
    wv = reinterpret_cast<const float4*>(tok == 1 ? w_ret : w_rew)[i];
    bv = reinterpret_cast<const float4*>(tok == 1 ? b_ret : b_rew)[i];
  }
}

// One token row: embed_ln(tok == 0 ? s_row : scal() * wv + bv), this thread's four channels; scal() reads the rtg /
// reward. kPads: s_row == nullptr is a zero state embedding (the step's instantiation is free of the check).
template <bool kPads, typename Scal>
__device__ __forceinline__ float4 embed_token_row_cta(int tok, int i, bool ok, const float* __restrict__ s_row,
                                                      Scal scal_of, float4 wv, float4 bv, float4 g, float4 bb, int d,
                                                      float eps, float* red) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ok) {
    if (tok == 0) {
      if (!kPads || s_row) v = reinterpret_cast<const float4*>(s_row)[i];
    } else {
      const float scal = scal_of();
      v = make_float4(fmaf(scal, wv.x, bv.x), fmaf(scal, wv.y, bv.y), fmaf(scal, wv.z, bv.z), fmaf(scal, wv.w, bv.w));
    }
  }
  const float mean = block_sum((v.x + v.y) + (v.z + v.w), red) / (float)d;
  const float a0 = v.x - mean, a1 = v.y - mean, a2 = v.z - mean, a3 = v.w - mean;
  const float rstd = rsqrtf(block_sum(ok ? (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3) : 0.f, red) / (float)d + eps);
  return make_float4(a0 * rstd * g.x + bb.x, a1 * rstd * g.y + bb.y, a2 * rstd * g.z + bb.z, a3 * rstd * g.w + bb.w);
}

// the step's embed kernel: one CTA per (b, tok) row; the token row is read once and both LayerNorms (embed_ln, then
// optionally block 0's pre-norm) run on registers.
__global__ void __launch_bounds__(1024) embed_tokens_cta_kernel(
    const float* __restrict__ s_emb, const float* __restrict__ rtg, const float* __restrict__ rew,
    const float* __restrict__ w_ret, const float* __restrict__ b_ret, const float* __restrict__ w_rew,
    const float* __restrict__ b_rew, const float* __restrict__ ln_w, const float* __restrict__ ln_b,
    float eps, float* __restrict__ x, int B, int d, unsigned* __restrict__ step_counter,
    unsigned* __restrict__ sample_counter,
    const float* __restrict__ ln0_w, float ln0_eps, float* __restrict__ xn0, __nv_bfloat16* __restrict__ a_hi,
    __nv_bfloat16* __restrict__ a_lo) {
  __shared__ float red[32];
  const int row = blockIdx.x, i = threadIdx.x;
  const bool ok = i < (d >> 2);
  const int b = row / 3, tok = row - 3 * b;
  // weights before the dependency wait
  float4 g, bb, wv, bv, g0 = make_float4(0.f, 0.f, 0.f, 0.f);
  embed_token_weights_cta(tok, i, ok, w_ret, b_ret, w_rew, b_rew, ln_w, ln_b, g, bb, wv, bv);
  if (ok && ln0_w) g0 = reinterpret_cast<const float4*>(ln0_w)[i];
  pdl_wait();
  if (step_counter && blockIdx.x == 0 && threadIdx.x == 0) *step_counter = *step_counter + 1;   // token ring slot
  if (sample_counter && blockIdx.x == 0 && threadIdx.x == 0) *sample_counter = *sample_counter + 1;   // sampler step
  pdl_trigger();
  float4 o = embed_token_row_cta<false>(
      tok, i, ok, s_emb + (int64_t)b * d, [&] { return (tok == 1) ? rtg[b] : (rew ? rew[b] : 0.f); }, wv, bv, g, bb, d,
      eps, red);
  if (ok) reinterpret_cast<float4*>(x + (int64_t)row * d)[i] = o;
  if (!ln0_w) return;
  if (!ok) o = make_float4(0.f, 0.f, 0.f, 0.f);
  const float mean = block_sum((o.x + o.y) + (o.z + o.w), red) / (float)d;
  const float a0 = o.x - mean, a1 = o.y - mean, a2 = o.z - mean, a3 = o.w - mean;
  const float rstd = rsqrtf(block_sum(ok ? (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3) : 0.f, red) / (float)d + ln0_eps);
  if (!ok) return;
  const float r[4] = {a0 * rstd * (1.f + g0.x), a1 * rstd * (1.f + g0.y), a2 * rstd * (1.f + g0.z), a3 * rstd * (1.f + g0.w)};
  if (xn0) reinterpret_cast<float4*>(xn0 + (int64_t)row * d)[i] = make_float4(r[0], r[1], r[2], r[3]);
  if (a_hi) {
    __nv_bfloat16 hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      hi[j] = __float2bfloat16_rn(r[j]);
      lo[j] = __float2bfloat16_rn(r[j] - __bfloat162float(hi[j]));
    }
    const int64_t base = (int64_t)row * d + 4 * i;
    *reinterpret_cast<uint2*>(a_hi + base) = *reinterpret_cast<uint2*>(hi);
    *reinterpret_cast<uint2*>(a_lo + base) = *reinterpret_cast<uint2*>(lo);
  }
}

void launch_embed_tokens(const float* s_emb, const float* rtg, const float* rew, const float* w_ret,
                         const float* b_ret, const float* w_rew, const float* b_rew, const float* ln_w,
                         const float* ln_b, float eps, float* x, int B, int d, unsigned* step_counter,
                         unsigned* sample_counter, const float* ln0_w, float ln0_eps, float* xn0, void* a_hi,
                         void* a_lo, cudaStream_t s) {
  const int rows = 3 * B;
  if (d <= 4096 && (d & 3) == 0) {
    const int threads = (((d >> 2) + 31) / 32) * 32;
    launch_k(embed_tokens_cta_kernel, dim3(rows), dim3(threads), 0, s, s_emb, rtg, rew, w_ret, b_ret, w_rew, b_rew, ln_w,
             ln_b, eps, x, B, d, step_counter, sample_counter, ln0_w, ln0_eps, xn0, (__nv_bfloat16*)a_hi, (__nv_bfloat16*)a_lo);
    return;
  }
  dim3 grid((rows + 7) / 8);
  launch_k(embed_tokens_kernel, grid, dim3(256), 0, s, s_emb, rtg, rew, w_ret, b_ret, w_rew, b_rew, ln_w, ln_b, eps,
           x, B, d, step_counter, sample_counter, ln0_w, ln0_eps, xn0, (__nv_bfloat16*)a_hi, (__nv_bfloat16*)a_lo);
}

// ---- sequence embed: the tokens of a prefill chunk straight from the caller's [B, Tn, ...] buffers ---------------
// Token row (k * Tc + t) * 3 + tok of the chunk reads env (perm ? perm[k] : k), timestep pos + t. Rows at or past the
// env's length (len[k] / len_div - pos) never touch caller memory: they are the tokens of a zero embedding, zero rtg
// and zero reward (finite; the prefill turns them into identity tokens through len).
// s_row: the row's state embedding (tok 0); scal: its rtg / reward (tok 1 / 2); nullptr = zero.
__device__ __forceinline__ void seq_embed_source(const SeqEmbedParams& p, int row, int tok, const float*& s_row,
                                                 const float*& scal) {
  const int kt = row / 3, k = kt / p.Tc, t = kt - k * p.Tc;
  s_row = scal = nullptr;
  const int n = p.len ? min(max(p.len[k] / p.len_div - p.pos, 0), p.Tc) : p.Tc;
  if (t >= n) return;
  const int64_t off = (int64_t)(p.perm ? p.perm[k] : k) * p.Tn + p.pos + t;
  if (tok == 0) s_row = p.s_emb + off * p.d;
  else scal = tok == 1 ? p.rtg + off : (p.rew ? p.rew + off : nullptr);
}

__global__ void __launch_bounds__(1024) seq_embed_tokens_kernel(SeqEmbedParams p) {
  __shared__ float red[32];
  const int row = blockIdx.x, i = threadIdx.x;
  const bool ok = i < (p.d >> 2);
  const int tok = row % 3;
  float4 g, bb, wv, bv;
  embed_token_weights_cta(tok, i, ok, p.w_ret, p.b_ret, p.w_rew, p.b_rew, p.ln_w, p.ln_b, g, bb, wv, bv);
  pdl_wait();
  pdl_trigger();
  const float *s_row, *scal;
  seq_embed_source(p, row, tok, s_row, scal);
  const float4 o = embed_token_row_cta<true>(tok, i, ok, s_row, [&] { return scal ? *scal : 0.f; }, wv, bv, g, bb, p.d,
                                             p.eps, red);
  if (ok) reinterpret_cast<float4*>(p.x + (int64_t)row * p.d)[i] = o;
}

// d > 4096: one warp per token row
__global__ void __launch_bounds__(256) seq_embed_tokens_warp_kernel(SeqEmbedParams p) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  if (row >= 3 * p.rows) return;
  const int tok = row % 3;
  const float *s_row, *scal;
  seq_embed_source(p, row, tok, s_row, scal);
  embed_token_row_warp<true>(tok, lane, s_row, scal ? *scal : 0.f, tok == 1 ? p.w_ret : p.w_rew,
                       tok == 1 ? p.b_ret : p.b_rew, p.ln_w, p.ln_b, p.eps, p.x + (int64_t)row * p.d, p.d);
}

void launch_seq_embed_tokens(const SeqEmbedParams& p, cudaStream_t s) {
  if (p.rows <= 0) return;
  const int64_t rows = 3 * (int64_t)p.rows;
  if (p.d <= 4096 && (p.d & 3) == 0) {
    launch_k(seq_embed_tokens_kernel, dim3((unsigned)rows), dim3((((p.d >> 2) + 31) / 32) * 32), 0, s, p);
    return;
  }
  launch_k(seq_embed_tokens_warp_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, s, p);
}

// zero-pad states [rows, K] -> bf16 hi/lo operand planes [rows, Kpad] of the embed_state GEMM (pad + split in one)
__global__ void pad_split_kernel(const float* __restrict__ in, int K, __nv_bfloat16* __restrict__ hi,
                                 __nv_bfloat16* __restrict__ lo, int Kpad, int rows) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_trigger();
  if (i >= (int64_t)rows * Kpad) return;
  const int r = (int)(i / Kpad), c = (int)(i - (int64_t)r * Kpad);
  const float v = c < K ? in[(int64_t)r * K + c] : 0.f;
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[i] = h;
  lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}
void launch_pad_split(const float* in, int K, void* hi, void* lo, int Kpad, int rows, cudaStream_t s) {
  const int64_t n = (int64_t)rows * Kpad;
  launch_k(pad_split_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, in, K, (__nv_bfloat16*)hi,
           (__nv_bfloat16*)lo, Kpad, rows);
}

__global__ void pad_rows_kernel(const float* __restrict__ in, int K, float* __restrict__ out, int Kpad,
                                int rows) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_trigger();
  if (i >= (int64_t)rows * Kpad) return;
  const int r = (int)(i / Kpad), c = (int)(i - (int64_t)r * Kpad);
  out[i] = c < K ? in[(int64_t)r * K + c] : 0.f;
}
void launch_pad_rows(const float* in, int K, float* out, int Kpad, int rows, cudaStream_t s) {
  const int64_t n = (int64_t)rows * Kpad;
  launch_k(pad_rows_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, in, K, out, Kpad, rows);
}

__global__ void copy_rows_kernel(const float* __restrict__ in, int64_t in_stride, float* __restrict__ out,
                                 int64_t out_stride, int rows, int d) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_trigger();
  if (i >= (int64_t)rows * d) return;
  const int r = (int)(i / d), c = (int)(i - (int64_t)r * d);
  out[(int64_t)r * out_stride + c] = in[(int64_t)r * in_stride + c];
}
void launch_copy_rows(const float* in, int64_t in_stride, float* out, int64_t out_stride, int rows, int d,
                      cudaStream_t s) {
  const int64_t n = (int64_t)rows * d;
  launch_k(copy_rows_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, s, in, in_stride, out, out_stride,
           rows, d);
}

// ------------------------------------------------------------------------------------------------
// Pre-cell kernel: CausalConv1d.step (ring window) + bias -> SiLU -> block-diagonal q/k/v
// (LinearHeadwiseExpand, 4x4 blocks) -> partial igate/fgate pre-activations.
// [ext-xlstm] mLSTMLayer.step / conv1d_step / mLSTMCell.step gate Linear(cat[q,k,v]) — SURVEY App. A.
// grid = (NCH channel chunks, B envs); one thread owns one 4-channel block for all T tokens, so the conv
// window lives in registers across the tokens of the step. Gate partial sums per chunk are written out
// and summed in fixed order by the state kernel (deterministic, no float atomics).
// ------------------------------------------------------------------------------------------------

template <int KS, int T, int NH>
__global__ void __launch_bounds__(128, 4) conv_qkv_gates_kernel(ConvQkvParams p) {
  constexpr int kMaxT = T;
  constexpr int kMaxNH = NH;
  __shared__ float red[2 * kMaxNH * kMaxT * 4];
  const int b = blockIdx.y;
  const int chunk = blockIdx.x;
  const int inner = p.inner;
  const int nblk = inner >> 2;                       // 4-channel blocks
  const int blk_per_chunk = (nblk + p.NCH - 1) / p.NCH;
  const int j = chunk * blk_per_chunk + threadIdx.x;
  const bool active = threadIdx.x < blk_per_chunk && j < nblk;
  const int c = 4 * (active ? j : 0);

  // ---- phase 1: conv window -> SiLU -> block-diagonal q/k/v for the T tokens -----------------------
  float q[kMaxT][4], k[kMaxT][4], v[kMaxT][4];
#pragma unroll
  for (int t = 0; t < kMaxT; ++t)
#pragma unroll
    for (int o = 0; o < 4; ++o) q[t][o] = k[t][o] = v[t][o] = 0.f;
  // Everything this thread needs that no kernel of the step writes (weights, and the conv window, which only
  // this kernel touches) is loaded BEFORE the dependency wait, so it overlaps the tail of proj_up.
  float win[KS][4];
  float cw[4][KS];
  float cbv[4] = {0.f, 0.f, 0.f, 0.f};
  float wq[16], wk[16], wv[16];
  float* cs = p.conv_state + (int64_t)b * KS * inner + c;
  if (active) {
    // rows 1..KS-1 of the state are the KS-1 most recent inputs (oldest first); row 0 is shifted out
#pragma unroll
    for (int r = 0; r < KS; ++r) {
      const float4 w4 = *reinterpret_cast<const float4*>(cs + (int64_t)r * inner);
      win[r][0] = w4.x; win[r][1] = w4.y; win[r][2] = w4.z; win[r][3] = w4.w;
    }
#pragma unroll
    for (int ch = 0; ch < 4; ++ch)
#pragma unroll
      for (int r = 0; r < KS; ++r) cw[ch][r] = p.conv_w[(int64_t)(c + ch) * KS + r];
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
  if (active) {
    float4 xm4[kMaxT];
#pragma unroll
    for (int t = 0; t < kMaxT; ++t)
      if (t < T) {
        const float* up = p.u + ((int64_t)b * T + t) * 2 * inner + c;
        xm4[t] = *reinterpret_cast<const float4*>(up);
        for (int z = 1; z < p.u_splits; ++z) {          // split-K planes of proj_up, added in plane order
          const float4 a4 = *reinterpret_cast<const float4*>(up + z * p.u_stride);
          xm4[t].x += a4.x; xm4[t].y += a4.y; xm4[t].z += a4.z; xm4[t].w += a4.w;
        }
      }
#pragma unroll
    for (int t = 0; t < kMaxT; ++t) {
      if (t < T) {
        const int64_t row = (int64_t)b * T + t;
        const float xm[4] = {xm4[t].x, xm4[t].y, xm4[t].z, xm4[t].w};
        // roll(-1); state[-1] = x
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
          for (int r = 0; r < KS; ++r) acc = fmaf(win[r][ch], cw[ch][r], acc);
          a[ch] = silu(acc + cbv[ch]);
        }
#pragma unroll
        for (int o = 0; o < 4; ++o) {
          float sq = 0.f, sk = 0.f, sv = 0.f;
#pragma unroll
          for (int dd = 0; dd < 4; ++dd) {
            sq = fmaf(a[dd], wq[4 * o + dd], sq);
            sk = fmaf(a[dd], wk[4 * o + dd], sk);
            sv = fmaf(xm[dd], wv[4 * o + dd], sv);
          }
          q[t][o] = sq; k[t][o] = sk; v[t][o] = sv;
        }
        // channel c of head h sits at (row*NH + h)*DH + (c - h*DH) == row*inner + c: (q,k) pairs interleaved
        float* qk = p.qk + (row * inner + c) * 2;
        *reinterpret_cast<float4*>(qk) = make_float4(q[t][0], k[t][0], q[t][1], k[t][1]);
        *reinterpret_cast<float4*>(qk + 4) = make_float4(q[t][2], k[t][2], q[t][3], k[t][3]);
        *reinterpret_cast<float4*>(p.v + row * inner + c) = make_float4(v[t][0], v[t][1], v[t][2], v[t][3]);
        *reinterpret_cast<float4*>(p.act + row * inner + c) = make_float4(a[0], a[1], a[2], a[3]);
      }
    }
    // write the window back: rows = last KS inputs, oldest first (reference conv_state layout)
#pragma unroll
    for (int r = 0; r < KS; ++r)
      *reinterpret_cast<float4*>(cs + (int64_t)r * inner) =
          make_float4(win[r][0], win[r][1], win[r][2], win[r][3]);
  }

  // ---- phase 2: partial igate / fgate pre-activations of this channel chunk --------------------------
  // g~ = W[:, c] . q + W[:, inner + c] . k + W[:, 2*inner + c] . v, per head, summed over the chunk's channels
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int h = 0; h < kMaxNH; ++h) {
    if (h < NH) {
      float gi[kMaxT], gf[kMaxT];
#pragma unroll
      for (int t = 0; t < kMaxT; ++t) gi[t] = gf[t] = 0.f;
      if (active) {
        const float* wi = p.wi + (int64_t)h * 3 * inner + c;
        const float* wf = p.wf + (int64_t)h * 3 * inner + c;
        const float4 iq = *reinterpret_cast<const float4*>(wi);
        const float4 ik = *reinterpret_cast<const float4*>(wi + inner);
        const float4 iv = *reinterpret_cast<const float4*>(wi + 2 * inner);
        const float4 fq = *reinterpret_cast<const float4*>(wf);
        const float4 fk = *reinterpret_cast<const float4*>(wf + inner);
        const float4 fv = *reinterpret_cast<const float4*>(wf + 2 * inner);
#pragma unroll
        for (int t = 0; t < kMaxT; ++t) {
          if (t < T) {
            float si = q[t][0] * iq.x + q[t][1] * iq.y + q[t][2] * iq.z + q[t][3] * iq.w;
            si += k[t][0] * ik.x + k[t][1] * ik.y + k[t][2] * ik.z + k[t][3] * ik.w;
            si += v[t][0] * iv.x + v[t][1] * iv.y + v[t][2] * iv.z + v[t][3] * iv.w;
            float sf = q[t][0] * fq.x + q[t][1] * fq.y + q[t][2] * fq.z + q[t][3] * fq.w;
            sf += k[t][0] * fk.x + k[t][1] * fk.y + k[t][2] * fk.z + k[t][3] * fk.w;
            sf += v[t][0] * fv.x + v[t][1] * fv.y + v[t][2] * fv.z + v[t][3] * fv.w;
            gi[t] = si;
            gf[t] = sf;
          }
        }
      }
      // warp reduce, then one slot per (gate, token, warp)
#pragma unroll
      for (int t = 0; t < kMaxT; ++t) {
        if (t < T) {
          const float si = warp_sum(gi[t]);
          const float sf = warp_sum(gf[t]);
          if (lane == 0) {
            red[((h * 2 + 0) * kMaxT + t) * 4 + wid] = si;
            red[((h * 2 + 1) * kMaxT + t) * 4 + wid] = sf;
          }
        }
      }
    }
  }
  __syncthreads();
  // thread x -> (h, gate, t): fixed-order sum over the (<= 4) warps
  const int nout = NH * 2 * T;
  if ((int)threadIdx.x < nout) {
    const int h = threadIdx.x / (2 * T);
    const int rem = threadIdx.x - h * 2 * T;
    const int g = rem / T, t = rem - g * T;
    float s = 0.f;
    for (int w = 0; w < nw; ++w) s += red[((h * 2 + g) * kMaxT + t) * 4 + w];
    float* gp = p.gate_part + (((int64_t)b * T + t) * p.NCH + chunk) * 2 * NH;
    gp[g * NH + h] = s;
  }
}

// Token-parallel variant (impl 1): one thread per (4-channel block, token). Token t's conv window is the last KS
// elements of [old window rows, x_0 .. x_t], so the tokens of a step do not depend on each other: the per-thread
// instruction chain is ~1/T of impl 0's (this kernel is latency-bound: a few warps per SM). Same arithmetic per
// element and the same summation order of the gate partials as impl 0 -> bit-identical outputs (tested).
// Measured on B200 (48M x 64 envs): 63.7 k vs 67.2 k env-steps/s for impl 0 — every thread re-loads the ~170 weights
// of its 4-channel block and up to KS rows of u, and the kernel is bound by those loads, not by the FMA chain.
// Not the default; kept as the record of that design point.
// blockDim = T * PC with PC = threads per token (multiple of 32, >= blocks per chunk); warps never straddle tokens.
template <int KS, int T, int NH>
__global__ void __launch_bounds__(512) conv_qkv_gates_tok_kernel(ConvQkvParams p) {
  __shared__ float red[2 * NH * T * 4];
  const int b = blockIdx.y;
  const int chunk = blockIdx.x;
  const int inner = p.inner;
  const int nblk = inner >> 2;
  const int blk_per_chunk = (nblk + p.NCH - 1) / p.NCH;
  const int PC = blockDim.x / T;
  const int t = threadIdx.x / PC;
  const int jj = threadIdx.x - t * PC;
  const int j = chunk * blk_per_chunk + jj;
  const bool active = jj < blk_per_chunk && j < nblk;
  const int c = 4 * (active ? j : 0);

  float win[KS][4];
  float cw[4][KS];
  float cbv[4] = {0.f, 0.f, 0.f, 0.f};
  float wq[16], wk[16], wv[16];
#pragma unroll
  for (int r = 0; r < KS; ++r)
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) win[r][ch] = 0.f;
  float* cs = p.conv_state + (int64_t)b * KS * inner + c;
  if (active) {
    // window row r of token t = element t + 1 + r of [old rows 0..KS-1, x_0, x_1, ...]; the old rows come first
#pragma unroll
    for (int r = 0; r < KS; ++r) {
      const int idx = t + 1 + r;
      if (idx < KS) {
        const float4 w4 = *reinterpret_cast<const float4*>(cs + (int64_t)idx * inner);
        win[r][0] = w4.x; win[r][1] = w4.y; win[r][2] = w4.z; win[r][3] = w4.w;
      }
    }
#pragma unroll
    for (int ch = 0; ch < 4; ++ch)
#pragma unroll
      for (int r = 0; r < KS; ++r) cw[ch][r] = p.conv_w[(int64_t)(c + ch) * KS + r];
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
  float q[4] = {0.f, 0.f, 0.f, 0.f}, k[4] = {0.f, 0.f, 0.f, 0.f}, v[4] = {0.f, 0.f, 0.f, 0.f};
  if (active) {
#pragma unroll
    for (int r = 0; r < KS; ++r) {
      const int idx = t + 1 + r;
      if (idx >= KS) {
        const float* up = p.u + ((int64_t)b * T + (idx - KS)) * 2 * inner + c;
        float4 x4 = *reinterpret_cast<const float4*>(up);
        for (int z = 1; z < p.u_splits; ++z) {          // split-K planes of proj_up, added in plane order
          const float4 a4 = *reinterpret_cast<const float4*>(up + z * p.u_stride);
          x4.x += a4.x; x4.y += a4.y; x4.z += a4.z; x4.w += a4.w;
        }
        win[r][0] = x4.x; win[r][1] = x4.y; win[r][2] = x4.z; win[r][3] = x4.w;
      }
    }
    const int64_t row = (int64_t)b * T + t;
    const float xm[4] = {win[KS - 1][0], win[KS - 1][1], win[KS - 1][2], win[KS - 1][3]};
    float a[4];
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
      float acc = 0.f;
#pragma unroll
      for (int r = 0; r < KS; ++r) acc = fmaf(win[r][ch], cw[ch][r], acc);
      a[ch] = silu(acc + cbv[ch]);
    }
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
    float* qk = p.qk + (row * inner + c) * 2;
    *reinterpret_cast<float4*>(qk) = make_float4(q[0], k[0], q[1], k[1]);
    *reinterpret_cast<float4*>(qk + 4) = make_float4(q[2], k[2], q[3], k[3]);
    *reinterpret_cast<float4*>(p.v + row * inner + c) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p.act + row * inner + c) = make_float4(a[0], a[1], a[2], a[3]);
  }

  // partial igate / fgate pre-activations of this (chunk, token): same expressions and order as impl 0
  const int lane = threadIdx.x & 31, wtok = jj >> 5;
  const int nwt = PC >> 5;
#pragma unroll
  for (int h = 0; h < NH; ++h) {
    float si = 0.f, sf = 0.f;
    if (active) {
      const float* wi = p.wi + (int64_t)h * 3 * inner + c;
      const float* wf = p.wf + (int64_t)h * 3 * inner + c;
      const float4 iq = *reinterpret_cast<const float4*>(wi);
      const float4 ik = *reinterpret_cast<const float4*>(wi + inner);
      const float4 iv = *reinterpret_cast<const float4*>(wi + 2 * inner);
      const float4 fq = *reinterpret_cast<const float4*>(wf);
      const float4 fk = *reinterpret_cast<const float4*>(wf + inner);
      const float4 fv = *reinterpret_cast<const float4*>(wf + 2 * inner);
      si = q[0] * iq.x + q[1] * iq.y + q[2] * iq.z + q[3] * iq.w;
      si += k[0] * ik.x + k[1] * ik.y + k[2] * ik.z + k[3] * ik.w;
      si += v[0] * iv.x + v[1] * iv.y + v[2] * iv.z + v[3] * iv.w;
      sf = q[0] * fq.x + q[1] * fq.y + q[2] * fq.z + q[3] * fq.w;
      sf += k[0] * fk.x + k[1] * fk.y + k[2] * fk.z + k[3] * fk.w;
      sf += v[0] * fv.x + v[1] * fv.y + v[2] * fv.z + v[3] * fv.w;
    }
    si = warp_sum(si);
    sf = warp_sum(sf);
    if (lane == 0) {
      red[((h * 2 + 0) * T + t) * 4 + wtok] = si;
      red[((h * 2 + 1) * T + t) * 4 + wtok] = sf;
    }
  }
  __syncthreads();
  // The window of the last token = the KS most recent inputs, oldest first. Written only AFTER the barrier: the other
  // tokens' threads of this 4-channel block read the old window rows in their prologue.
  if (active && t == T - 1) {
#pragma unroll
    for (int r = 0; r < KS; ++r)
      *reinterpret_cast<float4*>(cs + (int64_t)r * inner) = make_float4(win[r][0], win[r][1], win[r][2], win[r][3]);
  }
  const int nout = NH * 2 * T;
  if ((int)threadIdx.x < nout) {
    const int h = threadIdx.x / (2 * T);
    const int rem = threadIdx.x - h * 2 * T;
    const int g = rem / T, tt = rem - g * T;
    float s = 0.f;
    for (int w = 0; w < nwt; ++w) s += red[((h * 2 + g) * T + tt) * 4 + w];
    float* gp = p.gate_part + (((int64_t)b * T + tt) * p.NCH + chunk) * 2 * NH;
    gp[g * NH + h] = s;
  }
}

// Packed-fp32 variant (impl 2, KS = 4, NH <= 4): the kernel sits in the per-block chain of the env step with ~5 warps per
// SM, so what counts is the length of one thread's dependent instruction stream after the dependency wait. Against impl 0:
//   * conv, headwise q/k/v and gate dot products as FFMA2 / FMUL2 / FADD2 on fp32 pairs (channel pairs, output pairs,
//     the (igate, fgate) pair of a head) with every chain in impl 0's order: outputs are BIT-identical (tested);
//   * the gate weights (24 x NH values per thread) are loaded BEFORE the dependency wait like the other weights -- in
//     impl 0 their L2 round trip sits between phase 1 and phase 2 (occupancy is irrelevant here: up to 255 registers);
//   * the NH * 2 * T <= 32 partial sums of a warp are reduced by one transposing butterfly (31 shuffles, the pairwise
//     sums of warp_sum()) instead of NH * 2 * T warp_sum() trees (120 shuffles at NH = 4, T = 3).
template <int T, int NH>
__global__ void __launch_bounds__(128, 1) conv_qkv_gates_pk_kernel(ConvQkvParams p) {
  constexpr int KS = 4, NV = NH * 2 * T;
  static_assert(NV <= 32, "one butterfly per warp");
  __shared__ float red[NV * 4];
  const int b = blockIdx.y;
  const int chunk = blockIdx.x;
  const int inner = p.inner;
  const int nblk = inner >> 2;
  const int blk_per_chunk = (nblk + p.NCH - 1) / p.NCH;
  const int j = chunk * blk_per_chunk + threadIdx.x;
  const bool active = threadIdx.x < blk_per_chunk && j < nblk;
  const int c = 4 * (active ? j : 0);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nw = (blockDim.x + 31) >> 5;

  // everything no kernel of the step writes: conv window, taps, headwise blocks, gate weights -- before the wait
  f32x2 win[KS][2], cwp[KS][2], cbp[2];
  f32x2 hq[4][2], hk[4][2], hv[4][2];                      // [dd][output pair]
  f32x2 gw[NH][3][4];                                     // (igate, fgate) weight of [head][q|k|v][channel]
  float* cs = p.conv_state + (int64_t)b * KS * inner + c;
  {
    float4 w4[4];
#pragma unroll
    for (int r = 0; r < KS; ++r) {
      const float4 x4 = *reinterpret_cast<const float4*>(cs + (int64_t)r * inner);
      win[r][0] = pk2(x4.x, x4.y);
      win[r][1] = pk2(x4.z, x4.w);
    }
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) w4[ch] = *reinterpret_cast<const float4*>(p.conv_w + (int64_t)(c + ch) * KS);
    cwp[0][0] = pk2(w4[0].x, w4[1].x); cwp[0][1] = pk2(w4[2].x, w4[3].x);
    cwp[1][0] = pk2(w4[0].y, w4[1].y); cwp[1][1] = pk2(w4[2].y, w4[3].y);
    cwp[2][0] = pk2(w4[0].z, w4[1].z); cwp[2][1] = pk2(w4[2].z, w4[3].z);
    cwp[3][0] = pk2(w4[0].w, w4[1].w); cwp[3][1] = pk2(w4[2].w, w4[3].w);
    const float4 cb = *reinterpret_cast<const float4*>(p.conv_b + c);
    cbp[0] = pk2(cb.x, cb.y);
    cbp[1] = pk2(cb.z, cb.w);
    // headwise block W[o][dd] at wq[16 j + 4 o + dd]: pairs over o for a fixed dd
    const float* bq = p.wq + (int64_t)(c >> 2) * 16;
    const float* bk = p.wk + (int64_t)(c >> 2) * 16;
    const float* bv = p.wv + (int64_t)(c >> 2) * 16;
    float4 rq[4], rk[4], rv[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      rq[o] = reinterpret_cast<const float4*>(bq)[o];
      rk[o] = reinterpret_cast<const float4*>(bk)[o];
      rv[o] = reinterpret_cast<const float4*>(bv)[o];
    }
#define XL_COL(r, dd) (dd == 0 ? r.x : dd == 1 ? r.y : dd == 2 ? r.z : r.w)
#pragma unroll
    for (int dd = 0; dd < 4; ++dd) {
      hq[dd][0] = pk2(XL_COL(rq[0], dd), XL_COL(rq[1], dd)); hq[dd][1] = pk2(XL_COL(rq[2], dd), XL_COL(rq[3], dd));
      hk[dd][0] = pk2(XL_COL(rk[0], dd), XL_COL(rk[1], dd)); hk[dd][1] = pk2(XL_COL(rk[2], dd), XL_COL(rk[3], dd));
      hv[dd][0] = pk2(XL_COL(rv[0], dd), XL_COL(rv[1], dd)); hv[dd][1] = pk2(XL_COL(rv[2], dd), XL_COL(rv[3], dd));
    }
#undef XL_COL
#pragma unroll
    for (int h = 0; h < NH; ++h)
#pragma unroll
      for (int part = 0; part < 3; ++part) {
        const float4 wi = *reinterpret_cast<const float4*>(p.wi + (int64_t)(h * 3 + part) * inner + c);
        const float4 wf = *reinterpret_cast<const float4*>(p.wf + (int64_t)(h * 3 + part) * inner + c);
        gw[h][part][0] = pk2(wi.x, wf.x); gw[h][part][1] = pk2(wi.y, wf.y);
        gw[h][part][2] = pk2(wi.z, wf.z); gw[h][part][3] = pk2(wi.w, wf.w);
      }
  }
  pdl_wait();
  pdl_trigger();

  float4 xm4[T];
  if (p.u_splits <= 1) {
#pragma unroll
    for (int t = 0; t < T; ++t) xm4[t] = *reinterpret_cast<const float4*>(p.u + ((int64_t)b * T + t) * 2 * inner + c);
  } else {
    // split-K planes of proj_up, added in plane order; planes 1 and 2 are requested together with plane 0 (a plain loop
    // is scheduled load -> add -> load: one L2 round trip per plane)
    float4 p1[T], p2[T];
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const float* up = p.u + ((int64_t)b * T + t) * 2 * inner + c;
      xm4[t] = *reinterpret_cast<const float4*>(up);
      p1[t] = *reinterpret_cast<const float4*>(up + p.u_stride);
      p2[t] = *reinterpret_cast<const float4*>(up + (p.u_splits > 2 ? 2 : 1) * p.u_stride);
    }
#pragma unroll
    for (int t = 0; t < T; ++t) {
      xm4[t].x += p1[t].x; xm4[t].y += p1[t].y; xm4[t].z += p1[t].z; xm4[t].w += p1[t].w;
      if (p.u_splits > 2) { xm4[t].x += p2[t].x; xm4[t].y += p2[t].y; xm4[t].z += p2[t].z; xm4[t].w += p2[t].w; }
      const float* up = p.u + ((int64_t)b * T + t) * 2 * inner + c;
      for (int z = 3; z < p.u_splits; ++z) {
        const float4 a4 = *reinterpret_cast<const float4*>(up + z * p.u_stride);
        xm4[t].x += a4.x; xm4[t].y += a4.y; xm4[t].z += a4.z; xm4[t].w += a4.w;
      }
    }
  }
  f32x2 G[NH][T];
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int64_t row = (int64_t)b * T + t;
    const f32x2 x01 = pk2(xm4[t].x, xm4[t].y), x23 = pk2(xm4[t].z, xm4[t].w);
    // roll(-1); state[-1] = x; conv over the window, oldest first (fma(w, c, 0) == w * c)
    win[0][0] = win[1][0]; win[0][1] = win[1][1];
    win[1][0] = win[2][0]; win[1][1] = win[2][1];
    win[2][0] = win[3][0]; win[2][1] = win[3][1];
    win[3][0] = x01;       win[3][1] = x23;
    f32x2 a01 = fma2(win[0][0], cwp[0][0], 0ull), a23 = fma2(win[0][1], cwp[0][1], 0ull);
#pragma unroll
    for (int r = 1; r < KS; ++r) {
      a01 = fma2(win[r][0], cwp[r][0], a01);
      a23 = fma2(win[r][1], cwp[r][1], a23);
    }
    a01 = add2(a01, cbp[0]);
    a23 = add2(a23, cbp[1]);
    float a[4];
    unpk2(a01, a[0], a[1]);
    unpk2(a23, a[2], a[3]);
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) a[ch] = silu(a[ch]);
    const float xm[4] = {xm4[t].x, xm4[t].y, xm4[t].z, xm4[t].w};
    f32x2 q01 = 0ull, q23 = 0ull, k01 = 0ull, k23 = 0ull, v01 = 0ull, v23 = 0ull;
#pragma unroll
    for (int dd = 0; dd < 4; ++dd) {
      q01 = fma2(bc2(a[dd]), hq[dd][0], q01);  q23 = fma2(bc2(a[dd]), hq[dd][1], q23);
      k01 = fma2(bc2(a[dd]), hk[dd][0], k01);  k23 = fma2(bc2(a[dd]), hk[dd][1], k23);
      v01 = fma2(bc2(xm[dd]), hv[dd][0], v01); v23 = fma2(bc2(xm[dd]), hv[dd][1], v23);
    }
    float q[4], k[4], v[4];
    unpk2(q01, q[0], q[1]); unpk2(q23, q[2], q[3]);
    unpk2(k01, k[0], k[1]); unpk2(k23, k[2], k[3]);
    unpk2(v01, v[0], v[1]); unpk2(v23, v[2], v[3]);
    if (active) {
      // channel c of head h sits at (row*NH + h)*DH + (c - h*DH) == row*inner + c: (q,k) pairs interleaved
      float* qk = p.qk + (row * inner + c) * 2;
      *reinterpret_cast<float4*>(qk) = make_float4(q[0], k[0], q[1], k[1]);
      *reinterpret_cast<float4*>(qk + 4) = make_float4(q[2], k[2], q[3], k[3]);
      *reinterpret_cast<float4*>(p.v + row * inner + c) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(p.act + row * inner + c) = make_float4(a[0], a[1], a[2], a[3]);
    }
    // partial (igate, fgate) pre-activations: x1 w1, then + x0 w0, + x2 w2, + x3 w3 per part; q-, k-, v-sums added in order
#pragma unroll
    for (int h = 0; h < NH; ++h) {
      f32x2 sq = mul2(bc2(q[1]), gw[h][0][1]);
      sq = fma2(bc2(q[0]), gw[h][0][0], sq);
      sq = fma2(bc2(q[2]), gw[h][0][2], sq);
      sq = fma2(bc2(q[3]), gw[h][0][3], sq);
      f32x2 sk = mul2(bc2(k[1]), gw[h][1][1]);
      sk = fma2(bc2(k[0]), gw[h][1][0], sk);
      sk = fma2(bc2(k[2]), gw[h][1][2], sk);
      sk = fma2(bc2(k[3]), gw[h][1][3], sk);
      f32x2 sv = mul2(bc2(v[1]), gw[h][2][1]);
      sv = fma2(bc2(v[0]), gw[h][2][0], sv);
      sv = fma2(bc2(v[2]), gw[h][2][2], sv);
      sv = fma2(bc2(v[3]), gw[h][2][3], sv);
      G[h][t] = active ? add2(add2(sq, sk), sv) : 0ull;
    }
  }
  if (active) {
    // write the window back: rows = last KS inputs, oldest first (reference conv_state layout)
#pragma unroll
    for (int r = 0; r < KS; ++r) {
      float4 w4;
      unpk2(win[r][0], w4.x, w4.y);
      unpk2(win[r][1], w4.z, w4.w);
      *reinterpret_cast<float4*>(cs + (int64_t)r * inner) = w4;
    }
  }
  // value index (h * 2 + gate) * T + t, padded with zeros to 32: lane l ends with the warp total of value l
  float vals[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) vals[i] = 0.f;
#pragma unroll
  for (int h = 0; h < NH; ++h)
#pragma unroll
    for (int t = 0; t < T; ++t) unpk2(G[h][t], vals[(h * 2 + 0) * T + t], vals[(h * 2 + 1) * T + t]);
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) {
    const bool upper = (lane & m) != 0;
#pragma unroll
    for (int i = 0; i < m; ++i) {
      const float keep = upper ? vals[i + m] : vals[i];
      const float send = upper ? vals[i] : vals[i + m];
      vals[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
    }
  }
  if (lane < NV) red[lane * 4 + wid] = vals[0];
  __syncthreads();
  if ((int)threadIdx.x < NV) {
    const int h = threadIdx.x / (2 * T);
    const int rem = threadIdx.x - h * 2 * T;
    const int g = rem / T, t = rem - g * T;
    float s = 0.f;
    for (int w = 0; w < nw; ++w) s += red[threadIdx.x * 4 + w];
    float* gp = p.gate_part + (((int64_t)b * T + t) * p.NCH + chunk) * 2 * NH;
    gp[g * NH + h] = s;
  }
}

bool launch_conv_qkv_gates(const ConvQkvParams& p, cudaStream_t s) {
  const int nblk = p.inner / 4;
  const int per_chunk = (nblk + p.NCH - 1) / p.NCH;
  const int threads = ((per_chunk + 31) / 32) * 32;   // one thread per 4-channel block; <= 128 (host-checked)
  dim3 grid(p.NCH, p.B);
  if (p.impl == 2 && p.KS == 4 && threads <= 128) {
#define XL_CONV_PK_CASE(TV, NHV) \
  if (p.T == TV && p.NH == NHV) { launch_k(conv_qkv_gates_pk_kernel<TV, NHV>, grid, dim3(threads), 0, s, p); return true; }
    XL_CONV_PK_CASE(1, 4) XL_CONV_PK_CASE(2, 4) XL_CONV_PK_CASE(3, 4) XL_CONV_PK_CASE(4, 4)
    XL_CONV_PK_CASE(1, 2) XL_CONV_PK_CASE(3, 2) XL_CONV_PK_CASE(1, 1) XL_CONV_PK_CASE(3, 1)
#undef XL_CONV_PK_CASE
  }
  if (p.impl == 1 && threads * p.T <= 512) {
#define XL_CONV_TOK_CASE(KSV, TV, NHV) \
  if (p.KS == KSV && p.T == TV && p.NH == NHV) { launch_k(conv_qkv_gates_tok_kernel<KSV, TV, NHV>, grid, dim3(threads * TV), 0, s, p); return true; }
    XL_CONV_TOK_CASE(4, 1, 4) XL_CONV_TOK_CASE(4, 2, 4) XL_CONV_TOK_CASE(4, 3, 4) XL_CONV_TOK_CASE(4, 4, 4)
    XL_CONV_TOK_CASE(4, 3, 8) XL_CONV_TOK_CASE(4, 3, 2) XL_CONV_TOK_CASE(4, 3, 1)
#undef XL_CONV_TOK_CASE
  }
  // instantiated for the shipped presets (KS = 4, NH = 4; 1..4 tokens per step) plus NH = 1, 2, 8
#define XL_CONV_CASE(KSV, TV, NHV) \
  if (p.KS == KSV && p.T == TV && p.NH == NHV) { launch_k(conv_qkv_gates_kernel<KSV, TV, NHV>, grid, dim3(threads), 0, s, p); return true; }
  XL_CONV_CASE(4, 1, 4) XL_CONV_CASE(4, 2, 4) XL_CONV_CASE(4, 3, 4) XL_CONV_CASE(4, 4, 4)
  XL_CONV_CASE(4, 1, 8) XL_CONV_CASE(4, 3, 8) XL_CONV_CASE(4, 1, 2) XL_CONV_CASE(4, 3, 2)
  XL_CONV_CASE(4, 1, 1) XL_CONV_CASE(4, 3, 1) XL_CONV_CASE(2, 1, 4) XL_CONV_CASE(2, 3, 4)
  XL_CONV_CASE(3, 1, 4) XL_CONV_CASE(3, 3, 4)
#undef XL_CONV_CASE
  return false;
}

// ------------------------------------------------------------------------------------------------
// argmax over action logits + MinMaxTokenizer.inv_tokenize
// (multi_domain_discrete_dt_model.py:83-94; src/tokenizers_custom/minmax_tokenizer.py:31-47).
// torch.argmax semantics: first index of the maximum; NaN counts as the maximum.
// one warp per (b, action dim).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) argmax_tokens_kernel(const float* __restrict__ logits,
                                                            int64_t row_pitch, int B, int act_dim,
                                                            int num_actions, int discrete_actions,
                                                            int discrete, float bin_width, float min_val,
                                                            int32_t* __restrict__ tokens,
                                                            float* __restrict__ actions,
                                                            int32_t* __restrict__ ring,
                                                            const unsigned* __restrict__ step_counter,
                                                            int ring_slots, int64_t ring_slot_stride) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int nrows = discrete ? B : B * act_dim;
  pdl_wait();
  pdl_trigger();
  if (w >= nrows) return;
  const int b = discrete ? w : w / act_dim;
  const int j = discrete ? 0 : w - b * act_dim;
  const float* lg = logits + (int64_t)b * row_pitch + (int64_t)j * num_actions;
  const int bi = warp_argmax(lg, discrete ? discrete_actions : num_actions, lane);
  if (lane == 0) {
    // token ring: the step's tokens also land in slot (step - 1) % slots of the caller's ring, from where the
    // multi-GPU result gather picks them up without a copy between graph replays
    if (ring) ring[(int64_t)((*step_counter - 1u) % (unsigned)ring_slots) * ring_slot_stride + (int64_t)b * act_dim + j] = bi;
    if (discrete) {
      tokens[(int64_t)b * act_dim] = bi;
      actions[(int64_t)b * act_dim] = (float)bi;
    } else {
      tokens[(int64_t)b * act_dim + j] = bi;
      int t = bi - discrete_actions;
      if (t < 0) t = 0;
      actions[(int64_t)b * act_dim + j] = (float)t * bin_width + min_val;
    }
  }
}

void launch_argmax_tokens(const float* logits, int64_t row_pitch, int B, int act_dim, int num_actions,
                          int discrete_actions, int discrete, float bin_width, float min_val,
                          int32_t* tokens, float* actions, int32_t* ring, const unsigned* step_counter,
                          int ring_slots, int64_t ring_slot_stride, cudaStream_t s) {
  const int rows = discrete ? B : B * act_dim;
  dim3 grid((rows + 7) / 8);
  launch_k(argmax_tokens_kernel, grid, dim3(256), 0, s, logits, row_pitch, B, act_dim, num_actions,
           discrete_actions, discrete, bin_width, min_val, tokens, actions, ring, step_counter, ring_slots,
           ring_slot_stride);
}

__global__ void set_u32_kernel(unsigned* p, unsigned v) { *p = v; }
void launch_set_u32(unsigned* p, unsigned v, cudaStream_t s) { set_u32_kernel<<<1, 1, 0, s>>>(p, v); }

// ------------------------------------------------------------------------------------------------
// per-env state reset (past_key_values = None for the masked envs; evaluation.py:124,251,261)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) state_reset_kernel(float* C, float* n, float* m, float* conv,
                                                          const uint8_t* __restrict__ mask, int B,
                                                          int64_t c_per_env, int64_t n_per_env,
                                                          int64_t m_per_env, int64_t conv_per_env) {
  const int b = blockIdx.y;
  pdl_wait();
  pdl_trigger();
  if (mask && mask[b] == 0) return;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float4* c4 = reinterpret_cast<float4*>(C + (int64_t)b * c_per_env);
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t i = t0; i < c_per_env / 4; i += stride) c4[i] = z;
  for (int64_t i = t0; i < n_per_env; i += stride) n[(int64_t)b * n_per_env + i] = 0.f;
  for (int64_t i = t0; i < m_per_env; i += stride) m[(int64_t)b * m_per_env + i] = 0.f;
  for (int64_t i = t0; i < conv_per_env; i += stride) conv[(int64_t)b * conv_per_env + i] = 0.f;
}

void launch_state_reset(float* C, float* n, float* m, float* conv, const uint8_t* mask, int B,
                        int64_t c_per_env, int64_t n_per_env, int64_t m_per_env, int64_t conv_per_env,
                        cudaStream_t s) {
  dim3 grid(32, B);
  state_reset_kernel<<<grid, 256, 0, s>>>(C, n, m, conv, mask, B, c_per_env, n_per_env, m_per_env,
                                          conv_per_env);
}

// ---- ragged prefill: env permutation of the state and chunk rows ----------------------------------------
// grid = (CTAs per env, Bc compact envs, blocks). Every part is env-major with a fixed per-env size, so one part of one
// env is a contiguous run of bytes on both sides; runs whose size is a multiple of 16 B (all but m when NH < 4) go as
// 128-bit words. HBM-bound.
__device__ __forceinline__ void copy_run(const char* __restrict__ src, char* __restrict__ dst, size_t bytes, int64_t t0,
                                         int64_t stride) {
  if (bytes % 16 == 0) {
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    for (int64_t i = t0; i < (int64_t)(bytes / 16); i += stride) d4[i] = s4[i];
  } else {
    const float* s1 = reinterpret_cast<const float*>(src);
    float* d1 = reinterpret_cast<float*>(dst);
    for (int64_t i = t0; i < (int64_t)(bytes / 4); i += stride) d1[i] = s1[i];
  }
}

__global__ void __launch_bounds__(256) state_permute_kernel(char* caller, char* compact, const int32_t* __restrict__ perm,
                                                            StateCopyGeom g, int to_caller) {
  const int k = blockIdx.y, blk = blockIdx.z;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  pdl_wait();
  pdl_trigger();
  const int env[2] = {perm[k], k};
  const uint64_t below = blk >= 64 ? ~0ull : ((1ull << blk) - 1ull);
  const int ns = __popcll(g.slstm_mask & below);
  char* base[2];
#pragma unroll
  for (int j = 0; j < 2; ++j)
    base[j] = (j ? compact : caller) + (size_t)(blk - ns) * g.layer_bytes[j] + (size_t)ns * g.slayer_bytes[j];
  const int from = to_caller ? 1 : 0, to = 1 - from;
  auto run = [&](const size_t* off, size_t env_bytes, size_t plane) {
    // plane: bytes between the planes of one part per env of the batch (sLSTM (y, c, n, m)); 0 = one plane
    for (int p = 0; p < (plane ? 4 : 1); ++p)
      copy_run(base[from] + off[from] + p * plane * g.B[from] + env[from] * env_bytes,
               base[to] + off[to] + p * plane * g.B[to] + env[to] * env_bytes, env_bytes, t0, stride);
  };
  if ((g.slstm_mask >> blk) & 1ull) {
    run(g.s_off, g.s_env, g.s_env);
    run(g.sconv_off, g.sconv_env, 0);
  } else {
    run(g.c_off, g.c_env, 0);
    run(g.n_off, g.n_env, 0);
    run(g.m_off, g.m_env, 0);
    run(g.conv_off, g.conv_env, 0);
  }
}

void launch_state_permute(void* caller, void* compact, const int32_t* perm, int Bc, const StateCopyGeom& g,
                          int to_caller, cudaStream_t s) {
  // ~8 KiB of C per thread row of a CTA: enough CTAs in flight for HBM at a few envs, no more than 64 per (env, block)
  const size_t words = std::max(g.c_env, g.s_env * 4) / 16;
  const unsigned per = (unsigned)std::min<size_t>(64, std::max<size_t>(1, words / (256 * 32)));
  launch_k(state_permute_kernel, dim3(per, Bc, g.num_blocks), dim3(256), 0, s, (char*)caller, (char*)compact, perm, g,
           to_caller);
}

__global__ void __launch_bounds__(256) ragged_rows_kernel(float* caller, float* compact, const int32_t* __restrict__ perm,
                                                          const int32_t* __restrict__ len, int len_div, int S, int Sc,
                                                          int pos, int width, int to_caller) {
  const int k = blockIdx.y;
  pdl_wait();
  pdl_trigger();
  const int nk = min(max(len[k] / len_div - pos, 0), Sc);
  const int rows = to_caller ? nk : Sc;                       // the scatter writes valid rows only
  float* crow = compact + (int64_t)k * Sc * width;
  float* urow = caller + ((int64_t)perm[k] * S + pos) * width;
  const int64_t n = (int64_t)rows * width, valid = (int64_t)nk * width;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  if (width % 4 == 0) {
    for (int64_t i = t0; i < n / 4; i += stride) {
      if (to_caller) reinterpret_cast<float4*>(urow)[i] = reinterpret_cast<const float4*>(crow)[i];
      else reinterpret_cast<float4*>(crow)[i] = 4 * i < valid ? reinterpret_cast<const float4*>(urow)[i]
                                                              : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  } else {
    for (int64_t i = t0; i < n; i += stride) {
      if (to_caller) urow[i] = crow[i];
      else crow[i] = i < valid ? urow[i] : 0.f;
    }
  }
}

void launch_ragged_rows(float* caller, float* compact, const int32_t* perm, const int32_t* len, int len_div, int Bk,
                        int S, int Sc, int pos, int width, int to_caller, cudaStream_t s) {
  const int64_t words = ((int64_t)Sc * width + 3) / 4;
  const unsigned per = (unsigned)std::min<int64_t>(64, std::max<int64_t>(1, (words + 255) / 256));
  launch_k(ragged_rows_kernel, dim3(per, Bk), dim3(256), 0, s, caller, compact, perm, len, len_div, S, Sc, pos, width,
           to_caller);
}


// ---- L2 warm-up of the next block's matrix memory --------------------------------------------------
// Runs on a side stream while the latency-bound chain (finalize / proj_down / LN / proj_up / conv) of the
// current block leaves HBM idle: bulk L2 prefetches of the first `bytes` of the next block's C, so that the
// next state-stream launch finds part of its read stream in L2. Reads only; no ordering needed against it.
__global__ void l2_prefetch_kernel(const char* base, unsigned long long bytes, unsigned chunk, int evict_last) {
  const unsigned long long nchunks = (bytes + chunk - 1) / chunk;
  unsigned long long policy = 0;
  if (evict_last) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(policy));
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < nchunks;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long off = i * chunk;
    const unsigned sz = (unsigned)((bytes - off) < chunk ? (bytes - off) : chunk) & ~15u;
    if (!sz) continue;
    if (evict_last)   // keep the warmed lines resident until the state stream consumes them (its loads are evict_first)
      asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(base + off), "r"(sz), "l"(policy)
                   : "memory");
    else
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(base + off), "r"(sz) : "memory");
  }
}

void launch_l2_prefetch(const void* base, size_t bytes, int num_sms, int evict_last, cudaStream_t s) {
  if (!bytes) return;
  const unsigned chunk = 4096;
  l2_prefetch_kernel<<<num_sms, 64, 0, s>>>((const char*)base, (unsigned long long)bytes, chunk, evict_last);
}

}  // namespace xl
