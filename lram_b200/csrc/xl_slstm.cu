// sLSTM block step for xLSTM[a:b] stacks (xlstm_config.slstm_at, xlstm_ms_mediumplus.yaml:27).
// Replaces, for the recurrent inference path, what the reference gets from the third-party xlstm package's
// sLSTMLayer.step + its JIT-compiled sLSTM CUDA extension (src/algos/models/decision_xlstm.py:29-101 baby-sits
// that extension for pickling) and GatedFeedForward. The recurrent state is tiny ((y,c,n,m) [4,B,d] + the conv
// window), so nothing here is HBM-bound: the kernels are sized for latency (weights stream from L2).
//
// Row order everywhere: row = env * T + token (the fused step's [b][t] order). Tokens of one env are sequential
// through the recurrent term R y_{t-1}; everything else is token-parallel.
#include "xl_common.cuh"
#include "xl_internal.h"

namespace xl {

// ---- causal conv step over the T tokens of an env + swish ------------------------------------------
// conv_state [B,KS,d] oldest first (CausalConv1d.step: roll(-1), append, sum_k state[k]*w[c,k] + b).
template <int KS>
__global__ void slstm_conv_kernel(const float* __restrict__ xn, float* __restrict__ conv_state,
                                  const float* __restrict__ cw, const float* __restrict__ cb,
                                  float* __restrict__ xc, int B, int T, int d, const int32_t* __restrict__ len,
                                  int pos) {
  pdl_wait();
  pdl_trigger();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (c >= d) return;
  float w[KS], win[KS];
#pragma unroll
  for (int k = 0; k < KS; ++k) {
    w[k] = cw[(size_t)c * KS + k];
    win[k] = conv_state[((size_t)b * KS + k) * d + c];
  }
  const float bias = cb[c];
  const int nb = len ? min(max(len[b] - pos, 0), T) : T;   // ragged prefill: tokens t >= nb are pads (window kept)
  for (int t = nb; t < T; ++t) xc[((size_t)b * T + t) * d + c] = 0.f;
  for (int t = 0; t < nb; ++t) {
#pragma unroll
    for (int k = 0; k + 1 < KS; ++k) win[k] = win[k + 1];
    win[KS - 1] = xn[((size_t)b * T + t) * d + c];
    float y = 0.f;
#pragma unroll
    for (int k = 0; k < KS; ++k) y += win[k] * w[k];     // same left-to-right order as torch.sum over dim 1
    y += bias;
    xc[((size_t)b * T + t) * d + c] = silu(y);
  }
#pragma unroll
  for (int k = 0; k < KS; ++k) conv_state[((size_t)b * KS + k) * d + c] = win[k];
}

bool launch_slstm_conv(const float* xn, float* conv_state, const float* cw, const float* cb, float* xc, int B,
                       int T, int d, int KS, cudaStream_t s, const int32_t* len, int pos) {
  dim3 grid((d + 127) / 128, B), block(128);
  switch (KS) {
    case 2: launch_k(slstm_conv_kernel<2>, grid, block, 0, s, xn, conv_state, cw, cb, xc, B, T, d, len, pos); break;
    case 3: launch_k(slstm_conv_kernel<3>, grid, block, 0, s, xn, conv_state, cw, cb, xc, B, T, d, len, pos); break;
    case 4: launch_k(slstm_conv_kernel<4>, grid, block, 0, s, xn, conv_state, cw, cb, xc, B, T, d, len, pos); break;
    default: return false;
  }
  return true;
}

// ---- the four headwise (block-diagonal) gate projections --------------------------------------------
// pre[m, g, h*DH + o] = bias[h, g, o] + sum_k in_g[m, h*DH + k] * W_g[h, o, k]
// in_g = xc (conv branch) for g = 0 (i), 1 (f); xn for g = 2 (z), 3 (o). fp32 FMA, 64x64 tile, 4x4 per thread.
constexpr int kGT = 64, kGK = 16;
__global__ void __launch_bounds__(256) slstm_gates_kernel(const float* __restrict__ xc, const float* __restrict__ xn,
                                                          const float* __restrict__ w_i, const float* __restrict__ w_f,
                                                          const float* __restrict__ w_z, const float* __restrict__ w_o,
                                                          const float* __restrict__ bias, float* __restrict__ pre,
                                                          int M, int d, int NH, int DH) {
  __shared__ float sA[kGK][kGT + 1];
  __shared__ float sW[kGK][kGT + 1];
  const int g = blockIdx.z / NH, h = blockIdx.z % NH;
  const int m0 = blockIdx.x * kGT, o0 = blockIdx.y * kGT;
  const float* W = (g == 0 ? w_i : g == 1 ? w_f : g == 2 ? w_z : w_o) + (size_t)h * DH * DH;
  const float* A = (g < 2 ? xc : xn) + (size_t)h * DH;
  const int tid = threadIdx.x;
  const int tm = (tid / 16) * 4, to = (tid % 16) * 4;
  float acc[4][4] = {};
  pdl_wait();
  pdl_trigger();
  for (int k0 = 0; k0 < DH; k0 += kGK) {
    // 64 x 16 tiles of A (rows m) and W (rows o): thread loads 4 elements of each
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int idx = tid + r * 256;          // 0..1023
      const int row = idx / kGK, kk = idx % kGK;
      const int k = k0 + kk;
      sA[kk][row] = (m0 + row < M && k < DH) ? A[(size_t)(m0 + row) * d + k] : 0.f;
      sW[kk][row] = (o0 + row < DH && k < DH) ? W[(size_t)(o0 + row) * DH + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kGK; ++kk) {
      float a[4], w[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) { a[j] = sA[kk][tm + j]; w[j] = sW[kk][to + j]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] += a[i] * w[j];
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + tm + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int o = o0 + to + j;
      if (o < DH) pre[((size_t)m * 4 + g) * d + h * DH + o] = acc[i][j] + bias[((size_t)h * 4 + g) * DH + o];
    }
  }
}

void launch_slstm_gates(const float* xc, const float* xn, const float* w_i, const float* w_f, const float* w_z,
                        const float* w_o, const float* bias, float* pre, int M, int d, int NH, cudaStream_t s) {
  const int DH = d / NH;
  dim3 grid((M + kGT - 1) / kGT, (DH + kGT - 1) / kGT, 4 * NH);
  launch_k(slstm_gates_kernel, grid, dim3(256), 0, s, xc, xn, w_i, w_f, w_z, w_o, bias, pre, M, d, NH, DH);
}

// ---- one token of the sLSTM cell: raw = pre + R y_{t-1}; pointwise update --------------------------
// CTA = (32 outputs of one head) x (8 envs); 256 threads = 32 outputs x 8 slices of the reduction dim.
// R [NH, DH(in), 4, DH(out)]: for fixed (head, in) the 4 x DH outputs are contiguous -> each warp reads 128
// contiguous bytes per (in, gate). y_{t-1} comes from the state (t == 0) or from the previous token's output row;
// the new y only goes to y_out (the state's y is written by slstm_out_kernel after the last token), so CTAs of the
// same launch never read what another one writes.
constexpr int kCO = 32, kCE = 8, kCS = 8;
__global__ void __launch_bounds__(256) slstm_cell_kernel(const float* __restrict__ pre, const float* __restrict__ R,
                                                         float* __restrict__ st, float* __restrict__ y_out,
                                                         int B, int stB, int T, int t, int d, int NH, int DH,
                                                         const int32_t* __restrict__ len, int pos) {
  extern __shared__ float smem[];
  float* sy = smem;                         // [kCE][DH]
  float* red = smem + kCE * DH;             // [kCS][kCE][4][kCO]
  const int o0 = blockIdx.x * kCO, h = blockIdx.y, b0 = blockIdx.z * kCE;
  const int tid = threadIdx.x, o = tid % kCO, ds = tid / kCO;
  const size_t Bd = (size_t)stB * d;      // the state holds stB envs per part; st points at this slice's env 0
  pdl_wait();
  pdl_trigger();
  for (int idx = tid; idx < kCE * DH; idx += 256) {
    const int e = idx / DH, k = idx % DH, b = b0 + e;
    float v = 0.f;
    if (b < B) v = (t == 0) ? st[(size_t)b * d + h * DH + k] : y_out[((size_t)b * T + t - 1) * d + h * DH + k];
    sy[idx] = v;
  }
  __syncthreads();
  float acc[kCE][4];
#pragma unroll
  for (int e = 0; e < kCE; ++e) acc[e][0] = acc[e][1] = acc[e][2] = acc[e][3] = 0.f;
  const int per = (DH + kCS - 1) / kCS;
  const int k_lo = ds * per, k_hi = min(DH, k_lo + per);
  const bool o_ok = (o0 + o) < DH;
  const float* Rp = R + (size_t)h * DH * 4 * DH + o0 + o;
  if (o_ok) {
#pragma unroll 4
    for (int k = k_lo; k < k_hi; ++k) {
      const float* rk = Rp + (size_t)k * 4 * DH;
      const float r0 = __ldg(rk), r1 = __ldg(rk + DH), r2 = __ldg(rk + 2 * DH), r3 = __ldg(rk + 3 * DH);
#pragma unroll
      for (int e = 0; e < kCE; ++e) {
        const float yv = sy[e * DH + k];
        acc[e][0] += yv * r0; acc[e][1] += yv * r1; acc[e][2] += yv * r2; acc[e][3] += yv * r3;
      }
    }
  }
#pragma unroll
  for (int e = 0; e < kCE; ++e)
#pragma unroll
    for (int g = 0; g < 4; ++g) red[((ds * kCE + e) * 4 + g) * kCO + o] = acc[e][g];
  __syncthreads();
  // thread (e = ds, o): fixed-order sum over the 8 slices, then the pointwise update of element (b, h*DH + o0 + o)
  const int e = ds, b = b0 + e;
  if (b >= B || !o_ok) return;
  const int ch = h * DH + o0 + o;
  if (len && t >= len[b] - pos) {               // ragged prefill pad: state kept, y_{t-1} carried forward
    y_out[((size_t)b * T + t) * d + ch] = sy[e * DH + o0 + o];
    return;
  }
  float raw[4];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < kCS; ++q) s += red[((q * kCE + e) * 4 + g) * kCO + o];
    raw[g] = pre[(((size_t)b * T + t) * 4 + g) * d + ch] + s;
  }
  const size_t si = (size_t)b * d + ch;
  const float c = st[Bd + si], n = st[2 * Bd + si], m = st[3 * Bd + si];
  const float logfplusm = m + log_sigmoid(raw[1]);
  const float mnew = (n == 0.f) ? raw[0] : fmaxf(raw[0], logfplusm);
  const float og = 1.f / (1.f + expf(-raw[3]));
  const float ig = fminf(expf(raw[0] - mnew), 1.f);
  const float fg = fminf(expf(logfplusm - mnew), 1.f);
  const float cnew = fg * c + ig * tanhf(raw[2]);
  const float nnew = fg * n + ig;
  const float ynew = og * cnew / nnew;
  st[Bd + si] = cnew;
  st[2 * Bd + si] = nnew;
  st[3 * Bd + si] = mnew;
  y_out[((size_t)b * T + t) * d + ch] = ynew;
}

cudaError_t launch_slstm_cell(const float* pre, const float* R, float* st, float* y_out, int B, int stB, int T, int t,
                              int d, int NH, cudaStream_t s, const int32_t* len, int pos) {
  const int DH = d / NH;
  const size_t smem = sizeof(float) * ((size_t)kCE * DH + (size_t)kCS * kCE * 4 * kCO);
  if (cudaError_t e = ensure_dyn_smem<&slstm_cell_kernel>(smem); e != cudaSuccess) return e;
  dim3 grid((DH + kCO - 1) / kCO, NH, (B + kCE - 1) / kCE);
  return launch_k(slstm_cell_kernel, grid, dim3(256), smem, s, pre, R, st, y_out, B, stB, T, t, d, NH, DH, len, pos);
}

// ---- MultiHeadLayerNorm(y) -> residual add; carries y of the last token into the state -----------
// One CTA per row, one warp per head. x += GN_h(y) * (1 + w). part/splits: split-K planes of a preceding
// mLSTM proj_down that are still to be folded into x are NOT handled here (the block's first LayerNorm did).
__global__ void slstm_out_kernel(const float* __restrict__ y_out, const float* __restrict__ gn_w, float* __restrict__ x,
                                 float* __restrict__ st_y, int T, int d, int NH, int DH, float eps) {
  const int m = blockIdx.x, h = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  if (h >= NH) return;
  const float* yr = y_out + (size_t)m * d + h * DH;
  float s = 0.f;
  for (int k = lane; k < DH; k += 32) s += yr[k];
  const float mean = warp_sum(s) / (float)DH;
  float v = 0.f;
  for (int k = lane; k < DH; k += 32) { const float dlt = yr[k] - mean; v += dlt * dlt; }
  const float rstd = rsqrtf(warp_sum(v) / (float)DH + eps);
  const int b = m / T, t = m % T;
  for (int k = lane; k < DH; k += 32) {
    const int ch = h * DH + k;
    const float yv = yr[k];
    x[(size_t)m * d + ch] += (yv - mean) * rstd * (1.f + gn_w[ch]);
    if (t == T - 1) st_y[(size_t)b * d + ch] = yv;
  }
}

void launch_slstm_out(const float* y_out, const float* gn_w, float* x, float* st_y, int M, int T, int d, int NH,
                      float eps, cudaStream_t s) {
  launch_k(slstm_out_kernel, dim3(M), dim3(32 * NH), 0, s, y_out, gn_w, x, st_y, T, d, NH, d / NH, eps);
}

// ---- gated feed-forward middle: g = gelu(up[:, :ff]) * up[:, ff:] (exact erf GELU) ------------------
__global__ void ffn_gate_kernel(const float* __restrict__ up, float* __restrict__ out, __nv_bfloat16* __restrict__ hi,
                                __nv_bfloat16* __restrict__ lo, int M, int ff) {
  pdl_wait();
  pdl_trigger();
  const size_t n = (size_t)M * ff;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t m = i / ff, j = i % ff;
    const float a = up[m * 2 * ff + j], b = up[m * 2 * ff + ff + j];
    const float g = 0.5f * a * (1.f + erff(a * 0.70710678118654752440f)) * b;
    if (out) out[i] = g;
    if (hi) {
      const __nv_bfloat16 h16 = __float2bfloat16_rn(g);
      hi[i] = h16;
      lo[i] = __float2bfloat16_rn(g - __bfloat162float(h16));
    }
  }
}

void launch_ffn_gate(const float* up, float* out, void* hi, void* lo, int M, int ff, cudaStream_t s) {
  const size_t n = (size_t)M * ff;
  int blocks = (int)((n + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  launch_k(ffn_gate_kernel, dim3(blocks), dim3(256), 0, s, up, out, (__nv_bfloat16*)hi, (__nv_bfloat16*)lo, M, ff);
}

}  // namespace xl
