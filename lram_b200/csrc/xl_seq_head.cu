// Per-timestep head reduction of the sequence forward (xl_policy_forward): from the logits of a chunk's timesteps to
// tokens, actions and log-probabilities at their [B, Tn, ...] positions, in one launch per chunk.
// Token rule: warp_argmax, shared with the step's argmax kernel and the sampler's fallback, so a row yields the token the
// step would take from the same logits. Action decode: MinMaxTokenizer.inv_tokenize as argmax_tokens_kernel does it.
#include <cuda_runtime.h>

#include "xl_common.cuh"
#include "xl_internal.h"

namespace xl {

// One warp per (chunk row, action row j). Chunk row r is timestep tt = r % Tc of compact env k = r / Tc; it lands at
// timestep t = pos + tt of env b = perm ? perm[k] : k. With len (ragged), rows with t >= len[k] / len_div are pads of
// the chunk and write nothing. Discrete: row j = 0 reads the env's num_actions logits; j >= 1 write -1 / 0 / 0.
__global__ void __launch_bounds__(256) seq_head_kernel(SeqHeadParams p) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  pdl_wait();
  pdl_trigger();
  if (w >= (int64_t)p.rows * p.act_dim) return;
  const int r = (int)(w / p.act_dim), j = (int)(w - (int64_t)r * p.act_dim);
  const int k = r / p.Tc, t = p.pos + (r - k * p.Tc);
  if (p.len && t >= p.len[k] / p.len_div) return;
  const int b = p.perm ? p.perm[k] : k;
  const int64_t o = ((int64_t)b * p.Tn + t) * p.act_dim + j;     // [B, Tn, act_dim] position
  if (p.discrete && j > 0) {
    if (lane == 0) {
      if (p.tokens) p.tokens[o] = -1;
      if (p.actions) p.actions[o] = 0.f;
      if (p.logprobs) p.logprobs[o] = 0.f;
    }
    return;
  }
  const int n = p.num_actions;
  const float* lg = p.logits + (int64_t)r * p.n_out + (int64_t)j * n;
  // pass 1 (from L2): the row's copy to [B, Tn, n_out] and the lane maxima of the log-sum-exp; passes 2 and 3 (the argmax
  // and the exp sum) re-read the row from L1
  float* dst = p.out_logits ? p.out_logits + ((int64_t)b * p.Tn + t) * p.n_out + (int64_t)j * n : nullptr;
  float mx = -INFINITY;
  if (dst || p.logprobs) {
    for (int i = lane; i < n; i += 32) {
      const float v = lg[i];
      if (dst) dst[i] = v;
      mx = fmaxf(mx, v);
    }
  }
  if (p.tokens || p.actions) {
    const int bi = warp_argmax(lg, p.discrete ? p.discrete_actions : n, lane);
    if (lane == 0) {
      if (p.tokens) p.tokens[o] = bi;
      if (p.actions) {
        if (p.discrete) {
          p.actions[o] = (float)bi;
        } else {
          int tk = bi - p.discrete_actions;
          if (tk < 0) tk = 0;
          p.actions[o] = (float)tk * p.bin_width + p.min_val;
        }
      }
    }
  }
  if (p.logprobs) {
    // log_softmax at the target: (l[tgt] - max) - log(sum exp(l - max)), fp32, warp-shuffle reductions
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, s));
    float se = 0.f;
    for (int i = lane; i < n; i += 32) se += expf(lg[i] - mx);
    se = warp_sum(se);
    if (lane == 0) {
      const int tg = p.targets[o];
      float lp;
      if (tg < 0) lp = 0.f;
      else if (tg >= n) lp = __int_as_float(0x7fc00000);   // NaN
      else lp = (lg[tg] - mx) - logf(se);
      p.logprobs[o] = lp;
    }
  }
}

void launch_seq_head(const SeqHeadParams& p, cudaStream_t s) {
  if (p.rows <= 0) return;
  const int64_t warps = (int64_t)p.rows * p.act_dim;
  launch_k(seq_head_kernel, dim3((unsigned)((warps + 7) / 8)), dim3(256), 0, s, p);
}

}  // namespace xl
