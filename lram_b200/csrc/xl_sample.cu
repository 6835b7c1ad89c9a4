// Stochastic action selection on the device: `a_sample_kwargs` / sample_from_logits
// (src/algos/models/model_utils.py:7-32) for each env's own logit block, with a counter-based Philox4x32-10 draw in
// place of torch's global RNG. The contract (quantile cut, top-k, fp64 softmax, draw, fallbacks) is written down at
// xl_set_sampling in include/xlstm_b200.h; tests/test_gpu_sampling.py restates it on the host.
//
// One CTA per env, one warp per action row (1 row discrete, act_dim rows continuous). A row of <= 512 logits is
// sorted in registers (bitonic, 16 values per lane) for the order statistics the quantile and top-k need; the
// candidate set, the weights and the index-order prefix sums are then formed on the row as loaded (lane l holds
// indices 32c + l). The fp32 logits are exact in fp64, so the order statistics are taken on the fp32 values; the
// quantile, the weights and the sums are fp64.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/xlstm_b200.h"
#include "xl_common.cuh"
#include "xl_internal.h"

namespace xl {
namespace {

constexpr int kChunks = kSampleMaxActions / 32;   // row values per lane

// Philox4x32-10 (Salmon et al., SC'11; Random123's philox4x32_R(10, ...)): the key is bumped before rounds 2..10.
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    const uint32_t lo0 = 0xD2511F53u * c[0], hi0 = __umulhi(0xD2511F53u, c[0]);
    const uint32_t lo1 = 0xCD9E8D57u * c[2], hi1 = __umulhi(0xCD9E8D57u, c[2]);
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
  }
}

// Ascending bitonic sort of the warp's 512 values; element e = lane * 16 + r lives in v[r] of lane `lane`.
__device__ __forceinline__ void warp_sort512(float (&v)[kChunks], int lane) {
#pragma unroll
  for (int lk = 1; lk <= 9; ++lk) {
    const int k = 1 << lk;
#pragma unroll
    for (int lj = lk - 1; lj >= 0; --lj) {
      const int j = 1 << lj;
      if (j >= kChunks) {                         // partner in lane ^ (j / 16), same register
        const int lm = j / kChunks;
        const bool keep_min = ((lane & (k / kChunks)) == 0) != ((lane & lm) != 0);
#pragma unroll
        for (int r = 0; r < kChunks; ++r) {
          const float o = __shfl_xor_sync(0xffffffffu, v[r], lm);
          v[r] = keep_min ? fminf(v[r], o) : fmaxf(v[r], o);
        }
      } else {                                    // partner in register r ^ j of the same lane
#pragma unroll
        for (int r = 0; r < kChunks; ++r) {
          if (r & j) continue;
          const int p = r | j;
          const bool asc = k >= kChunks ? (lane & (k / kChunks)) == 0 : (r & k) == 0;
          const float a = fminf(v[r], v[p]), b = fmaxf(v[r], v[p]);
          v[r] = asc ? a : b;
          v[p] = asc ? b : a;
        }
      }
    }
  }
}

// sorted[p] (warp-uniform p) of a warp_sort512 result, in every lane
__device__ __forceinline__ float sorted_at(const float (&v)[kChunks], int p) {
  float x = 0.f;
#pragma unroll
  for (int r = 0; r < kChunks; ++r)
    if (r == (p & (kChunks - 1))) x = v[r];
  return __shfl_sync(0xffffffffu, x, p / kChunks);
}

__device__ __forceinline__ int warp_count(bool pred) { return __popc(__ballot_sync(0xffffffffu, pred)); }

__global__ void __launch_bounds__(32 * kSampleMaxRows) sample_tokens_kernel(
    const float* __restrict__ logits, int64_t row_pitch, int act_dim, int num_actions, int discrete_actions,
    int discrete, float bin_width, float min_val, int32_t* __restrict__ tokens, float* __restrict__ actions,
    int32_t* __restrict__ ring, const unsigned* __restrict__ ring_counter, int ring_slots, int64_t ring_slot_stride,
    const xl_sampling* __restrict__ prm, const unsigned* __restrict__ step_counter) {
  __shared__ double s_pct[kSampleMaxRows];
  __shared__ float s_max[kSampleMaxRows];
  __shared__ int s_nan[kSampleMaxRows];
  const int b = blockIdx.x, j = threadIdx.x >> 5, lane = threadIdx.x & 31, R = blockDim.x >> 5;
  const int n = num_actions;
  const float* lg = logits + (int64_t)b * row_pitch + (int64_t)j * num_actions;
  pdl_wait();
  pdl_trigger();
  const xl_sampling p = *prm;
  const bool use_p = p.top_p > 0.f, use_k = p.top_k > 0;

  // ---- phase 1: the row, its max, its quantile and its k-th largest value --------------------------------------
  float x[kChunks];
  bool has_nan = false;
  float mx = -INFINITY;
#pragma unroll
  for (int c = 0; c < kChunks; ++c) {
    const int i = 32 * c + lane;
    x[c] = i < n ? lg[i] : -INFINITY;
    has_nan |= x[c] != x[c];
    mx = fmaxf(mx, x[c]);
  }
  const bool row_nan = __any_sync(0xffffffffu, has_nan);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  double pct = 0.0;     // torch.quantile(row, top_p)
  float t_k = 0.f;      // n-k th order statistic = k-th largest value of the row
  if ((use_p || use_k) && !row_nan) {
    float v[kChunks];
#pragma unroll
    for (int c = 0; c < kChunks; ++c) v[c] = 32 * c + lane < n ? x[c] : INFINITY;   // padding sorts to the top
    warp_sort512(v, lane);
    if (use_p) {
      const double rank = (double)p.top_p * (double)(n - 1);
      const int lo = (int)floor(rank), hi = (int)ceil(rank);
      const double w = rank - (double)lo;
      const double a = sorted_at(v, lo), e = sorted_at(v, hi);
      // torch.lerp, unfused
      pct = w < 0.5 ? __dadd_rn(a, __dmul_rn(w, __dsub_rn(e, a))) : __dsub_rn(e, __dmul_rn(__dsub_rn(e, a), 1.0 - w));
    }
    if (use_k) t_k = sorted_at(v, n - p.top_k);
  }
  if (lane == 0) { s_pct[j] = pct; s_max[j] = mx; s_nan[j] = row_nan; }
  __syncthreads();

  // ---- phase 2: env-wide guard, candidates, weights, draw ------------------------------------------------------
  // the reference cuts only when (percentile != logits.max()).all() over the env's whole block; a NaN makes the
  // block max NaN, and nothing compares equal to it
  bool cut = use_p;
  if (cut) {
    bool any_nan = false;
    float bmax = -INFINITY;
    for (int r = 0; r < R; ++r) { any_nan |= s_nan[r] != 0; bmax = fmaxf(bmax, s_max[r]); }
    if (!any_nan)
      for (int r = 0; r < R; ++r) cut &= s_pct[r] != (double)bmax;
  }
  bool surv[kChunks];
  int S = 0;
#pragma unroll
  for (int c = 0; c < kChunks; ++c) {
    surv[c] = 32 * c + lane < n && (!cut || (double)x[c] > pct);
    S += warp_count(surv[c]);
  }
  int tok = -1;
  // NaN, nothing left after the cut, or no finite maximum: the reference's Categorical would raise; take the argmax
  const bool fallback = row_nan || S == 0 || !isfinite(mx);
  if (!fallback) {
    // top-k of the cut row: the survivors are its S largest values, so for k < S the k-th largest survivor is t_k;
    // among values equal to t_k the lowest indices fill the remaining places
    bool cand[kChunks];
    if (use_k && p.top_k < S) {
      int G = 0;
#pragma unroll
      for (int c = 0; c < kChunks; ++c) G += warp_count(32 * c + lane < n && x[c] > t_k);
      int ties = 0;
      const int need = p.top_k - G;
#pragma unroll
      for (int c = 0; c < kChunks; ++c) {
        const bool eq = 32 * c + lane < n && x[c] == t_k;
        const unsigned bal = __ballot_sync(0xffffffffu, eq);
        cand[c] = (32 * c + lane < n && x[c] > t_k) || (eq && ties + __popc(bal & ((1u << lane) - 1u)) < need);
        ties += __popc(bal);
      }
    } else {
#pragma unroll
      for (int c = 0; c < kChunks; ++c) cand[c] = surv[c];
    }
    // weights exp(temperature * (l - l_max)) and their running sums in index order
    const double T = (double)p.temperature, m = (double)mx;
    double part[kChunks];
    double carry = 0.0;
    int last = -1;
#pragma unroll
    for (int c = 0; c < kChunks; ++c) {
      double s = cand[c] ? exp(__dmul_rn(T, (double)x[c] - m)) : 0.0;
      const unsigned pos = __ballot_sync(0xffffffffu, s > 0.0);
      if (pos) last = 32 * c + 31 - __clz(pos);
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, s, o);
        if (lane >= o) s += t;
      }
      part[c] = carry + s;
      carry += __shfl_sync(0xffffffffu, s, 31);
    }
    const double Z = carry;
    uint32_t ctr[4] = {*step_counter - 1u, (uint32_t)(p.env_id_base + b * p.env_id_stride), (uint32_t)j, 0u};
    philox4x32_10(ctr, (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
    const double u = (double)((uint64_t)(ctr[0] >> 5) * 67108864ull + (ctr[1] >> 6)) * 0x1p-53;
    const double target = u * Z;
#pragma unroll
    for (int c = 0; c < kChunks; ++c) {
      const unsigned hit = __ballot_sync(0xffffffffu, 32 * c + lane < n && part[c] > target);
      if (hit && tok < 0) tok = 32 * c + __ffs(hit) - 1;
    }
    if (tok < 0) tok = last;   // u * Z rounded up to Z
  } else {
    tok = warp_argmax(lg, discrete ? discrete_actions : num_actions, lane);
  }
  if (lane == 0) {
    if (ring) ring[(int64_t)((*ring_counter - 1u) % (unsigned)ring_slots) * ring_slot_stride + (int64_t)b * act_dim + j] = tok;
    if (discrete) {
      tokens[(int64_t)b * act_dim] = tok;
      actions[(int64_t)b * act_dim] = (float)tok;
    } else {
      tokens[(int64_t)b * act_dim + j] = tok;
      int t = tok - discrete_actions;
      if (t < 0) t = 0;
      actions[(int64_t)b * act_dim + j] = (float)t * bin_width + min_val;
    }
  }
}

__global__ void set_sampling_kernel(xl_sampling* dst, xl_sampling p, unsigned* counter, unsigned v) {
  *dst = p;
  *counter = v;
}

}  // namespace

void launch_sample_tokens(const float* logits, int64_t row_pitch, int B, int act_dim, int num_actions,
                          int discrete_actions, int discrete, float bin_width, float min_val, int32_t* tokens,
                          float* actions, int32_t* ring, const unsigned* ring_counter, int ring_slots,
                          int64_t ring_slot_stride, const void* prm, const unsigned* step_counter, cudaStream_t s) {
  const int rows = discrete ? 1 : act_dim;
  launch_k(sample_tokens_kernel, dim3(B), dim3(32 * rows), 0, s, logits, row_pitch, act_dim, num_actions,
           discrete_actions, discrete, bin_width, min_val, tokens, actions, ring, ring_counter, ring_slots,
           ring_slot_stride, (const xl_sampling*)prm, step_counter);
}

void launch_set_sampling(void* dst, const void* params, unsigned* counter, unsigned counter_value, cudaStream_t s) {
  set_sampling_kernel<<<1, 1, 0, s>>>((xl_sampling*)dst, *(const xl_sampling*)params, counter, counter_value);
}

}  // namespace xl
