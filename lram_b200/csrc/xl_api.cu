// C ABI of libxlstm_b200.so (see include/xlstm_b200.h): handle, weight binding, state layout, and the
// orchestration of one env step (embed -> L x [LN, proj_up, conv/qkv/gates, state step, proj_down] -> LN ->
// head -> argmax/inv_tokenize). No torch types; no allocation on the step path.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <utility>
#include <vector>

#include "../../include/xlstm_b200.h"
#include "xl_internal.h"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define XL_CUDA(expr)                                                                          \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return fail(XL_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                  __LINE__);                                                                   \
  } while (0)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct BlockWeights {
  const void* w[XL_W_PER_BLOCK_COUNT];
};

// What a captured step graph is specific to: the entry that captured it, its arguments and its pointers (baked into
// the graph). Pointers an entry does not take are null.
struct GraphKey {
  enum Entry { kPolicyStep, kEncoderStep } entry;
  void* state;
  const void *in, *rtg, *rewards;             // in: the policy step's states, the encoder step's x_in
  void *tokens, *actions, *logits, *out;      // out: the policy step's hidden, the encoder step's x_out
  int B, T, mode;
  unsigned flags;
  bool operator==(const GraphKey& o) const {
    return entry == o.entry && state == o.state && in == o.in && rtg == o.rtg && rewards == o.rewards &&
           tokens == o.tokens && actions == o.actions && logits == o.logits && out == o.out && B == o.B && T == o.T &&
           mode == o.mode && flags == o.flags;
  }
};

struct GraphCacheEntry {
  GraphKey key;
  cudaGraphExec_t exec = nullptr;
  int64_t launches = 0;   // kernel launches the graph replays
};

}  // namespace

// words of the handle's counters area: [0] token ring step, [1] sampler step, [2] step word of xl_sample_actions;
// xl_sampling copies (32 B, 8-B aligned) of the armed sampler and of xl_sample_actions at kCntArmed / kCntUnit
constexpr int kCntRing = 0, kCntSample = 1, kCntUnitStep = 2, kCntArmed = 8, kCntUnit = 16;
constexpr int kSplitMax = 8;   // split-K planes of the skinny projections
constexpr size_t kSplitRows = 1024;   // split-K only pays (and has plane storage) up to this many rows

struct xl_handle {
  xl_config cfg;
  int device = 0;
  int num_sms = 148;
  int DH = 0, NCH = 0, Kpad = 0, head_out = 0, num_actions = 0;
  uint64_t slstm_mask = 0;             // bit i: block i is an sLSTM block (+ gated feed-forward)
  std::vector<BlockWeights> blocks;
  const void* pw[16];  // policy-level weights, index = id - XL_W_POST_NORM
  // workspace (device)
  char* ws = nullptr;
  size_t ws_bytes = 0;
  float *x = nullptr, *xn = nullptr, *u = nullptr, *qkv = nullptr, *act = nullptr, *gate_part = nullptr,
        *gated = nullptr, *partial = nullptr, *s_emb = nullptr, *states_pad = nullptr, *logits = nullptr,
        *d_states = nullptr, *d_rtg = nullptr, *d_rew = nullptr, *d_actions = nullptr, *xtok = nullptr, *hid = nullptr;
  float* d_embeds = nullptr;    // [B, d] state embeddings staged by the eager tail of xl_policy_*_embeds
  int32_t* d_tokens = nullptr;
  unsigned int* counters = nullptr;
  __nv_bfloat16 *a_hi = nullptr, *a_lo = nullptr;
  int64_t launches = 0;
  std::vector<GraphCacheEntry> graphs;
  size_t a_cap = 0;                    // elements per bf16 hi/lo plane
  int num_tickets = 0;
  cudaStream_t cap_stream = nullptr;   // graph capture never happens on the caller's (possibly legacy) stream
  cudaStream_t side = nullptr;         // the step's L2 warm-up and the tcgen05 cell's overlapped kernels run here,
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;   // forked from / joined to the caller's stream by these events
  int state_impl = 1;                  // 1 = one-shot TMA ring (default), 2 = persistent stream-K TMA ring, 0 = plain loads
  int state_stages = 0;                // impl 2 ring depth (0 = default)        (xl_set_option "state_stages")
  int state_ctas_per_sm = 0;           // impl 2 persistent CTAs per SM (0 = 1)  (xl_set_option "state_ctas_per_sm")
  int state_rows_split = 0;            // 0 = automatic                          (xl_set_option "state_rows_split")
  int fuse_ends = 1;                   // 1: pad+split of the states in one kernel, block 0's pre-norm inside the embed
                                       // kernel, post-norm of the action rows only + head operand split in one kernel
                                       // (4 launches fewer per env step); 0: the separate kernels ("fuse_ends")
  int up_fuse = 0;                     // 1: conv / q k v / gate partials run in the proj_up epilogue (fused 3-token step,
                                       // tcgen05 path, no split-K); 0: separate pre-cell kernel ("up_fuse"). Measured on
                                       // B200 (profiles/r02_chain_fusion.md): one launch fewer per block but 3 % SLOWER at
                                       // 48M x 64 envs and 9 % slower at 206M x 128 -- the 32-wide x_m tiles make 1.5x more
                                       // CTAs re-read the A planes from L2, which is what bounds these skinny GEMMs
  int gp_chunks = 16;                  // gate-partial chunks the workspace holds per row (>= NCH and >= inner/64)
  int state_fuse = 0;                  // finalize inside the state stream kernel, one thread-block cluster per (env, head):
                                       // 1 = every CTA normalises its 128 columns, GroupNorm statistics meet over DSMEM;
                                       // 2 = numerators are pushed to rank 0, which finalizes the head; 3 = measurement aid
                                       // (unfused kernel under the cluster shape); 0 = separate finalize kernel (default).
                                       // Measured (profiles/r02_chain_fusion.md): variant 2 wins 1-2 % at 206M x 128 and
                                       // 48M x 256, loses 5 % at 48M x 64 and 2 % at 110M x 256: cluster co-scheduling alone
                                       // costs 1.4 us per launch there, and the tails no longer overlap ("state_fuse")
  int small_state_fuse = 0;            // few-env path (M <= 16 rows): variant 2 over the head's slab x row-chunk tiles (one
                                       // cluster of <= 16 CTAs; 2..16 = cap). One launch fewer per block, yet measured
                                       // SLOWER where the launch chain is the step: 16M x 1 env 153 -> 189 us, 48M x 1
                                       // 285 -> 364 us; 206M x 1 and 48M x 4 gain 3 % (profiles/r02_chain_fusion.md s7).
                                       // 0 = separate finalize kernel (default)            ("small_state_fuse")
  int gemm_impl = 0;                   // 0 auto, 1 CUDA-core, 2 tcgen05      (xl_set_option "gemm_impl")
  int gemm_splitk = 8;                 // max split-K planes of proj_up / proj_down, 0/1 = off ("gemm_splitk")
  int gemm_up_bn = 0, gemm_up_splits = 0, gemm_down_bn = 0, gemm_down_splits = 0;   // 0 = cost model; A/B overrides
  int debug_skip = 0;                  // measurement aid: bit k set = do not launch kernel class k of every block
                                       // (1 LN, 2 proj_up, 4 conv/qkv, 8 state stream, 16 finalize, 32 proj_down);
                                       // results are garbage, only the step time is meaningful ("debug_skip")
  float *part_up = nullptr, *part_down = nullptr;   // split-K planes [kSplitMax][part_rows][2*inner | d]
  size_t part_rows = 0;
  int l2_prefetch_policy = 0;          // 1: warm with an L2 evict_last policy ("l2_prefetch_policy")
  int conv_impl = 2;                   // pre-cell kernel: 0 = thread per 4-channel block, 1 = thread per (block, token),
                                       // 2 (default) = as 0 on packed fp32 pairs, gate weights before the wait, butterfly
                                       // reduction (KS = 4, NH <= 4; other shapes run impl 0)
  int l2_prefetch_mb = -1;             // MiB of the NEXT block's C warmed into L2 on a side stream while the chain
                                       // of the current block runs; 0 = off, -1 = automatic ("l2_prefetch_mb"):
                                       // 48 MiB when one block's C is 100..300 MB (measured +2 % at 151 MB, 48M x 64
                                       // envs; -0.3 % at >= 1 GB, where nothing prefetched survives until it is read)
  // context-prefill workspace (lazily allocated by xl_prefill / xl_policy_prefill, grow-only)
  char* pf_buf = nullptr;
  int pf_rows = 0;                              // rows of every [rows, ...] buffer
  size_t pf_gsc_floats = 0;                     // floats of the gate-scan scratch pf_gsc
  float *pf_x = nullptr, *pf_xn = nullptr, *pf_u = nullptr, *pf_qkv = nullptr, *pf_act = nullptr, *pf_gp = nullptr,
        *pf_gated = nullptr, *pf_num = nullptr, *pf_qn = nullptr, *pf_f = nullptr, *pf_i = nullptr, *pf_m = nullptr,
        *pf_semb = nullptr, *pf_spad = nullptr, *pf_sin = nullptr, *pf_rtg = nullptr, *pf_rew = nullptr, *pf_gsc = nullptr;
  __nv_bfloat16 *pf_hi = nullptr, *pf_lo = nullptr;
  uint8_t *pf_pc = nullptr, *pf_pv = nullptr;   // prepared operands of the chunkwise tensor-core cell
  // ragged prefill (xl_prefill_ragged / xl_policy_prefill_ragged): compact state of the active envs (grow-only,
  // xl_state_bytes(h, active envs)) and the call's [perm | token lengths] index (host staging and device copy)
  char* rg_state = nullptr;
  size_t rg_state_bytes = 0;
  int32_t* rg_idx = nullptr;                    // device, 2 * max_batch
  std::vector<int32_t> rg_host;
  // sequence forward (xl_policy_forward): logits of one chunk's timesteps [rows, n_out] (grow-only)
  float* sq_logits = nullptr;
  size_t sq_logits_floats = 0;
  int prefill_rows = 16384;                     // rows (envs x tokens) per prefill chunk                  ("prefill_rows")
  char* pf_tc = nullptr;                        // workspace of the tcgen05 chunkwise cell (grow-only)
  size_t pf_tc_bytes = 0;
  int prefill_cell = 2;                         // 2: chunkwise tcgen05 cell (xl_prefill_tc.cu), 1: chunkwise mma.sync cell
                                                // (xl_prefill_mma.cu), 0: fp32 sequence cell            ("prefill_cell")
  int smallm = -1;                              // GEMV-style front (LN + proj_up + conv/qkv) and back (proj_down) kernels
                                                // ("smallm"): 1 = whenever B*T <= 16 rows, 0 = never, -1 = automatic: B*T <= 4
                                                // rows and d <= 1024, where they are measured faster (16M x 1 env: 168 vs 196 us,
                                                // 48M: 312 vs 359, 110M: 481 vs 506; 206M equal; slower from 2 envs on —
                                                // profiles/r01_lowlat_persistent.md)
  // token ring (xl_set_token_ring): every policy step also stores its tokens in slot (step % slots) of this caller-owned
  // device buffer [slots, B, act_dim]; the step counter lives in counters[0] and is advanced on the device
  int host_zero_copy = 1;        // xl_policy_step_host: kernels read the step's inputs from / write its results to the
                                 // caller's PINNED (mapped) host buffers directly instead of 4 staged DMA copies
                                 // ("host_zero_copy"); pageable buffers fall back to staging copies
  std::vector<std::pair<const void*, void*>> host_map;   // host pointer -> device alias (nullptr: not mapped)
  int32_t* tok_ring = nullptr;
  int tok_slots = 0;
  // sampler (xl_set_sampling): while armed, policy_back launches the sampling kernel instead of the argmax one; its
  // parameters and step counter live in the counters area (kCnt* below), written on the caller's stream
  bool sampling = false;
  bool profiling = false;
  std::vector<cudaEvent_t> prof_state;  // start/stop pairs around state-step launches
  std::vector<cudaEvent_t> prof_step;   // start/stop pairs around policy steps
};

namespace {

struct StateLayout {
  size_t c_off, n_off, m_off, conv_off, layer_bytes;      // mLSTM block slot
  size_t s_off, sconv_off, slayer_bytes;                   // sLSTM block slot: (y,c,n,m) [4,B,d] | conv [B,KS,d]
};

inline bool is_slstm(const xl_handle* h, int i) { return (h->slstm_mask >> i) & 1ull; }

StateLayout state_layout(const xl_handle* h, int B) {
  const xl_config& c = h->cfg;
  StateLayout L;
  size_t off = 0;
  L.c_off = off;
  off = align_up(off + sizeof(float) * (size_t)B * c.num_heads * h->DH * h->DH, 256);
  L.n_off = off;
  off = align_up(off + sizeof(float) * (size_t)B * c.num_heads * h->DH, 256);
  L.m_off = off;
  off = align_up(off + sizeof(float) * (size_t)B * c.num_heads, 256);
  L.conv_off = off;
  off = align_up(off + sizeof(float) * (size_t)B * c.conv_kernel * c.inner_dim, 256);
  L.layer_bytes = off;
  off = 0;
  L.s_off = off;
  off = align_up(off + sizeof(float) * (size_t)4 * B * c.embedding_dim, 256);
  L.sconv_off = off;
  off = align_up(off + sizeof(float) * (size_t)B * c.conv_kernel * c.embedding_dim, 256);
  L.slayer_bytes = off;
  return L;
}

// byte offset of block i's slot: blocks are packed back to back, each with the size of its kind
size_t layer_base(const xl_handle* h, const StateLayout& L, int i) {
  const uint64_t below = i >= 64 ? ~0ull : ((1ull << i) - 1ull);
  const int ns = __builtin_popcountll(h->slstm_mask & below);
  return (size_t)(i - ns) * L.layer_bytes + (size_t)ns * L.slayer_bytes;
}

int check_batch(const xl_handle* h, int B) {
  if (!h) return fail(XL_ERR_INVALID_ARG, "null handle");
  if (B <= 0 || B > h->cfg.max_batch)
    return fail(XL_ERR_INVALID_ARG, "B=%d outside [1, max_batch=%d]", B, h->cfg.max_batch);
  return XL_OK;
}

// Drops every captured step graph: they bake in weight pointers, options, the token ring and the sampler's kernel.
void clear_graphs(xl_handle* h) {
  for (auto& g : h->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  h->graphs.clear();
}

// The buffers a Linear and the block kernels work in: the step's (step_ws) or the prefill's (prefill_ws).
// a_cap: elements of the bf16 hi/lo operand planes a tcgen05 Linear may use.
struct Ws {
  float *x, *xn, *xtok, *hid, *u, *qkv, *act, *gate_part, *gated, *partial, *s_emb, *states_pad, *logits;
  __nv_bfloat16 *a_hi, *a_lo;
  size_t a_cap;
};

// The handle's step workspace for a step over B envs. The tcgen05 Linear of a step takes at most 4 tokens x
// max(inner, d) plane elements per env: which Linear path runs depends on B only, not on the planes' total size.
Ws step_ws(const xl_handle* h, int B) {
  const size_t kmax = std::max(h->cfg.inner_dim, h->cfg.embedding_dim);
  Ws w;
  w.x = h->x; w.xn = h->xn; w.xtok = h->xtok; w.hid = h->hid; w.u = h->u; w.qkv = h->qkv; w.act = h->act;
  w.gate_part = h->gate_part; w.gated = h->gated; w.partial = h->partial;
  w.s_emb = h->s_emb; w.states_pad = h->states_pad; w.logits = h->logits;
  w.a_hi = h->a_hi; w.a_lo = h->a_lo;
  w.a_cap = (size_t)B * 4 * kmax;
  return w;
}

// Linear layer dispatch. impl: 0 auto, 1 CUDA-core, 2 tensor-core.
// presplit: the bf16 hi/lo planes of A already sit in w.a_hi / w.a_lo (written by the producing kernel).
// bn / splits / split_stride: tile width and split-K of the tcgen05 kernel (0 / 1 / 0 = planned, no split).
int linear(xl_handle* h, const Ws& w, const float* A, const void* W, const float* bias, const float* residual,
           float* out, int M, int N, int K, int impl, cudaStream_t s, bool presplit = false, int bn = 0,
           int splits = 1, long long split_stride = 0) {
  if (K % 8 != 0) return fail(XL_ERR_UNSUPPORTED, "linear: K=%d must be a multiple of 8", K);
  const bool tc_ok = xl::gemm_tc_supported(M, N, K) && (size_t)M * K <= w.a_cap;
  if (impl == 2 && !tc_ok)
    return fail(XL_ERR_UNSUPPORTED, "linear: tcgen05 path needs K %% 64 == 0 and M*K <= %zu (got M=%d K=%d)",
                w.a_cap, M, K);
  if (impl == 2 || (impl == 0 && tc_ok)) {
    if (!presplit) {
      xl::launch_split_bf16(A, K, w.a_hi, w.a_lo, M, K, s);
      h->launches += 1;
    }
    XL_CUDA(xl::launch_gemm_tc(w.a_hi, w.a_lo, (const __nv_bfloat16*)W, bias, residual, out, M, N, K,
                               h->num_sms, bn, splits, split_stride, s));
    h->launches += 1;
    return XL_OK;
  }
  if (splits > 1) return fail(XL_ERR_INVALID_ARG, "linear: split-K needs the tcgen05 path");
  xl::launch_gemm_simple(A, (const __nv_bfloat16*)W, bias, residual, out, M, N, K, s);
  h->launches += 1;
  XL_CUDA(cudaGetLastError());
  return XL_OK;
}

// One step over all B envs of a state buffer laid out for B envs, on stream s.
struct Step {
  int B;
  Ws ws;
  cudaStream_t s;
};

Step make_step(const xl_handle* h, int B, cudaStream_t s) { return {B, step_ws(h, B), s}; }

// Gate-partial chunks of the small-batch front kernel (xl_smallm.cu) when it will run for this step, else 0.
int smallm_chunks(const xl_handle* h, const Step& sl, int T, unsigned flags) {
  const xl_config& c = h->cfg;
  if (!h->smallm || h->debug_skip || (flags & XL_FLAG_SIMPLE_GEMM)) return 0;
  if (h->smallm < 0 && (sl.B * T > 4 || c.embedding_dim > 1024)) return 0;
  return xl::smallm_pre_chunks(sl.B, T, c.embedding_dim, c.inner_dim, c.num_heads, c.conv_kernel);
}

constexpr unsigned kFlagHeadOnly = 1u << 28;    // internal: nobody reads the hidden states: post_blocks_norm only on the
                                                // action-token rows, fused with the head's operand split (policy_back)
constexpr unsigned kFlagLn0Done = 1u << 29;     // internal: the embed kernel already ran block 0's pre-norm (operands in place)
constexpr unsigned kFlagNoRing = 1u << 30;      // internal: steps run on behalf of xl_policy_prefill leave the token ring
                                                // and the sampler alone (argmax, no step counted)

struct BlockPlan {
  bool tc_up, tc_down;
  bool up_fused;                          // proj_up runs with the pre-cell epilogue (no conv/qkv kernel, NCH = inner/64)
  int impl;
  int up_bn, up_sp, down_bn, down_sp;     // tile width / split-K planes of proj_up and proj_down (sp = 1: none)
};

BlockPlan block_plan(const xl_handle* h, const Step& sl, int T, unsigned flags) {
  const xl_config& c = h->cfg;
  const int M = sl.B * T;
  BlockPlan p;
  p.impl = (flags & XL_FLAG_SIMPLE_GEMM) ? 1 : h->gemm_impl;
  // when the tensor-core Linear will run, the producers write its bf16 hi/lo operand planes directly
  p.tc_up = p.impl != 1 && xl::gemm_tc_supported(M, 2 * c.inner_dim, c.embedding_dim) &&
            (size_t)M * c.embedding_dim <= sl.ws.a_cap;
  p.tc_down = p.impl != 1 && xl::gemm_tc_supported(M, c.embedding_dim, c.inner_dim) &&
              (size_t)M * c.inner_dim <= sl.ws.a_cap;
  // split-K (planes summed by the consumer kernels): rows within the plane storage
  const bool can_split = (size_t)M <= h->part_rows && c.embedding_dim <= 4096 &&
                         !smallm_chunks(h, sl, T, flags);   // the fused front kernel reads a complete x
  const int max_sp = can_split ? std::min(std::max(h->gemm_splitk, 1), kSplitMax) : 1;
  p.up_bn = p.down_bn = 0;
  p.up_sp = p.down_sp = 1;
  if (p.tc_up) {
    xl::gemm_tc_plan(M, 2 * c.inner_dim, c.embedding_dim, h->num_sms, max_sp, &p.up_bn, &p.up_sp);
    if (h->gemm_up_bn) p.up_bn = h->gemm_up_bn;
    if (h->gemm_up_splits && can_split && (c.embedding_dim / 64) % h->gemm_up_splits == 0 &&
        h->gemm_up_splits <= kSplitMax)
      p.up_sp = h->gemm_up_splits;
  }
  p.up_fused = h->up_fuse && p.tc_up && !h->debug_skip && !smallm_chunks(h, sl, T, flags) &&
               xl::gemm_up_conv_chunks(c.inner_dim) <= h->gp_chunks &&
               xl::gemm_up_conv_supported(T, c.conv_kernel, c.num_heads, c.inner_dim, c.embedding_dim);
  if (p.up_fused) { p.up_bn = 64; p.up_sp = 1; }
  if (p.tc_down) {
    xl::gemm_tc_plan(M, c.embedding_dim, c.inner_dim, h->num_sms, max_sp, &p.down_bn, &p.down_sp);
    if (h->gemm_down_bn) p.down_bn = h->gemm_down_bn;
    if (h->gemm_down_splits && can_split && (c.inner_dim / 64) % h->gemm_down_splits == 0 &&
        h->gemm_down_splits <= kSplitMax)
      p.down_sp = h->gemm_down_splits;
  }
  return p;
}

xl::StateStepParams state_params(const xl_handle* h, void* state, const Step& sl, int i, int T, bool tc_down,
                                 int up_sp = 1, int small_nch = 0, bool up_fused = false) {
  const xl_config& c = h->cfg;
  const int inner = c.inner_dim, NH = c.num_heads, DH = h->DH;
  const StateLayout L = state_layout(h, sl.B);
  const BlockWeights& w = h->blocks[i];
  char* base = (char*)state + layer_base(h, L, i);
  const int M = sl.B * T;
  xl::StateStepParams sp;
  memset(&sp, 0, sizeof(sp));
  sp.C = (float*)(base + L.c_off);
  sp.n = (float*)(base + L.n_off);
  sp.m = (float*)(base + L.m_off);
  sp.qk = sl.ws.qkv;
  sp.v = sl.ws.qkv + (size_t)2 * M * inner;
  sp.gate_part = sl.ws.gate_part;
  sp.igate_b = (const float*)w.w[XL_W_IGATE_B];
  sp.fgate_b = (const float*)w.w[XL_W_FGATE_B];
  sp.outnorm_w = (const float*)w.w[XL_W_OUTNORM];
  sp.skip = (const float*)w.w[XL_W_SKIP];
  sp.act = sl.ws.act;
  sp.u = up_sp > 1 ? h->part_up : sl.ws.u;
  sp.u_splits = up_sp;
  sp.u_stride = (int64_t)M * 2 * inner;
  sp.out = tc_down ? nullptr : sl.ws.gated;
  sp.out_hi = tc_down ? sl.ws.a_hi : nullptr;
  sp.out_lo = tc_down ? sl.ws.a_lo : nullptr;
  sp.partial = sl.ws.partial;
  sp.B = sl.B; sp.T = T; sp.NH = NH; sp.DH = DH; sp.inner = inner; sp.NCH = h->NCH;
  if (small_nch) sp.NCH = small_nch;   // chunks of the small-batch front kernel (one per CTA cluster, <= 16)
  if (up_fused) sp.NCH = xl::gemm_up_conv_chunks(inner);   // one chunk per x_m tile of the proj_up epilogue
  sp.ln_eps = c.ln_eps; sp.cell_eps = c.cell_eps;
  sp.impl = h->state_impl; sp.num_layers = c.num_blocks;
  sp.stages = h->state_stages; sp.ctas_per_sm = h->state_ctas_per_sm; sp.rows_split = h->state_rows_split;
  sp.fuse_finalize = (h->debug_skip & (8 | 16)) ? 0 : h->state_fuse;
  // few-env path: the launch chain IS the step time, so the head's tiles form one cluster whose rank 0 finalizes
  if (small_nch && h->state_fuse == 0 && h->small_state_fuse) {
    sp.fuse_finalize = 2;
    sp.max_cluster = h->small_state_fuse > 1 ? h->small_state_fuse : 0;
  }
  return sp;
}

// block i, part 1: x_n = LN(x); u = x_n W_up^T; conv + SiLU + q/k/v + gate partials   (rows ordered [b][t])
int block_pre(xl_handle* h, void* state, const Step& sl, int i, int T, unsigned flags) {
  const xl_config& c = h->cfg;
  const int d = c.embedding_dim, inner = c.inner_dim, NH = c.num_heads;
  const int M = sl.B * T;
  const StateLayout L = state_layout(h, sl.B);
  const BlockPlan bp = block_plan(h, sl, T, flags);
  const BlockWeights& w = h->blocks[i];
  const Ws& ws = sl.ws;
  char* base = (char*)state + layer_base(h, L, i);
  if (const int nch = smallm_chunks(h, sl, T, flags)) {
    // M <= 16 rows: LN + proj_up + conv / q k v / gate partials as ONE GEMV-style kernel (xl_smallm.cu)
    xl::SmallPreParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.x = ws.x;
    sp.norm_w = (const float*)w.w[XL_W_XLSTM_NORM];
    sp.w_up = (const __nv_bfloat16*)w.w[XL_W_PROJ_UP];
    sp.conv_w = (const float*)w.w[XL_W_CONV_W]; sp.conv_b = (const float*)w.w[XL_W_CONV_B];
    sp.wq = (const float*)w.w[XL_W_Q_PROJ]; sp.wk = (const float*)w.w[XL_W_K_PROJ]; sp.wv = (const float*)w.w[XL_W_V_PROJ];
    sp.wi = (const float*)w.w[XL_W_IGATE_W]; sp.wf = (const float*)w.w[XL_W_FGATE_W];
    sp.conv_state = (float*)(base + L.conv_off);
    sp.u = ws.u; sp.qk = ws.qkv; sp.v = ws.qkv + (size_t)2 * M * inner; sp.act = ws.act;
    sp.gate_part = ws.gate_part;
    sp.B = sl.B; sp.T = T; sp.d = d; sp.inner = inner; sp.NH = NH; sp.NCH = nch;
    sp.ln_eps = c.ln_eps;
    XL_CUDA(xl::launch_smallm_pre(sp, sl.s));
    h->launches += 1;
    return XL_OK;
  }
  if (h->debug_skip & 1) {
  } else if (i == 0 && (flags & kFlagLn0Done)) {
    h->launches -= 1;    // block 0's pre-norm ran inside the embed kernel (policy_front): nothing to launch
  } else if (i > 0 && bp.down_sp > 1 && !is_slstm(h, i - 1)) {
    // the previous (mLSTM) block's proj_down left split-K planes: x += planes, then normalise
    xl::launch_ln_rows_reduce(ws.x, h->part_down, bp.down_sp, (int64_t)M * d, bp.tc_up ? nullptr : ws.xn, d,
                              (const float*)w.w[XL_W_XLSTM_NORM], c.ln_eps, M, d, bp.tc_up ? ws.a_hi : nullptr,
                              bp.tc_up ? ws.a_lo : nullptr, sl.s);
  } else {
    xl::launch_ln_rows(ws.x, d, bp.tc_up ? nullptr : ws.xn, d, (const float*)w.w[XL_W_XLSTM_NORM], nullptr, 1,
                       c.ln_eps, M, d, bp.tc_up ? ws.a_hi : nullptr, bp.tc_up ? ws.a_lo : nullptr, sl.s);
  }
  h->launches += 1;
  if (bp.up_fused) {
    // proj_up with the pre-cell epilogue: conv + SiLU + q/k/v + gate partials on the x_m tiles while they are on chip
    xl::UpEpiParams ep;
    ep.conv_state = (float*)(base + L.conv_off);
    ep.conv_w = (const float*)w.w[XL_W_CONV_W]; ep.conv_b = (const float*)w.w[XL_W_CONV_B];
    ep.wq = (const float*)w.w[XL_W_Q_PROJ]; ep.wk = (const float*)w.w[XL_W_K_PROJ]; ep.wv = (const float*)w.w[XL_W_V_PROJ];
    ep.wi = (const float*)w.w[XL_W_IGATE_W]; ep.wf = (const float*)w.w[XL_W_FGATE_W];
    ep.qk = ws.qkv; ep.v = ws.qkv + (size_t)2 * M * inner; ep.act = ws.act; ep.gate_part = ws.gate_part;
    ep.B = sl.B; ep.T = T; ep.inner = inner; ep.NCH = xl::gemm_up_conv_chunks(inner);
    XL_CUDA(xl::launch_gemm_up_conv(ws.a_hi, ws.a_lo, (const __nv_bfloat16*)w.w[XL_W_PROJ_UP], ws.u, M, d, ep, sl.s));
    h->launches += 1;
    return XL_OK;
  }
  int rc = (h->debug_skip & 2) ? 0 : linear(h, ws, ws.xn, w.w[XL_W_PROJ_UP], nullptr, nullptr,
                  bp.up_sp > 1 ? h->part_up : ws.u, M, 2 * inner,
                  d, bp.impl, sl.s, bp.tc_up, bp.up_bn, bp.up_sp, (long long)M * 2 * inner);
  if (rc) return rc;
  if (h->debug_skip & 4) return XL_OK;
  xl::ConvQkvParams cp;
  cp.u = bp.up_sp > 1 ? h->part_up : ws.u;
  cp.u_splits = bp.up_sp;
  cp.u_stride = (int64_t)M * 2 * inner;
  cp.conv_state = (float*)(base + L.conv_off);
  cp.conv_w = (const float*)w.w[XL_W_CONV_W];
  cp.conv_b = (const float*)w.w[XL_W_CONV_B];
  cp.wq = (const float*)w.w[XL_W_Q_PROJ];
  cp.wk = (const float*)w.w[XL_W_K_PROJ];
  cp.wv = (const float*)w.w[XL_W_V_PROJ];
  cp.wi = (const float*)w.w[XL_W_IGATE_W];
  cp.wf = (const float*)w.w[XL_W_FGATE_W];
  cp.qk = ws.qkv;
  cp.v = ws.qkv + (size_t)2 * M * inner;
  cp.act = ws.act;
  cp.gate_part = ws.gate_part;
  cp.B = sl.B; cp.T = T; cp.inner = inner; cp.NH = NH; cp.KS = c.conv_kernel; cp.NCH = h->NCH;
  cp.impl = h->conv_impl;
  if (!xl::launch_conv_qkv_gates(cp, sl.s))
    return fail(XL_ERR_UNSUPPORTED, "conv/qkv kernel not instantiated for KS=%d T=%d NH=%d", cp.KS, cp.T, cp.NH);
  h->launches += 1;
  return XL_OK;
}

// block i, part 2: the HBM-bound state stream (C update + partial numerators)
int block_state(xl_handle* h, void* state, const Step& sl, int i, int T, unsigned flags) {
  const BlockPlan bp = block_plan(h, sl, T, flags);
  const int small_nch = smallm_chunks(h, sl, T, flags);
  // (few-env path: fp32 g for the GEMV proj_down and no split-K planes -- the same parameters block_post() builds,
  // because the stream kernel may finalize the head itself)
  const xl::StateStepParams sp = small_nch ? state_params(h, state, sl, i, T, /*tc_down=*/false, 1, small_nch)
                                           : state_params(h, state, sl, i, T, bp.tc_down, bp.up_sp, 0, bp.up_fused);
  cudaEvent_t pe0 = nullptr, pe1 = nullptr;
  if (h->profiling) {
    XL_CUDA(cudaEventCreate(&pe0));
    XL_CUDA(cudaEventCreate(&pe1));
    XL_CUDA(cudaEventRecord(pe0, sl.s));
  }
  if (!(h->debug_skip & 8)) XL_CUDA(xl::launch_state_step(sp, h->num_sms, sl.s));
  h->launches += 1;
  if (h->profiling) {
    XL_CUDA(cudaEventRecord(pe1, sl.s));
    h->prof_state.push_back(pe0);
    h->prof_state.push_back(pe1);
  }
  return XL_OK;
}

// block i, part 3: n/m update + normalise + skip + output gate; x = x + gated W_down^T
int block_post(xl_handle* h, void* state, const Step& sl, int i, int T, unsigned flags) {
  const xl_config& c = h->cfg;
  const BlockPlan bp = block_plan(h, sl, T, flags);
  const int small_nch = smallm_chunks(h, sl, T, flags);
  const Ws& ws = sl.ws;
  const int M = sl.B * T;
  if (small_nch) {
    // M <= 16 rows: finalize emits fp32 g, then x += g W_down^T as warp GEMVs (xl_smallm.cu)
    xl::StateStepParams sp = state_params(h, state, sl, i, T, /*tc_down=*/false, 1, small_nch);
    const bool fused = xl::state_step_fuses_finalize(sp, h->num_sms);
    if (!fused) XL_CUDA(xl::launch_state_finalize(sp, h->num_sms, sl.s));
    xl::SmallDownParams dp;
    dp.g = ws.gated; dp.w_down = (const __nv_bfloat16*)h->blocks[i].w[XL_W_PROJ_DOWN]; dp.x = ws.x;
    dp.M = M; dp.d = c.embedding_dim; dp.inner = c.inner_dim;
    XL_CUDA(xl::launch_smallm_down(dp, sl.s));
    h->launches += fused ? 1 : 2;
    return XL_OK;
  }
  const xl::StateStepParams sp = state_params(h, state, sl, i, T, bp.tc_down, bp.up_sp, small_nch, bp.up_fused);
  if (!xl::state_step_fuses_finalize(sp, h->num_sms)) {      // else block_state's kernel has finalized already
    if (!(h->debug_skip & 16)) XL_CUDA(xl::launch_state_finalize(sp, h->num_sms, sl.s));
    h->launches += 1;
  }
  if (h->debug_skip & 32) return XL_OK;
  if (bp.down_sp > 1)   // planes; folded into x by the next LayerNorm (block_pre of block i+1 / final_norm)
    return linear(h, ws, ws.gated, h->blocks[i].w[XL_W_PROJ_DOWN], nullptr, nullptr, h->part_down, M,
                  c.embedding_dim, c.inner_dim, bp.impl, sl.s, bp.tc_down, bp.down_bn, bp.down_sp,
                  (long long)M * c.embedding_dim);
  return linear(h, ws, ws.gated, h->blocks[i].w[XL_W_PROJ_DOWN], nullptr, ws.x, ws.x, M, c.embedding_dim,
                c.inner_dim, bp.impl, sl.s, bp.tc_down, bp.down_bn);
}

// sLSTM block i (sLSTM layer + gated feed-forward) over the M = Bk*T rows of ws.x (rows [env][token]), envs
// [0, Bk) of a state holding Btot envs. pend_sp > 1: the previous mLSTM block left that many split-K
// proj_down planes, folded into x by this block's first LayerNorm. Workspace reuse: xn = LN(x), act = swish(conv),
// u = gate pre-activations [M,4,d], gated = y [M,d], qkv = feed-forward up projection [M,2ff].
// len / pos (ragged prefill): env b has clamp(len[b] - pos, 0, T) real tokens, pads after them
int slstm_block(xl_handle* h, void* state, const Ws& ws, int Btot, int Bk, int i, int T, unsigned flags,
                int pend_sp, cudaStream_t s, const int32_t* len = nullptr, int pos = 0) {
  const xl_config& c = h->cfg;
  const int d = c.embedding_dim, NH = c.num_heads, ff = c.ffn_dim, KS = c.conv_kernel, M = Bk * T;
  const StateLayout L = state_layout(h, Btot);
  const BlockWeights& w = h->blocks[i];
  char* base = (char*)state + layer_base(h, L, i);
  float* st = (float*)(base + L.s_off);                   // (y,c,n,m), part stride Btot*d
  float* conv = (float*)(base + L.sconv_off);
  const int impl = (flags & XL_FLAG_SIMPLE_GEMM) ? 1 : h->gemm_impl;
  const bool tc_up = impl != 1 && xl::gemm_tc_supported(M, 2 * ff, d) && (size_t)M * d <= ws.a_cap;
  const bool tc_down = impl != 1 && xl::gemm_tc_supported(M, d, ff) && (size_t)M * ff <= ws.a_cap;
  auto F = [&](int id) { return (const float*)w.w[id]; };
  if (pend_sp > 1)
    xl::launch_ln_rows_reduce(ws.x, h->part_down, pend_sp, (int64_t)M * d, ws.xn, d, F(XL_W_XLSTM_NORM), c.ln_eps, M,
                              d, nullptr, nullptr, s);
  else
    xl::launch_ln_rows(ws.x, d, ws.xn, d, F(XL_W_XLSTM_NORM), nullptr, 1, c.ln_eps, M, d, nullptr, nullptr, s);
  if (!xl::launch_slstm_conv(ws.xn, conv, F(XL_W_CONV_W), F(XL_W_CONV_B), ws.act, Bk, T, d, KS, s, len, pos))
    return fail(XL_ERR_UNSUPPORTED, "sLSTM conv kernel not instantiated for KS=%d", KS);
  xl::launch_slstm_gates(ws.act, ws.xn, F(XL_W_S_GATE_I), F(XL_W_S_GATE_F), F(XL_W_S_GATE_Z), F(XL_W_S_GATE_O),
                         F(XL_W_S_BIAS), ws.u, M, d, NH, s);
  for (int t = 0; t < T; ++t)
    XL_CUDA(xl::launch_slstm_cell(ws.u, F(XL_W_S_RECURRENT), st, ws.gated, Bk, Btot, T, t, d, NH, s, len, pos));
  xl::launch_slstm_out(ws.gated, F(XL_W_S_GROUP_NORM), ws.x, st, M, T, d, NH, c.ln_eps, s);
  xl::launch_ln_rows(ws.x, d, tc_up ? nullptr : ws.xn, d, F(XL_W_FFN_NORM), nullptr, 1, c.ln_eps, M, d,
                     tc_up ? ws.a_hi : nullptr, tc_up ? ws.a_lo : nullptr, s);
  h->launches += 5 + T;
  int rc = linear(h, ws, ws.xn, w.w[XL_W_FFN_UP], nullptr, nullptr, ws.qkv, M, 2 * ff, d, impl, s, tc_up);
  if (rc) return rc;
  xl::launch_ffn_gate(ws.qkv, tc_down ? nullptr : ws.gated, tc_down ? ws.a_hi : nullptr, tc_down ? ws.a_lo : nullptr,
                      M, ff, s);
  h->launches += 1;
  rc = linear(h, ws, ws.gated, w.w[XL_W_FFN_DOWN], nullptr, ws.x, ws.x, M, d, ff, impl, s, tc_down);
  if (rc) return rc;
  XL_CUDA(cudaGetLastError());
  return XL_OK;
}

// split-K planes the block before i leaves for i's first LayerNorm (1 = none)
int pending_planes(const xl_handle* h, const Step& sl, int i, int T, unsigned flags) {
  if (i == 0 || is_slstm(h, i - 1)) return 1;
  return block_plan(h, sl, T, flags).down_sp;
}

// post_blocks_norm over the M = B*T rows of ws.x left by run_blocks (folds the last block's split-K planes)
void final_norm(xl_handle* h, const Step& sl, int T, unsigned flags, float* out, int64_t out_stride) {
  const xl_config& c = h->cfg;
  const int d = c.embedding_dim, M = sl.B * T;
  const BlockPlan bp = block_plan(h, sl, T, flags);
  const float* post_w = (const float*)h->pw[XL_W_POST_NORM - XL_W_POST_NORM];
  if (bp.down_sp > 1 && !is_slstm(h, c.num_blocks - 1))
    xl::launch_ln_rows_reduce(sl.ws.x, h->part_down, bp.down_sp, (int64_t)M * d, out, out_stride, post_w, c.ln_eps,
                              M, d, nullptr, nullptr, sl.s);
  else
    xl::launch_ln_rows(sl.ws.x, d, out, out_stride, post_w, nullptr, 1, c.ln_eps, M, d, nullptr, nullptr, sl.s);
  h->launches += 1;
}

// One pass of the block stack over M = B*T rows held in ws.x (rows ordered [b][t]).
int run_blocks(xl_handle* h, void* state, const Step& sl, int T, unsigned flags) {
  const int L = h->cfg.num_blocks;
  // L2 warm-up of the next block's C on the side stream. Block 0 of the NEXT env step is warmed after the last block's
  // state kernel.
  const StateLayout lay = state_layout(h, sl.B);
  const size_t c_bytes = sizeof(float) * (size_t)sl.B * h->cfg.num_heads * h->DH * h->DH;
  int warm_mb = h->l2_prefetch_mb;
  if (warm_mb < 0) warm_mb = (c_bytes >= ((size_t)100 << 20) && c_bytes <= ((size_t)300 << 20)) ? 48 : 0;
  const bool warm = warm_mb > 0 && L > 1;
  const size_t warm_bytes = std::min(c_bytes, (size_t)warm_mb << 20);
  int rc = XL_OK;
  for (int i = 0; i < L && !rc; ++i) {
    if (is_slstm(h, i)) {
      rc = slstm_block(h, state, sl.ws, sl.B, sl.B, i, T, flags, pending_planes(h, sl, i, T, flags), sl.s);
      continue;
    }
    rc = block_pre(h, state, sl, i, T, flags);
    if (!rc) rc = block_state(h, state, sl, i, T, flags);
    if (!rc && warm) {
      XL_CUDA(cudaEventRecord(h->ev_fork, sl.s));
      XL_CUDA(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
      int nx = (i + 1) % L;
      while (is_slstm(h, nx) && nx != i) nx = (nx + 1) % L;        // next mLSTM block
      const char* next_c = (const char*)state + layer_base(h, lay, nx) + lay.c_off;
      xl::launch_l2_prefetch(next_c, warm_bytes, h->num_sms, h->l2_prefetch_policy, h->side);
      h->launches += 1;
    }
    if (!rc) rc = block_post(h, state, sl, i, T, flags);
  }
  if (warm) {   // join (also on the error path: a capture must not end with an unjoined stream)
    cudaEventRecord(h->ev_join, h->side);
    cudaStreamWaitEvent(sl.s, h->ev_join, 0);
  }
  if (rc) return rc;
  XL_CUDA(cudaGetLastError());
  return XL_OK;
}

// Encoder over x_in [B,T,d] -> x_out [B,T,d] (post_blocks_norm applied), single stream.
int run_encoder(xl_handle* h, void* state, const Step& sl, const float* x_in, float* x_out, int T, int mode,
                unsigned flags) {
  const xl_config& c = h->cfg;
  const int d = c.embedding_dim;
  const int B = sl.B;
  const Ws& ws = sl.ws;
  cudaStream_t s = sl.s;
  const float* post_w = (const float*)h->pw[XL_W_POST_NORM - XL_W_POST_NORM];
  if (mode == XL_MODE_FUSED || T == 1) {
    if (x_in != ws.x) {
      XL_CUDA(cudaMemcpyAsync(ws.x, x_in, sizeof(float) * (size_t)B * T * d, cudaMemcpyDeviceToDevice, s));
    }
    int rc = run_blocks(h, state, sl, T, flags);
    if (rc) return rc;
    if (!(flags & kFlagHeadOnly)) final_norm(h, sl, T, flags, x_out, d);
  } else if (mode == XL_MODE_PER_TOKEN) {
    // reference order: for token: for block  (decision_xlstm.py:161-165). x_in may alias x_out: token t's
    // input row is consumed (gathered) before its output row is written.
    const float* src = x_in;
    if (x_in == x_out) {
      XL_CUDA(cudaMemcpyAsync(ws.xtok, x_in, sizeof(float) * (size_t)B * T * d, cudaMemcpyDeviceToDevice, s));
      src = ws.xtok;
    }
    for (int t = 0; t < T; ++t) {
      xl::launch_copy_rows(src + (size_t)t * d, (int64_t)T * d, ws.x, d, B, d, s);
      h->launches += 1;
      int rc = run_blocks(h, state, sl, 1, flags);
      if (rc) return rc;
      final_norm(h, sl, 1, flags, x_out + (size_t)t * d, (int64_t)T * d);
    }
  } else {
    return fail(XL_ERR_INVALID_ARG, "unknown mode %d", mode);
  }
  XL_CUDA(cudaGetLastError());
  return XL_OK;
}

// Arguments of one policy step (device pointers for the WHOLE batch of B envs).
struct StepArgs {
  void* state;
  const float *states, *rtg, *rewards;
  int32_t* tokens;
  float *actions, *logits, *hidden;
  int B, mode;
  unsigned flags;
};

// embed_state Linear(204 -> d) on zero-padded K, (s, rtg, r) token embedding + embed_ln -> xt [B, 3, d]
int policy_front(xl_handle* h, const StepArgs& a, const Step& sl, float* xt) {
  const xl_config& c = h->cfg;
  const int d = c.embedding_dim;
  const int impl = (a.flags & XL_FLAG_SIMPLE_GEMM) ? 1 : h->gemm_impl;
  auto PW = [&](int id) { return h->pw[id - XL_W_POST_NORM]; };
  const Ws& ws = sl.ws;
  const float* s_emb = ws.s_emb;
  if (a.flags & XL_FLAG_STATE_EMBEDS) {
    // a.states already holds the state-token embeddings [B, d] (image observations: embed_image = ImpalaCNN,
    // discrete_decision_transformer_model.py:187-203, runs in PyTorch/cuDNN before this call)
    s_emb = a.states;
  } else {
    const bool tc = impl != 1 && xl::gemm_tc_supported(sl.B, d, h->Kpad) && (size_t)sl.B * h->Kpad <= ws.a_cap;
    if (tc) {       // zero-pad + bf16 hi/lo split in one kernel, straight into the GEMM's operand planes
      xl::launch_pad_split(a.states, c.state_dim, ws.a_hi, ws.a_lo, h->Kpad, sl.B, sl.s);
    } else {
      xl::launch_pad_rows(a.states, c.state_dim, ws.states_pad, h->Kpad, sl.B, sl.s);
    }
    h->launches += 1;
    int rc = linear(h, ws, ws.states_pad, PW(XL_W_EMBED_STATE_W), (const float*)PW(XL_W_EMBED_STATE_B), nullptr,
                    ws.s_emb, sl.B, d, h->Kpad, impl, sl.s, /*presplit=*/tc);
    if (rc) return rc;
  }
  // block 0's pre-norm rides on the embed kernel when the stack will consume it as is (kFlagLn0Done set by run_policy)
  const float* ln0_w = nullptr;
  float* xn0 = nullptr;
  void *hi0 = nullptr, *lo0 = nullptr;
  if (a.flags & kFlagLn0Done) {
    const BlockPlan bp = block_plan(h, sl, c.tokens_per_step, a.flags);
    ln0_w = (const float*)h->blocks[0].w[XL_W_XLSTM_NORM];
    if (bp.tc_up) { hi0 = ws.a_hi; lo0 = ws.a_lo; } else { xn0 = ws.xn; }
  }
  xl::launch_embed_tokens(s_emb, a.rtg, a.rewards,
                          (const float*)PW(XL_W_EMBED_RETURN_W), (const float*)PW(XL_W_EMBED_RETURN_B),
                          (const float*)PW(XL_W_EMBED_REWARD_W), (const float*)PW(XL_W_EMBED_REWARD_B),
                          (const float*)PW(XL_W_EMBED_LN_W), (const float*)PW(XL_W_EMBED_LN_B), c.embed_ln_eps, xt,
                          sl.B, d, (h->tok_ring && !(a.flags & kFlagNoRing)) ? h->counters + kCntRing : nullptr,
                          (h->sampling && !(a.flags & kFlagNoRing)) ? h->counters + kCntSample : nullptr,
                          ln0_w, c.ln_eps, xn0, hi0, lo0, sl.s);
  h->launches += 1;
  return XL_OK;
}

// action head on the rtg token of hid [B, T, d] -> logits -> argmax / inv_tokenize
int policy_back(xl_handle* h, const StepArgs& a, const Step& sl, const float* hid) {
  const xl_config& c = h->cfg;
  const int d = c.embedding_dim, T = c.tokens_per_step;
  const int impl = (a.flags & XL_FLAG_SIMPLE_GEMM) ? 1 : h->gemm_impl;
  auto PW = [&](int id) { return h->pw[id - XL_W_POST_NORM]; };
  const Ws& ws = sl.ws;
  cudaStream_t s = sl.s;
  const int B = sl.B;
  // gather row b*T + pos to a dense [B,d], then Linear(d -> 2192 / 274)
  float* xa = ws.s_emb;  // reuse [B,d]
  const bool head_only = (a.flags & kFlagHeadOnly) != 0;
  if (head_only) {
    // post_blocks_norm of the action-token rows only (+ the last proj_down's pending planes), emitted as the head
    // GEMM's bf16 hi/lo operand planes: one launch instead of norm-all-rows + gather + split
    const BlockPlan bp = block_plan(h, sl, T, a.flags);
    const int pend = is_slstm(h, c.num_blocks - 1) ? 1 : bp.down_sp;
    xl::launch_ln_rows_gather(ws.x, h->part_down, pend, (int64_t)B * T * d, (const float*)PW(XL_W_POST_NORM), c.ln_eps,
                              B, d, T, c.action_token_pos, ws.a_hi, ws.a_lo, s);
  } else {
    xl::launch_copy_rows(hid + (size_t)c.action_token_pos * d, (int64_t)T * d, xa, d, B, d, s);
  }
  h->launches += 1;
  const bool discrete = (a.flags & XL_FLAG_DISCRETE) != 0;
  // discrete branch only needs the first num_actions logits (multi_domain_discrete_dt_model.py:99-101)
  const int n_out = discrete ? h->num_actions : h->head_out;
  int rc;
  int32_t* ring = (h->tok_ring && !(a.flags & kFlagNoRing)) ? h->tok_ring : nullptr;
  const int64_t ring_stride = (int64_t)B * c.act_dim;
  const bool sample = h->sampling && !(a.flags & kFlagNoRing);
  const float bw = (c.tok_max_val - c.tok_min_val) / (float)c.action_channels;
  if (discrete) {
    rc = linear(h, ws, xa, PW(XL_W_HEAD_W), (const float*)PW(XL_W_HEAD_B), nullptr, ws.logits, B, n_out, d, impl, s,
                head_only);
    if (rc) return rc;
    if (a.logits) {
      XL_CUDA(cudaMemcpyAsync(a.logits, ws.logits, sizeof(float) * (size_t)B * n_out, cudaMemcpyDeviceToDevice, s));
    }
    if (sample)
      xl::launch_sample_tokens(ws.logits, n_out, B, c.act_dim, n_out, c.discrete_actions, 1, 0.f, 0.f, a.tokens,
                               a.actions, ring, h->counters + kCntRing, h->tok_slots, ring_stride,
                               h->counters + kCntArmed, h->counters + kCntSample, s);
    else
      xl::launch_argmax_tokens(ws.logits, n_out, B, c.act_dim, n_out, c.discrete_actions, 1, 0.f, 0.f, a.tokens,
                               a.actions, ring, h->counters + kCntRing, h->tok_slots, ring_stride, s);
  } else {
    float* lg = a.logits ? a.logits : ws.logits;
    rc = linear(h, ws, xa, PW(XL_W_HEAD_W), (const float*)PW(XL_W_HEAD_B), nullptr, lg, B, n_out, d, impl, s, head_only);
    if (rc) return rc;
    if (sample)
      xl::launch_sample_tokens(lg, h->head_out, B, c.act_dim, h->num_actions, c.discrete_actions, 0, bw, c.tok_min_val,
                               a.tokens, a.actions, ring, h->counters + kCntRing, h->tok_slots, ring_stride,
                               h->counters + kCntArmed, h->counters + kCntSample, s);
    else
      xl::launch_argmax_tokens(lg, h->head_out, B, c.act_dim, h->num_actions, c.discrete_actions, 0, bw,
                               c.tok_min_val, a.tokens, a.actions, ring, h->counters + kCntRing, h->tok_slots,
                               ring_stride, s);
  }
  h->launches += 1;
  return XL_OK;
}

int run_policy(xl_handle* h, const StepArgs& args, cudaStream_t s) {
  const int d = h->cfg.embedding_dim, T = h->cfg.tokens_per_step;
  const Step sl = make_step(h, args.B, s);
  float* xt = (args.mode == XL_MODE_FUSED) ? sl.ws.x : sl.ws.xtok;
  // launch-saving fusions of the step's head and tail (fused mode, multi-kernel stack)
  StepArgs a = args;
  if (h->fuse_ends && a.mode == XL_MODE_FUSED && !h->debug_skip) {
    if (!is_slstm(h, 0) && !smallm_chunks(h, sl, T, a.flags)) a.flags |= kFlagLn0Done;
    const int impl = (a.flags & XL_FLAG_SIMPLE_GEMM) ? 1 : h->gemm_impl;
    const int n_out = (a.flags & XL_FLAG_DISCRETE) ? h->num_actions : h->head_out;
    if (!a.hidden && impl != 1 && xl::gemm_tc_supported(a.B, n_out, d) && (size_t)a.B * d <= sl.ws.a_cap && d <= 4096)
      a.flags |= kFlagHeadOnly;
  }
  int rc = policy_front(h, a, sl, xt);
  if (rc) return rc;
  float* hid = a.hidden ? a.hidden : sl.ws.hid;
  rc = run_encoder(h, a.state, sl, xt, hid, T, a.mode, a.flags);
  if (rc) return rc;
  rc = policy_back(h, a, sl, hid);
  if (rc) return rc;
  XL_CUDA(cudaGetLastError());
  return XL_OK;
}

// ---- context prefill ----------------------------------------------------------------------------------
// Grows the workspace to `rows` rows and `gsc_floats` floats of gate-scan scratch (never shrinks either).
int ensure_prefill_ws(xl_handle* h, int rows, size_t gsc_floats) {
  if (rows <= h->pf_rows && gsc_floats <= h->pf_gsc_floats) return XL_OK;
  rows = std::max(rows, h->pf_rows);
  gsc_floats = std::max(gsc_floats, h->pf_gsc_floats);
  const xl_config& c = h->cfg;
  const size_t d = c.embedding_dim, inner = c.inner_dim, NH = c.num_heads, R = (size_t)rows;
  const size_t kmax = std::max(std::max(inner, d), (size_t)h->Kpad);
  size_t off = 0;
  auto carve = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  };
  const size_t o_x = carve(4 * R * d), o_xn = carve(4 * R * d), o_u = carve(4 * R * 2 * inner);
  const size_t o_qkv = carve(4 * R * 3 * inner), o_act = carve(4 * R * inner), o_gp = carve(4 * R * 16 * 2 * NH);
  const size_t o_gated = carve(4 * R * inner), o_num = carve(4 * R * inner), o_qn = carve(4 * R * NH);
  const size_t o_f = carve(4 * R * NH), o_i = carve(4 * R * NH), o_m = carve(4 * R * NH);
  const size_t o_semb = carve(4 * R * d), o_spad = carve(4 * R * h->Kpad), o_sin = carve(4 * R * c.state_dim);
  const size_t o_rtg = carve(4 * R), o_rew = carve(4 * R);
  const size_t o_gsc = carve(4 * gsc_floats);
  const size_t o_hi = carve(2 * R * kmax), o_lo = carve(2 * R * kmax);
  size_t pc_bytes = 0, pv_bytes = 0;
  if (xl::prefill_cell_mma_supported(h->DH)) xl::prefill_cell_mma_ws(rows, (int)NH, h->DH, &pc_bytes, &pv_bytes);
  const size_t o_pc = carve(pc_bytes), o_pv = carve(pv_bytes);
  XL_CUDA(cudaDeviceSynchronize());            // nothing may still be using the old workspace
  if (h->pf_buf) cudaFree(h->pf_buf);
  h->pf_buf = nullptr;
  h->pf_rows = 0;
  h->pf_gsc_floats = 0;
  cudaError_t e = cudaMalloc((void**)&h->pf_buf, off);
  if (e != cudaSuccess) return fail(XL_ERR_CUDA, "cudaMalloc(prefill workspace %zu B) failed: %s", off, cudaGetErrorString(e));
  char* b = h->pf_buf;
  h->pf_x = (float*)(b + o_x); h->pf_xn = (float*)(b + o_xn); h->pf_u = (float*)(b + o_u);
  h->pf_qkv = (float*)(b + o_qkv); h->pf_act = (float*)(b + o_act); h->pf_gp = (float*)(b + o_gp);
  h->pf_gated = (float*)(b + o_gated); h->pf_num = (float*)(b + o_num); h->pf_qn = (float*)(b + o_qn);
  h->pf_f = (float*)(b + o_f); h->pf_i = (float*)(b + o_i); h->pf_m = (float*)(b + o_m);
  h->pf_semb = (float*)(b + o_semb); h->pf_spad = (float*)(b + o_spad); h->pf_sin = (float*)(b + o_sin);
  h->pf_rtg = (float*)(b + o_rtg); h->pf_rew = (float*)(b + o_rew);
  h->pf_gsc = (float*)(b + o_gsc);
  h->pf_hi = (__nv_bfloat16*)(b + o_hi); h->pf_lo = (__nv_bfloat16*)(b + o_lo);
  h->pf_pc = (uint8_t*)(b + o_pc); h->pf_pv = (uint8_t*)(b + o_pv);
  h->pf_rows = rows;
  h->pf_gsc_floats = gsc_floats;
  return XL_OK;
}

int ensure_prefill_tc_ws(xl_handle* h, int B, int Sc) {
  const size_t need = xl::prefill_cell_tc_ws_bytes(B, Sc, h->cfg.num_heads, h->DH);
  if (need <= h->pf_tc_bytes) return XL_OK;
  XL_CUDA(cudaDeviceSynchronize());            // nothing may still be using the old workspace
  if (h->pf_tc) cudaFree(h->pf_tc);
  h->pf_tc = nullptr;
  h->pf_tc_bytes = 0;
  cudaError_t e = cudaMalloc((void**)&h->pf_tc, need);
  if (e != cudaSuccess) return fail(XL_ERR_CUDA, "cudaMalloc(prefill cell workspace %zu B) failed: %s", need, cudaGetErrorString(e));
  h->pf_tc_bytes = need;
  return XL_OK;
}

Ws prefill_ws(const xl_handle* h) {
  Ws w;
  memset(&w, 0, sizeof(w));
  w.x = h->pf_x; w.xn = h->pf_xn; w.u = h->pf_u; w.qkv = h->pf_qkv; w.act = h->pf_act; w.gate_part = h->pf_gp;
  w.gated = h->pf_gated; w.s_emb = h->pf_semb; w.states_pad = h->pf_spad;
  w.a_hi = h->pf_hi; w.a_lo = h->pf_lo;
  const size_t kmax = std::max(std::max((size_t)h->cfg.inner_dim, (size_t)h->cfg.embedding_dim), (size_t)h->Kpad);
  w.a_cap = (size_t)h->pf_rows * kmax;
  return w;
}

// The sequence cell that runs B envs x Sc tokens of this handle: 2 = tcgen05, 1 = mma.sync, 0 = fp32; -1 when none
// can. tcgen05 cell: whole 128-token chunks per (env, head) -- short runs of many envs (Sc < 64: more than half of
// every chunk would be padding) or a workspace beyond 8 GiB fall through to the 16-token mma.sync cell.
int seq_cell_choice(const xl_handle* h, int B, int Sc) {
  const int NH = h->cfg.num_heads, DH = h->DH;
  if (h->prefill_cell == 2 && xl::prefill_cell_tc_supported(DH) && Sc >= 64 &&
      xl::prefill_cell_tc_ws_bytes(B, Sc, NH, DH) <= ((size_t)8 << 30))
    return 2;
  if (h->prefill_cell >= 1 && xl::prefill_cell_mma_supported(DH) && Sc % xl::prefill_cell_mma_chunk() == 0) return 1;
  if (xl::prefill_cell_supported(DH) && Sc % 8 == 0) return 0;
  return -1;
}

// Gate scan + sequence cell of one mLSTM block over B envs x Sc tokens (rows [env][token]): the carried C / n / m_state
// advanced by the Sc tokens, per-token num [B*Sc, inner], qn [B*Sc, NH] and m [B*NH][Sc] (mseq) for the finalize.
// gate_part [B*Sc, NCH, 2*NH] partial gate pre-activations, biases nullable; len / pos: ragged chunk (see
// prefill_blocks). The prefill workspace must hold B*Sc rows and the gate-scan scratch. *cell (nullable) <- the cell
// that ran (seq_cell_choice).
int seq_cell(xl_handle* h, float* C, float* n, float* m_state, const float* q, const float* k, const float* v,
             const float* gate_part, const float* igate_b, const float* fgate_b, float* num, float* qn, float* mseq,
             int B, int Sc, int NCH, cudaStream_t s, const int32_t* len, int pos, int* cell) {
  const int NH = h->cfg.num_heads, DH = h->DH, inner = h->cfg.inner_dim;
  const int which = seq_cell_choice(h, B, Sc);
  if (which < 0) return fail(XL_ERR_UNSUPPORTED, "no sequence cell takes DH=%d over %d tokens", DH, Sc);
  xl::launch_gate_scan_seq(gate_part, igate_b, fgate_b, m_state, h->pf_f, h->pf_i, mseq, h->pf_gsc, B, Sc, NH, NCH, s,
                           len, pos);
  XL_CUDA(cudaGetLastError());
  if (which == 2) {
    if (int rcw = ensure_prefill_tc_ws(h, B, Sc)) return rcw;
    const xl::CellSideStream side = {h->side, h->ev_fork, h->ev_join};
    XL_CUDA(xl::launch_cell_tc(C, n, q, k, v, h->pf_f, h->pf_i, num, qn, h->pf_tc, B, Sc, NH, DH, inner, s, &side));
    h->launches += 6;
    XL_CUDA(cudaGetLastError());
  } else if (which == 1) {
    XL_CUDA(xl::launch_cell_mma(C, n, q, k, v, h->pf_f, h->pf_i, num, qn, h->pf_pc, h->pf_pv, B, Sc, NH, DH, inner, s));
    h->launches += 1;
  } else {
    XL_CUDA(xl::launch_cell_seq(C, n, q, k, v, h->pf_f, h->pf_i, num, qn, B, Sc, NH, DH, inner, s));
  }
  if (cell) *cell = which;
  return XL_OK;
}

// tokens per env in one prefill chunk: ~2048 rows per chunk over all envs, a multiple of 48 (whole (s, rtg, r)
// timesteps, whole 8-token stages of the fp32 cell and whole 16-token chunks of the tensor-core cell)
int prefill_chunk_tokens(const xl_handle* h, int B) {
  int sc = h->prefill_rows / B;
  if (sc < 48) sc = 48;
  return sc / 48 * 48;
}

// The block stack over the chunk held in pf_x [B*Sc, d] (rows [env][token]), in place; state advanced by Sc tokens.
// The state holds Btot >= B envs; the chunk belongs to its first B. Ragged prefill (len != nullptr, a device array of B
// token counts; the chunk starts at token pos of the context): env b advances by its clamp(len[b] - pos, 0, Sc) real
// tokens only, every env of the chunk having at least one.
int prefill_blocks(xl_handle* h, void* state, int Btot, int B, int Sc, unsigned flags, cudaStream_t s,
                   const int32_t* len = nullptr, int pos = 0) {
  const xl_config& c = h->cfg;
  const int d = c.embedding_dim, inner = c.inner_dim, NH = c.num_heads, DH = h->DH;
  const int M = B * Sc;
  const StateLayout L = state_layout(h, Btot);
  const Ws ws = prefill_ws(h);
  const int impl = (flags & XL_FLAG_SIMPLE_GEMM) ? 1 : h->gemm_impl;
  const bool tc_up = impl != 1 && xl::gemm_tc_supported(M, 2 * inner, d) && (size_t)M * d <= ws.a_cap;
  const bool tc_down = impl != 1 && xl::gemm_tc_supported(M, d, inner) && (size_t)M * inner <= ws.a_cap;
  for (int i = 0; i < c.num_blocks; ++i) {
    if (is_slstm(h, i)) {
      // no parallel form exists for the sLSTM: its cell runs token by token (Sc launches of a tiny kernel), the
      // rest of the block (conv, gate projections, GroupNorm, feed-forward) over the whole chunk
      int rcs = slstm_block(h, state, ws, Btot, B, i, Sc, flags, 1, s, len, pos);
      if (rcs) return rcs;
      continue;
    }
    const BlockWeights& w = h->blocks[i];
    char* base = (char*)state + layer_base(h, L, i);
    xl::launch_ln_rows(ws.x, d, tc_up ? nullptr : ws.xn, d, (const float*)w.w[XL_W_XLSTM_NORM], nullptr, 1, c.ln_eps,
                       M, d, tc_up ? ws.a_hi : nullptr, tc_up ? ws.a_lo : nullptr, s);
    h->launches += 1;
    XL_CUDA(cudaGetLastError());
    // GEMM-sized M: 128 x 256 tiles for proj_up (2/3 of the operand bytes per flop; measured -2 % on the 206M prefill)
    const int up_bn = h->gemm_up_bn ? h->gemm_up_bn : (M >= 1024 && (2 * inner) % 256 == 0 ? 256 : 0);
    int rc = linear(h, ws, ws.xn, w.w[XL_W_PROJ_UP], nullptr, nullptr, ws.u, M, 2 * inner, d, impl, s, tc_up, up_bn);
    if (rc) return rc;
    xl::ConvQkvParams cp;
    cp.u = ws.u;
    cp.u_splits = 1;
    cp.u_stride = 0;
    cp.conv_state = (float*)(base + L.conv_off);
    cp.conv_w = (const float*)w.w[XL_W_CONV_W];
    cp.conv_b = (const float*)w.w[XL_W_CONV_B];
    cp.wq = (const float*)w.w[XL_W_Q_PROJ];
    cp.wk = (const float*)w.w[XL_W_K_PROJ];
    cp.wv = (const float*)w.w[XL_W_V_PROJ];
    cp.wi = (const float*)w.w[XL_W_IGATE_W];
    cp.wf = (const float*)w.w[XL_W_FGATE_W];
    cp.qk = ws.qkv;
    cp.v = ws.qkv + (size_t)2 * M * inner;
    cp.act = ws.act;
    cp.gate_part = ws.gate_part;
    cp.B = B; cp.T = Sc; cp.inner = inner; cp.NH = NH; cp.KS = c.conv_kernel; cp.NCH = h->NCH;
    cp.impl = 0;
    if (!xl::launch_conv_qkv_gates_seq(cp, Sc, s, len, pos))
      return fail(XL_ERR_UNSUPPORTED, "sequence conv/qkv kernel not instantiated for KS=%d NH=%d", cp.KS, cp.NH);
    XL_CUDA(cudaGetLastError());
    rc = seq_cell(h, (float*)(base + L.c_off), (float*)(base + L.n_off), (float*)(base + L.m_off), cp.qk,
                  cp.qk + (size_t)M * inner, cp.v, ws.gate_part, (const float*)w.w[XL_W_IGATE_B],
                  (const float*)w.w[XL_W_FGATE_B], h->pf_num, h->pf_qn, h->pf_m, B, Sc, h->NCH, s, len, pos, nullptr);
    if (rc) return rc;
    XL_CUDA(xl::launch_finalize_seq(h->pf_num, h->pf_qn, h->pf_m, (const float*)w.w[XL_W_OUTNORM],
                                    (const float*)w.w[XL_W_SKIP], ws.act, ws.u, tc_down ? nullptr : ws.gated,
                                    tc_down ? ws.a_hi : nullptr, tc_down ? ws.a_lo : nullptr, B, Sc, NH, DH, inner,
                                    c.ln_eps, c.cell_eps, s));
    h->launches += 5;
    rc = linear(h, ws, ws.gated, w.w[XL_W_PROJ_DOWN], nullptr, ws.x, ws.x, M, d, inner, impl, s, tc_down,
                h->gemm_down_bn);
    if (rc) return rc;
  }
  XL_CUDA(cudaGetLastError());
  return XL_OK;
}

bool prefill_fast_path(const xl_handle* h) {
  return xl::prefill_cell_supported(h->DH) && h->cfg.conv_kernel == 4;
}

// ---- sequence plan -------------------------------------------------------------------------------------------------
// Every sequence call (context prefill, policy prefill, sequence forward) runs chunks {pos, Bk, n}: units
// [pos, pos + n) of the first Bk envs of the state the chunks advance, a unit being T tokens (1: encoder tokens;
// tokens_per_step: timesteps). Units from `tail` on run as eager steps.
// Uniform call (no lengths): all B envs of the caller's state, perm / len null.
// Ragged call: the active envs (length > 0) sorted by length, descending and stable: compact env k is caller env perm[k].
// Once sorted, the envs that still have tokens at position pos are a prefix Bk of the compact batch, so every chunk runs
// the sequence kernels on that prefix (same base pointers, smaller B) and pads each env's end up to the chunk's length
// with identity tokens. If the active envs already are envs 0..Bc-1 in that order, the chunks work on the caller's state
// in place; otherwise the state is gathered into a compact one of Bc envs and scattered back at the end.
struct SeqChunk {
  int pos, Bk, n;
};
struct SeqPlan {
  int T = 1;                          // tokens per unit
  std::vector<SeqChunk> chunks;
  int tail = 0;                       // first unit of the eager tail
  std::vector<int32_t> perm, len;     // ragged: len in units
  bool in_place = true;
  void* st = nullptr;                 // the state the chunks advance
  int Btot = 0;                       // envs of its layout
  const int32_t *d_perm = nullptr, *d_len = nullptr;   // ragged: device copies, d_len in tokens; uniform: null
};

int check_lengths(const int32_t* lengths, int B, int S, const char* what) {
  if (!lengths) return fail(XL_ERR_INVALID_ARG, "null lengths");
  for (int b = 0; b < B; ++b)
    if (lengths[b] < 0 || lengths[b] > S)
      return fail(XL_ERR_INVALID_ARG, "lengths[%d]=%d outside [0, %s=%d]", b, lengths[b], what, S);
  return XL_OK;
}

xl::StateCopyGeom state_copy_geom(const xl_handle* h, int B, int Bc) {
  const xl_config& c = h->cfg;
  xl::StateCopyGeom g;
  g.slstm_mask = h->slstm_mask;
  g.num_blocks = c.num_blocks;
  const int Bs[2] = {B, Bc};
  for (int j = 0; j < 2; ++j) {
    const StateLayout L = state_layout(h, Bs[j]);
    g.B[j] = Bs[j];
    g.layer_bytes[j] = L.layer_bytes; g.slayer_bytes[j] = L.slayer_bytes;
    g.c_off[j] = L.c_off; g.n_off[j] = L.n_off; g.m_off[j] = L.m_off; g.conv_off[j] = L.conv_off;
    g.s_off[j] = L.s_off; g.sconv_off[j] = L.sconv_off;
  }
  const size_t f = sizeof(float), NH = c.num_heads, DH = h->DH, KS = c.conv_kernel;
  g.c_env = f * NH * DH * DH; g.n_env = f * NH * DH; g.m_env = f * NH; g.conv_env = f * KS * c.inner_dim;
  g.s_env = f * c.embedding_dim; g.sconv_env = f * KS * c.embedding_dim;
  return g;
}

// Sort, upload the index, and gather the state when the active envs are not a sorted prefix.
int ragged_begin(xl_handle* h, void* state, const int32_t* lengths, int B, SeqPlan& p, cudaStream_t s) {
  for (int b = 0; b < B; ++b)
    if (lengths[b] > 0) p.perm.push_back(b);
  std::stable_sort(p.perm.begin(), p.perm.end(), [&](int a, int b) { return lengths[a] > lengths[b]; });
  const int Bc = (int)p.perm.size();
  for (int k = 0; k < Bc; ++k) {
    p.len.push_back(lengths[p.perm[k]]);
    p.in_place = p.in_place && p.perm[k] == k;
  }
  if (!h->rg_idx) XL_CUDA(cudaMalloc((void**)&h->rg_idx, sizeof(int32_t) * 2 * (size_t)h->cfg.max_batch));
  h->rg_host.assign(2 * (size_t)Bc, 0);
  for (int k = 0; k < Bc; ++k) {
    h->rg_host[k] = p.perm[k];
    h->rg_host[Bc + k] = p.len[k] * p.T;
  }
  XL_CUDA(cudaMemcpyAsync(h->rg_idx, h->rg_host.data(), sizeof(int32_t) * 2 * (size_t)Bc, cudaMemcpyHostToDevice, s));
  p.d_perm = h->rg_idx;
  p.d_len = h->rg_idx + Bc;
  if (p.in_place) {
    p.st = state;
    p.Btot = B;
    return XL_OK;
  }
  const size_t need = xl_state_bytes(h, Bc);
  if (need > h->rg_state_bytes) {
    XL_CUDA(cudaDeviceSynchronize());          // nothing may still be using the old buffer
    if (h->rg_state) cudaFree(h->rg_state);
    h->rg_state = nullptr;
    h->rg_state_bytes = 0;
    cudaError_t e = cudaMalloc((void**)&h->rg_state, need);
    if (e != cudaSuccess)
      return fail(XL_ERR_CUDA, "cudaMalloc(ragged prefill state %zu B) failed: %s", need, cudaGetErrorString(e));
    h->rg_state_bytes = need;
  }
  xl::launch_state_permute(state, h->rg_state, p.d_perm, Bc, state_copy_geom(h, B, Bc), 0, s);
  h->launches += 1;
  XL_CUDA(cudaGetLastError());
  p.st = h->rg_state;
  p.Btot = Bc;
  return XL_OK;
}

int ragged_end(xl_handle* h, void* state, int B, const SeqPlan& p, cudaStream_t s) {
  if (p.in_place) return XL_OK;
  const int Bc = (int)p.perm.size();
  xl::launch_state_permute(state, h->rg_state, p.d_perm, Bc, state_copy_geom(h, B, Bc), 1, s);
  h->launches += 1;
  XL_CUDA(cudaGetLastError());
  return XL_OK;
}

// Chunks of the shrinking active prefix: today's chunk length for Bk envs (prefill_chunk_tokens), cut to the longest
// remaining context rounded up to 8 units (16 where the chunkwise cells run: whole 16-token chunks of the mma.sync cell).
void ragged_chunks(const xl_handle* h, SeqPlan& p) {
  const int gran = (h->prefill_cell >= 1 && xl::prefill_cell_mma_supported(h->DH)) ? 16 : 8;
  const std::vector<int32_t>& len = p.len;
  int pos = 0, Bk = (int)len.size();
  while (pos < len[0]) {
    while (len[Bk - 1] <= pos) --Bk;
    const int cmax = prefill_chunk_tokens(h, Bk) / p.T;
    const int n = std::min(cmax, (len[0] - pos + gran - 1) / gran * gran);
    p.chunks.push_back({pos, Bk, n});
    pos += n;
  }
}

// Chunks of all B envs, each a multiple of 8 units (of 16 where the mma.sync cell runs; an 8-unit remainder takes the
// fp32 cell); the last S mod 8 units, and every unit of a shape without the sequence path, form the eager tail.
void uniform_chunks(const xl_handle* h, int B, int S, SeqPlan& p) {
  int pos = 0;
  if (prefill_fast_path(h)) {
    const int cmax = prefill_chunk_tokens(h, B) / p.T;
    while (S - pos >= 8) {
      int n = std::min(cmax, (S - pos) / 8 * 8);
      if (h->prefill_cell >= 1 && xl::prefill_cell_mma_supported(h->DH) && n >= 16) n = n / 16 * 16;
      p.chunks.push_back({pos, B, n});
      pos += n;
    }
  }
  p.tail = pos;
}

// The plan of one call of B envs x S units (lengths: host, or nullptr for a uniform call), the ragged state gathered,
// and the prefill workspace grown to its largest chunk: rows, and the gate-scan scratch of gate_pre_seq_kernel.
int seq_plan(xl_handle* h, void* state, const int32_t* lengths, int B, int S, SeqPlan& p, cudaStream_t s) {
  if (lengths) {
    if (int rc = ragged_begin(h, state, lengths, B, p, s)) return rc;
    ragged_chunks(h, p);
    p.tail = S;
  } else {
    p.st = state;
    p.Btot = B;
    uniform_chunks(h, B, S, p);
  }
  int rows = 0;
  size_t gsc = 0;
  for (const SeqChunk& ch : p.chunks) {
    rows = std::max(rows, ch.Bk * ch.n * p.T);
    gsc = std::max(gsc, xl::gate_scan_seq_scratch_floats(ch.Bk, ch.n * p.T, h->cfg.num_heads));
  }
  return ensure_prefill_ws(h, rows, gsc);
}

// Moves chunk ch's rows between a caller's [B, S, width] buffer and a chunk buffer [Bk, n, width]: to the chunk
// (to_caller 0; ragged pads zero-filled) or back to the caller (to_caller 1; ragged: valid rows only).
int chunk_rows(xl_handle* h, const SeqPlan& p, const SeqChunk& ch, float* caller, float* chunk, int S, int width,
               int to_caller, cudaStream_t s) {
  if (p.d_len) {
    xl::launch_ragged_rows(caller, chunk, p.d_perm, p.d_len, p.T, ch.Bk, S, ch.n, ch.pos, width, to_caller, s);
    h->launches += 1;
    return XL_OK;
  }
  const size_t cpitch = sizeof(float) * (size_t)S * width, kpitch = sizeof(float) * (size_t)ch.n * width;
  float* c = caller + (size_t)ch.pos * width;
  if (to_caller)
    XL_CUDA(cudaMemcpy2DAsync(c, cpitch, chunk, kpitch, kpitch, ch.Bk, cudaMemcpyDeviceToDevice, s));
  else
    XL_CUDA(cudaMemcpy2DAsync(chunk, kpitch, c, cpitch, kpitch, ch.Bk, cudaMemcpyDeviceToDevice, s));
  return XL_OK;
}

// ---- sequence forward: the action head of every timestep ----------------------------------------------------------
// The forward calls run the policy prefill and also emit the action outputs of every timestep from what each chunk (and
// each eager tail step) leaves behind, so their state is the prefill's.
struct SeqHead {
  xl_seq_outputs out;
  int discrete, n_out, Tn;
};

int ensure_seq_logits(xl_handle* h, size_t floats) {
  if (floats <= h->sq_logits_floats) return XL_OK;
  XL_CUDA(cudaDeviceSynchronize());            // nothing may still be using the old workspace
  if (h->sq_logits) cudaFree(h->sq_logits);
  h->sq_logits = nullptr;
  h->sq_logits_floats = 0;
  cudaError_t e = cudaMalloc((void**)&h->sq_logits, sizeof(float) * floats);
  if (e != cudaSuccess)
    return fail(XL_ERR_CUDA, "cudaMalloc(sequence logits %zu B) failed: %s", sizeof(float) * floats, cudaGetErrorString(e));
  h->sq_logits_floats = floats;
  return XL_OK;
}

// tokens / actions / logprobs / logits of `rows` timesteps whose logits sit in sq_logits (see xl::SeqHeadParams)
void seq_head_reduce(xl_handle* h, const SeqHead& hd, int rows, int Tc, int pos, const int32_t* perm,
                     const int32_t* len, cudaStream_t s) {
  const xl_config& c = h->cfg;
  xl::SeqHeadParams p;
  p.logits = h->sq_logits;
  p.rows = rows; p.Tc = Tc; p.pos = pos; p.Tn = hd.Tn;
  p.n_out = hd.n_out; p.act_dim = c.act_dim; p.num_actions = h->num_actions; p.discrete_actions = c.discrete_actions;
  p.discrete = hd.discrete;
  p.bin_width = hd.discrete ? 0.f : (c.tok_max_val - c.tok_min_val) / (float)c.action_channels;
  p.min_val = hd.discrete ? 0.f : c.tok_min_val;
  p.perm = perm; p.len = len; p.len_div = c.tokens_per_step;
  p.tokens = hd.out.tokens; p.actions = hd.out.actions; p.out_logits = hd.out.logits;
  p.targets = hd.out.targets; p.logprobs = hd.out.logprobs;
  xl::launch_seq_head(p, s);
  h->launches += 1;
}

// Head of one prefill chunk of Bk envs x Tc timesteps, after prefill_blocks: post_blocks_norm of the rtg-token rows of
// pf_x only (complete there: the prefill's proj_down leaves no split-K planes), emitted as the head's bf16 operand planes
// where the tcgen05 Linear runs; the head Linear over the chunk's Bk*Tc timesteps into sq_logits; the reduction.
int seq_head_chunk(xl_handle* h, const SeqHead& hd, int Bk, int Tc, int pos, const int32_t* perm, const int32_t* len,
                   unsigned flags, cudaStream_t s) {
  const xl_config& c = h->cfg;
  const int d = c.embedding_dim, T = c.tokens_per_step, rows = Bk * Tc;
  const Ws ws = prefill_ws(h);
  const int impl = (flags & XL_FLAG_SIMPLE_GEMM) ? 1 : h->gemm_impl;
  auto PW = [&](int id) { return h->pw[id - XL_W_POST_NORM]; };
  const float* post_w = (const float*)PW(XL_W_POST_NORM);
  int rc = ensure_seq_logits(h, (size_t)rows * hd.n_out);
  if (rc) return rc;
  const bool tc = impl != 1 && xl::gemm_tc_supported(rows, hd.n_out, d) && (size_t)rows * d <= ws.a_cap && d <= 4096;
  if (tc)
    xl::launch_ln_rows_gather(ws.x, nullptr, 1, 0, post_w, c.ln_eps, rows, d, T, c.action_token_pos, ws.a_hi, ws.a_lo, s);
  else
    xl::launch_ln_rows(ws.x + (size_t)c.action_token_pos * d, (int64_t)T * d, ws.xn, d, post_w, nullptr, 1, c.ln_eps,
                       rows, d, nullptr, nullptr, s);
  h->launches += 1;
  rc = linear(h, ws, ws.xn, PW(XL_W_HEAD_W), (const float*)PW(XL_W_HEAD_B), nullptr, h->sq_logits, rows, hd.n_out, d,
              impl, s, /*presplit=*/tc);
  if (rc) return rc;
  seq_head_reduce(h, hd, rows, Tc, pos, perm, len, s);
  XL_CUDA(cudaGetLastError());
  return XL_OK;
}

// Every output position of the call set to its past-the-length value (tokens -1, the rest 0): the ragged forward then
// writes only the timesteps its envs have.
int seq_clear_outputs(const xl_handle* h, const SeqHead& hd, int B, cudaStream_t s) {
  const size_t pos = (size_t)B * hd.Tn, A = h->cfg.act_dim;
  if (hd.out.tokens) XL_CUDA(cudaMemsetAsync(hd.out.tokens, 0xff, sizeof(int32_t) * pos * A, s));
  if (hd.out.actions) XL_CUDA(cudaMemsetAsync(hd.out.actions, 0, sizeof(float) * pos * A, s));
  if (hd.out.logprobs) XL_CUDA(cudaMemsetAsync(hd.out.logprobs, 0, sizeof(float) * pos * A, s));
  if (hd.out.logits) XL_CUDA(cudaMemsetAsync(hd.out.logits, 0, sizeof(float) * pos * hd.n_out, s));
  return XL_OK;
}

// encoder_only: the block stack + post_blocks_norm (what xl_encoder_step / xl_prefill read); otherwise also the
// policy-level embeddings and the action head (xl_policy_*).
int weights_ready(const xl_handle* h, bool encoder_only) {
  if (!h) return fail(XL_ERR_INVALID_ARG, "null handle");
  static const int s_ids[] = {XL_W_XLSTM_NORM, XL_W_CONV_W, XL_W_CONV_B, XL_W_S_GATE_I, XL_W_S_GATE_F, XL_W_S_GATE_Z,
                              XL_W_S_GATE_O, XL_W_S_RECURRENT, XL_W_S_BIAS, XL_W_S_GROUP_NORM, XL_W_FFN_NORM,
                              XL_W_FFN_UP, XL_W_FFN_DOWN};
  for (int i = 0; i < h->cfg.num_blocks; ++i) {
    if (is_slstm(h, i)) {
      for (int k : s_ids)
        if (!h->blocks[i].w[k]) return fail(XL_ERR_NOT_READY, "sLSTM block %d weight id %d not bound", i, k);
      continue;
    }
    for (int k = 0; k <= XL_W_PROJ_DOWN; ++k)
      if (!h->blocks[i].w[k]) return fail(XL_ERR_NOT_READY, "block %d weight id %d not bound", i, k);
  }
  const int last = encoder_only ? XL_W_POST_NORM : XL_W_HEAD_B;
  for (int id = XL_W_POST_NORM; id <= last; ++id)
    if (!h->pw[id - XL_W_POST_NORM]) return fail(XL_ERR_NOT_READY, "policy weight id %d not bound", id);
  return XL_OK;
}

// CUDA-graph replay of a step entry: replays the graph captured for `key`, or captures record(stream) -- which enqueues
// the step on the stream it is given -- into a new graph on cap_stream and launches it. At most 8 graphs are kept,
// the oldest evicted first. h->launches counts the graph's kernels on every launch; the capture itself counts none.
template <class Record>
int run_graph(xl_handle* h, const GraphKey& key, cudaStream_t s, Record&& record) {
  for (auto& g : h->graphs) {
    if (g.key == key) {
      XL_CUDA(cudaGraphLaunch(g.exec, s));
      h->launches += g.launches;
      return XL_OK;
    }
  }
  int rc = weights_ready(h, key.entry == GraphKey::kEncoderStep);
  if (rc) return rc;
  // make sure every lazy attribute (dynamic smem opt-in) is set before capture: one eager warm-up is NOT
  // done here because it would advance the state; attributes are set inside launch paths, which is legal
  // during capture (cudaFuncSetAttribute is not a stream operation).
  GraphCacheEntry g;
  g.key = key;
  cudaGraph_t graph = nullptr;
  const int64_t before = h->launches;
  XL_CUDA(cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal));
  rc = record(h->cap_stream);
  cudaError_t e = cudaStreamEndCapture(h->cap_stream, &graph);
  g.launches = h->launches - before;
  h->launches = before;
  if (rc) {
    if (graph) cudaGraphDestroy(graph);
    return rc;
  }
  if (e != cudaSuccess) return fail(XL_ERR_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(e));
  e = cudaGraphInstantiate(&g.exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) return fail(XL_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e));
  if (h->graphs.size() >= 8) {
    cudaGraphExecDestroy(h->graphs.front().exec);
    h->graphs.erase(h->graphs.begin());
  }
  h->graphs.push_back(g);
  XL_CUDA(cudaGraphLaunch(g.exec, s));
  h->launches += g.launches;
  return XL_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

int xl_abi_version(void) { return XL_ABI_VERSION; }
const char* xl_last_error(void) { return g_err; }

int xl_create(const xl_config* cfg, xl_handle** out) {
  if (!cfg || !out) return fail(XL_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  const xl_config& c = *cfg;
  if (c.embedding_dim <= 0 || c.embedding_dim % 8) return fail(XL_ERR_UNSUPPORTED, "embedding_dim %% 8 != 0");
  if (c.num_heads <= 0 || c.num_heads > 8) return fail(XL_ERR_UNSUPPORTED, "num_heads must be in [1,8]");
  if (c.inner_dim <= 0 || c.inner_dim % (4 * c.num_heads) || c.inner_dim % 8)
    return fail(XL_ERR_UNSUPPORTED, "inner_dim must be a multiple of 8 and of 4*num_heads");
  if (c.qkv_blocksize != 4) return fail(XL_ERR_UNSUPPORTED, "qkv_blocksize must be 4");
  if (c.conv_kernel < 2 || c.conv_kernel > 4) return fail(XL_ERR_UNSUPPORTED, "conv_kernel must be in [2,4]");
  if (c.tokens_per_step < 1 || c.tokens_per_step > 4) return fail(XL_ERR_UNSUPPORTED, "tokens_per_step in [1,4]");
  if (c.action_token_pos < 0 || c.action_token_pos >= c.tokens_per_step)
    return fail(XL_ERR_INVALID_ARG, "action_token_pos out of range");
  if (c.max_batch <= 0 || c.num_blocks <= 0) return fail(XL_ERR_INVALID_ARG, "max_batch/num_blocks <= 0");
  if (c.tokens_per_step != 3)
    return fail(XL_ERR_UNSUPPORTED, "policy token layout is (s, rtg, r): tokens_per_step must be 3");
  const int DH = c.inner_dim / c.num_heads;
  if (DH > 1024) return fail(XL_ERR_UNSUPPORTED, "head_dim > 1024");
  const uint64_t smask = ((uint64_t)c.slstm_mask_hi << 32) | c.slstm_mask_lo;
  if (smask) {
    if (c.num_blocks < 64 && (smask >> c.num_blocks)) return fail(XL_ERR_INVALID_ARG, "slstm_mask names a block >= num_blocks");
    if (c.num_blocks > 64) return fail(XL_ERR_UNSUPPORTED, "sLSTM stacks: num_blocks <= 64");
    if (c.embedding_dim % c.num_heads) return fail(XL_ERR_UNSUPPORTED, "sLSTM: embedding_dim %% num_heads != 0");
    if (c.ffn_dim <= 0 || c.ffn_dim % 8) return fail(XL_ERR_UNSUPPORTED, "sLSTM: ffn_dim must be a positive multiple of 8");
    if (2 * c.ffn_dim > 3 * c.inner_dim || c.ffn_dim > c.inner_dim || 4 * c.embedding_dim > 2 * c.inner_dim)
      return fail(XL_ERR_UNSUPPORTED, "sLSTM: ffn_dim %d / d %d do not fit the workspace of inner_dim %d", c.ffn_dim,
                  c.embedding_dim, c.inner_dim);
    if ((size_t)8 * (c.embedding_dim / c.num_heads) * 4 + 8 * 8 * 4 * 32 * 4 > 200 * 1024)
      return fail(XL_ERR_UNSUPPORTED, "sLSTM: head_dim too large for the cell kernel");
  }

  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(XL_ERR_NO_DEVICE, "no CUDA device: the xlstm_b200 path has no CPU fallback");
  }
  xl_handle* h = new (std::nothrow) xl_handle();
  if (!h) return fail(XL_ERR_INVALID_ARG, "out of host memory");
  h->cfg = c;
  h->DH = DH;
  h->slstm_mask = smask;
  {
    // gate pre-activations are produced as NCH partial sums (64 four-channel blocks per chunk), summed in
    // fixed order by the state kernels
    const int nblk = c.inner_dim / 4;
    int nch = (nblk + 63) / 64;
    if (nch < 1) nch = 1;
    if (nch > 16) nch = 16;
    h->NCH = nch;
    if ((nblk + nch - 1) / nch > 128) { delete h; return fail(XL_ERR_UNSUPPORTED, "inner_dim too large"); }
  }
  h->Kpad = (int)align_up((size_t)c.state_dim, 64);
  h->num_actions = c.discrete_actions + c.action_channels;
  h->head_out = h->num_actions * c.act_dim;
  h->blocks.resize(c.num_blocks);
  for (auto& b : h->blocks) memset(&b, 0, sizeof(b));
  memset(h->pw, 0, sizeof(h->pw));
  cudaGetDevice(&h->device);
  cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device);

  // workspace carve-up
  const size_t M = (size_t)c.max_batch * 4;  // up to 4 tokens per step
  const size_t B = (size_t)c.max_batch;
  const size_t d = c.embedding_dim, inner = c.inner_dim;
  size_t off = 0;
  auto carve = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  };
  const size_t o_x = carve(4 * M * d), o_xn = carve(4 * M * d), o_xtok = carve(4 * M * d);
  const size_t o_hid = carve(4 * M * d);
  const size_t o_u = carve(4 * M * 2 * inner), o_qkv = carve(4 * M * 3 * inner), o_act = carve(4 * M * inner);
  h->gp_chunks = std::max(16, xl::gemm_up_conv_chunks((int)inner));
  const size_t o_gp = carve(4 * M * h->gp_chunks * 2 * c.num_heads), o_gated = carve(4 * M * inner);
  const size_t o_part = carve(4 * B * c.num_heads * 32 * 4 * DH);  // RS <= 32, T <= 4
  const size_t o_semb = carve(4 * B * d), o_sp = carve(4 * B * h->Kpad), o_lg = carve(4 * B * h->head_out);
  const size_t o_ds = carve(4 * B * c.state_dim), o_dr = carve(4 * B), o_dw = carve(4 * B);
  const size_t o_da = carve(4 * B * c.act_dim), o_dt = carve(4 * B * c.act_dim);
  h->num_tickets = 4096;
  const size_t o_cnt = carve(4 * (size_t)h->num_tickets);

  size_t a_cap = M * (inner > d ? inner : d);
  if (a_cap < B * (size_t)h->Kpad) a_cap = B * (size_t)h->Kpad;
  if (a_cap < (size_t)1 << 20) a_cap = (size_t)1 << 20;   // room for xl_linear unit tests
  h->a_cap = a_cap;
  const size_t o_hi = carve(2 * a_cap), o_lo = carve(2 * a_cap);
  h->part_rows = M < kSplitRows ? M : kSplitRows;
  const size_t o_pu = carve(4 * (size_t)kSplitMax * h->part_rows * 2 * inner);
  const size_t o_pd = carve(4 * (size_t)kSplitMax * h->part_rows * d);
  const size_t o_de = carve(4 * B * d);   // last, so that the step's buffers keep their places
  h->ws_bytes = off;
  cudaError_t e = cudaMalloc((void**)&h->ws, h->ws_bytes);
  if (e != cudaSuccess) {
    delete h;
    return fail(XL_ERR_CUDA, "cudaMalloc(workspace %zu B) failed: %s", off, cudaGetErrorString(e));
  }
  cudaMemset(h->ws, 0, h->ws_bytes);
  cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking);
  cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
  h->x = (float*)(h->ws + o_x); h->xn = (float*)(h->ws + o_xn); h->xtok = (float*)(h->ws + o_xtok);
  h->hid = (float*)(h->ws + o_hid);
  h->u = (float*)(h->ws + o_u); h->qkv = (float*)(h->ws + o_qkv); h->act = (float*)(h->ws + o_act);
  h->gate_part = (float*)(h->ws + o_gp); h->gated = (float*)(h->ws + o_gated);
  h->partial = (float*)(h->ws + o_part); h->s_emb = (float*)(h->ws + o_semb);
  h->states_pad = (float*)(h->ws + o_sp); h->logits = (float*)(h->ws + o_lg);
  h->d_states = (float*)(h->ws + o_ds); h->d_rtg = (float*)(h->ws + o_dr); h->d_rew = (float*)(h->ws + o_dw);
  h->d_actions = (float*)(h->ws + o_da); h->d_tokens = (int32_t*)(h->ws + o_dt);
  h->counters = (unsigned int*)(h->ws + o_cnt);

  h->a_hi = (__nv_bfloat16*)(h->ws + o_hi); h->a_lo = (__nv_bfloat16*)(h->ws + o_lo);
  h->part_up = (float*)(h->ws + o_pu); h->part_down = (float*)(h->ws + o_pd);
  h->d_embeds = (float*)(h->ws + o_de);
  *out = h;
  return XL_OK;
}

void xl_destroy(xl_handle* h) {
  if (!h) return;
  clear_graphs(h);
  if (h->ws) cudaFree(h->ws);
  if (h->pf_tc) cudaFree(h->pf_tc);
  if (h->pf_buf) cudaFree(h->pf_buf);
  if (h->rg_state) cudaFree(h->rg_state);
  if (h->rg_idx) cudaFree(h->rg_idx);
  if (h->sq_logits) cudaFree(h->sq_logits);
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  if (h->side) cudaStreamDestroy(h->side);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  delete h;
}

int xl_state_dim_padded(const xl_handle* h) { return h ? h->Kpad : 0; }

int xl_bind_weight(xl_handle* h, int layer, int which, const void* dev_ptr, int dtype, int64_t numel) {
  if (!h || !dev_ptr) return fail(XL_ERR_INVALID_ARG, "null argument");
  const xl_config& c = h->cfg;
  const int64_t d = c.embedding_dim, inner = c.inner_dim, NH = c.num_heads, KS = c.conv_kernel;
  int64_t want = -1;
  int want_dtype = 0;
  if (layer >= 0) {
    if (layer >= c.num_blocks) return fail(XL_ERR_INVALID_ARG, "layer %d >= num_blocks", layer);
    const int64_t DHs = d / NH, ff = c.ffn_dim;
    if (is_slstm(h, layer)) switch (which) {
      case XL_W_XLSTM_NORM: case XL_W_CONV_B: case XL_W_S_GROUP_NORM: case XL_W_FFN_NORM: want = d; break;
      case XL_W_CONV_W: want = d * KS; break;
      case XL_W_S_GATE_I: case XL_W_S_GATE_F: case XL_W_S_GATE_Z: case XL_W_S_GATE_O: want = NH * DHs * DHs; break;
      case XL_W_S_RECURRENT: want = NH * DHs * 4 * DHs; break;
      case XL_W_S_BIAS: want = NH * 4 * DHs; break;
      case XL_W_FFN_UP: want = 2 * ff * d; want_dtype = 1; break;
      case XL_W_FFN_DOWN: want = d * ff; want_dtype = 1; break;
      default: return fail(XL_ERR_INVALID_ARG, "weight id %d does not belong to an sLSTM block (layer %d)", which, layer);
    }
    else switch (which) {
      case XL_W_XLSTM_NORM: want = d; break;
      case XL_W_PROJ_UP: want = 2 * inner * d; want_dtype = 1; break;
      case XL_W_Q_PROJ: case XL_W_K_PROJ: case XL_W_V_PROJ: want = inner * 4; break;
      case XL_W_CONV_W: want = inner * KS; break;
      case XL_W_CONV_B: want = inner; break;
      case XL_W_IGATE_W: case XL_W_FGATE_W: want = NH * 3 * inner; break;
      case XL_W_IGATE_B: case XL_W_FGATE_B: want = NH; break;
      case XL_W_OUTNORM: case XL_W_SKIP: want = inner; break;
      case XL_W_PROJ_DOWN: want = d * inner; want_dtype = 1; break;
      default: return fail(XL_ERR_INVALID_ARG, "unknown per-block weight id %d", which);
    }
  } else {
    switch (which) {
      case XL_W_POST_NORM: want = d; break;
      case XL_W_EMBED_STATE_W: want = d * h->Kpad; want_dtype = 1; break;
      case XL_W_EMBED_STATE_B: case XL_W_EMBED_RETURN_W: case XL_W_EMBED_RETURN_B:
      case XL_W_EMBED_REWARD_W: case XL_W_EMBED_REWARD_B: case XL_W_EMBED_LN_W: case XL_W_EMBED_LN_B:
        want = d; break;
      case XL_W_HEAD_W: want = (int64_t)h->head_out * d; want_dtype = 1; break;
      case XL_W_HEAD_B: want = h->head_out; break;
      default: return fail(XL_ERR_INVALID_ARG, "unknown policy weight id %d", which);
    }
  }
  if (numel != want) return fail(XL_ERR_INVALID_ARG, "weight %d (layer %d): numel %lld, expected %lld", which,
                                 layer, (long long)numel, (long long)want);
  if (dtype != want_dtype)
    return fail(XL_ERR_INVALID_ARG, "weight %d (layer %d): dtype %d, expected %d (0=fp32,1=bf16)", which, layer,
                dtype, want_dtype);
  if (((uintptr_t)dev_ptr) % 16) return fail(XL_ERR_INVALID_ARG, "weight pointer must be 16-byte aligned");
  if (layer >= 0) h->blocks[layer].w[which] = dev_ptr;
  else h->pw[which - XL_W_POST_NORM] = dev_ptr;
  clear_graphs(h);   // bound pointers are baked into cached graphs
  return XL_OK;
}

int xl_weights_ready(const xl_handle* h) { return weights_ready(h, false); }

int xl_encoder_weights_ready(const xl_handle* h) { return weights_ready(h, true); }

size_t xl_state_bytes(const xl_handle* h, int B) {
  if (!h || B <= 0) return 0;
  return layer_base(h, state_layout(h, B), h->cfg.num_blocks);
}

int xl_state_layout(const xl_handle* h, int B, int layer, int part, size_t* offset_bytes, size_t* size_bytes) {
  if (!h || !offset_bytes || !size_bytes) return fail(XL_ERR_INVALID_ARG, "null argument");
  if (layer < 0 || layer >= h->cfg.num_blocks || B <= 0) return fail(XL_ERR_INVALID_ARG, "bad layer/B");
  const StateLayout L = state_layout(h, B);
  const xl_config& c = h->cfg;
  size_t o, sz;
  if (is_slstm(h, layer)) {
    switch (part) {
      case XL_STATE_SLSTM: o = L.s_off; sz = sizeof(float) * (size_t)4 * B * c.embedding_dim; break;
      case XL_STATE_CONV: o = L.sconv_off; sz = sizeof(float) * (size_t)B * c.conv_kernel * c.embedding_dim; break;
      default: return fail(XL_ERR_INVALID_ARG, "state part %d does not exist in sLSTM block %d", part, layer);
    }
    *offset_bytes = layer_base(h, L, layer) + o;
    *size_bytes = sz;
    return XL_OK;
  }
  switch (part) {
    case XL_STATE_C: o = L.c_off; sz = sizeof(float) * (size_t)B * c.num_heads * h->DH * h->DH; break;
    case XL_STATE_N: o = L.n_off; sz = sizeof(float) * (size_t)B * c.num_heads * h->DH; break;
    case XL_STATE_M: o = L.m_off; sz = sizeof(float) * (size_t)B * c.num_heads; break;
    case XL_STATE_CONV: o = L.conv_off; sz = sizeof(float) * (size_t)B * c.conv_kernel * c.inner_dim; break;
    default: return fail(XL_ERR_INVALID_ARG, "bad state part %d", part);
  }
  *offset_bytes = layer_base(h, L, layer) + o;
  *size_bytes = sz;
  return XL_OK;
}

int xl_state_reset(xl_handle* h, void* state, const uint8_t* env_mask, int B, void* stream) {
  int rc = check_batch(h, B);
  if (rc) return rc;
  if (!state) return fail(XL_ERR_INVALID_ARG, "null state");
  cudaStream_t s = (cudaStream_t)stream;
  const StateLayout L = state_layout(h, B);
  const xl_config& c = h->cfg;
  if (!env_mask) {
    XL_CUDA(cudaMemsetAsync(state, 0, layer_base(h, L, c.num_blocks), s));
    return XL_OK;
  }
  for (int i = 0; i < c.num_blocks; ++i) {
    char* base = (char*)state + layer_base(h, L, i);
    if (is_slstm(h, i)) {
      const int64_t d = c.embedding_dim, Bd = (int64_t)B * d;
      float* st = (float*)(base + L.s_off);
      xl::launch_state_reset((float*)(base + L.sconv_off), st, st + Bd, st + 2 * Bd, env_mask, B,
                             (int64_t)c.conv_kernel * d, d, d, d, s);
      xl::launch_state_reset(nullptr, st + 3 * Bd, nullptr, nullptr, env_mask, B, 0, d, 0, 0, s);
      h->launches += 2;
      continue;
    }
    xl::launch_state_reset((float*)(base + L.c_off), (float*)(base + L.n_off), (float*)(base + L.m_off),
                           (float*)(base + L.conv_off), env_mask, B, (int64_t)c.num_heads * h->DH * h->DH,
                           (int64_t)c.num_heads * h->DH, c.num_heads, (int64_t)c.conv_kernel * c.inner_dim, s);
    h->launches += 1;
  }
  XL_CUDA(cudaGetLastError());
  return XL_OK;
}

int xl_encoder_step(xl_handle* h, void* state, const float* x_in, float* x_out, int B, int T, int mode,
                    unsigned flags, void* stream) {
  int rc = check_batch(h, B);
  if (rc) return rc;
  if (!state || !x_in || !x_out) return fail(XL_ERR_INVALID_ARG, "null argument");
  if (T < 1 || T > 4) return fail(XL_ERR_UNSUPPORTED, "T=%d outside [1,4]", T);
  cudaStream_t s = (cudaStream_t)stream;
  auto record = [&](cudaStream_t rs) {
    return run_encoder(h, state, make_step(h, B, rs), x_in, x_out, T, mode, flags & ~(unsigned)XL_FLAG_GRAPH);
  };
  if (!(flags & XL_FLAG_GRAPH) || h->profiling) {
    rc = weights_ready(h, true);
    return rc ? rc : record(s);
  }
  // the encoder-only swap of decision_xlstm.py:188-189 at small batch is launch-bound when its ~6 kernels per block
  // are enqueued eagerly
  const GraphKey key = {GraphKey::kEncoderStep, state, x_in, nullptr, nullptr, nullptr, nullptr, nullptr, x_out,
                        B, T, mode, flags};
  return run_graph(h, key, s, record);
}

int xl_mlstm_cell_step(xl_handle* h, float* C, float* n, float* m, const float* qkv, const float* igate,
                       const float* fgate, const float* outnorm_w, float* h_norm, float* h_raw, int B, int T,
                       int rows_split, int cols_per_cta, void* stream) {
  int rc = check_batch(h, B);
  if (rc) return rc;
  if (!C || !n || !m || !qkv || !igate || !fgate || !outnorm_w || !h_norm)
    return fail(XL_ERR_INVALID_ARG, "null argument");
  if (T < 1 || T > 4) return fail(XL_ERR_UNSUPPORTED, "T=%d outside [1,4]", T);
  if (rows_split > 32) return fail(XL_ERR_UNSUPPORTED, "rows_split > 32");
  const xl_config& c = h->cfg;
  cudaStream_t s = (cudaStream_t)stream;
  // pack the caller's gate pre-activations as a single "chunk": [M, 1, 2*NH]
  const int M = B * T, NH = c.num_heads;
  XL_CUDA(cudaMemcpy2DAsync(h->gate_part, sizeof(float) * 2 * NH, igate, sizeof(float) * NH, sizeof(float) * NH,
                            M, cudaMemcpyDeviceToDevice, s));
  XL_CUDA(cudaMemcpy2DAsync(h->gate_part + NH, sizeof(float) * 2 * NH, fgate, sizeof(float) * NH,
                            sizeof(float) * NH, M, cudaMemcpyDeviceToDevice, s));
  xl::StateStepParams sp;
  memset(&sp, 0, sizeof(sp));
  xl::launch_repack_qkv(qkv, h->qkv, h->qkv + (size_t)2 * M * c.inner_dim, M, c.inner_dim, s);
  sp.C = C; sp.n = n; sp.m = m; sp.qk = h->qkv; sp.v = h->qkv + (size_t)2 * M * c.inner_dim;
  sp.gate_part = h->gate_part;
  sp.outnorm_w = outnorm_w; sp.out = h_norm; sp.h_raw = h_raw;
  sp.partial = h->partial;
  sp.B = B; sp.T = T; sp.NH = NH; sp.DH = h->DH; sp.inner = c.inner_dim; sp.NCH = 1;
  sp.rows_split = rows_split; sp.cols_per_cta = cols_per_cta;
  sp.ln_eps = c.ln_eps; sp.cell_eps = c.cell_eps;
  sp.impl = h->state_impl; sp.num_layers = c.num_blocks;
  sp.stages = h->state_stages; sp.ctas_per_sm = h->state_ctas_per_sm;
  sp.fuse_finalize = h->state_fuse;
  cudaEvent_t pe0 = nullptr, pe1 = nullptr;
  if (h->profiling) {
    XL_CUDA(cudaEventCreate(&pe0));
    XL_CUDA(cudaEventCreate(&pe1));
    XL_CUDA(cudaEventRecord(pe0, s));
  }
  XL_CUDA(xl::launch_state_step(sp, h->num_sms, s));
  if (h->profiling) {
    XL_CUDA(cudaEventRecord(pe1, s));
    h->prof_state.push_back(pe0);
    h->prof_state.push_back(pe1);
  }
  if (!xl::state_step_fuses_finalize(sp, h->num_sms)) XL_CUDA(xl::launch_state_finalize(sp, h->num_sms, s));
  h->launches += 3;
  return XL_OK;
}

int xl_mlstm_cell_seq(xl_handle* h, float* C, float* n, float* m, const float* q, const float* k, const float* v,
                      const float* gates, const float* act, const float* u, const float* outnorm_w, const float* skip,
                      float* num, float* qn, float* mseq, float* out, int* cell, int B, int S, void* stream) {
  int rc = check_batch(h, B);
  if (rc) return rc;
  if (!C || !n || !m || !q || !k || !v || !gates || !act || !u || !outnorm_w || !skip || !num || !qn || !mseq || !out)
    return fail(XL_ERR_INVALID_ARG, "null argument");
  if (S < 1) return fail(XL_ERR_INVALID_ARG, "S=%d", S);
  const xl_config& c = h->cfg;
  const int which = seq_cell_choice(h, B, S);
  if (which != h->prefill_cell)
    return fail(XL_ERR_UNSUPPORTED, "prefill_cell %d cannot take DH=%d over %d tokens of %d envs", h->prefill_cell,
                h->DH, S, B);
  cudaStream_t s = (cudaStream_t)stream;
  rc = ensure_prefill_ws(h, B * S, xl::gate_scan_seq_scratch_floats(B, S, c.num_heads));
  if (rc) return rc;
  rc = seq_cell(h, C, n, m, q, k, v, gates, nullptr, nullptr, num, qn, mseq, B, S, 1, s, nullptr, 0, cell);
  if (rc) return rc;
  XL_CUDA(xl::launch_finalize_seq(num, qn, mseq, outnorm_w, skip, act, u, out, nullptr, nullptr, B, S, c.num_heads,
                                  h->DH, c.inner_dim, c.ln_eps, c.cell_eps, s));
  h->launches += 1;
  return XL_OK;
}

int xl_policy_step(xl_handle* h, void* state, const float* states, const float* rtg, const float* rewards,
                   int32_t* tokens, float* actions, float* logits, float* hidden, int B, int mode,
                   unsigned flags, void* stream) {
  int rc = check_batch(h, B);
  if (rc) return rc;
  if (!state || !states || !rtg || !tokens || !actions) return fail(XL_ERR_INVALID_ARG, "null argument");
  if (mode != XL_MODE_FUSED && mode != XL_MODE_PER_TOKEN) return fail(XL_ERR_INVALID_ARG, "unknown mode %d", mode);
  cudaStream_t s = (cudaStream_t)stream;
  StepArgs args;
  args.state = state; args.states = states; args.rtg = rtg; args.rewards = rewards; args.tokens = tokens;
  args.actions = actions; args.logits = logits; args.hidden = hidden; args.B = B; args.mode = mode; args.flags = flags;
  if (!(flags & XL_FLAG_GRAPH) || h->profiling) {     // profiling brackets eager launches with events: no replay
    rc = xl_weights_ready(h);
    if (rc) return rc;
    args.flags &= ~(unsigned)XL_FLAG_GRAPH;
    cudaEvent_t pe0 = nullptr, pe1 = nullptr;
    if (h->profiling) {
      XL_CUDA(cudaEventCreate(&pe0));
      XL_CUDA(cudaEventCreate(&pe1));
      XL_CUDA(cudaEventRecord(pe0, s));
    }
    rc = run_policy(h, args, s);
    if (h->profiling) {
      cudaEventRecord(pe1, s);
      h->prof_step.push_back(pe0);
      h->prof_step.push_back(pe1);
    }
    return rc;
  }
  const GraphKey key = {GraphKey::kPolicyStep, state, states, rtg, rewards, tokens, actions, logits, hidden,
                        B, 0, mode, flags};
  return run_graph(h, key, s, [&](cudaStream_t rs) { return run_policy(h, args, rs); });
}

int xl_policy_step_host(xl_handle* h, void* state, const float* h_states, const float* h_rtg,
                        const float* h_rewards, int32_t* h_tokens, float* h_actions, int B, int mode,
                        unsigned flags, void* stream) {
  int rc = check_batch(h, B);
  if (rc) return rc;
  if (!state || !h_states || !h_rtg || !h_tokens || !h_actions) return fail(XL_ERR_INVALID_ARG, "null argument");
  if (flags & XL_FLAG_STATE_EMBEDS)
    return fail(XL_ERR_UNSUPPORTED, "xl_policy_step_host takes raw states; state embeddings are device tensors "
                                    "(use xl_policy_step with XL_FLAG_STATE_EMBEDS)");
  cudaStream_t s = (cudaStream_t)stream;
  const xl_config& c = h->cfg;
  if (h->host_zero_copy) {
    // Pinned host memory is mapped into the device address space (UVA): the first kernel of the step reads the 52 KB
    // of states / rtg over PCIe itself and the argmax kernel stores the 4 KB of tokens / actions straight into the
    // caller's buffers — no DMA copy launches (each ~8-10 us of latency) around the graph launch, one stream
    // synchronisation at the end. The graph is keyed on the device aliases, so callers should reuse their buffers.
    auto alias = [&](const void* p) -> void* {
      for (auto& kv : h->host_map)
        if (kv.first == p) return kv.second;
      cudaPointerAttributes at;
      void* d = nullptr;
      if (cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeHost) d = at.devicePointer;
      cudaGetLastError();
      if (h->host_map.size() >= 64) h->host_map.erase(h->host_map.begin());
      h->host_map.emplace_back(p, d);
      return d;
    };
    void* ds = alias(h_states);
    void* dr = alias(h_rtg);
    void* dw = h_rewards ? alias(h_rewards) : nullptr;
    void* dt = alias(h_tokens);
    void* da = alias(h_actions);
    if (ds && dr && dt && da && (!h_rewards || dw)) {
      rc = xl_policy_step(h, state, (const float*)ds, (const float*)dr, (const float*)dw, (int32_t*)dt, (float*)da,
                          nullptr, nullptr, B, mode, flags, s);
      if (rc) return rc;
      XL_CUDA(cudaStreamSynchronize(s));
      return XL_OK;
    }
  }
  // (Measured and dropped in round 2: capturing these copies as nodes of the step's graph — one launch per env step —
  // made the end-to-end step 1.5x SLOWER on B200, 1.48 ms vs 0.99 ms at 48M x 64 envs; memcpy nodes to / from pinned
  // host memory serialise badly against the programmatic-dependent-launch kernel nodes. Plain async copies around the
  // graph launch it is.)
  XL_CUDA(cudaMemcpyAsync(h->d_states, h_states, sizeof(float) * (size_t)B * c.state_dim, cudaMemcpyHostToDevice, s));
  XL_CUDA(cudaMemcpyAsync(h->d_rtg, h_rtg, sizeof(float) * (size_t)B, cudaMemcpyHostToDevice, s));
  if (h_rewards) XL_CUDA(cudaMemcpyAsync(h->d_rew, h_rewards, sizeof(float) * (size_t)B, cudaMemcpyHostToDevice, s));
  rc = xl_policy_step(h, state, h->d_states, h->d_rtg, h_rewards ? h->d_rew : nullptr, h->d_tokens, h->d_actions,
                      nullptr, nullptr, B, mode, flags, s);
  if (rc) return rc;
  XL_CUDA(cudaMemcpyAsync(h_tokens, h->d_tokens, sizeof(int32_t) * (size_t)B * c.act_dim, cudaMemcpyDeviceToHost, s));
  XL_CUDA(cudaMemcpyAsync(h_actions, h->d_actions, sizeof(float) * (size_t)B * c.act_dim, cudaMemcpyDeviceToHost, s));
  XL_CUDA(cudaStreamSynchronize(s));
  return XL_OK;
}

// Tokens of one prefill chunk (Bk envs x Tc timesteps from timestep pos) straight from given state embeddings
// [B, Tn, d] into pf_x: one launch where raw states take a staging copy, pad_rows, the embed_state Linear and the embed
// kernel. perm / len as in launch_ragged_rows (nullptr: envs 0..Bk-1, every timestep valid).
static void seq_embed_chunk(xl_handle* h, const float* embeds, const float* rtg, const float* rewards,
                            const int32_t* perm, const int32_t* len, int Bk, int Tn, int Tc, int pos, cudaStream_t s) {
  const xl_config& c = h->cfg;
  auto PW = [&](int id) { return (const float*)h->pw[id - XL_W_POST_NORM]; };
  xl::SeqEmbedParams p;
  p.s_emb = embeds; p.rtg = rtg; p.rew = rewards;
  p.perm = perm; p.len = len; p.len_div = c.tokens_per_step;
  p.Tn = Tn; p.Tc = Tc; p.pos = pos; p.rows = Bk * Tc; p.d = c.embedding_dim;
  p.w_ret = PW(XL_W_EMBED_RETURN_W); p.b_ret = PW(XL_W_EMBED_RETURN_B);
  p.w_rew = PW(XL_W_EMBED_REWARD_W); p.b_rew = PW(XL_W_EMBED_REWARD_B);
  p.ln_w = PW(XL_W_EMBED_LN_W); p.ln_b = PW(XL_W_EMBED_LN_B); p.eps = c.embed_ln_eps;
  p.x = prefill_ws(h).x;
  xl::launch_seq_embed_tokens(p, s);
  h->launches += 1;
}

// One call of the sequence path; each entry point below only fills this in.
struct SeqCall {
  enum Input { kTokens, kStates, kEmbeds };
  const char* fn;                     // the entry point, for messages
  Input in;                           // x: encoder tokens [B, S, d], raw states [B, S, state_dim] or state embeddings [B, S, d]
  void* state;
  const float *x, *rtg, *rewards;     // rtg / rewards [B, S] of the policy forms (rewards nullable)
  const int32_t* lengths;             // host [B] in units, or nullptr
  int B, S;                           // S in units: tokens (encoder) or timesteps (policy)
  unsigned flags;
  void* stream;
  bool ragged = false;                // lengths are required (the _ragged entries)
  float* y_out = nullptr;             // encoder: post_blocks_norm hidden states [B, S, d], nullable
  bool head = false;                  // forward entries: the action outputs of every timestep go to *out
  const xl_seq_outputs* out = nullptr;
  SeqCall(const char* fn, Input in, void* state, const float* x, const float* rtg, const float* rewards,
          const int32_t* lengths, int B, int S, unsigned flags, void* stream)
      : fn(fn), in(in), state(state), x(x), rtg(rtg), rewards(rewards), lengths(lengths), B(B), S(S), flags(flags),
        stream(stream) {}
};

// Validate; all lengths full -> the uniform call; plan; per chunk: stage the inputs, the block stack, the outputs;
// scatter the state back; the eager tail of a uniform call.
static int run_seq(xl_handle* h, SeqCall c) {
  const bool enc = c.in == SeqCall::kTokens;
  if (c.head) {
    if (!h) return fail(XL_ERR_INVALID_ARG, "null handle");
    if (!c.out) return fail(XL_ERR_INVALID_ARG, "null outputs");
    if (c.out->logprobs && !c.out->targets) return fail(XL_ERR_INVALID_ARG, "logprobs need targets");
  }
  if (c.in == SeqCall::kStates && (c.flags & XL_FLAG_STATE_EMBEDS))   // they would be read as [B, S, state_dim] rows
    return fail(XL_ERR_UNSUPPORTED, "%s takes raw states; state embeddings go through xl_policy_prefill_embeds / "
                                    "xl_policy_forward_embeds", c.fn);
  if (c.in == SeqCall::kEmbeds) {
    if (!h) return fail(XL_ERR_INVALID_ARG, "null handle");
    if ((uintptr_t)c.x % 16)
      return fail(XL_ERR_INVALID_ARG, "state_embeds must be 16-byte aligned (rows are loaded as float4)");
    c.flags |= XL_FLAG_STATE_EMBEDS;
  }
  int rc = check_batch(h, c.B);
  if (rc) return rc;
  if (!c.state || !c.x || (!enc && !c.rtg)) return fail(XL_ERR_INVALID_ARG, "null argument");
  const char* unit = enc ? "S" : "Tn";
  if (c.S <= 0) return fail(XL_ERR_INVALID_ARG, "%s=%d must be positive", unit, c.S);
  if ((c.lengths || c.ragged) && (rc = check_lengths(c.lengths, c.B, c.S, unit))) return rc;
  if ((rc = weights_ready(h, enc))) return rc;
  cudaStream_t s = (cudaStream_t)c.stream;
  const xl_config& cf = h->cfg;
  const int B = c.B, S = c.S, d = cf.embedding_dim, sd = cf.state_dim;
  SeqHead hd;
  const SeqHead* head = nullptr;
  if (c.head) {
    hd.out = *c.out;
    hd.discrete = (c.flags & XL_FLAG_DISCRETE) ? 1 : 0;
    hd.n_out = hd.discrete ? h->num_actions : h->head_out;
    hd.Tn = S;
    head = &hd;
  }
  const int32_t* lengths = c.lengths;
  if (lengths) {
    const int nfull = (int)std::count(lengths, lengths + B, S), nzero = (int)std::count(lengths, lengths + B, 0);
    if (nfull == B) {
      lengths = nullptr;          // the uniform call, bit for bit
    } else {
      if (nzero < B && !prefill_fast_path(h))
        return fail(XL_ERR_UNSUPPORTED, "ragged prefill needs the sequence path (conv_kernel 4, a cell plan for DH=%d)",
                    h->DH);
      // output positions past an env's length keep these values (y_out 0; tokens -1, the rest 0)
      if (c.y_out) XL_CUDA(cudaMemsetAsync(c.y_out, 0, sizeof(float) * (size_t)B * S * d, s));
      if (head && (rc = seq_clear_outputs(h, hd, B, s))) return rc;
      if (nzero == B) return XL_OK;
    }
  }
  SeqPlan p;
  p.T = enc ? 1 : cf.tokens_per_step;
  if ((rc = seq_plan(h, c.state, lengths, B, S, p, s))) return rc;
  auto gather = [&](const SeqChunk& ch, const float* src, float* dst, int width) {
    return chunk_rows(h, p, ch, const_cast<float*>(src), dst, S, width, 0, s);
  };
  const Ws ws = prefill_ws(h);
  const int impl = (c.flags & XL_FLAG_SIMPLE_GEMM) ? 1 : h->gemm_impl;
  auto PW = [&](int id) { return (const float*)h->pw[id - XL_W_POST_NORM]; };
  for (const SeqChunk& ch : p.chunks) {
    const int rows = ch.Bk * ch.n;
    if (c.in == SeqCall::kTokens) {
      if ((rc = gather(ch, c.x, ws.x, d))) return rc;
    } else if (c.in == SeqCall::kEmbeds) {
      seq_embed_chunk(h, c.x, c.rtg, c.rewards, p.d_perm, p.d_len, ch.Bk, S, ch.n, ch.pos, s);
    } else {
      // the chunk's timesteps [Bk, n, state_dim], [Bk, n], then embed: rows (env, timestep) -> tokens
      // (env, timestep, {s, rtg, r}) == the env's sequence order
      if ((rc = gather(ch, c.x, h->pf_sin, sd)) || (rc = gather(ch, c.rtg, h->pf_rtg, 1)) ||
          (c.rewards && (rc = gather(ch, c.rewards, h->pf_rew, 1))))
        return rc;
      xl::launch_pad_rows(h->pf_sin, sd, ws.states_pad, h->Kpad, rows, s);
      h->launches += 1;
      rc = linear(h, ws, ws.states_pad, PW(XL_W_EMBED_STATE_W), PW(XL_W_EMBED_STATE_B), nullptr,
                  ws.s_emb, rows, d, h->Kpad, impl, s);
      if (rc) return rc;
      xl::launch_embed_tokens(ws.s_emb, h->pf_rtg, c.rewards ? h->pf_rew : nullptr, PW(XL_W_EMBED_RETURN_W),
                              PW(XL_W_EMBED_RETURN_B), PW(XL_W_EMBED_REWARD_W), PW(XL_W_EMBED_REWARD_B),
                              PW(XL_W_EMBED_LN_W), PW(XL_W_EMBED_LN_B), cf.embed_ln_eps, ws.x, rows, d, nullptr, nullptr,
                              nullptr, 0.f, nullptr, nullptr, nullptr, s);
      h->launches += 1;
    }
    if ((rc = prefill_blocks(h, p.st, p.Btot, ch.Bk, ch.n * p.T, c.flags, s, p.d_len, ch.pos * p.T))) return rc;
    if (c.y_out) {
      xl::launch_ln_rows(h->pf_x, d, h->pf_xn, d, PW(XL_W_POST_NORM), nullptr, 1, cf.ln_eps, rows, d, nullptr, nullptr,
                         s);
      h->launches += 1;
      if ((rc = chunk_rows(h, p, ch, c.y_out, h->pf_xn, S, d, 1, s))) return rc;
    }
    if (head && (rc = seq_head_chunk(h, hd, ch.Bk, ch.n, ch.pos, p.d_perm, p.d_len, c.flags, s))) return rc;
    XL_CUDA(cudaGetLastError());
  }
  if ((rc = ragged_end(h, c.state, B, p, s))) return rc;
  // the eager tail (uniform calls only): fused encoder steps of <= 4 tokens ...
  if (enc) {
    const Step sl = make_step(h, B, s);
    for (int pos = p.tail; pos < S;) {
      const SeqChunk ch = {pos, B, std::min(4, S - pos)};
      if ((rc = gather(ch, c.x, sl.ws.x, d))) return rc;
      if ((rc = run_encoder(h, c.state, sl, sl.ws.x, sl.ws.hid, ch.n, XL_MODE_FUSED, c.flags))) return rc;
      if (c.y_out && (rc = chunk_rows(h, p, ch, c.y_out, sl.ws.hid, S, d, 1, s))) return rc;
      pos += ch.n;
    }
    return XL_OK;
  }
  // ... or ordinary fused policy steps with their outputs discarded; a forward reduces each step's logits as a chunk
  // of one timestep
  if (head && p.tail < S && (rc = ensure_seq_logits(h, (size_t)B * hd.n_out))) return rc;
  const bool embeds = c.in == SeqCall::kEmbeds;
  float* stage = embeds ? h->d_embeds : h->d_states;
  for (int pos = p.tail; pos < S; ++pos) {
    const SeqChunk ch = {pos, B, 1};
    if ((rc = gather(ch, c.x, stage, embeds ? d : sd)) || (rc = gather(ch, c.rtg, h->d_rtg, 1)) ||
        (c.rewards && (rc = gather(ch, c.rewards, h->d_rew, 1))))
      return rc;
    StepArgs a;
    a.state = c.state; a.states = stage; a.rtg = h->d_rtg; a.rewards = c.rewards ? h->d_rew : nullptr;
    a.tokens = h->d_tokens; a.actions = h->d_actions; a.logits = head ? h->sq_logits : nullptr; a.hidden = nullptr;
    a.B = B; a.mode = XL_MODE_FUSED; a.flags = (c.flags & ~(unsigned)XL_FLAG_GRAPH) | kFlagNoRing;
    if ((rc = run_policy(h, a, s))) return rc;
    if (head) seq_head_reduce(h, hd, B, 1, pos, nullptr, nullptr, s);
  }
  return XL_OK;
}

int xl_prefill(xl_handle* h, void* state, const float* x_in, float* y_out, int B, int S, unsigned flags, void* stream) {
  SeqCall c("xl_prefill", SeqCall::kTokens, state, x_in, nullptr, nullptr, nullptr, B, S, flags, stream);
  c.y_out = y_out;
  return run_seq(h, c);
}

int xl_prefill_ragged(xl_handle* h, void* state, const float* x_in, float* y_out, const int32_t* lengths, int B, int S,
                      unsigned flags, void* stream) {
  SeqCall c("xl_prefill_ragged", SeqCall::kTokens, state, x_in, nullptr, nullptr, lengths, B, S, flags, stream);
  c.ragged = true;
  c.y_out = y_out;
  return run_seq(h, c);
}

int xl_policy_prefill(xl_handle* h, void* state, const float* states, const float* rtg, const float* rewards, int B,
                      int Tn, unsigned flags, void* stream) {
  return run_seq(h, SeqCall("xl_policy_prefill", SeqCall::kStates, state, states, rtg, rewards, nullptr, B, Tn, flags,
                            stream));
}

int xl_policy_prefill_ragged(xl_handle* h, void* state, const float* states, const float* rtg, const float* rewards,
                             const int32_t* lengths, int B, int Tn, unsigned flags, void* stream) {
  SeqCall c("xl_policy_prefill_ragged", SeqCall::kStates, state, states, rtg, rewards, lengths, B, Tn, flags, stream);
  c.ragged = true;
  return run_seq(h, c);
}

int xl_policy_forward(xl_handle* h, void* state, const float* states, const float* rtg, const float* rewards,
                      const int32_t* lengths, int B, int Tn, const xl_seq_outputs* out, unsigned flags, void* stream) {
  SeqCall c("xl_policy_forward", SeqCall::kStates, state, states, rtg, rewards, lengths, B, Tn, flags, stream);
  c.head = true;
  c.out = out;
  return run_seq(h, c);
}

int xl_policy_prefill_embeds(xl_handle* h, void* state, const float* state_embeds, const float* rtg,
                             const float* rewards, const int32_t* lengths, int B, int Tn, unsigned flags,
                             void* stream) {
  return run_seq(h, SeqCall("xl_policy_prefill_embeds", SeqCall::kEmbeds, state, state_embeds, rtg, rewards, lengths, B,
                            Tn, flags, stream));
}

int xl_policy_forward_embeds(xl_handle* h, void* state, const float* state_embeds, const float* rtg,
                             const float* rewards, const int32_t* lengths, int B, int Tn, const xl_seq_outputs* out,
                             unsigned flags, void* stream) {
  SeqCall c("xl_policy_forward_embeds", SeqCall::kEmbeds, state, state_embeds, rtg, rewards, lengths, B, Tn, flags,
            stream);
  c.head = true;
  c.out = out;
  return run_seq(h, c);
}

int xl_linear(xl_handle* h, const float* A, const void* W_bf16, const float* bias, const float* residual,
              float* out, int M, int N, int K, int impl, void* stream) {
  if (!h || !A || !W_bf16 || !out) return fail(XL_ERR_INVALID_ARG, "null argument");
  if (M <= 0 || N <= 0 || K <= 0) return fail(XL_ERR_INVALID_ARG, "bad GEMM shape");
  Ws w = step_ws(h, h->cfg.max_batch);
  w.a_cap = h->a_cap;                  // a stand-alone Linear may use the whole operand planes
  return linear(h, w, A, W_bf16, bias, residual, out, M, N, K, impl, (cudaStream_t)stream);
}

int xl_set_token_ring(xl_handle* h, int32_t* ring, int slots, int next_slot, void* stream) {
  if (!h) return fail(XL_ERR_INVALID_ARG, "null handle");
  if (ring && (slots <= 0 || next_slot < 0 || next_slot >= slots))
    return fail(XL_ERR_INVALID_ARG, "token ring: slots=%d next_slot=%d", slots, next_slot);
  if (ring != h->tok_ring || (ring && slots != h->tok_slots)) {
    clear_graphs(h);   // the ring pointer is baked into captured graphs
    h->tok_ring = ring;
    h->tok_slots = ring ? slots : 0;
  }
  if (ring) {
    xl::launch_set_u32(h->counters + kCntRing, (unsigned)next_slot, (cudaStream_t)stream);
    XL_CUDA(cudaGetLastError());
  }
  return XL_OK;
}

static int check_sampling(const xl_handle* h, const xl_sampling* p) {
  if (!(p->temperature > 0.f) || !std::isfinite(p->temperature))
    return fail(XL_ERR_INVALID_ARG, "sampling: temperature %g must be finite and > 0", (double)p->temperature);
  if (!(p->top_p >= 0.f && p->top_p <= 1.f)) return fail(XL_ERR_INVALID_ARG, "sampling: top_p %g outside [0, 1]", (double)p->top_p);
  if (p->top_k < 0 || p->top_k > h->num_actions)
    return fail(XL_ERR_INVALID_ARG, "sampling: top_k %d outside [0, num_actions=%d]", p->top_k, h->num_actions);
  if (p->env_id_base < 0 || p->env_id_stride < 1)
    return fail(XL_ERR_INVALID_ARG, "sampling: env_id_base %d must be >= 0 and env_id_stride %d >= 1", p->env_id_base,
                p->env_id_stride);
  if (h->num_actions > xl::kSampleMaxActions || h->cfg.act_dim > xl::kSampleMaxRows)
    return fail(XL_ERR_UNSUPPORTED, "sampling: num_actions %d > %d or act_dim %d > %d", h->num_actions,
                xl::kSampleMaxActions, h->cfg.act_dim, xl::kSampleMaxRows);
  return XL_OK;
}

int xl_set_sampling(xl_handle* h, const xl_sampling* params, uint32_t step0, void* stream) {
  if (!h) return fail(XL_ERR_INVALID_ARG, "null handle");
  if (params) {
    int rc = check_sampling(h, params);
    if (rc) return rc;
  }
  if (h->sampling != (params != nullptr)) {
    // the sampling kernel and the counter advance are baked into captured graphs; the parameters are not
    clear_graphs(h);
    h->sampling = params != nullptr;
  }
  if (params) {
    xl::launch_set_sampling(h->counters + kCntArmed, params, h->counters + kCntSample, step0, (cudaStream_t)stream);
    XL_CUDA(cudaGetLastError());
  }
  return XL_OK;
}

int xl_sample_actions(xl_handle* h, const float* logits, int B, unsigned flags, const xl_sampling* params,
                      uint32_t step, int32_t* tokens, float* actions, void* stream) {
  int rc = check_batch(h, B);
  if (rc) return rc;
  if (!logits || !params || !tokens || !actions) return fail(XL_ERR_INVALID_ARG, "null argument");
  rc = check_sampling(h, params);
  if (rc) return rc;
  const xl_config& c = h->cfg;
  cudaStream_t s = (cudaStream_t)stream;
  const bool discrete = (flags & XL_FLAG_DISCRETE) != 0;
  // the kernel draws for (*counter - 1)
  xl::launch_set_sampling(h->counters + kCntUnit, params, h->counters + kCntUnitStep, step + 1u, s);
  const float bw = (c.tok_max_val - c.tok_min_val) / (float)c.action_channels;
  xl::launch_sample_tokens(logits, discrete ? h->num_actions : h->head_out, B, c.act_dim, h->num_actions,
                           c.discrete_actions, discrete ? 1 : 0, discrete ? 0.f : bw, discrete ? 0.f : c.tok_min_val,
                           tokens, actions, nullptr, nullptr, 1, 0, h->counters + kCntUnit, h->counters + kCntUnitStep, s);
  h->launches += 2;
  XL_CUDA(cudaGetLastError());
  return XL_OK;
}

int xl_set_option(xl_handle* h, const char* name, int value) {
  if (!h || !name) return fail(XL_ERR_INVALID_ARG, "null argument");
  if (!strcmp(name, "state_impl")) {
    if (value < 0 || value > 2) return fail(XL_ERR_INVALID_ARG, "state_impl must be 0, 1 or 2");
    h->state_impl = value;
  } else if (!strcmp(name, "state_stages")) {
    if (value < 0 || value > 8) return fail(XL_ERR_INVALID_ARG, "state_stages must be in [0, 8]");
    h->state_stages = value;
  } else if (!strcmp(name, "state_ctas_per_sm")) {
    if (value < 0 || value > 2) return fail(XL_ERR_INVALID_ARG, "state_ctas_per_sm must be in [0, 2]");
    h->state_ctas_per_sm = value;
  } else if (!strcmp(name, "state_rows_split")) {
    if (value < 0 || value > 32) return fail(XL_ERR_INVALID_ARG, "state_rows_split must be in [0, 32]");
    h->state_rows_split = value;
  } else if (!strcmp(name, "host_zero_copy")) {
    h->host_zero_copy = value ? 1 : 0;
  } else if (!strcmp(name, "gemm_cluster")) {
    if (value != 1 && value != 2 && value != 4) return fail(XL_ERR_INVALID_ARG, "gemm_cluster must be 1, 2 or 4");
    xl::g_gemm_cluster = value;          // process-wide
  } else if (!strcmp(name, "gemm_2cta")) {
    if (value < -1 || value > 2)
      return fail(XL_ERR_INVALID_ARG, "gemm_2cta must be -1 (automatic), 0, 1 (2-SM tiles) or 2 (persistent 2-SM)");
    xl::g_gemm_2cta = value;             // process-wide
  } else if (!strcmp(name, "gemm_bm")) {
    if (value != 0 && value != 64 && value != 128) return fail(XL_ERR_INVALID_ARG, "gemm_bm must be 0, 64 or 128");
    xl::g_gemm_bm = value;               // process-wide
  } else if (!strcmp(name, "gemm_m64_layout")) {
    xl::gemm_tc_set_m64_layout(value);   // process-wide probe
  } else if (!strcmp(name, "fuse_ends")) {
    h->fuse_ends = value ? 1 : 0;
  } else if (!strcmp(name, "up_fuse")) {
    h->up_fuse = value ? 1 : 0;
  } else if (!strcmp(name, "small_state_fuse")) {
    if (value < 0 || value > 16) return fail(XL_ERR_INVALID_ARG, "small_state_fuse must be in [0, 16]");
    h->small_state_fuse = value;     // 0 off, 1 on (clusters of <= 16 CTAs), 2..16 = on with that cluster cap
  } else if (!strcmp(name, "state_fuse")) {
    if (value < 0 || value > 3)
      return fail(XL_ERR_INVALID_ARG, "state_fuse must be 0 (separate finalize kernel), 1 (cluster, symmetric), "
                                      "2 (cluster, rank 0 finalizes) or 3 (unfused kernel under the cluster shape)");
    h->state_fuse = value;
  } else if (!strcmp(name, "prefill_cell")) {
    if (value < 0 || value > 2)
      return fail(XL_ERR_INVALID_ARG, "prefill_cell must be 0 (fp32 sequence cell), 1 (chunkwise mma.sync) or 2 (chunkwise tcgen05)");
    h->prefill_cell = (int)value;
  } else if (!strcmp(name, "prefill_rows")) {
    if (value < 48 || value > 32768) return fail(XL_ERR_INVALID_ARG, "prefill_rows must be in [48, 32768]");
    h->prefill_rows = value;
  } else if (!strcmp(name, "prefill_conv_run")) {
    if (value < 4 || value > 64 || value % 4) return fail(XL_ERR_INVALID_ARG, "prefill_conv_run must be a multiple of 4 in [4, 64]");
    xl::g_prefill_conv_run = value;           // process-wide: tokens per CTA of the sequence conv/qkv kernel
  } else if (!strcmp(name, "prefill_conv")) {
    if (value < 0 || value > 2) return fail(XL_ERR_INVALID_ARG, "prefill_conv must be 0 (scalar), 1 (packed fp32) or 2 (packed + SFU SiLU)");
    xl::g_prefill_conv_impl = value;          // process-wide A/B of the sequence conv/qkv/gates kernel
  } else if (!strcmp(name, "prefill_conv_persist")) {
    xl::g_prefill_conv_persist = value ? 1 : 0;   // process-wide A/B: packed conv kernel persistent over the token runs
  } else if (!strcmp(name, "prefill_scan_split")) {
    if (value != 2 && value != 4) return fail(XL_ERR_INVALID_ARG, "prefill_scan_split must be 2 or 4");
    xl::g_prefill_scan_split = value;             // process-wide A/B: 8 or 16 epilogue warps in the chunk update + scan kernel
  } else if (!strcmp(name, "prefill_tc_overlap")) {
    xl::g_prefill_tc_overlap = value ? 1 : 0;     // process-wide A/B: S GEMM / P~ / n scan on a side stream beside the chunk scan
  } else if (!strcmp(name, "prefill_prep")) {
    xl::g_prefill_prep = value ? 1 : 0;       // process-wide A/B of the chunk preparation kernel (1 = single-read tile kernel)
  } else if (!strcmp(name, "prefill_tc_fused")) {
    xl::g_prefill_tc_fused = value ? 1 : 0;   // process-wide A/B: chunk update + scan in one kernel (1) or through HBM (0)
  } else if (!strcmp(name, "pdl")) {
    xl::g_use_pdl = value ? 1 : 0;       // process-wide: programmatic dependent launch of every kernel
  } else if (!strcmp(name, "l2_prefetch_mb")) {
    if (value < -1 || value > 4096) return fail(XL_ERR_INVALID_ARG, "l2_prefetch_mb must be in [-1, 4096] (-1 = automatic)");
    h->l2_prefetch_mb = value;
  } else if (!strcmp(name, "l2_prefetch_policy")) {
    h->l2_prefetch_policy = value ? 1 : 0;
  } else if (!strcmp(name, "gemm_splitk")) {
    if (value < 0 || value > kSplitMax) return fail(XL_ERR_INVALID_ARG, "gemm_splitk must be in [0, %d]", kSplitMax);
    h->gemm_splitk = value;
  } else if (!strcmp(name, "gemm_up_bn") || !strcmp(name, "gemm_down_bn")) {
    if (value != 0 && value != 32 && value != 64 && value != 128 && value != 256)
      return fail(XL_ERR_INVALID_ARG, "%s must be 0, 32, 64, 128 or 256", name);
    (name[5] == 'u' ? h->gemm_up_bn : h->gemm_down_bn) = value;
  } else if (!strcmp(name, "gemm_up_splits") || !strcmp(name, "gemm_down_splits")) {
    if (value < 0 || value > kSplitMax) return fail(XL_ERR_INVALID_ARG, "%s must be in [0, %d]", name, kSplitMax);
    (name[5] == 'u' ? h->gemm_up_splits : h->gemm_down_splits) = value;
  } else if (!strcmp(name, "conv_impl")) {
    if (value < 0 || value > 2) return fail(XL_ERR_INVALID_ARG, "conv_impl must be 0, 1 or 2");
    h->conv_impl = value;
  } else if (!strcmp(name, "smallm")) {
    if (value < -1 || value > 1) return fail(XL_ERR_INVALID_ARG, "smallm must be -1 (automatic), 0 or 1");
    h->smallm = value;
#ifdef XL_DEBUG_OPTIONS
  } else if (!strcmp(name, "debug_skip")) {
    // measurement aid (marginal cost of a kernel class): results are garbage while set. Compiled in only with
    // -DXL_DEBUG_OPTIONS (XL_DEBUG_OPTIONS=1 python -m lram_b200.build --force); absent from the product library.
    h->debug_skip = value;
#endif
  } else if (!strcmp(name, "gemm_impl")) {
    if (value < 0 || value > 2) return fail(XL_ERR_INVALID_ARG, "gemm_impl must be 0, 1 or 2");
    h->gemm_impl = value;
  } else {
    return fail(XL_ERR_INVALID_ARG, "unknown option %s", name);
  }
  clear_graphs(h);
  return XL_OK;
}

int xl_profile_begin(xl_handle* h) {
  if (!h) return fail(XL_ERR_INVALID_ARG, "null handle");
  h->profiling = true;
  return XL_OK;
}

int xl_profile_end(xl_handle* h, double* state_kernel_ms, int64_t* state_kernel_launches, double* step_ms) {
  if (!h || !state_kernel_ms || !state_kernel_launches || !step_ms) return fail(XL_ERR_INVALID_ARG, "null argument");
  h->profiling = false;
  double a = 0.0, b = 0.0;
  auto drain = [](std::vector<cudaEvent_t>& v, double& acc) -> cudaError_t {
    cudaError_t err = cudaSuccess;
    for (size_t i = 0; i + 1 < v.size(); i += 2) {
      float ms = 0.f;
      cudaError_t e = cudaEventSynchronize(v[i + 1]);
      if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, v[i], v[i + 1]);
      if (e != cudaSuccess) err = e;
      acc += ms;
      cudaEventDestroy(v[i]);
      cudaEventDestroy(v[i + 1]);
    }
    return err;
  };
  const int64_t n = (int64_t)h->prof_state.size() / 2;
  cudaError_t e1 = drain(h->prof_state, a);
  cudaError_t e2 = drain(h->prof_step, b);
  h->prof_state.clear();
  h->prof_step.clear();
  *state_kernel_ms = a;
  *state_kernel_launches = n;
  *step_ms = b;
  if (e1 != cudaSuccess || e2 != cudaSuccess) return fail(XL_ERR_CUDA, "profile events: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
  return XL_OK;
}

int64_t xl_launch_count(xl_handle* h) {
  if (!h) return 0;
  const int64_t v = h->launches;
  h->launches = 0;
  return v;
}

}  // extern "C"
