/*
 * xlstm_b200 — C ABI of the B200-native recurrent-inference path for LRAM's xLSTM policy.
 *
 * Plain C: pointers, sizes, ints. No torch / C++ types cross this boundary. Every device pointer is owned
 * by the caller (PyTorch tensors' data_ptr()); the library owns only the opaque handle and a scratch
 * workspace sized at xl_create(). All work is enqueued on the caller's stream; nothing synchronises unless
 * the entry point says so (only the *_host call does). A handle is not thread-safe (the reference is
 * single-threaded per process, one process per GPU: src/algos/builder.py:25-29).
 *
 * Each entry point cites the reference interface (file:line under ml-jku/LRAM, or the third-party `xlstm`
 * v1.0.x symbol the reference calls at that line) it replaces.
 *
 * Return value: 0 on success, negative xl_status otherwise; message via xl_last_error() (thread local).
 */
#ifndef XLSTM_B200_H
#define XLSTM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

#define XL_ABI_VERSION 3

typedef enum {
  XL_OK = 0,
  XL_ERR_INVALID_ARG = -1,
  XL_ERR_UNSUPPORTED = -2,
  XL_ERR_CUDA = -3,
  XL_ERR_NOT_READY = -4, /* weights missing */
  XL_ERR_NO_DEVICE = -5
} xl_status;

typedef struct xl_handle xl_handle;

/* Shapes of the policy. Mirrors xLSTMConfig.xlstm_config (src/algos/models/decision_xlstm.py:104-133,
 * configs/agent_params/huggingface/xlstm_*.yaml) and the multi-domain model kwargs
 * (configs/agent_params/model_kwargs/multi_domain.yaml:1-11). */
typedef struct {
  int32_t embedding_dim;      /* d                                              */
  int32_t num_blocks;         /* L (mLSTM blocks unless listed in slstm_mask)   */
  int32_t num_heads;          /* NH                                             */
  int32_t inner_dim;          /* ceil(2d/64)*64                                 */
  int32_t conv_kernel;        /* KS = 4                                         */
  int32_t qkv_blocksize;      /* 4 (only 4 is supported)                        */
  int32_t state_dim;          /* 204 (max_state_dim)                            */
  int32_t act_dim;            /* 8   (max_act_dim)                              */
  int32_t action_channels;    /* 256 (tokenizer vocab)                          */
  int32_t discrete_actions;   /* 18  (tokenizer shift)                          */
  int32_t tokens_per_step;    /* 3: (s, rtg, r)                                 */
  int32_t action_token_pos;   /* 1: action is read at the rtg token             */
  int32_t max_batch;          /* largest B any call will use (workspace sizing) */
  float ln_eps;               /* 1e-5 xlstm LayerNorm / MultiHeadLayerNorm      */
  float cell_eps;             /* 1e-6 recurrent_step_stabilized_simple          */
  float embed_ln_eps;         /* 1e-5 nn.LayerNorm                              */
  float tok_min_val;          /* -1 MinMaxTokenizer                             */
  float tok_max_val;          /* +1                                             */
  /* xLSTM[a:b] stacks (xlstm_config.slstm_at, configs/agent_params/huggingface/xlstm_ms_mediumplus.yaml:27;
   * README.md:188-190): bit i set = block i is an sLSTM block (sLSTM layer + gated feed-forward).          */
  uint32_t slstm_mask_lo;     /* blocks 0..31                                   */
  uint32_t slstm_mask_hi;     /* blocks 32..63                                  */
  int32_t ffn_dim;            /* ceil(1.3 d / 64) * 64 (slstm_block.feedforward.proj_factor); 0 = no sLSTM */
} xl_config;

/* Weight slots. Names in comments are the reference's state_dict keys. `layer` = block index, or -1 for
 * policy-level tensors. dtype: 0 = fp32, 1 = bf16. GEMM matrices must be bf16, everything else fp32. */
typedef enum {
  /* per block: encoder.layers.blocks.{i}.*                                                  shape */
  XL_W_XLSTM_NORM = 0,     /* xlstm_norm.weight (gamma = 1 + w)                         fp32 [d]              */
  XL_W_PROJ_UP = 1,        /* xlstm.proj_up.weight                                      bf16 [2*inner, d]     */
  XL_W_Q_PROJ = 2,         /* xlstm.q_proj.weight                                       fp32 [inner/4, 4, 4]  */
  XL_W_K_PROJ = 3,         /* xlstm.k_proj.weight                                       fp32 [inner/4, 4, 4]  */
  XL_W_V_PROJ = 4,         /* xlstm.v_proj.weight                                       fp32 [inner/4, 4, 4]  */
  XL_W_CONV_W = 5,         /* xlstm.conv1d.conv.weight                                  fp32 [inner, 1, KS]   */
  XL_W_CONV_B = 6,         /* xlstm.conv1d.conv.bias                                    fp32 [inner]          */
  XL_W_IGATE_W = 7,        /* xlstm.mlstm_cell.igate.weight                             fp32 [NH, 3*inner]    */
  XL_W_IGATE_B = 8,        /* xlstm.mlstm_cell.igate.bias                               fp32 [NH]             */
  XL_W_FGATE_W = 9,        /* xlstm.mlstm_cell.fgate.weight                             fp32 [NH, 3*inner]    */
  XL_W_FGATE_B = 10,       /* xlstm.mlstm_cell.fgate.bias                               fp32 [NH]             */
  XL_W_OUTNORM = 11,       /* xlstm.mlstm_cell.outnorm.weight (gamma = 1 + w)           fp32 [inner]          */
  XL_W_SKIP = 12,          /* xlstm.learnable_skip                                      fp32 [inner]          */
  XL_W_PROJ_DOWN = 13,     /* xlstm.proj_down.weight                                    bf16 [d, inner]       */
  /* sLSTM block (blocks in slstm_mask): encoder.layers.blocks.{i}.*; shares XL_W_XLSTM_NORM, XL_W_CONV_W
   * ([d,1,KS]) and XL_W_CONV_B ([d]) with the mLSTM slots. DHs = d / NH.                                     */
  XL_W_S_GATE_I = 14,      /* xlstm.fgate.weight  -> INPUT-gate pre-activation (sic, see oracle) fp32 [NH, DHs, DHs] */
  XL_W_S_GATE_F = 15,      /* xlstm.igate.weight  -> FORGET-gate pre-activation (sic)       fp32 [NH, DHs, DHs] */
  XL_W_S_GATE_Z = 16,      /* xlstm.zgate.weight                                        fp32 [NH, DHs, DHs]   */
  XL_W_S_GATE_O = 17,      /* xlstm.ogate.weight                                        fp32 [NH, DHs, DHs]   */
  XL_W_S_RECURRENT = 18,   /* xlstm.slstm_cell._recurrent_kernel_  [head, in, gate, out] fp32 [NH, DHs, 4, DHs] */
  XL_W_S_BIAS = 19,        /* xlstm.slstm_cell._bias_                                   fp32 [NH, 4, DHs]     */
  XL_W_S_GROUP_NORM = 20,  /* xlstm.group_norm.weight (gamma = 1 + w)                   fp32 [d]              */
  XL_W_FFN_NORM = 21,      /* ffn_norm.weight (gamma = 1 + w)                           fp32 [d]              */
  XL_W_FFN_UP = 22,        /* ffn.proj_up.weight                                        bf16 [2*ffn_dim, d]   */
  XL_W_FFN_DOWN = 23,      /* ffn.proj_down.weight                                      bf16 [d, ffn_dim]     */
  XL_W_PER_BLOCK_COUNT = 24,
  /* policy level (layer = -1) */
  XL_W_POST_NORM = 32,     /* encoder.layers.post_blocks_norm.weight (gamma = 1 + w)    fp32 [d]              */
  XL_W_EMBED_STATE_W = 33, /* embed_state.weight, K zero-padded to xl_state_dim_padded() bf16 [d, Kpad]       */
  XL_W_EMBED_STATE_B = 34, /* embed_state.bias                                          fp32 [d]              */
  XL_W_EMBED_RETURN_W = 35,/* embed_return.weight                                       fp32 [d] (=[d,1])     */
  XL_W_EMBED_RETURN_B = 36,/* embed_return.bias                                         fp32 [d]              */
  XL_W_EMBED_REWARD_W = 37,/* embed_rewards.weight                                      fp32 [d]              */
  XL_W_EMBED_REWARD_B = 38,/* embed_rewards.bias                                        fp32 [d]              */
  XL_W_EMBED_LN_W = 39,    /* embed_ln.weight                                           fp32 [d]              */
  XL_W_EMBED_LN_B = 40,    /* embed_ln.bias                                             fp32 [d]              */
  XL_W_HEAD_W = 41,        /* action_net.0.weight                                       bf16 [274*8, d]       */
  XL_W_HEAD_B = 42         /* action_net.0.bias                                         fp32 [274*8]          */
} xl_weight_id;

/* Pieces of the recurrent state (`past_key_values`, src/algos/models/decision_xlstm.py:163,168-169:
 * {"block_i": {"mlstm_state": (C, n, m), "conv_state": (conv,)}}), all fp32, resident in ONE caller-owned
 * buffer, layer-major so that one block's C is a single contiguous stream:
 *   for i in 0..L-1:  C[B,NH,DH/W,DH,W] | n[B,NH,DH] | m[B,NH] | conv[B,KS,inner]   (each 256-B aligned)
 * C is SLAB-MAJOR: the reference's C[b,h,dk,dv] lives at [b][h][dv / W][dk][dv % W] with W = 128 when
 * DH % 128 == 0 (else W = DH, i.e. the reference's row-major layout). Every [32 x 128] tile the state kernel
 * streams is then 16 contiguous KB (measured +4-5 % HBM throughput over row-major tiles). n, m and conv keep
 * the reference's layouts. lram_b200.engine.c_to_slab / c_from_slab convert. */
/* An sLSTM block's slot holds  slstm[4,B,d] = (y, c, n, m) | conv[B,KS,d]  instead (the reference's
 * {"slstm_state": [4,B,d], "conv_state": (conv,)}); blocks are packed back to back, so the offset of a block
 * depends on the kinds of the blocks before it — always ask xl_state_layout(). */
typedef enum { XL_STATE_C = 0, XL_STATE_N = 1, XL_STATE_M = 2, XL_STATE_CONV = 3, XL_STATE_SLSTM = 4 } xl_state_part;

/* step modes */
#define XL_MODE_PER_TOKEN 0 /* reference order: for token: for block (decision_xlstm.py:161-165)          */
#define XL_MODE_FUSED 1     /* for block: all tokens_per_step tokens; C is read/written once per env step  */

/* flags for xl_policy_step */
#define XL_FLAG_DISCRETE 1u   /* discrete-action branch: argmax over logits[:discrete_actions]             */
#define XL_FLAG_GRAPH 2u      /* replay the step from a cached CUDA graph (pointers must stay the same)    */
#define XL_FLAG_SIMPLE_GEMM 4u/* force the CUDA-core GEMM (debug / small M)                               */
#define XL_FLAG_STATE_EMBEDS 8u /* xl_policy_step: `states` is fp32 [B, d] = state-token embeddings already
                                 * computed by the caller (image observations: embed_image / ImpalaCNN,
                                 * discrete_decision_transformer_model.py:187-203, image_encoders.py:10-66, stays in
                                 * PyTorch/cuDNN); the embed_state Linear is skipped. The sequence calls take
                                 * embeddings through xl_policy_prefill_embeds / xl_policy_forward_embeds       */

int xl_abi_version(void);
const char* xl_last_error(void);

/* Build a handle for `cfg` on the current CUDA device. Allocates the scratch workspace (activations for
 * max_batch * tokens_per_step rows). Replaces: xLSTMEncoder.__init__ (decision_xlstm.py:124-136) building
 * xLSTMBlockStack, plus the policy's embed/head modules (multi_domain_discrete_dt_model.py:12-81). */
int xl_create(const xl_config* cfg, xl_handle** out);
void xl_destroy(xl_handle* h);

/* Padded K of the state embedding GEMM (multiple of 64). Host code zero-pads embed_state.weight to it. */
int xl_state_dim_padded(const xl_handle* h);

/* Bind one device-resident weight tensor (no copy; pointer must outlive the handle).
 * Replaces load_state_dict of the keys listed at xl_weight_id (loader: decision_transformer_sb3.py:1120-1184). */
int xl_bind_weight(xl_handle* h, int layer, int which, const void* dev_ptr, int dtype, int64_t numel);
/* 0 when every slot is bound, XL_ERR_NOT_READY (+message naming the first missing slot) otherwise. */
int xl_weights_ready(const xl_handle* h);
/* Same, but only for what xl_encoder_step / xl_prefill read: every block + post_blocks_norm. This is the state of a
 * handle that replaces ONLY `self.encoder` (the swap at decision_xlstm.py:188-189) while the reference policy keeps
 * its own embeddings and action head. */
int xl_encoder_weights_ready(const xl_handle* h);

/* Size / layout of the state buffer for B envs. */
size_t xl_state_bytes(const xl_handle* h, int B);
int xl_state_layout(const xl_handle* h, int B, int layer, int part, size_t* offset_bytes, size_t* size_bytes);

/* Zero the state of the envs whose env_mask[b] != 0 (device uint8 [B]); env_mask == NULL resets all.
 * Equivalent to `model.past_key_values = None` (src/callbacks/evaluation.py:124,251,261) per env:
 * zero C, n, m (m starts at 0, not -inf) and the conv window. */
int xl_state_reset(xl_handle* h, void* state, const uint8_t* env_mask, int B, void* stream);

/* Multi-GPU result gather without a copy between steps. The reference gathers evaluation results across ranks with
 * gather_object (src/utils/misc.py:159-191); here every xl_policy_step* additionally stores its int32 action tokens in
 * slot (n % slots) of the caller-owned device ring [slots, B, act_dim], n = steps since the ring was (re)armed +
 * next_slot; the caller all-gathers ranges of slots whenever it likes. The slot index advances ON THE DEVICE (inside a
 * captured graph too). ring == NULL disarms. Calling it again with the same ring only re-seeks to next_slot (enqueued on
 * `stream`); a different ring drops the cached graphs. B must stay the same between arming and gathering. */
int xl_set_token_ring(xl_handle* h, int32_t* ring, int slots, int next_slot, void* stream);

/* Stochastic action selection on the device: the reference's `a_sample_kwargs` (sample_from_logits,
 * src/algos/models/model_utils.py:7-32, called once per env at discrete_decision_transformer_sb3.py:62-63) with a
 * counter-based random stream. While armed, every xl_policy_step* picks its tokens by this contract instead of the
 * argmax; steps that xl_policy_prefill runs internally still take the argmax and do not count as steps here.
 *
 * For env b and action row j, take the row l[0..n) of logits, n = num_actions (discrete: the env's logits; continuous:
 * row j of its [act_dim, num_actions] block). In fp64:
 *  1. top_p > 0: percentile = torch.quantile(l, top_p): rank = (double)top_p * (n - 1), lo = floor(rank),
 *     hi = ceil(rank), w = rank - lo, with v = sorted(l): w < 0.5 ? v[lo] + w (v[hi] - v[lo])
 *     : v[hi] - (v[hi] - v[lo]) (1 - w). If percentile != max for EVERY row of the env, max taken over the env's
 *     whole logit block (a NaN anywhere in the block makes it NaN), every l_i <= percentile becomes -inf.
 *  2. top_k > 0: the k largest of the resulting row stay candidates, ties at the boundary to the lowest indices;
 *     -inf positions among them have weight 0.
 *  3. w_i = exp(temperature * (l_i - l_max)) over the candidates, Z = sum w_i (index order). u in [0, 1) from
 *     Philox4x32-10 with counter (step, global_env_id, j, 0) and key (seed & 0xffffffff, seed >> 32):
 *     u = ((x0 >> 5) * 2^26 + (x1 >> 6)) * 2^-53. The token is the first candidate, in index order, whose running sum
 *     exceeds u * Z.
 *  4. global_env_id = env_id_base + b * env_id_stride (b counts the envs of the call). With envs sharded as
 *     env i -> rank i mod N, base = rank and stride = N give every env the draws it gets on one GPU running all envs.
 *  5. step: a device counter, set to step0 here and advanced once per policy step on the device (inside a captured
 *     graph too); a step draws with the value it finds, so the first step after arming uses step0.
 *  6. A row containing NaN, or with no finite maximum among its candidates (everything cut, all -inf, or +inf), yields
 *     the argmax token (first index of the max of the first discrete_actions logits when discrete, of all num_actions
 *     otherwise; NaN counts as the max), where the reference would raise.
 * tokens / actions / token ring then hold the sampled tokens exactly as they hold the argmax ones (discrete: actions =
 * (float)token; continuous: max(token - discrete_actions, 0) * bin_width + min_val).
 * Rejected with XL_ERR_INVALID_ARG: temperature <= 0 or not finite, top_p outside [0, 1], top_k < 0 or > num_actions,
 * env_id_base < 0, env_id_stride < 1; XL_ERR_UNSUPPORTED: num_actions > 512 or act_dim > 8. */
typedef struct {
  float temperature;     /* 1.0 (the reference multiplies the logits by it)  */
  float top_p;           /* 0.5; 0 = no quantile cut                          */
  int32_t top_k;         /* 0 = no top-k cut                                  */
  int32_t env_id_base;   /* global id of the call's env 0                     */
  int32_t env_id_stride; /* global id step between consecutive envs           */
  uint64_t seed;
} xl_sampling;
/* params == NULL disarms: steps go back to the argmax. step0 = counter value of the next step. The parameters and the
 * counter are written on `stream` into the handle's device memory, so changing them needs no graph re-capture; arming
 * or disarming changes the step's kernels and drops the cached graphs. */
int xl_set_sampling(xl_handle* h, const xl_sampling* params, uint32_t step0, void* stream);
/* Unit-parity entry: sample B rows of given logits (discrete: [B, num_actions]; continuous: [B, act_dim*num_actions])
 * at an explicit step; tokens [B, act_dim] / actions [B, act_dim] as xl_policy_step writes them. Leaves the armed
 * sampler and its counter alone. */
int xl_sample_actions(xl_handle* h, const float* logits, int B, unsigned flags, const xl_sampling* params,
                      uint32_t step, int32_t* tokens, float* actions, void* stream);

/* xLSTMEncoder.forward(inputs_embeds=x_in, past_key_values=state, use_cache=True)
 * (src/algos/models/decision_xlstm.py:138-169) == T x xLSTMBlockStack.step + post_blocks_norm.
 * x_in, x_out: fp32 [B, T, d] (may alias). State updated in place. 1 <= T <= 4. */
int xl_encoder_step(xl_handle* h, void* state, const float* x_in, float* x_out, int B, int T, int mode,
                    unsigned flags, void* stream);

/* mLSTMCell.step's recurrent_step_stabilized_simple + MultiHeadLayerNorm alone ([ext-xlstm], reached via
 * decision_xlstm.py:163), for unit parity. qkv: fp32 [B*T, 3, inner] (q | k | v); igate, fgate: fp32
 * [B*T, NH] pre-activations (bias already added). C (slab-major, see xl_state_part), n [B,NH,DH], m [B,NH]
 * updated in place.
 * h_norm: fp32 [B*T, inner] = GroupNorm_NH(h) * (1 + outnorm_w[inner]); h_raw (nullable): un-normalised h.
 * rows_split / cols_per_cta: 0 = automatic tiling. */
int xl_mlstm_cell_step(xl_handle* h, float* C, float* n, float* m, const float* qkv, const float* igate,
                       const float* fgate, const float* outnorm_w, float* h_norm, float* h_raw, int B, int T,
                       int rows_split, int cols_per_cta, void* stream);

/* The sequence-path counterpart of xl_mlstm_cell_step, for unit parity: the gate scan and the sequence cell that a
 * context prefill of B envs x S tokens runs (chosen by the "prefill_cell" option under the same conditions), then the
 * sequence finalize. C (slab-major), n [B,NH,DH], m [B,NH] updated in place by S tokens.
 *   q, k, v   fp32 [B*S, inner] (rows [env][token], q and k unscaled)
 *   gates     fp32 [B*S, 2, NH] pre-activations (input gates, then forget gates; bias already added)
 *   act       fp32 [B*S, inner] a = silu(conv); u fp32 [B*S, 2*inner] (only the z half u[:, inner:] is read)
 *   outnorm_w, skip fp32 [inner]
 *   num  fp32 [B*S, inner] q^T C per token (un-normalised); qn fp32 [B*S, NH] q.n per token; mseq fp32 [B*NH, S] m
 *   out  fp32 [B*S, inner] (MultiHeadLayerNorm(h) + skip * a) * silu(z), h = num / (max(|qn|, exp(-m)) + cell_eps)
 *   cell (host, nullable) <- the cell that ran: 0 = fp32, 1 = mma.sync, 2 = tcgen05.
 * XL_ERR_UNSUPPORTED (nothing launched) when the cell "prefill_cell" selects cannot take DH and S: the tcgen05 cell
 * needs S >= 64, the mma.sync cell S % 16 == 0, the fp32 cell S % 8 == 0. */
int xl_mlstm_cell_seq(xl_handle* h, float* C, float* n, float* m, const float* q, const float* k, const float* v,
                      const float* gates, const float* act, const float* u, const float* outnorm_w, const float* skip,
                      float* num, float* qn, float* mseq, float* out, int* cell, int B, int S, void* stream);

/* One env step of the whole policy for B envs with device-resident inputs:
 * MultiDomainDiscreteDecisionXLSTMModel.forward on the inference-cache path (online_decision_transformer_
 * model.py:326-390 -> compute_hidden_states :392-461 -> encoder -> get_predictions discrete_decision_
 * transformer_model.py:368-383 -> multi_domain_discrete_dt_model.py:83-108) + MinMaxTokenizer.inv_tokenize
 * (src/tokenizers_custom/minmax_tokenizer.py:31-47).
 *   states  fp32 [B, state_dim]  (already zero-padded to 204: src/algos/decision_xlstm.py:16-19)
 *                                or fp32 [B, d] state embeddings with XL_FLAG_STATE_EMBEDS
 *   rtg     fp32 [B]             returns-to-go of this timestep
 *   rewards fp32 [B] or NULL     reward token input; NULL = 0 (what the reference feeds, evaluation.py:132)
 *   tokens  int32 [B, act_dim]   argmax (or, armed, sampled: xl_set_sampling) action tokens (continuous) / first
 *                                column (discrete)
 *   actions fp32 [B, act_dim]    inv_tokenized actions (continuous) / token as float (discrete)
 *   logits  fp32 [B, act_dim*num_actions] or NULL;  hidden fp32 [B, T, d] or NULL (last_hidden_state) */
int xl_policy_step(xl_handle* h, void* state, const float* states, const float* rtg, const float* rewards,
                   int32_t* tokens, float* actions, float* logits, float* hidden, int B, int mode,
                   unsigned flags, void* stream);

/* Same, with HOST buffers (pinned recommended): copies inputs H2D, runs the step, copies tokens+actions
 * D2H and synchronises the stream. This is the call the batched rollout loop makes once per env step
 * (replacement for src/callbacks/evaluation.py:134-141,152-154: predict + .cpu() + .to(device)). */
int xl_policy_step_host(xl_handle* h, void* state, const float* h_states, const float* h_rtg,
                        const float* h_rewards, int32_t* h_tokens, float* h_actions, int B, int mode,
                        unsigned flags, void* stream);

/* Context prefill of the encoder: x_in fp32 [B, S, d] (already embedded tokens), y_out fp32 [B, S, d] or NULL
 * (last_hidden_state of every token). Leaves `state` exactly where S calls of xLSTMBlockStack.step would
 * (src/algos/models/decision_xlstm.py:161-165; this is what the reference's `chunkwise_step` hook :158-159
 * asks of layers.step with S > 1). Runs layer-major over chunks of tokens: the projections are tcgen05 GEMMs
 * over all rows of a chunk; the mLSTM cell is the chunkwise form over 128-token chunks with every contraction a batched
 * tcgen05 GEMM over the (env, head, chunk) triples (xl_prefill_tc.cu; options "prefill_cell", "prefill_rows").
 * Allocates / grows private workspaces on first use (synchronises the device then); B <= max_batch. */
int xl_prefill(xl_handle* h, void* state, const float* x_in, float* y_out, int B, int S, unsigned flags, void* stream);

/* Same for the whole policy: Tn timesteps of context per env, states fp32 [B, Tn, state_dim], rtg fp32 [B, Tn],
 * rewards fp32 [B, Tn] or NULL (= 0). Embeds every timestep into its (s, rtg, r) tokens
 * (online_decision_transformer_model.py:522-530,588-612) and prefills the 3*Tn tokens; no action outputs
 * (a context only warms the state: src/callbacks/evaluation.py:213-237 `persist_context`; xl_policy_forward below
 * returns them). XL_FLAG_STATE_EMBEDS: XL_ERR_UNSUPPORTED, state untouched (embeddings: xl_policy_prefill_embeds). */
int xl_policy_prefill(xl_handle* h, void* state, const float* states, const float* rtg, const float* rewards, int B,
                      int Tn, unsigned flags, void* stream);

/* Ragged context prefill: a context length per env. lengths is a HOST int32 [B] array (tokens for xl_prefill_ragged,
 * timesteps for xl_policy_prefill_ragged); the buffers keep the shapes above ([B, S, d]; [B, Tn, state_dim], [B, Tn]).
 *  - Env b's state ends exactly where lengths[b] recurrent steps over its first lengths[b] tokens (timesteps) would
 *    leave it, the promise xl_prefill makes, per env. lengths[b] == 0 leaves every byte of env b's state unchanged.
 *  - Inputs at positions >= lengths[b] are never read (they may hold NaN).
 *  - y_out (nullable): row t < lengths[b] holds that token's last_hidden_state; every other row is written as 0.
 *  - Every length == S (Tn): this IS xl_prefill / xl_policy_prefill (bit-identical). Every length 0: the state is left
 *    alone, y_out zeroed, XL_OK.
 *  - XL_ERR_INVALID_ARG before any device work: lengths NULL, a length < 0 or > S (Tn), and the checks of the uniform
 *    calls. XL_ERR_UNSUPPORTED (state untouched) for lengths that are neither all S nor all 0 when the shape has no
 *    sequence path (conv_kernel != 4, or a head dim without a cell plan); no shipped preset is affected.
 *  - The policy form's work never advances the sampler's step counter or the token ring slot (as xl_policy_prefill),
 *    and it rejects XL_FLAG_STATE_EMBEDS as xl_policy_prefill does.
 * Work goes to the envs that have tokens: the active envs are sorted by length (descending, stable) and each chunk runs
 * on the prefix of them that still has tokens, an env's end padded up to the chunk with identity tokens (forget gate 1,
 * input gate 0, conv window and sLSTM state kept). When the active envs are not already envs 0..B'-1 in that order, their
 * state slots are gathered into a library-owned compact state of xl_state_bytes(h, B') bytes (grow-only, freed by
 * xl_destroy; growing it synchronises the device) and scattered back at the end. Not graph-capturable. */
int xl_prefill_ragged(xl_handle* h, void* state, const float* x_in, float* y_out, const int32_t* lengths, int B, int S,
                      unsigned flags, void* stream);
int xl_policy_prefill_ragged(xl_handle* h, void* state, const float* states, const float* rtg, const float* rewards,
                             const int32_t* lengths, int B, int Tn, unsigned flags, void* stream);

/* Outputs of xl_policy_forward. Every pointer is device memory and nullable (NULL = not wanted). */
typedef struct {
  int32_t* tokens;          /* [B, Tn, act_dim]  argmax action tokens per timestep, as xl_policy_step's tokens      */
  float* actions;           /* [B, Tn, act_dim]  as xl_policy_step's actions                                       */
  float* logits;            /* [B, Tn, n_out]    n_out = act_dim * num_actions (discrete: num_actions)             */
  const int32_t* targets;   /* [B, Tn, act_dim]  action tokens to score                                            */
  float* logprobs;          /* [B, Tn, act_dim]  log-probability of targets; needs targets                         */
} xl_seq_outputs;

/* Sequence forward of the policy: the per-timestep action outputs of whole trajectories in one chunkwise pass. This is
 * MultiDomainDiscreteDecisionXLSTMModel.forward(use_inference_cache=False) over [B, Tn] timesteps, every timestep read
 * at its rtg token (SURVEY.md a10/a11), with the state advanced as xl_policy_prefill advances it.
 *  - Inputs: those of xl_policy_prefill: states fp32 [B, Tn, state_dim], rtg fp32 [B, Tn], rewards fp32 [B, Tn] or NULL
 *    (= 0). lengths NULL: every env has Tn timesteps; otherwise a HOST int32 [B] array of values in [0, Tn], as for
 *    xl_policy_prefill_ragged.
 *  - Outputs at (b, t), t < lengths[b]: what xl_policy_step returns at that timestep (sampler disarmed) when env b is
 *    stepped from `state` over its timesteps 0..t. The logits agree to the error of the chunkwise prefill against
 *    recurrent steps; tokens are equal except where the top two logits of a row are closer than that error. Timesteps
 *    that run as eager steps (see below) are bit-identical to xl_policy_step.
 *  - State after the call: bit-identical to xl_policy_prefill (lengths NULL) or xl_policy_prefill_ragged (lengths) on the
 *    same arguments: the same kernels and chunks run, and the head only reads the residual stream.
 *  - logprobs[b,t,j] = log_softmax(row)[targets[b,t,j]], in fp32 with the row maximum subtracted. The row is the one the
 *    sampler draws from: row j of the [act_dim, num_actions] logit block (discrete: all num_actions logits of the env,
 *    not only the discrete_actions the argmax reads; column 0 only). A target < 0 gives 0 (padded action dims past an env's own act_dim); a target >= num_actions gives NaN.
 *  - XL_FLAG_DISCRETE: the token rule and column meaning of xl_policy_step (argmax over the first discrete_actions logits,
 *    actions = (float)token) in column 0; columns >= 1 of tokens / actions / logprobs hold -1 / 0 / 0.
 *  - Past an env's length (t >= lengths[b]): tokens -1, actions, logits and logprobs 0. Inputs there are never read. An
 *    env with length 0 keeps every byte of its state slot.
 *  - Always the argmax: the armed sampler is not used, and neither its step counter nor the token ring slot advances
 *    (as xl_policy_prefill).
 *  - Chunk flow: per chunk of the prefill, post_blocks_norm of the rtg-token rows only (as the head's bf16 operand
 *    planes), the action head as one tcgen05 Linear over the chunk's timesteps into a library-owned logits workspace
 *    (grow-only, chunk timesteps x n_out floats, freed by xl_destroy; growing it synchronises the device), then one
 *    reduction kernel per chunk: argmax, inv_tokenize, log-sum-exp and the scatter to [B, Tn, ...]. The last
 *    Tn mod 8 timesteps of a uniform call (all of them on shapes without the sequence path) run as eager policy steps.
 *  - XL_ERR_INVALID_ARG: out NULL, logprobs without targets, and the checks of xl_policy_prefill(_ragged).
 *    XL_ERR_UNSUPPORTED: XL_FLAG_STATE_EMBEDS; lengths that are neither all Tn nor all 0 on shapes without the sequence
 *    path (as xl_policy_prefill_ragged; state and outputs untouched). Not graph-capturable. State embeddings:
 *    xl_policy_forward_embeds below. */
int xl_policy_forward(xl_handle* h, void* state, const float* states, const float* rtg, const float* rewards,
                      const int32_t* lengths, int B, int Tn, const xl_seq_outputs* out, unsigned flags, void* stream);

/* Context prefill and sequence forward from state embeddings (image observations: the ImpalaCNN embed_image output of
 * every frame, discrete_decision_transformer_model.py:187-203, or the reference's img_is_encoded inputs :185-186).
 *  - state_embeds: device fp32 [B, Tn, d], 16-byte aligned: the state-token embedding of every timestep, as
 *    xl_policy_step takes it with XL_FLAG_STATE_EMBEDS (the embed_state Linear is skipped). rtg, rewards: as for
 *    xl_policy_prefill. lengths: NULL (every env has Tn timesteps) or a HOST int32 [B] array as for
 *    xl_policy_prefill_ragged.
 *  - Results: those of xl_policy_prefill / xl_policy_prefill_ragged / xl_policy_forward with each timestep's state token
 *    replaced by the given embedding. Outputs at (b, t) are what xl_policy_step(XL_FLAG_STATE_EMBEDS) returns when env b
 *    is stepped over its timesteps 0..t; timesteps that run as eager steps (the last Tn mod 8 of a uniform call) are
 *    bit-identical to those steps. The state after xl_policy_forward_embeds is bit-identical to
 *    xl_policy_prefill_embeds on the same arguments.
 *  - Inherited from the calls above: inputs past lengths[b] are never read (they may hold NaN); an env with length 0
 *    keeps every byte of its state slot; outputs past the length are -1 / 0; lengths all Tn are the uniform call
 *    (bit-identical); always the argmax; the sampler step counter and the token ring slot do not move; not
 *    graph-capturable; on shapes without the sequence path, lengths that are neither all Tn nor all 0 give
 *    XL_ERR_UNSUPPORTED with state and outputs untouched.
 *  - Each chunk's tokens come from one kernel (seq_embed_tokens_kernel) that reads the embedding, rtg and reward of
 *    every (env, timestep) row from these buffers and applies embed_ln, writing the prefill's token rows; it shares its
 *    per-row arithmetic with the step's embed kernel, so a state token gets the bits xl_policy_step gives it.
 *  - Flags: XL_FLAG_DISCRETE and XL_FLAG_SIMPLE_GEMM as for xl_policy_forward; XL_FLAG_STATE_EMBEDS is accepted and
 *    redundant.
 *  - XL_ERR_INVALID_ARG before any device work: a null required pointer, state_embeds not 16-byte aligned, logprobs
 *    without targets, and the checks of xl_policy_prefill(_ragged). */
int xl_policy_prefill_embeds(xl_handle* h, void* state, const float* state_embeds, const float* rtg,
                             const float* rewards, const int32_t* lengths, int B, int Tn, unsigned flags,
                             void* stream);
int xl_policy_forward_embeds(xl_handle* h, void* state, const float* state_embeds, const float* rtg,
                             const float* rewards, const int32_t* lengths, int B, int Tn, const xl_seq_outputs* out,
                             unsigned flags, void* stream);

/* out[M,N] = A[M,K] @ W[N,K]^T (+ bias[N]) (+ residual[M,N]); A fp32, W bf16, fp32 accumulate.
 * The nn.Linear of proj_up / proj_down / embed_state / action_net. impl: 0 auto, 1 CUDA-core, 2 tcgen05. */
int xl_linear(xl_handle* h, const float* A, const void* W_bf16, const float* bias, const float* residual,
              float* out, int M, int N, int K, int impl, void* stream);

/* Implementation switches for A/B measurements (defaults in brackets):
 *   "state_impl": [1] one-shot TMA ring, 2 persistent stream-K TMA ring, 0 register-batched global loads
 *   "state_stages" / "state_ctas_per_sm": ring depth and persistent CTAs per SM of impl 2 (0 = default)
 *   "state_rows_split": row chunks per (env, head) of impl 0/1 (0 = automatic)
 *   "gemm_impl":  [0] auto (tcgen05 when K % 64 == 0), 1 CUDA-core, 2 tcgen05
 *   "gemm_splitk": [8] max split-K planes of proj_up / proj_down (cost model picks <= this; 0/1 = off). Each
 *                  split CTA writes its partial tile to its own plane; the consumer kernels (LayerNorm,
 *                  conv/qkv, finalize) add the planes in order: no atomics, bit-reproducible
 *   "gemm_up_bn" / "gemm_up_splits" / "gemm_down_bn" / "gemm_down_splits": [0 = cost model] force tile width
 *                  (32/64/128) and split-K factor of the two projections
 *   "pdl": [1] programmatic dependent launch of every kernel (process-wide)
 *   "l2_prefetch_mb": [-1 = automatic] MiB of the next block's C warmed into L2 on a side stream while the current
 *                   block's latency-bound chain runs (0 = off; automatic = 48 when a block's C is 100..300 MB)
 *   "state_fuse": [0] finalize (n/m update, GroupNorm, output gate) inside the state stream kernel through one
 *                   thread-block cluster per (env, head): 1 = every CTA finishes its 128 columns, statistics over DSMEM;
 *                   2 = numerators pushed to rank 0, which finalizes the head. One launch fewer per block; measured
 *                   +1-2 % at 206M x 128 / 48M x 256 envs, -5 % at 48M x 64 (profiles/r02_chain_fusion.md)
 *   "small_state_fuse": [0] few-env path (B*T <= 16 rows, see "smallm"): variant 2 of "state_fuse" over the head's
 *                   slab x row-chunk tiles (one cluster of <= 16 CTAs; 2..16 = cluster cap). One launch fewer per block;
 *                   measured slower at 16M / 48M x 1 env (+3 us per block), 3 % faster at 206M x 1 and 48M x 4
 *   "up_fuse": [0] conv + SiLU + q/k/v + gate partials in the proj_up epilogue (gemm_up_conv_kernel); one launch fewer
 *                   per block, x_m never leaves the chip; measured 3-9 % slower (more CTAs re-read the A planes from L2)
 *   "gemm_bm": [0] 64 = 64-row tcgen05 tiles for proj_up / proj_down (bit-identical; measured 1 % slower at 48M x 64)
 *   "gemm_2cta": [-1 = automatic] 2-SM Linear: a CTA pair computes 256 x 256 tiles with tcgen05.mma.cta_group::2, each CTA
 *                   staging its 128 A rows and half of the W tile; 2 = persistent pairs with a double-buffered TMEM
 *                   accumulator (the epilogue of a tile overlaps the MMAs of the next), 1 = one tile per pair, 0 = never,
 *                   automatic = the persistent form for M >= 2048 rows (context prefill: -7 %). Bit-identical to the 1-SM kernel
 *   "fuse_ends": [1] pad+split of the states in one kernel, block 0's pre-norm inside the embed kernel, post-norm of the
 *                   action-token rows only fused with the head's operand split (3-4 launches fewer per env step)
 *   "conv_impl": [2] pre-cell kernel (conv + SiLU + q/k/v + gate partials): 0 = one thread per 4-channel block walking
 *                   the step's tokens in sequence; 1 = one thread per (4-channel block, token) (measured 5 % slower on the
 *                   48M x 64 step: 3x the per-thread weight loads); 2 = as 0 on packed fp32 pairs (FFMA2), gate weights loaded
 *                   before the dependency wait, one butterfly reduction per warp (+3 % on that step; KS = 4 and NH <= 4, other
 *                   shapes run 0). All three give bit-identical outputs
 *   "smallm": [-1 = automatic] LN + proj_up + conv/qkv as one GEMV-style kernel and proj_down as another (4 kernels
 *                   per block instead of 6, fp32 activations against bf16 weights on CUDA cores). 1 = whenever
 *                   B*T <= 16 rows, 0 = never, automatic = B*T <= 4 rows and d <= 1024 (one env: -14 % step latency)
 *   "prefill_cell": [2] sequence cell of the context prefill: 2 = chunkwise on tcgen05 (128-token chunks, head dims that
 *                   are multiples of 128), 1 = chunkwise on mma.sync (16-token chunks), 0 = fp32 token-order cell
 *   "prefill_rows": [16384] rows (envs x tokens) per prefill chunk; "prefill_conv_run": [16] tokens per thread run of the
 *                   sequence conv/qkv kernel; "prefill_tc_fused": [1] chunk update + scan in one kernel (0 = through HBM)
 *   "prefill_conv": [2] sequence conv/qkv/gates kernel of the prefill (process-wide): 0 = scalar fp32, 1 = packed fp32 pairs
 *                   (FFMA2; bit-identical to 0), 2 = 1 with the SFU SiLU (~2 ulp); "prefill_conv_persist": [1] that kernel
 *                   walks the token runs with 2 CTAs per SM (weights staged once per CTA) instead of one CTA per 64 tokens
 *   "prefill_prep": [1] chunk operand planes from one read of q, k, v through a shared-memory tile (0 = three-pass kernel;
 *                   bit-identical); "prefill_tc_overlap": [1] S = QK^T, P~ and the n scan on a side stream beside the chunk
 *                   update + scan when that kernel leaves >= 32 SMs idle (bit-identical); "prefill_scan_split": [2] epilogue warps
 *                   per TMEM lane quarter of that kernel (4 = 16 warps: bit-identical, measured 9 % slower)
 *   measurement / probe switches (A/B records under profiles/; none changes results):
 *   "l2_prefetch_policy": [0] 1 = warm-up with an L2 evict_last policy; "host_zero_copy": [1] xl_policy_step_host reads and
 *                   writes pinned host buffers through their device aliases (0 = staged copies);
 *   "gemm_cluster": [1] 2 / 4 = A tile TMA-multicast across a cluster of column-tile CTAs (process-wide; measured slower);
 *   "gemm_m64_layout": [0] probe of the TMEM row layout of 64-row UMMA tiles (tests only);
 *   "debug_skip": only in -DXL_DEBUG_OPTIONS builds (skips kernel classes to read their marginal cost; results garbage) */
int xl_set_option(xl_handle* h, const char* name, int value);

/* Counters for bench.py: kernels launched by this handle since the last call (reset on read). */
int64_t xl_launch_count(xl_handle* h);

/* Measurement aid for bench.py: between begin and end, every EAGER (non-graph) launch of the mLSTM state-step
 * kernel is bracketed by CUDA events on the launching stream, and every xl_policy_step by another pair.
 * xl_profile_end synchronises those events and returns the summed state-kernel time, the number of its
 * launches, and the summed step time (all ms). */
int xl_profile_begin(xl_handle* h);
int xl_profile_end(xl_handle* h, double* state_kernel_ms, int64_t* state_kernel_launches, double* step_ms);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* XLSTM_B200_H */
