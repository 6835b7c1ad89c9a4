// Internal launcher declarations shared by the translation units of libxlstm_b200.so.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace xl {

extern int g_use_pdl;   // programmatic dependent launch of every kernel (xl_common.cuh); xl_set_option("pdl")

// ---- xl_elementwise.cu ---------------------------------------------------------------------------
// LayerNorm over the last dim for `rows` rows. gamma = (residual_weight ? 1 + w : w), optional bias.
// in row r at in + r*in_stride, out row r at out + r*out_stride. Optional bf16 hi/lo split outputs
// (row-major [rows, d], dense) for the tensor-core GEMM A operand.
void launch_ln_rows(const float* in, int64_t in_stride, float* out, int64_t out_stride, const float* w,
                    const float* bias, int residual_weight, float eps, int rows, int d, void* a_hi,
                    void* a_lo, cudaStream_t s);
// Same, but first folds a split-K proj_down into the residual stream: x[r] += sum_z part[z*part_stride + r*d]
// (planes added in order z = 0..splits-1; x dense [rows, d], updated in place), then normalises x. d <= 4096.
void launch_ln_rows_reduce(float* x, const float* part, int splits, int64_t part_stride, float* out,
                           int64_t out_stride, const float* w, float eps, int rows, int d, void* a_hi, void* a_lo,
                           cudaStream_t s);

// Token embedding of one timestep: rows (b, tok) of [B,3,d]:
//   tok 0 = s_emb[b] (state Linear output incl. bias), tok 1 = rtg[b]*w_ret + b_ret,
//   tok 2 = rew[b]*w_rew + b_rew (rew == nullptr -> 0), then embed_ln (weight, bias).
void launch_embed_tokens(const float* s_emb, const float* rtg, const float* rew, const float* w_ret,
                         const float* b_ret, const float* w_rew, const float* b_rew, const float* ln_w,
                         const float* ln_b, float eps, float* x, int B, int d, unsigned* step_counter,
                         unsigned* sample_counter, const float* ln0_w, float ln0_eps, float* xn0, void* a_hi,
                         void* a_lo, cudaStream_t s);
// ln0_w != nullptr: also the first block's pre-norm of the produced rows -> xn0 (fp32) and/or bf16 hi/lo planes
// step_counter / sample_counter (nullable): incremented once per launch (token ring slot / sampler step)
void launch_pad_split(const float* in, int K, void* hi, void* lo, int Kpad, int rows, cudaStream_t s);
void launch_ln_rows_gather(const float* x, const float* part, int splits, int64_t part_stride, const float* w,
                           float eps, int rows, int d, int row_mul, int row_off, void* a_hi, void* a_lo,
                           cudaStream_t s);

// zero-pad states [B, K] -> [B, Kpad]
void launch_pad_rows(const float* in, int K, float* out, int Kpad, int rows, cudaStream_t s);
// copy rows with strides (token gather / scatter in per-token mode)
void launch_copy_rows(const float* in, int64_t in_stride, float* out, int64_t out_stride, int rows, int d,
                      cudaStream_t s);

struct ConvQkvParams {
  const float* u;       // [M, 2*inner]  (x_m | z) from proj_up; u_splits > 1: sum of that many split-K planes
  int u_splits;         // 0/1 = one plane
  int64_t u_stride;     // elements between planes
  float* conv_state;    // [B, KS, inner] in/out
  const float* conv_w;  // [inner, KS]
  const float* conv_b;  // [inner]
  const float* wq;      // [inner/4, 4, 4]
  const float* wk;
  const float* wv;
  const float* wi;      // [NH, 3*inner]
  const float* wf;      // [NH, 3*inner]
  float* qk;            // [M, NH, DH, 2]  (q, k) interleaved per channel
  float* v;             // [M, inner]
  float* act;           // [M, inner]   a = silu(conv)
  float* gate_part;     // [M, NCH, 2*NH]  partial gate pre-activations per channel chunk
  int B, T, inner, NH, KS, NCH;
  int impl;             // step path only: 0 = one thread per 4-channel block (tokens in sequence), 1 = one thread per
                        // (4-channel block, token)
};
// false when (KS, T, NH) has no instantiation
bool launch_conv_qkv_gates(const ConvQkvParams& p, cudaStream_t s);

// argmax over action logits + inv_tokenize.
// continuous: logits [B, act_dim*num_actions] -> tokens [B, act_dim], actions = max(tok-shift,0)*bw+min
// discrete:   tokens[b*act_dim] = argmax(logits[b, :discrete_actions]); actions[b*act_dim] = (float)token
// logits row b starts at logits + b*row_pitch.
void launch_argmax_tokens(const float* logits, int64_t row_pitch, int B, int act_dim, int num_actions,
                          int discrete_actions, int discrete, float bin_width, float min_val,
                          int32_t* tokens, float* actions, int32_t* ring, const unsigned* step_counter,
                          int ring_slots, int64_t ring_slot_stride, cudaStream_t s);
void launch_set_u32(unsigned* p, unsigned v, cudaStream_t s);

// ---- xl_sample.cu --------------------------------------------------------------------------------
// Stochastic action selection (xl_set_sampling; contract in include/xlstm_b200.h): drop-in for launch_argmax_tokens
// with the same layouts. prm points at a device copy of the parameters; the step drawn for is *step_counter - 1;
// env b's global id is prm->env_id_base + (env_offset + b) * prm->env_id_stride. num_actions <= kSampleMaxActions,
// act_dim <= kSampleMaxRows.
constexpr int kSampleMaxActions = 512;
constexpr int kSampleMaxRows = 8;
void launch_sample_tokens(const float* logits, int64_t row_pitch, int B, int act_dim, int num_actions,
                          int discrete_actions, int discrete, float bin_width, float min_val, int32_t* tokens,
                          float* actions, int32_t* ring, const unsigned* ring_counter, int ring_slots,
                          int64_t ring_slot_stride, const void* prm, const unsigned* step_counter, int env_offset,
                          cudaStream_t s);
// stream-ordered write of the parameters (an xl_sampling) to dst and of `counter_value` to *counter
void launch_set_sampling(void* dst, const void* params, unsigned* counter, unsigned counter_value, cudaStream_t s);

void launch_state_reset(float* C, float* n, float* m, float* conv, const uint8_t* mask, int B,
                        int64_t c_per_env, int64_t n_per_env, int64_t m_per_env, int64_t conv_per_env,
                        cudaStream_t s);

// Geometry of two state buffers of the same handle for the ragged prefill: [0] = the caller's state (B[0] envs),
// [1] = the compact state (B[1] envs). Offsets are bytes within a block's slot (state_layout of xl_api.cu); *_env are
// bytes per env of each part (s_env: per plane of the sLSTM's [4, B, d] planes).
struct StateCopyGeom {
  uint64_t slstm_mask;
  int num_blocks;
  int B[2];
  size_t layer_bytes[2], slayer_bytes[2];
  size_t c_off[2], n_off[2], m_off[2], conv_off[2], s_off[2], sconv_off[2];
  size_t c_env, n_env, m_env, conv_env, s_env, sconv_env;
};
// Every part of every block of env perm[k] of the caller's state <-> env k of the compact state, k < Bc.
// to_caller = 0: gather (caller -> compact); 1: scatter (compact -> caller). One launch, 128-bit accesses where a part's
// per-env size allows them.
void launch_state_permute(void* caller, void* compact, const int32_t* perm, int Bc, const StateCopyGeom& g,
                          int to_caller, cudaStream_t s);
// Ragged prefill row gather / scatter of one chunk. Compact row (k, t), k < Bk, t < Sc, <-> caller row
// (perm[k], pos + t) of a [*, S, width] buffer; n_k = clamp(len[k] / len_div - pos, 0, Sc) rows of env k are valid.
// to_caller = 0: compact[k, t] = t < n_k ? caller[perm[k], pos + t] : 0 (pad rows zero-filled, the caller's never read);
// 1: caller[perm[k], pos + t] = compact[k, t] for t < n_k only.
void launch_ragged_rows(float* caller, float* compact, const int32_t* perm, const int32_t* len, int len_div, int Bk,
                        int S, int Sc, int pos, int width, int to_caller, cudaStream_t s);

// ---- xl_seq_head.cu ------------------------------------------------------------------------------
// Per-timestep head reduction of xl_policy_forward over the logits of one chunk: argmax token (warp_argmax), action,
// log-probability of the target and a copy of the logit row, each written to its [B, Tn, ...] position.
struct SeqHeadParams {
  const float* logits;          // [rows, n_out] chunk rows: row r = timestep pos + r % Tc of compact env r / Tc
  int rows, Tc, pos, Tn;
  int n_out, act_dim, num_actions, discrete_actions, discrete;
  float bin_width, min_val;
  const int32_t* perm;          // compact env k -> caller env perm[k]; nullptr = identity
  const int32_t* len;           // ragged: env k's valid timesteps are t < len[k] / len_div (others skipped); nullptr = all
  int len_div;
  int32_t* tokens;              // [B, Tn, act_dim] (nullable, as every output below)
  float* actions;               // [B, Tn, act_dim]
  float* out_logits;            // [B, Tn, n_out]
  const int32_t* targets;       // [B, Tn, act_dim] (needed with logprobs)
  float* logprobs;              // [B, Tn, act_dim]
};
void launch_seq_head(const SeqHeadParams& p, cudaStream_t s);

// Embedded (s, rtg, r) tokens of one prefill chunk from given state embeddings (xl_policy_forward_embeds /
// xl_policy_prefill_embeds), with the step embed kernel's per-row arithmetic: x row (k * Tc + t) * 3 + tok from caller
// env perm[k], timestep pos + t. Rows past the env's length read nothing and are the tokens of zeros (see
// xl_elementwise.cu).
struct SeqEmbedParams {
  const float* s_emb;           // [B, Tn, d] state-token embeddings (16-byte aligned)
  const float* rtg;             // [B, Tn]
  const float* rew;             // [B, Tn] or nullptr (= 0)
  const int32_t* perm;          // compact env k -> caller env perm[k]; nullptr = identity
  const int32_t* len;           // env k's valid timesteps are t < len[k] / len_div - pos; nullptr = all Tc
  int len_div, Tn, Tc, pos;
  int rows, d;                  // rows = Bk * Tc timesteps
  const float *w_ret, *b_ret, *w_rew, *b_rew, *ln_w, *ln_b;
  float eps;
  float* x;                     // [Bk, Tc, 3, d]
};
void launch_seq_embed_tokens(const SeqEmbedParams& p, cudaStream_t s);

// bulk L2 prefetch of [base, base+bytes) (side stream, plain launch; see xl_elementwise.cu)
void launch_l2_prefetch(const void* base, size_t bytes, int num_sms, int evict_last, cudaStream_t s);

// ---- xl_state_step.cu ----------------------------------------------------------------------------
struct StateStepParams {
  float* C;                 // [B, NH, DH/Wc, DH, Wc] slab-major (Wc = 128 when DH % 128 == 0, else DH)
  float* n;                 // [B, NH, DH]
  float* m;                 // [B, NH]
  const float* qk;          // [M, NH, DH, 2]  (q, k) pairs, unscaled
  const float* v;           // [M, inner]
  const float* gate_part;   // [M, NCH, 2*NH]  (i gates first NH, f gates next NH), summed in order
  const float* igate_b;     // [NH] or nullptr
  const float* fgate_b;     // [NH] or nullptr
  const float* outnorm_w;   // [inner] (gamma = 1 + w)
  const float* skip;        // [inner] or nullptr  -> out = h_norm when nullptr
  const float* act;         // [M, inner]   (used when skip != nullptr)
  const float* u;           // [M, 2*inner] (z = u[:, inner:]) (used when skip != nullptr)
  int u_splits;             // split-K planes of u to add (0/1 = one plane), u_stride elements apart
  int64_t u_stride;
  float* out;               // [M, inner]  (h_norm + skip*a) * silu(z), or h_norm
  void* out_hi;             // optional bf16 hi/lo split of `out`
  void* out_lo;
  float* h_raw;             // optional [M, inner] un-normalised h
  float* partial;           // scratch [B*NH, RS, T, DH]
  int B, T, NH, DH, inner, NCH;
  int rows_split;           // RS
  int cols_per_cta;         // multiple of 4, <= 128, divides DH
  int impl;                 // 2 = persistent TMA ring (default), 1 = one-shot TMA ring, 0 = register-batched loads
  int stages;               // impl 2: ring depth (0 = default)
  int ctas_per_sm;          // impl 2: persistent CTAs per SM (0 = 1)
  int meta_slots;           // impl 2: depth of the segment-metadata ring (0 = 3)
  // impl 2 stream-K partition (filled by the launchers): grid G, tiles per CTA q (+1 for the first r CTAs),
  // partial slots per item. sk_grid == 0 -> rows_split layout of impl 0/1.
  int sk_grid, sk_q, sk_r, sk_smax;
  int num_layers;           // blocks sharing the L2 with this one (cache-policy choice); 0 = 1
  int max_cluster;          // leader variant: most CTAs (slabs x row chunks) per cluster, 0 = 16 (the opt-in maximum)
  int fuse_finalize;        // 1: let the stream kernel finalize inside a cluster per (env, head) when the tiling allows
                            // (state_step_fuses_finalize); launch_state_finalize must then NOT be called
  float ln_eps, cell_eps;
};
// Kernel 1 (stream C, emit partial numerators) and kernel 2 (n/m update, normalise, gate). Both pick the
// same tiling when rows_split / cols_per_cta are 0. Return cudaError.
cudaError_t launch_state_step(StateStepParams p, int num_sms, cudaStream_t s);
bool state_step_fuses_finalize(StateStepParams p, int num_sms);
cudaError_t launch_state_finalize(StateStepParams p, int num_sms, cudaStream_t s);
void state_step_auto_tiling(int B, int NH, int DH, int num_sms, int* rows_split, int* cols_per_cta);
void launch_repack_qkv(const float* qkv, float* qk, float* v, int M, int inner, cudaStream_t s);

// ---- xl_slstm.cu ---------------------------------------------------------------------------------
// sLSTM block (xLSTM[a:b] stacks). Rows ordered [env][token], T tokens per env; DHs = d / NH.
// Ragged prefill (len != nullptr): env b of the launch has n_b = clamp(len[b] - pos, 0, T) real tokens; the tokens
// after them are identity pads that change no state (len == nullptr: all T tokens are real).
// conv step over the T tokens + swish: xc [M,d]; conv_state [B,KS,d] in/out. false: KS not instantiated
bool launch_slstm_conv(const float* xn, float* conv_state, const float* cw, const float* cb, float* xc, int B,
                       int T, int d, int KS, cudaStream_t s, const int32_t* len = nullptr, int pos = 0);
// pre [M,4,d] (gate-major i,f,z,o) = bias + headwise projections (i,f from xc; z,o from xn); W_* [NH,DHs,DHs],
// bias [NH,4,DHs]
void launch_slstm_gates(const float* xc, const float* xn, const float* w_i, const float* w_f, const float* w_z,
                        const float* w_o, const float* bias, float* pre, int M, int d, int NH, cudaStream_t s);
// token t of every env: raw = pre + R y_{t-1}, pointwise update of (c,n,m) in st [4,stB,d] (st points at the
// slice's first env, B envs processed); y -> y_out [M,d]. A pad token (t >= n_b) leaves (c,n,m) alone and carries
// y_{t-1} into its y_out row, so that slstm_out stores the y of the env's last real token.
cudaError_t launch_slstm_cell(const float* pre, const float* R, float* st, float* y_out, int B, int stB, int T, int t,
                              int d, int NH, cudaStream_t s, const int32_t* len = nullptr, int pos = 0);
// x += MultiHeadLayerNorm(y_out) (gamma = 1 + w); st_y [B,d] <- y of each env's last token
void launch_slstm_out(const float* y_out, const float* gn_w, float* x, float* st_y, int M, int T, int d, int NH,
                      float eps, cudaStream_t s);
// gated feed-forward middle: gelu(up[:, :ff]) * up[:, ff:] -> fp32 out and/or bf16 hi/lo planes [M, ff]
void launch_ffn_gate(const float* up, float* out, void* hi, void* lo, int M, int ff, cudaStream_t s);

// ---- xl_prefill.cu -------------------------------------------------------------------------------
// Sequence (context prefill) versions of the per-block kernels; rows are ordered [env][token] with S tokens
// per env. S % 8 == 0.
// Ragged prefill (len != nullptr, the chunk starting at token pos of the context): env b has n_b = clamp(len[b] - pos,
// 0, S) real tokens, then identity pads (lf = 0, i~ = -inf: f = 1, i = 0, m carried, so every cell leaves C and n as
// they are). Every env of such a launch has n_b >= 1. len == nullptr: all S tokens are real, results as before.
bool prefill_cell_supported(int DH);
// conv + SiLU + q/k/v + gate partials over the chunk, then conv_state <- last KS inputs (ragged: the last KS rows of
// the old window followed by the env's n_b inputs). p.qk receives the q plane [M, inner] followed by the k plane
// [M, inner] (M = B*S). false: no instantiation
bool launch_conv_qkv_gates_seq(const ConvQkvParams& p, int S, cudaStream_t s, const int32_t* len = nullptr,
                               int pos = 0);
// m/f/i per token ([B*NH][S] each) from the gate partials; m_state [B*NH] in/out; scratch: gate_scan_seq_scratch_floats()
size_t gate_scan_seq_scratch_floats(int B, int S, int NH);
void launch_gate_scan_seq(const float* gate_part, const float* igate_b, const float* fgate_b, float* m_state,
                          float* fseq, float* iseq, float* mseq, float* scratch, int B, int S, int NH, int NCH,
                          cudaStream_t s, const int32_t* len = nullptr, int pos = 0);
// C / n advanced over the S tokens on chip; num [B*S, inner] = q^T C, qn [B*S, NH] = q.n per token
cudaError_t launch_cell_seq(float* C, float* n, const float* q, const float* k, const float* v, const float* fseq,
                            const float* iseq, float* num, float* qn, int B, int S, int NH, int DH, int inner,
                            cudaStream_t s);
// chunkwise tensor-core sequence cell (xl_prefill_mma.cu): prep kernel + mma.sync cell kernel; S % 16 == 0
bool prefill_cell_mma_supported(int DH);
int prefill_cell_mma_chunk();
void prefill_cell_mma_ws(int rows, int NH, int DH, size_t* common_bytes, size_t* vblk_bytes);
cudaError_t launch_cell_mma(float* C, float* n, const float* q, const float* k, const float* v, const float* fseq,
                            const float* iseq, float* num, float* qn, void* common, void* vblk, int B, int S, int NH,
                            int DH, int inner, cudaStream_t s);
// chunkwise sequence cell on tcgen05 (xl_prefill_tc.cu): 128-token chunks, every contraction a batched tcgen05 GEMM over
// the (env, head, chunk) triples of the run; any S >= 1 (a ragged last chunk is padded with neutral gates)
extern int g_gemm_2cta;
extern int g_prefill_tc_fused;
extern int g_prefill_conv_run;
extern int g_prefill_conv_impl;
extern int g_prefill_conv_persist;
extern int g_prefill_prep;
bool prefill_cell_tc_supported(int DH);
int prefill_cell_tc_chunk();
size_t prefill_cell_tc_ws_bytes(int B, int S, int NH, int DH);
extern int g_prefill_tc_overlap;
extern int g_prefill_scan_split;
// side stream + fork/join events (caller-owned) for the kernels of the cell that may run beside the chunk update + scan
struct CellSideStream {
  cudaStream_t stream;
  cudaEvent_t fork, join;
};
cudaError_t launch_cell_tc(float* C, float* n, const float* q, const float* k, const float* v, const float* fseq,
                           const float* iseq, float* num, float* qn, void* ws, int B, int S, int NH, int DH, int inner,
                           cudaStream_t s, const CellSideStream* side = nullptr);
cudaError_t launch_finalize_seq(const float* num, const float* qn, const float* mseq, const float* outnorm_w,
                                const float* skip, const float* act, const float* u, float* out, void* out_hi,
                                void* out_lo, int B, int S, int NH, int DH, int inner, float ln_eps, float cell_eps,
                                cudaStream_t s);

// ---- xl_smallm.cu --------------------------------------------------------------------------------
// Front half of an mLSTM block for M = B*T <= 16 rows as one GEMV-style kernel: LN + proj_up + conv/SiLU +
// headwise q/k/v + gate partials (one chunk per CTA that owns x_m columns). Outputs in the layouts the state-stream
// and finalize kernels read.
struct SmallPreParams {
  const float* x;               // [M, d] residual stream
  const float* norm_w;          // [d] (gamma = 1 + w)
  const __nv_bfloat16* w_up;    // [2*inner, d]
  const float *conv_w, *conv_b, *wq, *wk, *wv, *wi, *wf;
  float* conv_state;            // [B, 4, inner] in/out
  float* u;                     // [M, 2*inner]: only the z half is written
  float* qk;                    // [M, inner, 2]
  float* v;                     // [M, inner]
  float* act;                   // [M, inner]
  float* gate_part;             // [M, NCH, 2*NH], one chunk per cluster of CTAs
  int B, T, d, inner, NH, NCH;  // NCH = smallm_pre_chunks() <= 16
  float ln_eps;
};
int smallm_pre_chunks(int B, int T, int d, int inner, int NH, int KS);   // 0 = shape not supported
cudaError_t launch_smallm_pre(const SmallPreParams& p, cudaStream_t s);
// Back half: x[M,d] += g[M,inner] W_down[d,inner]^T as warp GEMVs (no split-K planes, x complete on exit).
struct SmallDownParams {
  const float* g;               // [M, inner] fp32 (finalize kernel output)
  const __nv_bfloat16* w_down;  // [d, inner]
  float* x;                     // [M, d] in/out
  int M, d, inner;
};
cudaError_t launch_smallm_down(const SmallDownParams& p, cudaStream_t s);

// ---- xl_gemm.cu ----------------------------------------------------------------------------------
// out[M,N] = A[M,K] W[N,K]^T (+bias) (+residual), A fp32, W bf16, CUDA cores, fp32 accumulate.
void launch_gemm_simple(const float* A, const __nv_bfloat16* W, const float* bias, const float* residual,
                        float* out, int M, int N, int K, cudaStream_t s);

// ---- xl_gemm_tc.cu -------------------------------------------------------------------------------
// Pre-cell epilogue of the up-projection (fused 3-token step): what conv_qkv_gates_kernel computes, done on the x_m
// tile while it is still on chip. Row tiles hold whole envs (42 envs x 3 tokens = 126 rows); gate partials come out
// per 32-channel tile: gate_part [M, NCH = gemm_up_conv_chunks(inner) = inner/32, 2*NH].
struct UpEpiParams {
  float* conv_state;           // [B, 4, inner] in/out
  const float *conv_w, *conv_b, *wq, *wk, *wv, *wi, *wf;
  float *qk, *v, *act, *gate_part;
  int B, T, inner, NCH;
};
bool gemm_up_conv_supported(int T, int KS, int NH, int inner, int d);
int gemm_up_conv_chunks(int inner);
cudaError_t launch_gemm_up_conv(const void* a_hi, const void* a_lo, const __nv_bfloat16* W, float* u, int M, int d,
                                const UpEpiParams& ep, cudaStream_t s);

// tcgen05 path: A given as bf16 hi/lo planes (A = hi + lo), W bf16, fp32 accumulate in TMEM.
bool gemm_tc_supported(int M, int N, int K);
extern int g_gemm_cluster;                     // 1 off, 2 / 4: A-tile multicast across column-tile CTAs ("gemm_cluster")
extern int g_gemm_bm;                          // 0 automatic, 64 / 128 forced ("gemm_bm")
void gemm_tc_set_m64_layout(int contiguous);   // probe of the M = 64 TMEM accumulator layout ("gemm_m64_layout")
void launch_split_bf16(const float* in, int64_t in_stride, void* hi, void* lo, int rows, int K, cudaStream_t s);
// bn = tile width (128/64/32, 0 = planned). splits > 1 = split-K: CTA z writes its raw partial tile to the plane
// out + z*split_stride (bias/residual must be null); the consumer kernels add the planes in order.
cudaError_t launch_gemm_tc(const void* a_hi, const void* a_lo, const __nv_bfloat16* W, const float* bias,
                           const float* residual, float* out, int M, int N, int K, int num_sms, int bn, int splits,
                           long long split_stride, int low_smem, cudaStream_t s);
// cost model: tile width and split-K factor (<= max_splits, dividing K/64)
void gemm_tc_plan(int M, int N, int K, int num_sms, int max_splits, int* bn_out, int* splits_out);

}  // namespace xl
