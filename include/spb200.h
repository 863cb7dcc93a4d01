/* spb200.h -- C ABI of libspb200.so, the sm_100a kernel library behind scoreperformer_b200.
 *
 * The reference (ilya16/ScorePerformer) has no FFI: its hot path is PyTorch eager code behind the nn.Module API of
 * `scoreperformer.models` (SURVEY.md section 8b).  This header is therefore the *new* bottom layer: each entry point
 * replaces the PyTorch library calls made by the reference lines cited next to it.  A maintainer binds it with
 * ctypes (see INTEGRATION.md); scoreperformer_b200/lib.py is exactly that binding.
 *
 * Conventions
 *   - every function returns 0 on success or a negative code (-1 bad argument, -2 CUDA runtime error, -3 driver API
 *     error) and never throws; `spb_last_error()` returns the message for the calling thread;
 *   - all pointers are DEVICE pointers owned by the caller (PyTorch tensors); the library allocates nothing;
 *   - `stream` is the caller's current CUDA stream (cudaStream_t passed as void*); no call synchronises;
 *   - bf16 buffers are `void*`, fp32 are `float*`, masks are `uint8_t*` (torch.bool), tokens/labels `int64_t*`;
 *   - "ACCUMULATED" outputs are added to (the caller zero-initialises), everything else is overwritten;
 *   - dropout masks come from a counter hash of (seed + *rng_offset, element index); `rng_offset` (device uint64, may be NULL) lets
 *     CUDA-graph replays draw fresh masks; the backward regenerates the forward's mask from the same pair;
 *   - functions are re-entrant; the only global state is the cached driver entry point for TMA descriptor encoding.
 */
#ifndef SPB200_H
#define SPB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* spb_stream_t; /* cudaStream_t */

int spb_abi_version(void);
const char* spb_last_error(void);

/* fp32 -> bf16 cast (autocast's weight/activation casts); optionally zeroes rows where rowmask is false. */
int spb_cast_f32_bf16(const float* src, void* dst, int64_t n, const uint8_t* rowmask, int row_len, spb_stream_t stream);

/* out fp32 [n_cols] += column sums of x [n_rows, ld] (bias gradients of every Linear). */
int spb_colsum(const void* x, int x_fp32, int ld, float* out, int n_rows, int n_cols, spb_stream_t stream);

/* C[M,N] = alpha * op(A) op(B)^T (+bias[n]) (*rowmask[m]) (+residual[m,n]);  tcgen05/TMEM/TMA GEMM, bf16 in, fp32 accumulate.
 *   trans_a = 0: A is row-major [M,K] (lda);  1: A is stored [K,M] (lda)        -- wgrad's dY^T
 *   trans_b = 0: B is row-major [N,K] (ldb), i.e. an nn.Linear weight;  1: stored [K,N] (ldb)   -- dgrad / wgrad
 *   c_fp32: output dtype; split_k: 0 auto, 1 off, >1 forced (fp32 C only); accumulate: add into C (fp32 only);
 *   alpha: optional device scalar.
 * Replaces: nn.Linear / F.linear / `@` in modules/transformer/attention.py:135-137,214, feedforward.py:19-21,56-61,
 * modules/layers.py:41-47, models/scoreperformer/embeddings.py:134-143,253-255,345-353 and their autograd backward. */
int spb_gemm_bf16(const void* A, const void* B, void* C, int M, int N, int K, int trans_a, int trans_b, int lda, int ldb, int ldc,
                  const float* bias, const float* residual, int ldr, const uint8_t* rowmask, int c_fp32, int split_k, int accumulate,
                  const float* alpha, spb_stream_t stream);

/* spb_gemm_bf16 with a bf16 C (no residual / split-K) whose epilogue also emits the per-head row dots
 *   rowdot_out[(b*H + h)*T + t] = sum_{c in head h} C[b*T + t, c] * X[b*T + t, c]     (N == H*64, X bf16 [M, ld_x])
 * = attention backward's delta = rowsum(dO * O), produced while dO = dY Wo is written (then call spb_attention_bwd with
 * delta_ready = 1). */
int spb_gemm_bf16_rowdot(const void* A, const void* B, void* C, int M, int N, int K, int trans_a, int trans_b, int lda, int ldb, int ldc,
                         const float* bias, const uint8_t* rowmask, const float* alpha, const void* X, int ld_x, float* rowdot_out, int T,
                         int H, spb_stream_t stream);

/* LayerNorm / AdaptiveLayerNorm over the last dim (256, 512, 1280 or 1536); pass (w,b) or gb = [gamma | beta] bf16 [n, 2*dim].
 * Replaces nn.LayerNorm and modules/layers.py:31-47. */
int spb_layer_norm_fwd(const void* x, int x_fp32, int ldx, const float* w, const float* b, const void* gb, int ldgb, void* y, int y_fp32,
                       int ldy, float* mean, float* rstd, int n_rows, int dim, float eps, spb_stream_t stream);
/* dx (= LN backward, + dres if given); dw/db ACCUMULATED (affine) or dgb written (adaptive); optional dx16 = bf16 copy of dx with
 * rows where dx16_rowmask is false zeroed (the operand of the next backward GEMM). */
int spb_layer_norm_bwd(const void* dy, int lddy, const void* x, int x_fp32, int ldx, const float* mean, const float* rstd, const float* w,
                       const void* gb, int ldgb, const float* dres, int lddres, void* dx, int dx_fp32, int lddx, float* dw, float* db,
                       void* dgb, int lddgb, void* dx16, int lddx16, const uint8_t* dx16_rowmask, int n_rows, int dim,
                       spb_stream_t stream);

/* GLU(SiLU) + dropout: u bf16 [n, 2*hidden] -> h bf16 [n, hidden] (modules/transformer/feedforward.py:13-22,56-61). */
int spb_glu_fwd(const void* u, void* h, int n_rows, int hidden, float dropout_p, uint64_t seed, const uint64_t* rng_offset,
                spb_stream_t stream);
/* du bf16 [n, 2*hidden]; dbias fp32 [2*hidden] ACCUMULATED (may be NULL). */
int spb_glu_bwd(const void* dh, const void* u, void* du, float* dbias, int n_rows, int hidden, float dropout_p, uint64_t seed,
                const uint64_t* rng_offset, spb_stream_t stream);

/* One new position of B scores through a whole AdaLN decoder stack in ONE persistent kernel (cache path of
 * modules/transformer/transformer.py:161-186,219-221; attention.py:139-197; feedforward.py:13-64; layers.py:31-47): phases separated
 * by a grid barrier, weights streamed from L2 once per step, the KV cache appended and read in place.  ptrs = HOST array of device
 * pointers, 9 per layer: wqkv bf16 [384,256], wo bf16 [256,256], logslopes fp32 [4], w1 bf16 [2048,256], b1 fp32 [2048], w2 bf16
 * [256,1024], kv cache bf16 [B, cap, 128], wqkv^T bf16 [256,384], wo^T bf16 [256,256] (the per-row products stream the transposes).  w_ada / b_ada: (gamma-1 | beta) rows of the 2*depth+1 AdaLN linears.  pos_dev: device
 * int64 position.  Scratch: bf16 gb [B,(2*depth+1)*512], qkv [B,384], o [B,256], hmid [B,1024]; fp32 xres [B,256]; barrier uint32.
 * hid_out fp32 [depth, B, 256] (may be NULL) = inputs of the attention layers; out fp32 [B,256]; out_bf16 (may be NULL) its bf16 copy;
 * gb_all bf16 [B, T_all, (2*depth+1)*512] (may be NULL) = the AdaLN terms of all positions prepared ahead (read at *pos_dev + 1).
 * front (HOST array of 8 device pointers, may be NULL): x = LN(x1 Wf^T + p2) Wc^T + c2 replaces x_in (TupleTransformer.embed_inputs,
 * transformer.py:158-185, for the cached step): x1 bf16 [B,1536], Wf bf16 [256,1536], p2 fp32 [B,256], scratch fp32 [B,256],
 * LayerNorm weight / bias fp32 [256], Wc^T bf16 [256,256], c2 fp32 [B,256].
 * barrier_is_zero: the caller guarantees *barrier == 0 (spb_sample_fields' `advance` clears it at the end of a note-step), so no memset
 * node is enqueued.  dim 256, 4 heads x 64, hidden 1024. */
int spb_decode_stack_step(const float* x_in, const float* style, int S, const void* w_ada, const float* b_ada, const void* const* ptrs,
                          int depth, const uint8_t* key_mask, const long long* pos_dev, int B, int cap, void* gb, void* qkv, void* o,
                          void* hmid, float* xres, float* hid_out, float* out, void* out_bf16, unsigned* barrier, float eps,
                          const void* gb_all, int T_all, const void* const* front, int barrier_is_zero, spb_stream_t stream);
/* dst_k[b, :] = src_k[b, *pos_dev + shift_k, :] for n <= 8 row-major [B, T, row_bytes_k] arrays in one launch (host arrays of device
 * pointers / sizes / shifts; positions clamped to [0, T)): the inputs a note-step of the rendering loop (wrappers.py:409-431) reads at
 * its device-side position. */
int spb_gather_at_pos(const void* const* srcs, void* const* dsts, const int* row_bytes, const int* shifts, int n, const long long* pos_dev,
                      int B, int T, spb_stream_t stream);
/* Start of a streaming call of a render session that keeps staged weights across calls, one launch: hashes the bit patterns of
 * n_tensors tensors (table = DEVICE int64 [n_tensors, 3]: device address, number of 32-bit words, index of its first word) into
 *     fingerprint = sum over words i of splitmix64((i << 32) | word_i)  mod 2^64
 * (order-independent, so CTAs combine with integer atomics), then state[3] = (fingerprint != state[0]) and state[0] = fingerprint.
 * state: device uint64 [4]; state[1] and state[2] must be zero on entry and are zero again on return.  Also clears advance[0..1] (the
 * counter of spb_sample_fields and the grid-barrier word of spb_decode_stack_step) and sets *pos_dev = start. */
int spb_session_begin(const long long* table, int n_tensors, unsigned long long* state, unsigned* advance, long long* pos_dev,
                      long long start, spb_stream_t stream);

/* Tied heads of the rendered fields + sampling in one launch (modules/sampling.py:12-59, wrappers.py:358-397): per listed field
 * (host int arrays: field index, first table row, vocabulary <= 256, top-k <= 32; k = 1 is greedy) logits = e_f . table_f^T stay in
 * registers, tokens [0, n_banned) are never emitted, and the drawn token is written to tokens[b, *pos_dev + 1, field] (int64 [B,T,F]).
 * advance (uint32 [2], may be NULL; [0] must be zero): the last CTA to finish does *pos_dev += 1 and clears advance[0] and advance[1]
 * (= the grid-barrier word of spb_decode_stack_step when the two are laid out together), ending the note-step without further launches. */
int spb_sample_fields(const void* e, int ld_e, const void* table, const int* fields, const int* offsets, const int* vocab, const int* topk,
                      int n_fields, int n_banned, float temperature, uint64_t seed, const long long* pos_dev, long long* tokens, int B,
                      int T, int F, unsigned* advance, spb_stream_t stream);
/* spb_sample_fields with the other logit filters of modules/sampling.py and per-field bans (wrappers.py:358-397 filter_key_ids).  Per
 * listed field, host arrays (each may be NULL = off for every field): top_p[i] >= 0 samples from the nucleus of that threshold (0 keeps
 * the arg-max only; < 0 = off); top_a_ratio[i] > 0 keeps the tokens whose probability is at least max_prob^top_a_pow[i] * top_a_ratio[i]
 * (max_prob of the score's own row; <= 0 = off); a field with neither samples top-k with topk[i].  At most one filter per field, finite
 * parameters.  ban_bits[8 i .. 8 i + 7] is a 256-bit set of tokens field i never emits, applied together with [0, n_banned) before
 * the filter (at least one token must remain).  Both filters see the softmax at temperature 1; the kept tokens are drawn from at
 * `temperature`.  With every filter off the draws equal spb_sample_fields'. */
int spb_sample_fields_filtered(const void* e, int ld_e, const void* table, const int* fields, const int* offsets, const int* vocab,
                               const int* topk, int n_fields, int n_banned, float temperature, uint64_t seed, const long long* pos_dev,
                               long long* tokens, int B, int T, int F, unsigned* advance, const float* top_p, const float* top_a_pow,
                               const float* top_a_ratio, const uint32_t* ban_bits, spb_stream_t stream);

/* Device side of the collator (data/collators/performance.py:239-255 MixedLM mask_sequence, score_performance.py:186-234): expands a
 * packed batch -- uint16 tokens, int32 segment ids [3, n] (bars | beats | onsets), uint8 directions, int32 lengths -- into the int64
 * tensors and bool masks the model consumes, and derives masked tokens / labels from the performance tokens.  ignore_dims /
 * ignore_ids are bit sets (mask_ignore_token_dims / mask_ignore_token_ids, ids < 32).  Optional groups are NULL in and out. */
int spb_unpack_batch(const uint16_t* perf, const uint16_t* score, const int32_t* segs, const uint8_t* dirs, const int32_t* perf_len,
                     const int32_t* score_len, int64_t* o_perf, int64_t* o_masked, int64_t* o_labels, int64_t* o_score, int64_t* o_segs,
                     int64_t* o_dirs, uint8_t* o_perf_mask, uint8_t* o_score_mask, int B, int T, int Fp, int Fs, int Fd,
                     uint32_t ignore_dims, uint32_t ignore_ids, int mask_token, long long label_pad, int label_pad_ignored_dims,
                     spb_stream_t stream);

/* Fused feed-forward sub-layer forward: out = resid + W2 . dropout(value * silu(gate)), [value | gate] = xn W1^T + b1
 * (modules/transformer/feedforward.py:13-22,35-64 inside the pre-norm residual of transformer.py:139-232).  One tcgen05 kernel:
 * the [n, 2*hidden] pre-activation and the [n, hidden] activation stay in TMEM / shared memory.  xn bf16 [n, dim]; w1 bf16
 * [2*hidden, dim] (value rows, then gate rows); b1 fp32 [2*hidden]; w2 bf16 [dim, hidden]; resid fp32 or NULL; out fp32.
 * u_save (bf16 [n, 2*hidden]) / h_save (bf16 [n, hidden]) are optional side outputs for the backward (same dropout mask function
 * as spb_glu_fwd / spb_glu_bwd).  Built for dim 256, hidden 1024. */
int spb_ffn_fwd(const void* xn, int ld_xn, const void* w1, const float* b1, const void* w2, const float* resid, int ld_res, float* out,
                int ld_out, void* u_save, void* h_save, int n_rows, int dim, int hidden, float dropout_p, uint64_t seed,
                const uint64_t* rng_offset, spb_stream_t stream);

/* Fused feed-forward sub-layer backward, data path (the autograd of feedforward.py:13-22,35-64): dh = dy W2 stays on chip,
 * du = GLU'(u) . mask . dh is written once (du may be u itself: in place), dxn = du W1, db1 += column sums of du.  One tcgen05
 * kernel of CTA pairs.  dy bf16 [n, dim]; w2t bf16 [hidden, dim] = the out-projection weight TRANSPOSED (spb_transpose_bf16);
 * w1 bf16 [2*hidden, dim]; u bf16 [n, 2*hidden] as saved by spb_ffn_fwd; db1 fp32 [2*hidden] or NULL; dxn bf16 [n, ld_dxn].
 * The weight gradients (du^T xn, dy^T h) remain spb_gemm_bf16 calls.  Dropout arguments as given to spb_ffn_fwd. */
int spb_ffn_bwd(const void* dy, int ld_dy, const void* w2t, const void* w1, const void* u, void* du, float* db1, void* dxn, int ld_dxn,
                int n_rows, int dim, int hidden, float dropout_p, uint64_t seed, const uint64_t* rng_offset, spb_stream_t stream);
/* dst[z][c, r] = srcs[z][r, c] for n_mats (<= 16) contiguous bf16 matrices [rows, cols]; srcs is a HOST array of device pointers,
 * dst one buffer [n_mats, cols, rows] (all out-projection weights of a stack in one launch). */
int spb_transpose_bf16(const void* const* srcs, int n_mats, void* dst, int rows, int cols, spb_stream_t stream);

/* dst_i[0:n_i] += src_i[0:n_i] (fp32) for n_pairs tensors in one launch; dsts / srcs / sizes are HOST arrays.  Adds the slices of a
 * batched AdaLN weight-gradient GEMM into the gradients of the per-norm nn.Linear parameters (modules/layers.py:31-47). */
int spb_multi_add_f32(float* const* dsts, const float* const* srcs, const int* sizes, int n_pairs, spb_stream_t stream);

/* dst_i = src_i (nbytes_i bytes, device to device) for n_pairs buffers in one launch; host arrays of device pointers / sizes.  Feeds
 * the tensors of a collated batch (data/collators/score_performance.py:186-234) into the static inputs of the captured step. */
int spb_multi_copy(void* const* dsts, const void* const* srcs, const long long* nbytes, int n_pairs, spb_stream_t stream);

/* Computed per-field tables W_f = index rows {discrete ids} + MLP(token_values) (modules/transformer/embeddings.py:124-143,199-211),
 * all fields in one launch.  ptrs is a HOST array of device pointers, 7 per field for the forward (index_weight [V,128], token_values
 * [V], discrete mask [V] fp32 0/1, W0 [128], b0 [128], W1 [128,128], b1 [128]) and 12 per field for the backward (+ the five gradient
 * buffers d_index_weight, dW0, db0, dW1, db1, all ACCUMULATED into). */
int spb_table_build_fwd(const int* field_sizes, int n_fields, const void* const* ptrs, float* table, spb_stream_t stream);
int spb_table_build_bwd(const int* field_sizes, int n_fields, const void* const* ptrs, const float* dtable, spb_stream_t stream);

/* Fused SPMuple tuple-token embedding: out[n, F*128] = LayerNorm(cat_f table[off_f + tokens[n,f]]) in bf16.
 * table fp32 [sum V_f, 128] is the concatenation of the computed per-field tables (modules/transformer/embeddings.py:91-143).
 * Replaces models/scoreperformer/embeddings.py:121-143 (12 gathers + cat + LayerNorm). */
int spb_embed_ln_fwd(const int64_t* tokens, int ld_tok, const float* table, const int* field_sizes, int n_fields, const float* w,
                     const float* b, void* out, int ld_out, float* mean, float* rstd, int n_rows, float eps, spb_stream_t stream);
/* dtable / dw / db ACCUMULATED; c1, c2 fp32 [n] scratch.  PAD rows (token 0) receive no gradient (padding_idx=0). */
int spb_embed_ln_bwd(const void* dy, int ld_dy, const int64_t* tokens, int ld_tok, const float* table, const int* field_sizes,
                     int n_fields, const float* w, const float* mean, const float* rstd, float* c1, float* c2, float* dtable, float* dw,
                     float* db, int n_rows, spb_stream_t stream);

/* Fused MQA attention with learned-slope ALiBi, key padding, causal mask and dropout; qkv bf16 [B*T, ld] = q(H*64) | k(64) | v(64).
 * lse fp32 [B,H,T] is saved for the backward.  Replaces modules/transformer/attend.py:58-126 + attention.py:139-197. */
int spb_attention_fwd(const void* qkv, int ld, const uint8_t* key_mask, const float* logslopes, void* out, int ld_out, float* lse, int B,
                      int T, int H, int dim_head, int causal, float dropout_p, uint64_t seed, const uint64_t* rng_offset,
                      spb_stream_t stream);
/* tcgen05/TMEM/TMA implementation of the same forward (4 heads x dim 64): 32 positions x 4 heads form the 128-row MMA tile, the
 * softmax runs one row per thread out of TMEM.  mask_bits_scratch: uint32 [B, ceil(T/32)] (written when key_mask != NULL; the
 * tcgen05 backward reads it again).  edist (fp32 [B,H,T] or NULL): E_i[|i-j|] under the attention weights, the forward-side
 * statistic spb_attention_bwd_tc needs for the ALiBi slope gradient (modules/transformer/embeddings.py:318-325). */
int spb_attention_fwd_tc(const void* qkv, int ld, const uint8_t* key_mask, uint32_t* mask_bits_scratch, const float* logslopes, void* out,
                         int ld_out, float* lse, float* edist, int B, int T, int H, int dim_head, int causal, float dropout_p,
                         uint64_t seed, const uint64_t* rng_offset, spb_stream_t stream);
/* tcgen05/TMEM/TMA backward: dQ, dK, dV and d(logslope) in one kernel (a CTA owns 128 keys and walks the query tiles; the five
 * contractions S, dP, dV, dK, dQ are tcgen05.mma chains with TMEM accumulators; dQ leaves through TMA tensor reduce-adds).
 * mask_bits / edist: side outputs of spb_attention_fwd_tc (mask_bits NULL = no padding); delta fp32 [B,H,T] = rowsum(dO * O)
 * (spb_gemm_bf16_rowdot); dq_acc: fp32 [B*T, H*64] scratch that must be ZERO on entry and is zero again on return;
 * dqkv bf16 [B*T, ld_dqkv] receives dq | dk | dv; dlogslopes fp32 [H] ACCUMULATED.  Autograd of attend.py:58-126. */
int spb_attention_bwd_tc(const void* qkv, int ld, const uint32_t* mask_bits, const float* logslopes, const void* dout, int ld_do,
                         const float* lse, const float* delta, const float* edist, float* dq_acc, void* dqkv, int ld_dqkv,
                         float* dlogslopes, int B, int T, int H, int dim_head, int causal, float dropout_p, uint64_t seed,
                         const uint64_t* rng_offset, spb_stream_t stream);
/* dqkv bf16 [B*T, ld_dqkv] in the qkv column layout; delta fp32 [B,H,T] scratch; dlogslopes fp32 [H] ACCUMULATED. */
int spb_attention_bwd(const void* qkv, int ld, const uint8_t* key_mask, const float* logslopes, const void* out, const void* dout,
                      int ld_out, const float* lse, float* delta, void* dqkv, int ld_dqkv, float* dlogslopes, int B, int T, int H,
                      int dim_head, int causal, float dropout_p, uint64_t seed, const uint64_t* rng_offset, int delta_ready,
                      spb_stream_t stream);

/* KV-cached incremental decode (one new query per sequence): q bf16 [B, H*64]; kv cache bf16 rows of (k | v); the query sits at
 * position q_pos.  Replaces the cached path of attention.py:155-156 / transformer.py:161-186 without the per-step torch.cat.
 * pos_dev (optional): device int64 holding q_pos -- n_keys is then the cache capacity, which makes the launch replayable from a
 * CUDA graph; append_kv: first copy columns [H*64, H*64+128) of every q row (the new k | v) into cache row q_pos (nothing when a
 * device position is outside the cache; a host q_pos outside [0, n_keys) is rejected).  Returns -1 when the H * n_keys fp32 scores
 * exceed the device's shared memory per block. */
int spb_attention_decode(const void* q, int ld_q, void* kv, int ld_kv, long long kv_batch_stride, const uint8_t* key_mask,
                         int mask_stride, const float* logslopes, void* out, int ld_out, int B, int H, int dim_head, int n_keys,
                         int q_pos, const int64_t* pos_dev, int append_kv, spb_stream_t stream);

/* One level of the hierarchical MMD-VAE style encoder (models/scoreperformer/mmd_transformer.py:304-368):
 * segmented mean over cat(hidden*mask, style[:, :w_style]) -> Linear -> latents_mask -> broadcast back into style[:, col0:col0+z].
 * pooled fp32 [B*S,320] and counts int32 [B*S] must be zeroed; segments == NULL selects mode 'mean' (S == 2, slot 1). */
int spb_latent_level_fwd(const float* hidden, const float* style_in, int ld_style, const uint8_t* mask, const int64_t* segments,
                         const float* W, const float* bias, float* pooled, int* counts, float* latents, uint8_t* lmask, float* style_out,
                         int col0, int B, int T, int S, int d_hidden, int w_style, int z, spb_stream_t stream);
int spb_latent_level_bwd(float* d_style, int ld_style, int col0, const float* dlat_direct, const uint8_t* mask, const int64_t* segments,
                         const float* W, const float* pooled, const int* counts, const uint8_t* lmask, float* dlat, float* dpooled,
                         float* d_hidden, float* dW, float* dbias, int B, int T, int S, int d_hidden_dim, int w_style, int z,
                         spb_stream_t stream);

/* Fused pairwise-RBF MMD (mmd_transformer.py:505-534): loss and d loss / d y in one pass, no [n,n,d] tensor. */
int spb_mmd_fwd_bwd(const float* z_prior, const float* y, const uint8_t* w, int n_z, int n_y, int d, float* coef, float* loss,
                    float* grad_y, spb_stream_t stream);

/* Masked cross-entropy over one field's logits (models/scoreperformer/wrappers.py:49-59): loss_sum/count ACCUMULATED,
 * optional unscaled dlogits = softmax - onehot (bf16) and argmax. */
int spb_ce_rows(const float* logits, int ld, const int64_t* labels, int ld_lab, int V, long long ignore_index, float* loss_sum,
                float* count, void* dlogits, int ld_d, int* argmax_out, int n_rows, spb_stream_t stream);

/* Tied head of one tuple field fused with its cross-entropy (embeddings.py:345-353 + wrappers.py:49-59): the [n, V] logits
 * e_f . table_f^T stay in tensor memory; only loss_sum / count (ACCUMULATED), the optional bf16 gradient rows
 * dlogits = softmax - onehot (zero for ignored labels; columns [V, ld_d) zeroed) and the optional argmax leave the SM.
 * e bf16 [n, lde] (the field's 128 columns), table bf16 [V, ldt], V <= 256.
 * stats (fp32 [3], ACCUMULATED, may be NULL) = the ScorePerformerEvaluator's sums over the labelled rows
 * (models/scoreperformer/evaluator.py:38-46,72-104): #(argmax == label), sum |tv[argmax] - tv[label]|,
 * sum_v softmax_v |tv[label] - tv[v]|, with tv = token_values (fp32 [V]; NULL leaves the two distances at 0). */
int spb_head_ce(const void* e, int lde, const void* table, int ldt, int V, const int64_t* labels, int ld_lab, long long ignore_index,
                float* loss_sum, float* count, void* dlogits, int ld_d, int* argmax, const float* token_values, float* stats,
                int n_rows, spb_stream_t stream);

/* Optimiser step on the flat buffers (experiments/optimizers.py:151-169): clip_grad_norm_(max_norm) + AdamW + bf16 shadow
 * refresh in one pass.  grad_norm = device scalar ||g||_2 before grad_scale (null / max_norm <= 0: no clipping);
 * step = device int64 with the 1-based step number; lr_dev = optional device scalar overriding lr (schedules under graph replay). */
int spb_adamw_step(float* p, const float* g, float* m, float* v, void* shadow_bf16, int64_t n, const float* grad_norm, float grad_scale,
                   float max_norm, float lr, float beta1, float beta2, float eps, float weight_decay, const int64_t* step,
                   const float* lr_dev, spb_stream_t stream);

/* Direction-classifier heads (models/classifiers/model.py:74-82,202-216): Dropout -> Linear(in_dim, C_g) -> weighted CE. */
int spb_clf_heads(const float* x, int ldx, const uint8_t* rowmask, const int64_t* labels, int ld_lab, const float* W, const float* bias,
                  const float* class_w, const int* n_classes, int n_heads, float* num, float* den, const float* dlogit_scale, float* dW,
                  float* db, float* dl_scratch, int n_rows, int in_dim, float dropout_p, uint64_t seed, const uint64_t* rng_offset, int backward,
                  spb_stream_t stream);
int spb_clf_logits(const float* x, int ldx, const float* W, const float* bias, float* out, int n_rows, int in_dim, int total,
                   spb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SPB200_H */
