/* rbr_b200.h — C-ABI of the B200-native (sm_100a) review-encoder hot path.
 *
 * The reference (H263/review-based-recommender) has no FFI of its own: its hot path is the
 * PyTorch nn.Module code cited beside each entry point below (paths relative to the reference
 * root).  Each function replaces the library calls those lines make on the GPU.  The host side
 * (review-based-recommender_b200/*.py) binds this library with ctypes; INTEGRATION.md shows the
 * stub a reference maintainer would add.
 *
 * Conventions (SURVEY.md §8b):
 *   - plain pointers and int64 sizes only; every data pointer is a DEVICE pointer unless named host_*;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy default
 *     stream) and never synchronises the device, allocates or frees caller-visible memory;
 *   - scratch memory is passed in (`ws`, `ws_bytes`) and sized by the matching *_workspace_bytes();
 *   - return value: 0 = ok, negative = error (RBR_E*); rbr_last_error() gives a thread-local message;
 *   - `*_grad` outputs are ACCUMULATED INTO (+=): the caller zero-fills them once per step
 *     (this is what lets several launches and both document sides share one gradient buffer);
 *   - token / id tensors are int64 row-major exactly as torch.LongTensor lays them out; masks are
 *     1 byte per element (torch.bool); floats are fp32 row-major contiguous.
 *   - there is no CPU implementation behind any of these symbols.
 */
#ifndef RBR_B200_H_
#define RBR_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RBR_OK 0
#define RBR_EINVAL (-1)      /* bad argument (null pointer, unsupported shape)            */
#define RBR_ECUDA (-2)       /* a CUDA runtime call or kernel launch failed               */
#define RBR_EWORKSPACE (-3)  /* workspace too small                                       */
#define RBR_EUNSUPPORTED (-4)/* shape outside what the selected kernel variant supports   */

/* precision of the conv contraction */
#define RBR_PREC_FP32 0 /* fp32 CUDA-core implicit GEMM, matches the reference within 1e-5          */
#define RBR_PREC_BF16 1 /* bf16 operands on tcgen05 tensor cores, fp32 accumulate in TMEM (1e-2)    */

/* activation fused after the conv, before max-over-time */
#define RBR_ACT_RELU 0 /* NgramFeat: nn.ReLU  (models/deepconn/layers.py:108)                       */
#define RBR_ACT_TANH 1 /* D-ATT:     nn.Tanh  (models/dual_att/layers.py:39,69,73,77)               */

/* `flags` of the conv entry points (per call; the library keeps no process-wide switches) */
#define RBR_CONV_TC_SINGLE_CTA 1 /* bf16 forward: only the single-CTA cp.async tensor-core kernel (A/B timing, tests)        */
#define RBR_CONV_TC_PAIR_ONLY 2  /* bf16 forward: only the CTA-pair TMA kernel; RBR_EUNSUPPORTED when the shape is outside it */
#define RBR_CONV_BWD_DENSE_TC 4  /* backward: force the dense tensor-core formulation (short documents) where the shape allows;
                                    default = chosen by shape                                                                  */
#define RBR_CONV_BWD_SPARSE 8    /* backward: force the arg-max-sparse CUDA-core formulation                                   */
#define RBR_IDS_I32 16           /* `ids` points to int32 token ids (staged input pipeline, SURVEY §8f-3) instead of int64     */
#define RBR_IDS_U16 64           /* `ids` points to uint16 token ids (staged input pipeline when the vocabulary has <= 65536 rows) */
#define RBR_MASK_FROM_IDS 32     /* mask == NULL means mask = (ids != 0) — utils.py:30-42's get_mask — instead of "all true"   */

int rbr_version(void);
const char* rbr_last_error(void);
/* Number of out-of-range token/id values seen by any kernel since the last call (they are treated as
 * padding rows); synchronises `stream`.  The reference raises IndexError / a device assert instead. */
int rbr_consume_oob_count(void* stream);
/* Cumulative number of CUDA kernels this library has launched in this process (host-side counter,
 * incremented at every launch site); bench.py reports the delta over its timed region. */
int64_t rbr_launch_count(void);

/* ---- K1: embedding row gather -------------------------------------------------------------------
 * Replaces nn.Embedding forward: WordEmbedding.forward, models/deepconn/layers.py:22-24
 * (same code at models/narre/narre.py:22-24, models/dual_att/layers.py:21-23).
 * out[t, :] = table[ids[t], :], bit-exact.                                                          */
int rbr_gather_fwd(const float* table, int64_t vocab, int64_t emb, const int64_t* ids, int64_t n_tokens,
                   float* out, void* stream);

/* ---- K1b: dense embedding gradient (warp-segmented scatter-add) ----------------------------------
 * Replaces aten::embedding_dense_backward, i.e. the autograd backward of layers.py:23.
 * table_grad[ids[t], :] += grad_rows[t, :] for ids[t] != padding_idx (padding_idx < 0: no padding row). */
int64_t rbr_embgrad_workspace_bytes(int64_t n_tokens, int64_t vocab);
int rbr_embgrad_scatter_add(const int64_t* ids, const float* grad_rows, int64_t n_tokens, int64_t emb,
                            int64_t vocab, int64_t padding_idx, float* table_grad, void* ws, int64_t ws_bytes,
                            void* stream);

/* ---- K0: bf16 shadow of the embedding table and packed conv weights (operand staging for K2) -----
 * shadow[v, 0:emb_pad] = bf16(table[v, 0:emb]) zero-padded; emb_pad = rbr_emb_pad(emb).             */
int64_t rbr_emb_pad(int64_t emb);
int rbr_table_to_bf16(const float* table, int64_t vocab, int64_t emb, void* shadow_bf16, void* stream);
/* Packed conv weights: one opaque buffer holding (a) fp32 [k][E][Hpad] for the fp32 conv, (b) fp32
 * [H][k][E] for the backward, (c) bf16 K-major UMMA operand tiles for the tensor-core conv.
 * weight is nn.Conv1d's [H, E, k] (models/deepconn/layers.py:44).                                    */
int64_t rbr_conv_pack_bytes(int64_t emb, int64_t filters, int64_t ksize);
int rbr_conv_pack(const float* weight, int64_t emb, int64_t filters, int64_t ksize, void* packed, void* stream);

/* ---- K2: fused  mask → Conv1d(same padding) → activation → max-over-time --------------------------
 * Replaces NgramFeat.forward, models/deepconn/layers.py:123-136 (masked_tensor utils.py:58-60,
 * transpose, MyConv1d :54-58, nn.ReLU, nn.MaxPool1d(seq_len) :107-109) together with the embedding
 * gather that feeds it (deepconn.py:43-47): the [N,L,E] activations are never materialised.
 *   ids   [n_docs, doc_len] int64 token ids;  mask [n_docs, doc_len] bytes or NULL (NULL = all true)
 *   table fp32 [vocab, emb] (RBR_PREC_FP32) — shadow_bf16 from rbr_table_to_bf16 (RBR_PREC_BF16)
 *   pad   symmetric zero padding of the conv ((k-1)/2 for NgramFeat, 0 for D-ATT's global convs);
 *         the pooled window is all doc_len + 2*pad - k + 1 output positions, padded tokens included
 *   gate  optional fp32 multiplier applied to every (unmasked) token row before the conv:
 *         gate_mode 0 = none, 1 = per token [n_docs, doc_len], 2 = per doc [n_docs]  (D-ATT gates)
 *   feat  [n_docs, feat_ld] fp32, columns [0, filters) written;  argmax [n_docs, feat_ld] int32 with
 *         the FIRST position attaining the max (nn.MaxPool1d tie rule);  pool_raw (optional, same shape):
 *         the pooled value before bias and activation, gate included (gate * conv_nobias(x) at the arg-max;
 *         needed by the backward of a gated conv).
 *   ids   int64 (torch.LongTensor) or, with RBR_IDS_I32 / RBR_IDS_U16 in `flags`, int32 / uint16; RBR_MASK_FROM_IDS: see above.
 *   RBR_PREC_BF16 shapes outside both tensor-core kernels fall back to the fp32 kernel when `table` is given.
 *   ws / ws_bytes: optional scratch of rbr_conv_fwd_workspace_bytes(n_docs) bytes (NULL: none).  With it, short-document
 *   batches (NARRE pads every user / item to 10 reviews: all-padding "documents") are first scanned for documents without
 *   any unmasked token; those get act(bias) / arg-max 0 directly — exactly what the conv over their all-zero rows yields —
 *   and only the others are tiled onto the tensor cores.  Long-document batches (DeepCoNN) are scanned for each document's
 *   last unmasked token, and the 128-position tiles lying entirely in the padding tail are skipped (every position from
 *   len + pad on reads zero rows only and yields the bias again: neither the max nor its first position changes).                                */
int64_t rbr_conv_fwd_workspace_bytes(int64_t n_docs);
/* The same plus room for the row-index table of a (doc_len, ksize, pad) conv: with a scratch of at least this size the call
 * first resolves every staged position of every document to its word-table row (int32, -1 = reads as zeros: outside the document,
 * masked out, or an id outside the table) in one coalesced pass, and the tensor-core kernel bulk-copies each tile's 136
 * indices from that table instead of chasing ids and masks (HBM misses of several microseconds under its own gather traffic)
 * on its critical path.  Results are identical with either scratch size.                                                        */
int64_t rbr_conv_fwd_workspace_bytes2(int64_t n_docs, int64_t doc_len, int64_t ksize, int64_t pad);
/* Tiling plan of the CTA-pair kernel for a shape (host-only, launches nothing; used by the CPU tests of the tiling logic):
 * out[0..15] = {available, passes, filters/pass, filters/CTA, 64-wide K blocks, K steps, gather4 groups per stage, stage bytes,
 * ring stages, resident weight bytes per CTA, short-document mode, documents per tile, document row stride, tiles per document,
 * shared-memory bytes, TMEM columns}.                                                                                         */
int rbr_conv_tc2_plan(int64_t emb, int64_t filters, int64_t ksize, int64_t doc_len, int64_t pad, int64_t n_docs, int64_t* out);
int rbr_conv_act_maxpool_fwd(int precision, int activation, const void* table, const void* shadow_bf16,
                             int64_t vocab, int64_t emb, const void* ids, const uint8_t* mask,
                             const float* gate, int gate_mode, int64_t n_docs, int64_t doc_len,
                             const void* packed, const float* bias, int64_t filters, int64_t ksize,
                             int64_t pad, float* feat, int32_t* argmax, float* pool_raw, int64_t feat_ld,
                             void* ws, int64_t ws_bytes, int flags, void* stream);
/* Timing experiments only.  With RBR_TC2_DEBUG=4 in the environment the CTA-pair conv kernel accumulates per-CTA cycle
 * counters; this copies out[cta][12] = {MMA warp total, its wait for operands, its wait for a free accumulator, producer warp 0
 * total, its wait for a free ring slot, epilogue warp 0 total, its wait for a finished accumulator, tiles, epilogue warp 0's
 * TMEM loads + column max, its per-document finalisation, producer warp 0's per-tile prologue, 0} of the last launch (synchronises the device). */
int rbr_debug_conv_tc2_prof(int64_t* out, int n_ctas);

/* ---- K2b: arg-max-sparse backward of K2 ------------------------------------------------------------
 * Replaces aten::convolution_backward + max_pool1d backward + relu backward + masked_fill backward +
 * embedding_dense_backward (the autograd reverse of layers.py:123-136 and :23).  After max-over-time
 * only ONE position per (doc, filter) carries gradient, so
 *   weight_grad[h,:,j] += g[n,h] * x[n, t*+j-pad, :],  bias_grad[h] += g[n,h],
 *   table_grad[ids[n, t*+j-pad], :] += g[n,h] * W[h,:,j]            (mask true, id != padding_idx)
 * with g = feat_grad * act'(feat), t* = argmax[n,h].
 * The call may be split: weight_grad == bias_grad == NULL computes only the table (and gate) part, table_grad == NULL
 * (with gate_grad == NULL) only the weight/bias part — data-parallel training finishes the table gradients of all
 * document sides first so that their all-reduce overlaps the weight-gradient kernels (parallel.py).
 * gate / gate_grad: as in the forward; gate_grad (same shape as gate, +=) receives d loss / d gate =
 * sum_h g * conv_nobias(x) = sum_h g * pool_raw / gate (0 where the gate saturated to exactly 0: no cancellation, no
 * inf/NaN), which is why a gated backward also needs the forward's `pool_raw` (NULL when gate_mode == 0). */
int64_t rbr_conv_bwd_workspace_bytes(int64_t n_docs, int64_t filters, int64_t ksize, int64_t emb, int64_t vocab);
int rbr_conv_act_maxpool_bwd(int precision, int activation, const void* table, const void* shadow_bf16,
                             int64_t vocab, int64_t emb, const void* ids, const uint8_t* mask,
                             const float* gate, int gate_mode, int64_t n_docs, int64_t doc_len,
                             const void* packed, int64_t filters, int64_t ksize, int64_t pad,
                             const float* feat, const int32_t* argmax, const float* feat_grad,
                             const float* pool_raw, int64_t feat_ld,
                             int64_t padding_idx, float* weight_grad, float* bias_grad, float* table_grad,
                             float* gate_grad, void* ws, int64_t ws_bytes, int flags, void* stream);

/* ---- K2c: the same backward as two tensor-core GEMMs over a token x filter-tap coefficient matrix (bf16 precision) ------
 * Replaces the same autograd nodes as K2b (conv dgrad + wgrad, pool / relu / mask backward, embedding_dense_backward).
 * Every document side of a step accumulates C[v][h*k+j] += g[n,h] for the token id v that tap j of (n, h)'s arg-max window
 * reads (rbr_conv_bwd_cmat_scatter, one call per side; also bias_grad[h] += g[n,h] when bias_grad != NULL); then
 *   table_grad[v,:]   += sum_hj C[v][hj] * W[hj,:]      (the bf16-rounded conv weights of `packed`; row padding_idx skipped)
 *   weight_grad[h,:,j] += sum_v C[v][h*k+j] * x[v,:]    (x = shadow_bf16)
 * run as tcgen05 GEMMs (rbr_conv_bwd_cmat_finish; C is split into bf16 hi + lo halves, fp32 accumulation).
 * C is kept as rbr_conv_bwd_cmat_chunks() FILTER BLOCKS of at most ~80 MB, each small enough to stay mostly L2-resident while the atomics of
 * its (doc, filter) items land in it (an atomic that misses L2 costs a random DRAM read + write-back).  Per step and block c:
 *   rbr_conv_bwd_cmat_begin(c)            zero-fills the block (the write allocates it in L2 without a DRAM read)
 *   rbr_conv_bwd_cmat_scatter(side, c)    once per document side — the sides may run on different streams
 *   rbr_conv_bwd_cmat_finish(1, c)        splits the block into the bf16 hi|lo operand while it is still in L2
 * then rbr_conv_bwd_cmat_finish(2 / 4, -1) for the two gradients.  chunk = -1 means "every block" in all three calls.
 * Bit 2 computes table rows [row_lo, row_hi) (cut on multiples of 128; 0, 0 = all): data-parallel training produces the
 * gradient in row slices and starts the all-reduce of each slice while the next one is still being computed.
 * `ws`: rbr_conv_bwd_cmat_workspace_bytes() bytes that the CALLER ZERO-FILLS ONCE (the weight scratch is left zeroed again
 * by bit 4).
 * `what`: 1 = close the accumulation of block `chunk` (split C; required once per block after its scatters, before 2 / 4),
 * 2 = table gradient, 4 = weight gradient — data-parallel training runs 1|2, starts the table all-reduce, then 4; 8 (with 2) =
 * the table gradient is OVERWRITTEN (every row and column is written, the padding row with zeros) instead of accumulated
 * into: the caller then need not zero-fill table_grad, and the epilogue stores without reading (halves its HBM traffic).
 * Shapes: emb % 4 == 0, emb <= 448 (the weight GEMM's shared-memory ring outgrows 227 KB at rbr_emb_pad(emb) = 512),
 * filters <= 1024, ksize <= 8, round_up(filters*ksize, 64) <= 4096, vocab * round_up(filters*ksize, 64) * 4 bytes <= 3 GiB,
 * no gate (rbr_conv_bwd_cmat_supported; otherwise use K2b).                                                             */
int rbr_conv_bwd_cmat_supported(int64_t vocab, int64_t emb, int64_t filters, int64_t ksize);
int64_t rbr_conv_bwd_cmat_workspace_bytes(int64_t vocab, int64_t emb, int64_t filters, int64_t ksize);
int rbr_conv_bwd_cmat_chunks(int64_t vocab, int64_t emb, int64_t filters, int64_t ksize);
int rbr_conv_bwd_cmat_begin(int chunk, int64_t vocab, int64_t emb, int64_t filters, int64_t ksize, void* ws, int64_t ws_bytes,
                            void* stream);
int rbr_conv_bwd_cmat_scatter(const void* ids, const uint8_t* mask, int64_t n_docs, int64_t doc_len, int64_t vocab, int64_t emb,
                              int64_t filters, int64_t ksize, int64_t pad, int activation, const float* feat,
                              const int32_t* argmax, const float* feat_grad, int64_t feat_ld, float* bias_grad, int chunk,
                              void* ws, int64_t ws_bytes, int flags, void* stream);
int rbr_conv_bwd_cmat_finish(int what, int chunk, int64_t row_lo, int64_t row_hi, const void* shadow_bf16, const void* packed,
                             int64_t vocab, int64_t emb, int64_t filters, int64_t ksize, int64_t padding_idx, float* table_grad,
                             float* weight_grad, void* ws, int64_t ws_bytes, void* stream);

/* ---- K8: the alternate encoder arch="HierPooling" ---------------------------------------------------------------------
 * Replaces HierPooling.forward (models/deepconn/layers.py:81-98: F.avg_pool1d(kernel k, stride 1) over time, then F.max_pool1d
 * over the whole pooled length) applied to the masked, transposed embeddings (NgramFeat.forward, layers.py:131-133), together
 * with the embedding gather: pooled[n,e] = max_t mean_{j<k} x[n,t+j,e], argmax = the FIRST window start attaining it.  The
 * optional Linear(E → out) and the ReLU that follow stay library ops.  Backward: table_grad[ids[n,t*+j], e] += grad[n,e] / k
 * for the k rows of the arg-max window (mask true, id != padding_idx).  1 <= k <= 8.                                   */
int rbr_hier_pool_fwd(const float* table, int64_t vocab, int64_t emb, const void* ids, const uint8_t* mask, int64_t n_docs,
                      int64_t doc_len, int64_t ksize, float* pooled, int32_t* argmax, int flags, void* stream);
int rbr_hier_pool_bwd(const void* ids, const uint8_t* mask, int64_t n_docs, int64_t doc_len, int64_t vocab, int64_t emb,
                      int64_t ksize, int64_t padding_idx, const int32_t* argmax, const float* pooled_grad, float* table_grad,
                      int flags, void* stream);

/* ---- K9: SimpleSiamese's masked average pooling fused with the embedding gather ------------------------------------------
 * Replaces word_embedding → transpose → MaskedAvgPooling1d.forward (models/simple_siamese/layers.py:90-110, called at
 * simple_siamese.py:59-64): out[n,:] = sum_t mask[n,t] * table[ids[n,t],:] / (sum_t mask[n,t] + 1e-8).
 * Backward: table_grad[ids[n,t],:] += mask[n,t] * out_grad[n,:] / (len + 1e-8), padding row skipped.  emb % 4 == 0.     */
int rbr_masked_avg_pool_fwd(const float* table, int64_t vocab, int64_t emb, const void* ids, const uint8_t* mask, int64_t n_docs,
                            int64_t doc_len, float* out, int flags, void* stream);
int rbr_masked_avg_pool_bwd(const void* ids, const uint8_t* mask, int64_t n_docs, int64_t doc_len, int64_t vocab, int64_t emb,
                            int64_t padding_idx, const float* out_grad, float* table_grad, int flags, void* stream);

/* ---- K3: fused NARRE review-level attention --------------------------------------------------------
 * Replaces LinearAttention.forward, models/narre/narre.py:40-64 (dropout excluded: applied by the caller).
 *   feat [B,R,H], other_id [B,R] int64, W_rv [H,A], W_id [A,A], h [A], b_1 [A], b_2 [1], ebd_vals [n_ids, A]
 *   out [B,H], scores [B,R]                                                                           */
int rbr_narre_attn_fwd(const float* feat, const int64_t* other_id, int64_t batch, int64_t reviews, int64_t hidden,
                       int64_t att, const float* W_rv, const float* W_id, const float* h, const float* b_1,
                       const float* b_2, const float* ebd_vals, int64_t n_ids, float* out, float* scores,
                       void* stream);
/* out_grad [B,H], scores_grad [B,R] or NULL → feat_grad [B,R,H] (written), parameter grads (+=).      */
int rbr_narre_attn_bwd(const float* feat, const int64_t* other_id, int64_t batch, int64_t reviews, int64_t hidden,
                       int64_t att, const float* W_rv, const float* W_id, const float* h, const float* b_1,
                       const float* b_2, const float* ebd_vals, int64_t n_ids, int64_t padding_idx,
                       const float* scores, const float* out_grad, const float* scores_grad, float* feat_grad,
                       float* W_rv_grad, float* W_id_grad, float* h_grad, float* b_1_grad, float* b_2_grad,
                       float* ebd_vals_grad, void* stream);

/* ---- K3 on tensor cores: both attention sides in ONE launch (csrc/attn_tc.cu) ---------------------------------------------
 * Same function as rbr_narre_attn_fwd / _bwd for n_sides (1 or 2) independent LinearAttention modules at once — NARRE's
 * user_att and item_att (models/narre/narre.py:184-185) — given as arrays of n_sides pointers per argument.  A CTA owns a
 * tile of samples; feat@W_rv, e@W_id and the four backward contractions run as mma.sync TF32 in the 3xTF32 scheme (fp32-grade
 * accuracy).  Returns RBR_EUNSUPPORTED for shapes outside it (att > 32, hidden > 512, reviews > 64): use K3 then.       */
int rbr_narre_attn_pair_supported(int64_t reviews, int64_t hidden, int64_t att);
int rbr_narre_attn_pair_fwd(int n_sides, const float* const* feat, const int64_t* const* other_id, int64_t batch, int64_t reviews,
                            int64_t hidden, int64_t att, const float* const* W_rv, const float* const* W_id, const float* const* h,
                            const float* const* b_1, const float* const* b_2, const float* const* ebd_vals, const int64_t* n_ids,
                            float* const* out, float* const* scores, void* stream);
int rbr_narre_attn_pair_bwd(int n_sides, const float* const* feat, const int64_t* const* other_id, int64_t batch, int64_t reviews,
                            int64_t hidden, int64_t att, const float* const* W_rv, const float* const* W_id, const float* const* h,
                            const float* const* b_1, const float* const* b_2, const float* const* ebd_vals, const int64_t* n_ids,
                            const int64_t* padding_idx, const float* const* scores, const float* const* out_grad,
                            const float* const* scores_grad, float* const* feat_grad, float* const* W_rv_grad,
                            float* const* W_id_grad, float* const* h_grad, float* const* b_1_grad, float* const* b_2_grad,
                            float* const* ebd_vals_grad, void* stream);

/* ---- K4: fused LastFeat ×2 + FM head (+ MSE loss) --------------------------------------------------
 * Replaces LastFeat.forward (models/deepconn/layers.py:156-165) for the user and the item side,
 * FM.forward (layers.py:188-209) and nn.MSELoss (trainer/train_deepconn_pp.py:140,164).
 *   u_text/i_text [B,H]; u_id/i_id [B] int64; W [H,K], b [K], ebd [users|items, K]; fm_h [K];
 *   user_bias [users], item_bias [items]; g_bias [1].
 *   drop_p in [0,1): FM dropout (0 = eval); the keep-mask is a counter hash of (drop_seed, sample, k) —
 *   it cannot bit-match torch's Philox stream, parity tests run with drop_p = 0.  drop_seed_dev (optional DEVICE pointer) is
 *   added to drop_seed inside the kernel: a step counter living on the device, so that a CUDA-graph replay of the step draws
 *   a new mask every time (graphs.py); the backward must be given the same pair.
 *   pred [B];  u_lat/i_lat [B,K] saved for the backward.
 *   ratings may be NULL; otherwise loss_sum[0] += grad_scale * sum (pred-rating)^2 (the caller zero-fills it) and
 *   pred_grad[b] = 2*(pred-rating)*grad_scale  (grad_scale = 1/B for MSELoss 'mean': loss_sum is then the loss). */
int rbr_head_fwd(const float* u_text, const float* i_text, const int64_t* u_id, const int64_t* i_id, int64_t batch,
                 int64_t hidden, int64_t latent, const float* Wu, const float* bu, const float* ebd_u,
                 const float* Wi, const float* bi, const float* ebd_i, const float* fm_h, const float* user_bias,
                 const float* item_bias, const float* g_bias, int64_t users, int64_t items, float drop_p,
                 uint64_t drop_seed, const uint64_t* drop_seed_dev, float* pred, float* u_lat, float* i_lat,
                 const float* ratings, float grad_scale, float* loss_sum, float* pred_grad, void* stream);
/* pred_grad [B] → u_text_grad/i_text_grad [B,H] (written) and parameter grads (+=).  Each of the four id tables has its
 * own padding row (nn.Embedding(padding_idx=...) of LastFeat.ebd ×2, FM.user_bias, FM.item_bias; < 0: none), which gets
 * no gradient.
 * rbr_head_dropout_mask (test/debug aid): writes the keep-scale the kernels apply, keep[b,k] in {0, 1/(1-p)}, for the same
 * (drop_p, drop_seed, drop_seed_dev) triple.                                                            */
int rbr_head_dropout_mask(int64_t batch, int64_t latent, float drop_p, uint64_t drop_seed, const uint64_t* drop_seed_dev,
                          float* keep, void* stream);
int rbr_head_bwd(const float* u_text, const float* i_text, const int64_t* u_id, const int64_t* i_id, int64_t batch,
                 int64_t hidden, int64_t latent, const float* Wu, const float* Wi, const float* fm_h,
                 const float* u_lat, const float* i_lat, float drop_p, uint64_t drop_seed, const uint64_t* drop_seed_dev,
                 int64_t ebd_u_padding_idx, int64_t ebd_i_padding_idx, int64_t user_bias_padding_idx,
                 int64_t item_bias_padding_idx, int64_t users, int64_t items, const float* pred_grad, float* u_text_grad, float* i_text_grad, float* Wu_grad, float* bu_grad,
                 float* ebd_u_grad, float* Wi_grad, float* bi_grad, float* ebd_i_grad, float* fm_h_grad,
                 float* user_bias_grad, float* item_bias_grad, float* g_bias_grad, void* stream);

/* ---- K5: D-ATT gates -------------------------------------------------------------------------------
 * Replaces LocalAttention.attn = Conv1d(E,1,k=window,pad=(window-1)/2)+Sigmoid (models/dual_att/layers.py:34-36,49)
 * → gate_local [n_docs, doc_len], and GlobalAttention.attn = Conv1d(E,1,k=doc_len)+Sigmoid (layers.py:65-67,83)
 * → gate_global [n_docs] (one scalar per document), computed from the token ids and the fp32 table.  The gated
 * convolutions themselves are rbr_conv_act_maxpool_fwd with RBR_ACT_TANH and gate_mode 1 (local, k=1) / 2 (global).
 *   w_local [1,E,window], b_local [1], w_global [1,E,doc_len], b_global [1]  (nn.Conv1d layouts).
 * Backward: gate_*_grad are d loss / d gate (filled by rbr_conv_act_maxpool_bwd's gate_grad); produces the four
 * parameter gradients (+=) and the gates' contribution to the table gradient (+=, padding row skipped).
 * `flags`: RBR_IDS_I32 when `ids` are int32 (D-ATT has no masks).                                                   */
int64_t rbr_datt_gate_workspace_bytes(int64_t n_docs, int64_t doc_len, int64_t emb, int64_t window, int64_t vocab);
int rbr_datt_gate_fwd(const float* table, int64_t vocab, int64_t emb, const void* ids, int64_t n_docs,
                      int64_t doc_len, const float* w_local, const float* b_local, int64_t window,
                      const float* w_global, const float* b_global, float* gate_local, float* gate_global,
                      void* ws, int64_t ws_bytes, int flags, void* stream);
int rbr_datt_gate_bwd(const float* table, int64_t vocab, int64_t emb, const void* ids, int64_t n_docs,
                      int64_t doc_len, const float* w_local, int64_t window, const float* w_global,
                      const float* gate_local, const float* gate_global, const float* gate_local_grad,
                      const float* gate_global_grad, int64_t padding_idx, float* w_local_grad, float* b_local_grad,
                      float* w_global_grad, float* b_global_grad, float* table_grad, void* ws, int64_t ws_bytes,
                      int flags, void* stream);

/* ---- K7: fused global-norm clip + Adam over flat parameter / gradient buffers (SURVEY §8f-1) -----------------------------
 * Replaces nn.utils.clip_grad_norm_(model.parameters(), max_norm) + torch.optim.Adam.step()
 * (trainer/train_deepconn_pp.py:135,167-168).  params / grads / exp_avg / exp_avg_sq: flat fp32 buffers of n_floats elements
 * with the same layout (every parameter a 256-byte aligned slot; gaps hold zeros and stay zero).
 *   clip = min(1, max_norm / (||grads||_2 + 1e-6))  (max_norm <= 0: no clipping);  sumsq_dev: 1 double of device scratch
 *   Adam (no amsgrad, no weight decay) with bias corrections from the DEVICE step counter step_dev[0], which the call
 *   increments first — a CUDA-graph replay of the trainer step therefore advances the optimizer correctly.
 *   grad_norm_out (optional, device): the unclipped gradient norm clip_grad_norm_ returns.
 *   shadow_bf16 (optional): the bf16 shadow of the word table (rows of rbr_emb_pad(emb) elements), rewritten from the updated
 *   parameters of the slice [table_off, table_off + table_rows*emb) — the next forward needs no rbr_table_to_bf16.        */
int rbr_clip_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n_floats, float lr,
                       float beta1, float beta2, float eps, float max_norm, double* sumsq_dev, int64_t* step_dev,
                       float* grad_norm_out, int64_t table_off, int64_t table_rows, int64_t emb, void* shadow_bf16,
                       void* stream);

/* ---- K6: data-parallel gradient all-reduce through the NVSwitch (NVLS multimem) ------------------------------
 * Replaces nn.DataParallel's gradient reduce_add (trainer/train_deepconn_pp.py:129-131) for one-process-per-GPU training:
 * `multicast_ptr` is the NVLS multicast address of the flat gradient arena (symmetric memory, same offset on every GPU).
 * Each rank calls this on its own stream; it reduces elements [rank, rank+1) * n/world across ALL GPUs inside the switch
 * (multimem.ld_reduce, fp32 add), multiplies by `scale` (1/world for the mean) and broadcasts the result to every GPU
 * (multimem.st).  The caller issues a cross-GPU barrier on the stream before (all gradients written) and after (all
 * slices broadcast) the call.
 * max_ctas <= 0 selects the default grid (32 CTAs: link-bound from 16 up, leaves the SMs to concurrent kernels).           */
int rbr_multimem_allreduce_f32(void* multicast_ptr, int64_t n_floats, int rank, int world, float scale, int max_ctas,
                               void* stream);
/* The same exchange with plain peer loads / stores instead of the switch reduction: `peer_ptrs` is a HOST array of `world`
 * device addresses (rank order; every GPU's copy of the arena, peer-mapped — torch symmetric memory's buffer_ptrs), the range
 * [offset_floats, offset_floats + n_floats) is reduced.  Each rank sums ITS 1/world slice over all copies in rank order, scales
 * and writes the result into every copy: (world-1)/world * N link bytes per GPU and direction instead of ~(1 + 1/world) * N.
 * Same barrier contract as above.  world in {2, 4, 8}; max_ctas <= 0: 64 CTAs.                                                  */
int rbr_p2p_allreduce_f32(const void* peer_ptrs, int64_t offset_floats, int64_t n_floats, int rank, int world, float scale,
                          int max_ctas, void* stream);

/* ---- K10: per-row top-k of a factorised score matrix (full-catalogue recommendation) --------------------------------
 * score[r, i] = sum_c A[r, c] * B[i, c] + row_bias[r] + col_bias[i]  (A [n_rows, dim], B [n_items, dim] fp32 row-major;
 * row_bias [n_rows] / col_bias [n_items], either may be NULL = 0).  For each row, the k eligible items with the largest
 * score, ordered by score descending then item id ascending, go to out_scores / out_items [n_rows, k]; the n_rows x n_items
 * scores are never materialised.  Eligible: every i < n_items not listed in excl_idx[excl_ptr[r] : excl_ptr[r+1]]
 * (CSR, each row's list sorted ascending without duplicates; both NULL = nothing excluded).  With fewer than k eligible
 * items the remaining slots hold item -1, score -inf.  A NaN score is never returned (scores enter by strict '>').
 * fp32-grade: each returned score is within ~1e-6 of |score|-scale of the exact dot product (3-piece bf16 split of both
 * operands, six tcgen05 products).  The FM head is such a product: relu(u*i) = relu(u)*relu(i) + relu(-u)*relu(-i).
 * Limits: 1 <= k <= 256, 1 <= dim <= 512, 1 <= n_items < 2^31; else RBR_EUNSUPPORTED.  The two queries are host-only and
 * launch nothing; rbr_factor_topk_slices gives the number of item slices the call splits each row's scan into (one CTA
 * per 128 rows and slice; a second kernel merges the slices' sorted lists, a copy when there is one slice).            */
int64_t rbr_factor_topk_workspace_bytes(int64_t n_rows, int64_t n_items, int64_t dim, int64_t k);
int64_t rbr_factor_topk_slices(int64_t n_rows, int64_t n_items, int64_t dim, int64_t k);
int rbr_factor_topk(const float* A, const float* row_bias, int64_t n_rows, const float* B, const float* col_bias,
                    int64_t n_items, int64_t dim, const int64_t* excl_ptr, const int64_t* excl_idx, int64_t k,
                    float* out_scores, int64_t* out_items, void* ws, int64_t ws_bytes, void* stream);

/* ---- K11: exact full-catalogue rank of target items under a factorised score matrix ----------------------------------
 * The score is K10's, from the same split operands, tcgen05 shape, K-step order, bias order and key (score descending,
 * then item id ascending), so the results are bit-consistent with rbr_factor_topk on the same inputs.  Row r's targets are
 * tgt_idx[tgt_ptr[r] : tgt_ptr[r+1]] (CSR, each row sorted ascending without duplicates, ids in [0, n_items), disjoint from
 * the row's exclusions; n_targets = tgt_ptr[n_rows]; at most max_targets per row — a caller with longer rows splits them
 * into several rows with the same A row, row bias and exclusions).  Exclusions as in rbr_factor_topk.  For each target t:
 *   out_ranks[p]  = #{ eligible i : key(r, i) >= key(r, t) }, i.e. the 1-based position of t in rbr_factor_topk's output
 *                   for k = infinity (other targets of the row are ordinary competitors; NaN and -inf scores never count);
 *                   -1 when t's own score is NaN or -inf;
 *   out_scores[p] = t's score, bit-identical to the score rbr_factor_topk returns for (r, t).
 * Item slices as in K10; per-slice counts are integers, so the result does not depend on the slice count.
 * Limits: 1 <= dim <= 512, 1 <= n_items < 2^31, 1 <= max_targets <= 64; else RBR_EUNSUPPORTED.  The workspace query is
 * host-only and launches nothing; the call never synchronises.                                                       */
int64_t rbr_factor_rank_workspace_bytes(int64_t n_rows, int64_t n_items, int64_t dim, int64_t n_targets, int64_t max_targets);
int rbr_factor_rank(const float* A, const float* row_bias, int64_t n_rows, const float* B, const float* col_bias,
                    int64_t n_items, int64_t dim, const int64_t* excl_ptr, const int64_t* excl_idx, const int64_t* tgt_ptr,
                    const int64_t* tgt_idx, int64_t n_targets, int64_t max_targets, int64_t* out_ranks, float* out_scores,
                    void* ws, int64_t ws_bytes, void* stream);

/* ---- K12: token attributions of a predicted rating from the per-entity feature cache ---------------------------------
 * After max-over-time (NgramFeat.forward, models/deepconn/layers.py:123-136; MyConv1d :54-58 with nn.Conv1d's [H, E, k]
 * weights, :44) feature (n, h) depends on the one window starting at t*[n,h] - pad, t* = the forward's first arg-max.
 *
 * rbr_conv_window_contrib: the tap contributions of that window,
 *   contrib[n * contrib_ld + h*ksize + j] = sum_e W[h,e,j] * x[n, argmax[n * argmax_ld + h] + j - pad, e]
 * in fp32 from the fp32 `table` and the fp32 [H][k][E] copy of W inside `packed` (rbr_conv_pack), whatever precision the
 * forward ran in.  x rows read as zeros exactly where the forward's do: outside the document, where the mask is false (mask
 * NULL: all true, or ids != 0 with RBR_MASK_FROM_IDS) and for ids outside [0, vocab).  `ids` as in K2 (RBR_IDS_I32 /
 * RBR_IDS_U16).  Several convs share one [n_docs, sum_c H_c * k_c] output through pointer offsets (argmax + first filter
 * column, contrib + first tap column) and the leading dimensions.  One table-row read per (n, h, j).
 *
 * rbr_explain_attrib: for n_rows (pair, side) rows — row p covers the docs_per_entity consecutive cached documents starting at
 * ent_row[p] (DeepCoNN 1, NARRE R reviews), each doc_len tokens — with g [n_rows, docs_per_entity, Htot] = d pred / d feat:
 *   attr[r, t] = sum_{h : feat > 0} sum_{j : t*[r,h] + j - pad = t} g[r,h] * contrib[r,h,j]    (gradient x input on x)
 * over the n_conv convs given by host_convs = {filters, ksize, pad} per conv (their filter columns are consecutive in
 * feat / argmax / g, Htot = sum of filters; their taps consecutive in contrib).  Writes
 *   text_total [n_rows]           sum_{h : feat > 0} g * sum_j contrib (= the sum of the map);
 *   top_pos / top_attr [n_rows, m]    the m windows of `width` consecutive positions with the largest summed attribution,
 *                                     greedily without overlap, ties to the lower start, never across a document boundary;
 *   bottom_pos / bottom_attr          the same for the smallest sums; positions are flat (r * doc_len + t), slots without a
 *                                     window left hold -1 / NaN;
 *   map [n_rows, docs_per_entity * doc_len] (optional: NULL = not written), review_attr [n_rows, docs_per_entity] (optional).
 * The map is built on chip with fixed-point integer atomics: results are bit-identical between calls and independent of the
 * batch and the row order.  A row whose ent_row lies outside [0, n_docs - docs_per_entity] gets NaN / -1.
 * Limits (rbr_explain_supported, host-only): 1 <= docs_per_entity * doc_len <= 16384, 1 <= m <= 32, 1 <= width <= 16,
 * 1 <= n_conv <= 8; otherwise rbr_explain_attrib returns RBR_EUNSUPPORTED.                                              */
int rbr_explain_supported(int64_t positions, int64_t m, int64_t width, int64_t n_conv);
int rbr_conv_window_contrib(const float* table, int64_t vocab, int64_t emb, const void* ids, const uint8_t* mask,
                            int64_t n_docs, int64_t doc_len, const void* packed, int64_t filters, int64_t ksize, int64_t pad,
                            const int32_t* argmax, int64_t argmax_ld, float* contrib, int64_t contrib_ld, int flags,
                            void* stream);
int rbr_explain_attrib(const int64_t* ent_row, int64_t n_rows, int64_t docs_per_entity, int64_t doc_len, const float* g,
                       const float* feat, const int32_t* argmax, int64_t feat_ld, const float* contrib, int64_t contrib_ld,
                       int64_t n_docs, int64_t n_conv, const int64_t* host_convs, int64_t m, int64_t width, float* text_total,
                       int64_t* top_pos, float* top_attr, int64_t* bottom_pos, float* bottom_attr, float* map,
                       float* review_attr, void* stream);
/* rbr_explain_attrib_ex: rbr_explain_attrib (which is this call with dense_coef = dense_vec = NULL) with
 *   feat NULL (in either call): every filter counts (no liveness predicate: D-ATT's tanh features);
 *   a dense term (dense_coef non-NULL): for document r of the row (cached document ent_row[p] + r),
 *     attr[r, t] += (sum_h g[r, h] * dense_coef[doc * dense_coef_ld + h]) * dense_vec[doc * dense_vec_ld + t]
 *   where the scalar is reduced in float64 in a fixed order; each product enters the map (and the total) as one more
 *   fixed-point term, and the scale bound counts it, so results stay bit-identical across calls, batches and row orders.
 * Limits as above; with a dense term also docs_per_entity * 8 bytes more shared memory (RBR_EUNSUPPORTED past 227 KB).     */
int rbr_explain_attrib_ex(const int64_t* ent_row, int64_t n_rows, int64_t docs_per_entity, int64_t doc_len, const float* g,
                          const float* feat, const int32_t* argmax, int64_t feat_ld, const float* contrib, int64_t contrib_ld,
                          int64_t n_docs, int64_t n_conv, const int64_t* host_convs, const float* dense_coef,
                          int64_t dense_coef_ld, const float* dense_vec, int64_t dense_vec_ld, int64_t m, int64_t width,
                          float* text_total, int64_t* top_pos, float* top_attr, int64_t* bottom_pos, float* bottom_attr,
                          float* map, float* review_attr, void* stream);

/* ---- K12 for D-ATT: gradient x input through both attention gates and the FC stack ----------------------------------------
 * D-ATT (models/dual_att/layers.py:25-89, dual_att.py:31-61): per side, gl = sigmoid(local gate conv, k = window, pad
 * (window-1)/2) per token, gg = sigmoid(global gate conv, k = doc_len) per document; features f = max_t tanh(conv(gate * x))
 * of a k = 1 conv on gl * x (l_out filters) and k = 2, 3, 4 convs on gg * x (g_out filters each, no padding), at the
 * forward's first arg-max t*.  x = the table row of each token (zero for ids outside the table; no masks).  With
 * d = 1 - f^2 and g = d pred / d f, gradient x input on x is the sum of
 *   local filter h:  g d gl[t*] (W_h . x[t*]) at t*, and g d (W_h . x[t*]) gl(1-gl)[t*] (w_l[:, j] . x[t* + j - pad]) at
 *                    t* + j - pad (the gate's taps);
 *   global filter h: g d gg (W_h[:, j] . x[t* + j]) at t* + j, and g d (sum_j W_h[:, j] . x[t* + j]) gg(1-gg) (w_g[:, s] . x[s])
 *                    at every position s.
 * Everything but g depends on the entity alone.
 *
 * rbr_datt_explain_contrib: those per-entity terms of n_docs documents, in fp32 from the fp32 table and the fp32 weight
 * copies inside `packed_*` (rbr_conv_pack of the four conv weights: local [l_out, E, 1], global [g_out, E, 2 / 3 / 4]),
 * whatever precision the forward ran in:
 *   contrib [n_docs, contrib_ld >= l_out * window + g_out * 9]: the local filters as one width-`window` conv with pad
 *     (window-1)/2 (column h * window + j; the direct term is folded into the centre tap), then the three global convs as
 *     pad-0 convs (columns h * k + j) — rbr_explain_attrib's layout for convs {l_out, window, (window-1)/2}, {g_out, 2, 0},
 *     {g_out, 3, 0}, {g_out, 4, 0};
 *   gate_coef [n_docs, coef_ld >= l_out + 3 g_out]: d * sum_j c_j on the global filters, 0 on the local ones;
 *   gate_vec [n_docs, vec_ld >= doc_len]: gg(1-gg) (w_g[:, s] . x[s]).
 * w_local_t [window][emb] and w_global_t [doc_len][emb] are the gate weights transposed (nn.Conv1d's [1, E, k] → [k, E]).
 * gate_local [n_docs, doc_len], gate_global [n_docs], feat / argmax [n_docs, feat_ld] (filter columns local, conv k=2, 3, 4)
 * are the forward's (rbr_datt_gate_fwd, rbr_conv_act_maxpool_fwd).  `flags`: RBR_IDS_I32 for int32 ids.
 * Limits: window odd and <= 16, doc_len >= 4; else RBR_EUNSUPPORTED before any launch.
 * The per-pair map is then rbr_explain_attrib_ex with feat NULL, g, this contrib and the dense term (gate_coef, gate_vec).
 *
 * rbr_datt_fc_grads: g for n_pairs pairs (u_ids[p], i_ids[p]) and both sides:
 *   g_user[p] = W0^T (user_mask[u] * W3^T item_out[i]),  g_item[p] = W0^T (item_mask[i] * W3^T user_out[u])
 * with user_out / item_out [n_users / n_items, out_dim] the cached FC outputs, user_mask / item_mask [*, hidden] (uint8 / bool)
 * the cached hidden ReLU masks 1[z > 0], w0 = fc.0.weight [hidden, in_dim], w3 = fc.3.weight [out_dim, hidden]; outputs
 * [n_pairs, in_dim].  Tensor cores at fp32 grade (3xTF32 mma.sync); every element is reduced in a fixed order, so results are
 * bit-identical whatever the batch, the chunking or the pair order.  Ids outside the tables give zero rows.
 * Limits: 1 <= hidden <= 768; else RBR_EUNSUPPORTED before any launch.                                                      */
int rbr_datt_explain_contrib(const float* table, int64_t vocab, int64_t emb, const void* ids, int64_t n_docs, int64_t doc_len,
                             const float* w_local_t, int64_t window, const float* w_global_t, const void* packed_local,
                             int64_t l_out, const void* packed_g2, const void* packed_g3, const void* packed_g4, int64_t g_out,
                             const float* gate_local, const float* gate_global, const float* feat, const int32_t* argmax,
                             int64_t feat_ld, float* contrib, int64_t contrib_ld, float* gate_coef, int64_t coef_ld,
                             float* gate_vec, int64_t vec_ld, int flags, void* stream);
int rbr_datt_fc_grads(const int64_t* u_ids, const int64_t* i_ids, int64_t n_pairs, const float* user_out, int64_t n_users,
                      const float* item_out, int64_t n_items, int64_t out_dim, const uint8_t* user_mask,
                      const uint8_t* item_mask, int64_t hidden, const float* w0, int64_t in_dim, const float* w3,
                      float* g_user, float* g_item, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RBR_B200_H_ */
