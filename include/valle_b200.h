/*
 * valle_b200.h -- C ABI of libvalle_b200.so: the sm_100a (B200) VALL-E decoding engine.
 *
 * Drop-in boundary (SURVEY.md section 8b).  Every entry point takes raw device pointers,
 * explicit sizes and a cudaStream_t (passed as void*); there are no torch / C++ types in any
 * signature and no C++ exception crosses the ABI.  Return value: 0 = ok, non-zero = error
 * code (message through vb_last_error(), thread-local).  OWNERSHIP: every buffer (weights,
 * KV cache, workspaces, outputs) is allocated and freed by the caller (PyTorch on the Python
 * side); the library allocates no persistent device memory and keeps no pointer past a call,
 * except inside the explicit opaque `vb_decoder_t` handle (created / destroyed in pairs),
 * which only stores the caller's pointers.
 *
 * Each function cites the reference interface (lifeiteng/vall-e, file:line under
 * /root/reference) whose arithmetic it replaces.  Host-side callers mirror the reference's
 * Python classes (valle_b200/modules, valle_b200/models); INTEGRATION.md shows the ctypes
 * stub a reference maintainer would add.
 */
#ifndef VALLE_B200_H_
#define VALLE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VB_ABI_VERSION 5

enum vb_status { VB_OK = 0, VB_ERR_ARG = 1, VB_ERR_CUDA = 2, VB_ERR_UNSUPPORTED = 3 };
/* storage type of the big matrices / activations.  Accumulation is always fp32. */
enum vb_dtype { VB_F32 = 0, VB_BF16 = 1 };
enum vb_epilogue { VB_EPI_NONE = 0, VB_EPI_RELU = 1, VB_EPI_RESIDUAL = 2 };
/* attention visibility rule */
enum vb_mask_mode {
  VB_MASK_FULL = 0,    /* NAR: every row of a sequence sees the whole sequence (valle.py:1125-1127) */
  VB_MASK_VALLE_AR = 1, /* AR inference: text rows see all text, audio rows see text + causal audio
                           (valle.py:1010-1033): kv_len(i) = max(S, i + 1) */
  /* padded training batches (valle.py:804-861,908-925): every sequence is [text padded to
     seg1_start | audio padded]; valid keys are text [0, text_lens[b]) and audio
     [seg1_start, seg1_start + seg1_lens[b]). */
  VB_MASK_PADDED_AR = 2, /* + text rows see text only, audio rows causal (the merged
                            attn_mask | key_padding_mask of valle.py:835-861) */
  VB_MASK_PADDED = 3,    /* key padding only (NAR training, valle.py:921-925) */
  VB_MASK_DENSE = 4      /* vb_attention only: an arbitrary boolean attn_mask [L, L] shared by all sequences and
                            heads, non-zero byte = blocked (the tensor form of activation.py:199-431 `attn_mask`);
                            exact-order CUDA-core kernel */
};

typedef void *vb_stream_t; /* cudaStream_t */

int vb_abi_version(void);
const char *vb_last_error(void);
/* number of kernels this library has launched in the calling process (bench.py gpu_launches) */
int64_t vb_launch_count(void);
/* Tuning / A-B switch `name` (the VB_* knobs listed in INTEGRATION.md) for this process; takes precedence over the
 * environment variable of the same name.  Values are read when kernels are launched (or captured). */
int vb_tune_set(const char *name, int value);
/* Profiling builds only (libvalle_b200_trace.so, compiled with -DVB_TRACE): bind a device ring
 * buf[cap] / counter; the kernels of the AR decode step then append (globaltimer_ns << 8 | id) stamps
 * (tools/trace_ar_step.py).  The product library returns VB_ERR_UNSUPPORTED. */
int vb_trace_bind(unsigned long long *buf, unsigned int *counter, unsigned int cap);

/* ------------------------------------------------------------------------------------------
 * a10  TokenEmbedding (valle/modules/embedding.py:21-47) and the 8-codebook sum composed by the
 *      caller (valle/models/valle.py:1064,1110-1113,1134).
 *   out[r,:] (=|+=) sum_{j<n_tables} tables[j][ tokens[r*tok_row_stride + j*tok_tab_stride] , :]
 *   summed in table order j = 0..n_tables-1 (same association order as the reference).
 *   tables: HOST array of n_tables device pointers to fp32 [vocab_j, d].
 *   table_rows: NULL or HOST array of the n_tables vocabulary sizes.  nn.Embedding raises IndexError for
 *   an id outside [0, vocab_j) (embedding.py:46); with table_rows given such an id is clamped (no
 *   out-of-bounds read) and *err_flag (device int32, may be NULL) is OR-ed with 1 for the host to report.
 *   out_rows: NULL or device int32 [n_rows] destination row of each input row (ragged packing).
 *   accumulate = 0: out = sum ; 1: out += sum
 * ---------------------------------------------------------------------------------------- */
int vb_embed_sum(const int64_t *tokens, int64_t tok_row_stride, int64_t tok_tab_stride,
                 const float *const *tables, const int32_t *table_rows, int n_tables, int64_t n_rows, int d,
                 float *out, int64_t out_row_stride, const int32_t *out_rows, int accumulate,
                 int32_t *err_flag, vb_stream_t stream);

/* a11  SinePositionalEmbedding.forward (embedding.py:93-97, scale=False):
 *   out[orow(r),:] = in[r,:] + alpha[0] * pe[pos(r), :], pos(r) = positions ? positions[r] : pos0 + r,
 *   orow(r) = out_rows ? out_rows[r] : r   (pe = fp32 table built on the CPU,
 *   embedding.py:75-91; product and sum rounded separately as the reference does). */
int vb_add_pe(const float *in, int64_t in_row_stride, const float *pe, int64_t pos0,
              const int32_t *positions, const float *alpha, int64_t n_rows, int d, float *out,
              int64_t out_row_stride, const int32_t *out_rows, vb_stream_t stream);

/* a8 / a9  LayerNorm.forward (transformer.py:57-74) and AdaptiveLayerNorm.forward
 *   (transformer.py:93-108).  y = LN(x; gamma, beta, eps); if ada_wb != NULL:
 *   y = ada_wb[0:d] * y + ada_wb[d:2d]  (weight | bias split order of transformer.py:96-101).
 *   rows: optional gather list (device int32 [n_rows]) of source rows, NULL = identity.
 *   out_dtype VB_F32 / VB_BF16. */
int vb_layernorm(const float *x, int64_t x_row_stride, const int32_t *rows, int64_t n_rows, int d,
                 const float *gamma, const float *beta, const float *ada_wb, float eps, void *out,
                 int out_dtype, vb_stream_t stream);

/* AdaptiveLayerNorm.project_layer for one stage embedding (transformer.py:96-100):
 *   out[2d] = W[2d,d] * emb[d] + b[2d]   (fp32) */
int vb_adaln_project(const float *W, const float *b, const float *emb, int d, float *out,
                     vb_stream_t stream);

/* a6/a7/a12  F.linear with fused epilogue (QKV in-proj, out-proj, FFN linear1/linear2,
 *   predict layers; transformer.py:332-334, activation.py:408, valle.py:1039,1128):
 *   C[M,N] = epi( A[M,K] * W[N,K]^T + bias[N] )
 *   VB_EPI_NONE / VB_EPI_RELU: C has dtype c_dtype.  VB_EPI_RESIDUAL: C is fp32 and is
 *   accumulated in place (C += ...), i.e. the residual add of transformer.py:297-302.
 *   a_dtype must equal w_dtype.  bf16 operands use the tcgen05/TMEM kernel when M is large,
 *   fp32 operands the exact-order SIMT kernel. */
int vb_linear(const void *A, int a_dtype, int64_t lda, const void *W, int w_dtype, const float *bias,
              void *C, int c_dtype, int64_t ldc, int64_t M, int N, int K, int epilogue,
              void *workspace, size_t workspace_bytes, vb_stream_t stream);

/* a7  scaled-dot-product attention of F.multi_head_attention_forward over packed, ragged
 *   sequences.  qkv: [M, 3d] (Q|K|V column blocks, head h = columns [h*hd,(h+1)*hd) of each
 *   block), cu_seqlens: device int32 [B+1] row offsets, text_lens: device int32 [B] (only for
 *   VB_MASK_VALLE_AR).  out: [M, d].  If kcache != NULL the K and V rows are also written to
 *   the caches ([B, H, cache_cap, hd], dtype = dtype) at their sequence position.
 *   dense_mask: device uint8 [>= max_seqlen rows, dense_ld] for VB_MASK_DENSE (NULL otherwise). */
int vb_attention(const void *qkv, int dtype, int64_t M, int B, int n_head, int head_dim,
                 const int32_t *cu_seqlens, const int32_t *text_lens, const int32_t *seg1_lens, int seg1_start,
                 int max_seqlen, int mask_mode, void *out, void *kcache, void *vcache,
                 int64_t cache_seq_stride, int cache_cap, const uint8_t *dense_mask, int64_t dense_ld,
                 vb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Decoder stack handle (transformer.py:337-406 TransformerEncoder of pre-LN
 * TransformerEncoderLayer, transformer.py:178-334).  Stores the caller's pointers only.
 * ---------------------------------------------------------------------------------------- */
typedef struct vb_layer_params {
  const void *in_proj_w;   /* [3d, d]  wdtype  self_attn.in_proj_weight */
  const float *in_proj_b;  /* [3d]     f32 */
  const void *out_proj_w;  /* [d, d] */
  const float *out_proj_b; /* [d] */
  const void *lin1_w;      /* [dff, d] */
  const float *lin1_b;     /* [dff] */
  const void *lin2_w;      /* [d, dff] */
  const float *lin2_b;     /* [d] */
  const float *norm1_w, *norm1_b; /* [d] LayerNorm affine (inner norm for AdaLN) */
  const float *norm2_w, *norm2_b;
} vb_layer_params;

typedef struct vb_decoder_desc {
  int32_t d_model, n_head, n_layer, d_ff;
  int32_t wdtype;                /* vb_dtype of the matrices and of activations/KV cache */
  const vb_layer_params *layers; /* host array [n_layer] */
  const float *final_norm_w, *final_norm_b; /* [d] */
} vb_decoder_desc;

typedef struct vb_decoder *vb_decoder_t;

int vb_decoder_create(const vb_decoder_desc *desc, vb_decoder_t *out);
void vb_decoder_destroy(vb_decoder_t dec);

/* bytes of scratch vb_decoder_forward needs for M rows */
size_t vb_decoder_forward_workspace(const vb_decoder_desc *desc, int64_t M);

/* a5/a6  TransformerEncoder.forward WITHOUT the final norm over packed ragged sequences
 *   (prefill of the AR decoder, a NAR pass, the training forward).
 *   x: fp32 [M, d] residual stream, updated in place.
 *   ada_wb: NULL (LayerNorm) or fp32 [(2*n_layer+1), 2d] AdaLN (weight|bias) rows for the
 *   current stage: row 2l = layer l norm1, 2l+1 = layer l norm2, last = final norm.
 *   kcache/vcache: NULL or [n_layer, B, H, cache_cap, hd] caches filled for later decoding. */
int vb_decoder_forward(vb_decoder_t dec, float *x, int64_t M, int B, const int32_t *cu_seqlens,
                       const int32_t *text_lens, const int32_t *seg1_lens, int seg1_start, int max_seqlen,
                       int mask_mode, const float *ada_wb,
                       void *kcache, void *vcache, int64_t cache_layer_stride,
                       int64_t cache_seq_stride, int cache_cap, void *workspace,
                       size_t workspace_bytes, vb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a2 / f2  Training: VALLE.forward with gradients (valle/models/valle.py:762-959; loss.backward() at
 *     valle/bin/trainer.py:674).  The backward functions produce what torch.autograd produces for the reference's
 *     modules; parameter gradients are fp32 and ACCUMULATED (+=) into caller-zeroed buffers.
 * ---------------------------------------------------------------------------------------- */
/* bytes of the activation store vb_decoder_forward_train fills for M rows (per layer: layer input, LN1 out, q|k|v,
 * attention out, post-attention residual, LN2 out, FFN hidden; plus one [M, d] scratch row block) */
size_t vb_decoder_train_save_bytes(const vb_decoder_desc *desc, int64_t M);
/* vb_decoder_forward (no KV cache) that keeps the activations the backward pass needs in `save`.
 * dropout_p > 0 = training mode of valle/modules/transformer.py:315-334 and of the attention inside
 * F.multi_head_attention_forward (activation.py:408-427, `dropout_p=self.dropout` when training): Bernoulli masks with
 * keep probability 1 - p, survivors scaled by 1 / (1 - p), on the attention probabilities, on both sub-layer outputs
 * ahead of the residual add and on the FFN hidden.  The masks are a stateless hash of (dropout_seed, layer, site,
 * element index): vb_decoder_backward called with the same (p, seed) regenerates them, nothing is stored.  The
 * reference draws its masks from torch's generator inside the kernels this library replaces, so individual masks
 * differ from the reference's while their distribution does not. */
int vb_decoder_forward_train(vb_decoder_t dec, float *x, int64_t M, int B, const int32_t *cu_seqlens,
                             const int32_t *text_lens, const int32_t *seg1_lens, int seg1_start, int max_seqlen,
                             int mask_mode, const float *ada_wb, void *save, size_t save_bytes, float dropout_p,
                             uint64_t dropout_seed, vb_stream_t stream);
/* nn.Dropout on a contiguous tensor (embedding.py:97 after the positional encoding): out[i] = in[i] / (1 - p) where
 * the hash of (seed, stream_id, i) keeps element i, else 0; in == out allowed.  Its own backward: the same call on
 * the gradient. */
int vb_dropout(const void *in, void *out, int dtype, int64_t n, float p, uint64_t seed, uint32_t stream_id,
               vb_stream_t stream);

typedef struct vb_layer_grads { /* fp32 gradient buffers of one layer, same shapes as vb_layer_params; NULL = skip */
  float *in_proj_w, *in_proj_b, *out_proj_w, *out_proj_b, *lin1_w, *lin1_b, *lin2_w, *lin2_b;
  float *norm1_w, *norm1_b, *norm2_w, *norm2_b;
} vb_layer_grads;
typedef struct vb_layer_wt { /* the four matrices TRANSPOSED, storage dtype (operands of the input-gradient GEMMs) */
  const void *in_proj_wt;  /* [d, 3d] */
  const void *out_proj_wt; /* [d, d] */
  const void *lin1_wt;     /* [d, dff] */
  const void *lin2_wt;     /* [dff, d] */
} vb_layer_wt;

size_t vb_decoder_backward_workspace(const vb_decoder_desc *desc, int64_t M);
/* Backward of vb_decoder_forward_train.  dx: fp32 [M, d], gradient w.r.t. the stack output on entry, w.r.t. the
 * stack input on return.  ada_wb / dada_wb: the AdaLN (weight|bias) rows of the forward call and their gradient
 * ([(2*n_layer+1), 2d], rows 2l / 2l+1 touched here), both NULL for a LayerNorm stack.  wt / grads: host arrays
 * [n_layer].  dropout_p / dropout_seed: the values of the forward call. */
int vb_decoder_backward(vb_decoder_t dec, float *dx, int64_t M, int B, const int32_t *cu_seqlens,
                        const int32_t *text_lens, const int32_t *seg1_lens, int seg1_start, int max_seqlen,
                        int mask_mode, const float *ada_wb, float *dada_wb, const void *save, const vb_layer_wt *wt,
                        const vb_layer_grads *grads, void *workspace, size_t workspace_bytes, float dropout_p,
                        uint64_t dropout_seed, vb_stream_t stream);

/* LayerNorm / AdaptiveLayerNorm backward (transformer.py:57-108) of y = vb_layernorm(x rows): dx[xrow(r), :] +=
 * d/dx, optional copy of the updated dx rows in copy_dtype ([*, d] dense), dgamma / dbeta / dada_wb (2d: weight |
 * bias) accumulated; any gradient pointer may be NULL. */
int vb_layernorm_backward(const float *x, int64_t x_row_stride, const int32_t *rows, int64_t n_rows, int d,
                          const float *gamma, const float *beta, const float *ada_wb, float eps, const float *dy,
                          int64_t dy_row_stride, float *dx, int64_t dx_row_stride, void *dx_copy, int copy_dtype,
                          float *dgamma, float *dbeta, float *dada_wb, vb_stream_t stream);
/* F.cross_entropy backward: dlogits[r, 0:n_vocab] = grad_scale * grad_rows[r] * (softmax - onehot(target)), 0 for
 * ignored rows; columns [n_vocab, n_out) are zero-filled (K padding of the following GEMMs). */
int vb_cross_entropy_backward(const float *logits, int64_t ld_logits, const int64_t *targets, int64_t n_rows,
                              int n_vocab, int64_t ignore_index, const float *grad_rows, float grad_scale, void *dlogits,
                              int out_dtype, int64_t ld_out, int n_out, vb_stream_t stream);
/* nn.Embedding backward of vb_embed_sum: table_grads[j][tokens[r, j], :] += dy[dy_row(r), :] */
int vb_embed_backward(const int64_t *tokens, int64_t tok_row_stride, int64_t tok_tab_stride, float *const *table_grads,
                      const int32_t *table_rows, int n_tables, int64_t n_rows, int d, const float *dy,
                      int64_t dy_row_stride, const int32_t *dy_rows, vb_stream_t stream);
/* out[0] += sum_r <a[r, :], b[pos(r), :]>: gradient of the SinePositionalEmbedding alpha (embedding.py:93-97) */
int vb_rowdot_accumulate(const float *a, int64_t a_row_stride, const float *b, int64_t pos0, const int32_t *positions,
                         int64_t n_rows, int d, float *out, vb_stream_t stream);
/* AdaptiveLayerNorm.project_layer backward for one (weight|bias) row: dW[2d, d] += dwb (x) emb, db[2d] += dwb,
 * demb[d] += W^T dwb */
int vb_adaln_project_backward(const float *W, const float *emb, const float *dwb, int d, float *dW, float *db,
                              float *demb, vb_stream_t stream);
size_t vb_linear_backward_workspace(int dtype, int64_t M, int N, int K);
/* Gradients of Y[M,N] = X[M,K] W[N,K]^T + b (vb_linear): dX = dY W computed as linear(dY, Wt) with Wt = W^T [K, N]
 * (dx_epilogue VB_EPI_NONE, or VB_EPI_RESIDUAL to accumulate into an fp32 dX), dW[N,K] += dY^T X, db[N] += column
 * sums of dY.  X / dY / Wt share `dtype`; N and K multiples of 64 (pad with zero columns). */
int vb_linear_backward(const void *X, int dtype, int64_t ldx, const void *Wt, const void *dY, int64_t lddy, void *dX,
                       int dx_dtype, int64_t lddx, int dx_epilogue, float *dW, float *db, int64_t M, int N, int K,
                       void *workspace, size_t workspace_bytes, vb_stream_t stream);
size_t vb_attention_backward_workspace(int64_t M, int n_head);
/* Backward of vb_attention: qkv / out / dout as in the forward call, dqkv [M, 3d] = (dQ | dK | dV), same dtype */
int vb_attention_backward(const void *qkv, const void *out, const void *dout, int dtype, int64_t M, int B, int n_head,
                          int head_dim, const int32_t *cu_seqlens, const int32_t *text_lens, const int32_t *seg1_lens,
                          int seg1_start, int max_seqlen, int mask_mode, void *dqkv, void *workspace,
                          size_t workspace_bytes, vb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a1  AR sampling loop of VALLE.inference (valle.py:1012-1057) with a growing KV cache,
 *     batched over B independent utterances.  All loop state lives on the device.
 * ---------------------------------------------------------------------------------------- */
/* A LayerNorm folded into the projection that consumes it (bf16 decode chain, valle/modules/transformer.py:296-302:
 * `x + sa(norm1(x))`, `x + ff(norm2(x))`, valle/models/valle.py:1039 `ar_predict_layer(norm(x))`):
 *   LayerNorm(x) W^T + b = rstd (x wf^T - mean c) + dvec,  wf[n,k] = W[n,k] gamma[k],  c[n] = sum_k wf[n,k],
 *   dvec[n] = b[n] + sum_k beta[k] W[n,k]
 * so the decode step multiplies the RAW fp32 residual rows (rounded to bf16 on the fly) by wf and the consumer of the
 * product applies the row moments: the residual + LayerNorm launches between the projections disappear.
 * Built by vb_ln_fold_build; all-NULL = not folded. */
typedef struct vb_ln_fold {
  const void *wf;     /* bf16 [N, K] */
  const float *c;     /* fp32 [N] */
  const float *dvec;  /* fp32 [N] */
} vb_ln_fold;

/* W: bf16 [N, K]; gamma, beta: fp32 [K] LayerNorm affine; bias: fp32 [N] or NULL; outputs as in vb_ln_fold */
int vb_ln_fold_build(const void *W, int N, int K, const float *gamma, const float *beta, const float *bias,
                     void *wf, float *c, float *dvec, vb_stream_t stream);

/* hands the decoder the folded in_proj (norm1) and linear1 (norm2) of every layer (host arrays [n_layer], copied);
 * NULL, NULL switches the folded decode chain off again.  bf16 decoders only; used by vb_ar_decode_step. */
int vb_decoder_set_decode_fold(vb_decoder_t dec, const vb_ln_fold *qkv, const vb_ln_fold *ffn1);

typedef struct vb_ar_state {
  int32_t B;
  int32_t tok_stride;         /* row stride of `tokens` */
  const int32_t *text_len;    /* [B] S_b */
  const int32_t *prompt_len;  /* [B] Tp_b */
  const int32_t *max_new;     /* [B] stop when n_gen > max_new (reference: 16*S_b, valle.py:1047) */
  int32_t *n_gen;             /* [B] tokens generated so far */
  int32_t *finished;          /* [B] 0 running, 1 stopped, 2 stopped at step 0 (valle.py:1049) */
  int32_t *tokens;            /* [B, tok_stride] generated first-codebook ids */
  float *x_cur;               /* [B, d] input row of the next decode step */
  float *logits;              /* [B, n_vocab_pad] fp32 logits of the last step (for sampling) */
  void *kcache, *vcache;      /* [n_layer, B, H, cache_cap, hd] */
  int64_t cache_layer_stride, cache_seq_stride; /* in elements */
  int32_t cache_cap;
  int32_t n_active_out_unused;
  /* seeded sampling on the device (vb_ar_head.greedy == 2), [B] each; NULL otherwise */
  const uint64_t *seed;       /* per-utterance seed s_b */
  const int32_t *top_k;       /* per-utterance top_k (<= 0: no filter) */
  const float *temperature;   /* per-utterance temperature (finite, > 0) */
} vb_ar_state;

typedef struct vb_ar_head {
  const void *predict_w;      /* [n_vocab, d] ar_predict_layer.weight (wdtype), no bias */
  int32_t n_vocab;            /* 1025 */
  int32_t eos_id;             /* 1024 */
  const float *audio_emb;     /* fp32 [n_vocab, d] ar_audio_embedding */
  const float *alpha;         /* ar_audio_position.alpha (device scalar) */
  const float *pe;            /* fp32 [pe_rows, d] sine table */
  int32_t pe_rows;
  int32_t greedy;             /* 1: argmax + stop rule + append on device; 0: logits only;
                                 2: seeded sampling + stop rule + append on device (below) */
  vb_ln_fold fold;            /* final LayerNorm folded into predict_w (all-NULL: separate LayerNorm launch) */
} vb_ar_head;

/* Seeded sampling (greedy == 2; vb_ar_state.seed / top_k / temperature set; n_vocab <= 1280).  The draw of utterance b
 * at decode step t = n_gen[b] depends only on its logits row, s_b = seed[b], t, top_k[b] and temperature[b] -- not on
 * its batch slot, the batch size or any other row:
 *   1. z_i = logits_i / T  (IEEE fp32 division; valle.py:1297-1298 `logits / temperature`)
 *   2. top_k > 0: k = min(top_k, n_vocab); keep every z_i >= (k-th largest z), ties with the k-th value included
 *      (top_k_top_p_filtering, valle.py:1254-1260); top_k <= 0: keep all
 *   3. Gumbel-max over the kept ids: h = mix64(s_b, t, i) >> 40 (24 bits; mix64 = the splitmix64 finaliser of the
 *      dropout masks, z = s + t * 0x9E3779B97F4A7C15 + i * 0xD1342543DE82EF95 then xor-shift-multiply), u = (h + 0.5)
 *      2^-24, e = -log(u) in fp32 (logf(u) for h < 2^23, else log1pf(-(2^24 - 1 - h + 0.5) 2^-24): both arguments are
 *      exact), key_i = z_i - logf(e); sample = argmax key, lowest id on an exact tie.  This is a draw from
 *      softmax(filtered z), as torch.multinomial(softmax(...), 1) draws.
 *   4. stop rule unchanged (valle.py:1044-1048): argmax(logits) == eos, or sample == eos, or the cap. */

/* bytes of scratch for vb_ar_head_step / vb_ar_decode_step.  The buffer must not be shared between
 * concurrently running streams. */
size_t vb_ar_step_workspace(const vb_decoder_desc *desc, int B, int cache_cap);

/* final LayerNorm + ar_predict_layer on rows h[B,d] (valle.py:1039), then (greedy) the stop
 * rule of valle.py:1044-1048 and the append of valle.py:1057 + next-row embedding
 * (valle.py:1013-1015).  Used after prefill and at the end of every decode step. */
int vb_ar_head_step(vb_decoder_t dec, const vb_ar_head *head, const float *h, vb_ar_state *st,
                    void *workspace, size_t workspace_bytes, vb_stream_t stream);

/* one decode step for all B rows: 12 x (LN -> QKV -> KV append -> single-query attention over
 * the cache -> out-proj -> LN -> FFN), then vb_ar_head_step.  Safe to capture in a CUDA graph
 * (no host reads; launch geometry depends only on B and cache_cap).  bf16 decoders with
 * vb_decoder_set_decode_fold + head->fold run the LayerNorm-folded chain (6 launches per layer; the
 * residual stream is assembled by bulk reductions whose order over the split-K slabs is not fixed:
 * last-bit differences between runs, VB_DECODE_FOLD=0 selects the fixed-order 8-launch chain). */
int vb_ar_decode_step(vb_decoder_t dec, const vb_ar_head *head, vb_ar_state *st, void *workspace,
                      size_t workspace_bytes, vb_stream_t stream);

/* after sampling on the host side (top_k != 1): push tokens[B] chosen by the caller
 * (valle.py:1040-1057 with torch's own RNG), applying the same stop rule. */
int vb_ar_push_tokens(const vb_ar_head *head, vb_ar_state *st, const int64_t *sampled, int d,
                      vb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a1  NAR stage tail (valle.py:1128-1134): samples = argmax(logits) over rows, written to
 *     codes[r*code_row_stride] (int64), and (if next_emb != NULL) y_emb[yrow(r),:] += next_emb[sample],
 *     yrow(r) = y_rows ? y_rows[r] : r.
 * ---------------------------------------------------------------------------------------- */
int vb_nar_argmax_accumulate(const float *logits, int64_t n_rows, int n_vocab, int64_t ld_logits,
                             int64_t *codes, int64_t code_row_stride, const float *next_emb,
                             float *y_emb, int64_t y_row_stride, const int32_t *y_rows, int d,
                             vb_stream_t stream);

/* a2  F.cross_entropy of VALLE.forward (valle.py:877,936-941), per row:
 *   loss[r] = logsumexp(logits[r,:]) - logits[r, targets[r]], 0 where targets[r] == ignore_index
 *   (pass ignore_index = -1 for none).  The caller sums (reduction="sum"). */
int vb_cross_entropy(const float *logits, int64_t ld_logits, const int64_t *targets, int64_t n_rows,
                     int n_vocab, int64_t ignore_index, float *loss, vb_stream_t stream);

/* gather rows: dst[r,:] = src[rows[r],:], a zero row where rows[r] < 0  (fp32): "last position" / target slices, and
 * the shifted copies (zero 'same' padding at the sequence ends) that turn the kernel-5 Conv1d of the text pre-net
 * (valle/models/valle.py:97-113,182-204) into one vb_linear over [rows, 5 d] */
int vb_gather_rows(const float *src, int64_t src_row_stride, const int32_t *rows, int64_t n_rows,
                   int d, float *dst, int64_t dst_row_stride, vb_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * a13  AudioTokenizer.encode / .decode (valle/data/tokenizer.py:211-254) -> PyPI `encodec`
 *      EncodecModel.encodec_model_24khz() at 6 kbps: SEANet conv stacks, 2-layer LSTM, 8-stage RVQ.
 *      fp32, activations [B, C, T] (time contiguous).
 * ---------------------------------------------------------------------------------------- */
/* SConv1d: y = conv1d(pad(act(x))) + bias (+ residual); act = ELU if pre_elu; padding (pad_left,
 * pad_right) reflect or zero.  wp: the conv weight [Cout, Cin, K] (weight-norm already folded,
 * tokenizer.py:181-208) PRE-PACKED channel-fastest as [Cin, K, Cout].
 * phase > 1 -- the causal SConvTranspose1d with K == 2*stride and the right padding trimmed, as a stride-1 K=2
 * convolution onto Cout = C * phase "phase channels" c' = c * phase + r: wp[ci][0][c'] = w_T[ci][c][r + phase],
 * wp[ci][1][c'] = w_T[ci][c][r] (w_T [Cin, C, 2*phase] the transposed-conv weight), pad_left = 1 (zero), bias [C];
 * output channel c' is stored to out[b, c, t * phase + r], out [B, C, Tout * phase]. */
int vb_conv1d(const float *x, int B, int Cin, int Tin, const float *wp, const float *bias, int Cout, int K,
              int stride, int dilation, int pad_left, int pad_right, int reflect, int pre_elu,
              const float *residual, float *out, int Tout, int phase, vb_stream_t stream);
/* one LSTM layer over T steps: xproj [T, B, 4H] = W_ih x + b_ih + b_hh (gate order i,f,g,o),
 * whh_t [H, 4H] = W_hh^T, h_seq [T, B, H] out, c_state [B * H + 64] floats of scratch (cell state of the
 * step-wise path / grid-barrier word of the persistent kernel).  B <= 64: all T steps run in one cooperative
 * launch (the W_hh slices stay in shared memory); larger batches fall back to one launch per step. */
int vb_lstm_layer(const float *xproj, const float *whh_t, int T, int B, int H, float *h_seq, float *c_state,
                  vb_stream_t stream);
/* residual VQ encode of rows x [n_rows, dim]: per stage idx = argmax -(|r|^2 - 2 r.e + |e|^2), r -= e_idx.
 * codebooks [n_q, n_codes, dim], codebooks_t [n_q, dim, n_codes], codebook_sq [n_q, n_codes];
 * The code of row r (sequence s = r / rows_per_seq, frame f = r % rows_per_seq) and stage q is written to
 * codes[s*code_seq_stride + f*code_row_stride + q*code_q_stride] (int64): [B, n_q, T] codes of a whole batch in one
 * launch with rows_per_seq = T, strides (n_q*T, 1, T); rows_per_seq <= 0: one sequence. */
int vb_rvq_encode(const float *x, int64_t n_rows, int dim, int n_q, int n_codes, const float *codebooks,
                  const float *codebooks_t, const float *codebook_sq, int64_t *codes, int64_t code_row_stride,
                  int64_t code_q_stride, int64_t rows_per_seq, int64_t code_seq_stride, vb_stream_t stream);
/* out = in.permute(p0, p1, p2) for a contiguous [d0, d1, d2] fp32 tensor */
int vb_permute3(const float *in, int d0, int d1, int d2, int p0, int p1, int p2, float *out, vb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VALLE_B200_H_ */
