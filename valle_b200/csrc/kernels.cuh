// Internal launcher declarations shared by the translation units of libvalle_b200.so.
#pragma once
#include "common.cuh"

namespace vb {

// Visibility rule of one query row (see vb_mask_mode): key c is seen iff c < lim0 or s1 <= c < hi1.
// Training-mode dropout (valle/modules/transformer.py:329,333-334, activation.py attention dropout, embedding.py:97):
// a stateless Bernoulli mask keyed by (seed of the forward call, stream id of the site, element index), so the backward
// pass regenerates the mask of the forward pass instead of storing it.  splitmix64 finaliser; keep <=> hash >= thresh
// with thresh = p * 2^32.  tests/test_backward_gpu.py holds the same function in numpy.
// The seeded AR sampler (sample.cu) draws its uniforms from the same hash, keyed by (utterance seed, decode step, id).
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t seed, uint64_t stream, uint64_t idx) {
  uint64_t z = seed + stream * 0x9E3779B97F4A7C15ull + idx * 0xD1342543DE82EF95ull;
  z ^= z >> 30;
  z *= 0xBF58476D1CE4E5B9ull;
  z ^= z >> 27;
  z *= 0x94D049BB133111EBull;
  z ^= z >> 31;
  return z;
}
struct DropCfg {
  uint64_t seed;
  uint32_t stream;     // site id: (layer << 2) | {0 attention probabilities, 1 after out-proj, 2 FFN hidden, 3 after FFN}
  uint32_t thresh;     // 0 = dropout off
  float inv_keep;      // 1 / (1 - p)
  int64_t lmax;        // attention only: index = ((b * H + h) * lmax + q) * lmax + k
};
__host__ __device__ __forceinline__ bool drop_keep(const DropCfg &c, uint64_t idx) {
  return (uint32_t)(mix64(c.seed, c.stream, idx) >> 32) >= c.thresh;
}
inline DropCfg make_drop(float p, uint64_t seed, uint32_t stream, int64_t lmax = 0) {
  DropCfg c{};
  if (p > 0.f) {
    c.seed = seed;
    c.stream = stream;
    const double t = (double)p * 4294967296.0;
    c.thresh = t >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)t;
    c.inv_keep = 1.f / (1.f - p);
    c.lmax = lmax;
  }
  return c;
}

struct RowMask {
  int lim0, s1, hi1;
  __device__ __forceinline__ bool ok(int c) const { return c < lim0 || (c >= s1 && c < hi1); }
};
__device__ __forceinline__ RowMask make_row_mask(int mode, int qr, int L, int S, int seg1_start, int seg1_len) {
  RowMask m{0, 0, 0};
  if (qr >= L) return m;
  if (mode == VB_MASK_FULL) {
    m.lim0 = L; m.s1 = L; m.hi1 = L;
  } else if (mode == VB_MASK_VALLE_AR) {
    m.lim0 = max(S, qr + 1); m.s1 = L; m.hi1 = L;
  } else if (mode == VB_MASK_PADDED_AR) {
    m.lim0 = S; m.s1 = seg1_start;
    m.hi1 = qr >= seg1_start ? seg1_start + min(seg1_len, qr - seg1_start + 1) : seg1_start;
  } else {  // VB_MASK_PADDED
    m.lim0 = S; m.s1 = seg1_start; m.hi1 = seg1_start + seg1_len;
  }
  return m;
}

// L2 prefetch of a slice of an upcoming layer's K and V cache, issued by the otherwise idle warps of the
// split-K decode projections (gemm_decode.cu) while their weight tiles stream: the projection chain is latency
// bound and leaves HBM mostly idle, the KV-cache attention that follows is HBM bound -- the slice [lo_pct, hi_pct)
// of every (utterance, head) stream is pulled into the 126 MB L2 ahead of it.  Only a hint: the lengths may be
// one step stale (read before the dependency wait), which changes what is prefetched, never what is computed.
struct KvPrefetch {
  const void *kbase, *vbase;  // caches of the target layer ([B, H, cap, 64]) or nullptr
  int64_t seq_stride_bytes;   // bytes between utterances
  int B, H, cap, row_bytes;   // row_bytes = 64 * element size
  const int32_t *text_len, *prompt_len, *n_gen;
  int lo_pct, hi_pct;
};
// worker = one warp; `n_workers` warps of the grid share the streams.  Lane i of a warp fetches the lengths of the
// warp's i-th stream up front (the three dependent global loads per stream would otherwise serialise the loop).
__device__ __forceinline__ void kv_prefetch(const KvPrefetch &pf, int worker, int n_workers) {
  if (pf.kbase == nullptr) return;
  const int lane = threadIdx.x & 31;
  const int n_streams = 2 * pf.B * pf.H;
  int kv_mine = 0;
  {
    const int s_mine = worker + lane * n_workers;
    if (s_mine < n_streams) {
      const int b = (s_mine >> 1) / pf.H;
      kv_mine = min(pf.text_len[b] + pf.prompt_len[b] + pf.n_gen[b], pf.cap);
    }
  }
  for (int i = 0, sidx = worker; sidx < n_streams; ++i, sidx += n_workers) {
    int kv;
    if (i < 32) {
      kv = __shfl_sync(0xffffffffu, kv_mine, i);
    } else {
      const int b = (sidx >> 1) / pf.H;
      kv = min(pf.text_len[b] + pf.prompt_len[b] + pf.n_gen[b], pf.cap);
    }
    const int pair = sidx >> 1;
    const int b = pair / pf.H, h = pair - b * pf.H;
    const int r_lo = kv * pf.lo_pct / 100, r_hi = kv * pf.hi_pct / 100;
    const char *p = (const char *)((sidx & 1) ? pf.vbase : pf.kbase) + (int64_t)b * pf.seq_stride_bytes +
                    ((int64_t)h * pf.cap + r_lo) * pf.row_bytes;
    const int lines = ((r_hi - r_lo) * pf.row_bytes) >> 7;  // 128-byte lines
    for (int l = lane; l < lines; l += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + ((int64_t)l << 7)));
  }
}

struct LnParams {
  const float *gamma, *beta, *ada_wb;  // ada_wb: NULL or [2d] (weight | bias)
  float eps;
};

struct QkvScatter {
  int d, head_dim;
  float *q;  // [B, d] fp32
  void *kcache, *vcache;  // this layer's cache base
  int64_t cache_seq_stride;
  int cache_cap;
  const int32_t *text_len, *prompt_len, *n_gen;
  const int32_t *finished;  // NULL or [B]: rows that have stopped keep their cache untouched
};

// gemm_simt.cu
int launch_gemm_simt(const void *A, int a_dtype, int64_t lda, const void *W, const float *bias, void *C,
                     int c_dtype, int64_t ldc, int64_t M, int N, int K, int epi, cudaStream_t s);
int launch_gemv(const float *x, int64_t ldx, int B, const void *W, int w_dtype, const float *bias,
                int N, int K, float *out, int64_t ldo, const LnParams *ln, int epi_mode,
                const QkvScatter *qkv, cudaStream_t s);

// gemm_tcgen05.cu
bool tcgen05_gemm_supported(int64_t M, int N, int K, int64_t lda, int64_t ldc);
int launch_gemm_tcgen05(const bf16 *A, int64_t lda, const bf16 *W, const float *bias, void *C,
                        int c_dtype, int64_t ldc, int64_t M, int N, int K, int epi, cudaStream_t s);

// gemm_decode.cu (swap-AB split-K tcgen05 projections for B <= 64 decode rows, bf16)
enum { DG_F32 = 0, DG_RESIDUAL = 1, DG_RELU_BF16 = 2, DG_QKV = 3 };
constexpr int kMaxForcedSplits = 16;  // cap of a caller-chosen split-K count (sizes the partial workspace)
size_t gemm_decode_workspace(int d_model, int d_ff);
int launch_gemm_decode(const bf16 *act, int B, int64_t ld_act, const bf16 *W, int N, int K, int force_splits,
                       const float *bias, int mode, float *out_f32, bf16 *out_bf16, int64_t ld_out,
                       const QkvScatter *qkv, float *partials, size_t partial_bytes, int *out_splits, int *out_ldp,
                       const KvPrefetch *pf, bool pdl, cudaStream_t s, bool red_add = false);
// LayerNorm folded into the projection (decode chain without the residual + LayerNorm launches):
//   moments of the fp32 rows, stats[split][64][2] = (sum x, sum x^2) over the split's k-range, next to the partials
struct LnFoldStats {
  const float *stats;  // NULL: the partials are plain (no folded LayerNorm)
  const float *c;      // [N]  sum_k wf[n,k]
  int splits, d;       // splits of the producing projection, LayerNorm width
  float eps;
  int copies;          // every tile row of the producing grid stores its own copy of the moments:
                       // stats[copy][split][64][2]; consumers spread over the copies (no L2 hot spot)
};
constexpr int kLnFoldMaxCopies = 32;
// Called by every lane of a (converged) warp whose threads share the row b: lane s fetches split s's pair, the warp
// adds them up by shuffles -- ONE L2 round trip.  (A per-thread loop over the splits, however it is unrolled, ends up
// as `splits` dependent round trips under the register caps of the consumer kernels: 2.3 us in the attention prologue.)
__device__ __forceinline__ float2 ln_fold_moments_load(const LnFoldStats &f, int b, int which) {
  const int lane = threadIdx.x & 31;
  const float *st = f.stats + (int64_t)(which % f.copies) * f.splits * 64 * 2;
  float2 m = make_float2(0.f, 0.f);
  if (lane < f.splits) m = __ldcg(reinterpret_cast<const float2 *>(st + ((int64_t)lane * 64 + b) * 2));
  return m;
}
__device__ __forceinline__ void ln_fold_moments_finish(const LnFoldStats &f, float2 m, float &mean, float &rstd) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    m.x += __shfl_xor_sync(0xffffffffu, m.x, o);
    m.y += __shfl_xor_sync(0xffffffffu, m.y, o);
  }
  mean = m.x / (float)f.d;
  rstd = rsqrtf(fmaxf(m.y / (float)f.d - mean * mean, 0.f) + f.eps);
}
__device__ __forceinline__ void ln_fold_moments(const LnFoldStats &f, int b, int which, float &mean, float &rstd) {
  ln_fold_moments_finish(f, ln_fold_moments_load(f, b, which), mean, rstd);
}
int launch_gemm_decode_x(const float *x, int B, int64_t ldx, const bf16 *Wf, int N, int K, int force_splits,
                         float *partials, size_t partial_bytes, float *stats, int *out_splits, int *out_ldp,
                         int *out_copies, const KvPrefetch *pf, bool pdl, cudaStream_t s);
int launch_ln_fold(const bf16 *W, int N, int K, const float *gamma, const float *beta, const float *bias, bf16 *wf,
                   float *c, float *dvec, cudaStream_t s);

// attention.cu
int launch_attention_varlen(const void *qkv, int dtype, int64_t M, int B, int n_head, int head_dim,
                            const int32_t *cu_seqlens, const int32_t *text_lens, const int32_t *seg1_lens,
                            int seg1_start, int max_seqlen, int mask_mode, void *out, void *kcache, void *vcache,
                            int64_t cache_seq_stride, int cache_cap, const uint8_t *dense_mask, int64_t dense_ld,
                            cudaStream_t s, const DropCfg *drop = nullptr);
// attention_mma.cu (bf16 tensor-core flash attention)
int launch_attention_mma(const bf16 *qkv, int64_t M, int B, int n_head, const int32_t *cu_seqlens,
                         const int32_t *text_lens, const int32_t *seg1_lens, int seg1_start, int max_seqlen,
                         int mask_mode, bf16 *out, bf16 *kcache,
                         bf16 *vcache, int64_t cache_seq_stride, int cache_cap, int tail_of_128, cudaStream_t s);
// attention_tcgen05.cu (bf16 flash attention on tcgen05/TMEM; no KV-cache fill)
bool attention_tcgen05_enabled();
int launch_attention_tcgen05(const bf16 *qkv, int64_t M, int B, int n_head, const int32_t *cu_seqlens,
                             const int32_t *text_lens, const int32_t *seg1_lens, int seg1_start, int max_seqlen,
                             int mask_mode, bf16 *out, int skip_partial, cudaStream_t s);
size_t attn_decode_workspace(int B, int n_head, int head_dim, int cache_cap);
int launch_attn_decode(const float *q, const float *qkv_part, int qkv_splits, int qkv_ldp, const float *qkv_bias,
                       int B, int n_head, int head_dim, void *kcache, void *vcache, int dtype,
                       int64_t cache_seq_stride, int cache_cap, const int32_t *text_len, const int32_t *prompt_len,
                       const int32_t *n_gen, const int32_t *finished, float *out, void *out16, void *workspace,
                       bool pdl, cudaStream_t s, const LnFoldStats *fold = nullptr);

// decode_fused.cu
int launch_relu_reduce(const float *partials, int splits, int ldp, const float *bias, int B, int N, bf16 *out16,
                       int64_t ldo, bool pdl, cudaStream_t s, const LnFoldStats *fold = nullptr);
int launch_ln_reduce(float *x, int64_t ldx, int B, int d, const float *partials, int splits, int ldp,
                     const float *bias, const float *gamma, const float *beta, float eps, bf16 *out16,
                     bool pdl, cudaStream_t s);

// backward.cu
int launch_transpose_pad(const void *in, int dtype, int64_t ld_in, int64_t R, int C, void *out, int64_t ld_out,
                         cudaStream_t s);
int launch_colsum(const void *in, int dtype, int64_t ld, int64_t R, int N, float *out, cudaStream_t s);
int launch_relu_bwd(void *dh, const void *h, int dtype, int64_t n, float scale, cudaStream_t s);
int attention_backward(const void *qkv, const void *out, const void *dout, int dtype, int64_t M, int B, int n_head,
                       int head_dim, const int32_t *cu_seqlens, const int32_t *text_lens, const int32_t *seg1_lens,
                       int seg1_start, int max_seqlen, int mask_mode, void *dqkv, void *workspace, size_t workspace_bytes,
                       const DropCfg *drop, cudaStream_t s);
// out[i] = keep(i) ? in[i] / (1 - p) : 0 (in place allowed); x[i] += keep(i) ? t[i] / (1 - p) : 0
int launch_dropout(const void *in, void *out, int dtype, int64_t n, const DropCfg &cfg, cudaStream_t s);
int launch_dropout_add(float *x, const float *t, int64_t n, const DropCfg &cfg, cudaStream_t s);
int launch_cast_from_f32(const float *in, void *out, int dtype, int64_t n, cudaStream_t s);

// sample.cu
int launch_ar_sample(float *logits, int64_t ld_logits, const float *partials, int splits, int ldp,
                     const vb_ar_head *head, vb_ar_state *st, int d, const int64_t *forced, int reduce_only, bool pdl,
                     cudaStream_t s, const LnFoldStats *fold = nullptr);

}  // namespace vb
