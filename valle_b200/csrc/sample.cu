// Device-side tails of the AR loop and of a NAR stage.
//   * ar_sample_kernel: argmax over the 1025 logits -- or, in the seeded mode, a top-k / temperature draw keyed by
//     (utterance seed, step, id) -- the stop rule of valle/models/valle.py:1044-1048
//     (argmax==EOS or sample==EOS or n_new > 16*S), the append of :1057 and the embedding + sine PE
//     of the appended token (:1013-1015) so the next decode step needs no host round trip
//     (the reference syncs to the host once per token).
//   * nar_argmax_accumulate_kernel: samples = argmax(logits) (:1130) and
//     y_emb[:, Tp:] += nar_audio_embeddings[i+1](samples) (:1133-1134).
#include <math_constants.h>

#include "common.cuh"
#include "kernels.cuh"

namespace vb {

struct ArgMax {
  float v;
  int i;
};
__device__ __forceinline__ ArgMax better(ArgMax a, ArgMax b) {
  // larger value wins; on ties the smaller index (torch.argmax returns the first maximum)
  return (b.v > a.v || (b.v == a.v && b.i < a.i)) ? b : a;
}
__device__ __forceinline__ ArgMax warp_argmax(ArgMax a) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ArgMax b;
    b.v = __shfl_xor_sync(0xffffffffu, a.v, o);
    b.i = __shfl_xor_sync(0xffffffffu, a.i, o);
    a = better(a, b);
  }
  return a;
}

// ---- seeded sampling (vb_ar_head.greedy == 2; the semantics are spelled out in include/valle_b200.h) ----
constexpr int kSeededCols = 5;  // ids per thread: n_vocab <= 5 * 256
struct SeededDraw {             // [B] device arrays, all NULL when the launch does not sample
  const uint64_t *seed;
  const int32_t *top_k;
  const float *temperature;
};

// order-preserving map of a non-NaN float onto uint32 (-0.0 and +0.0 map to the same key, as they compare equal)
__device__ __forceinline__ uint32_t float_order_key(float z) {
  const uint32_t u = __float_as_uint(z == 0.f ? 0.f : z);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float order_key_float(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// k-th largest key of the row (thread tid holds ids tid + 256 j, those < n_vocab count), 1 <= k <= n_vocab: radix
// select over the key bits, most significant byte first, one 256-bin shared-memory histogram per byte.  Called by all
// 256 threads of the CTA.
__device__ uint32_t block_kth_largest(const uint32_t (&key)[kSeededCols], int n_vocab, int k) {
  __shared__ uint32_t hist[256];
  __shared__ int wsum[8];
  __shared__ uint32_t s_digit;
  __shared__ int s_krem;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t prefix = 0, pmask = 0;
  int krem = k;  // rank still to find among the ids that match `prefix` on the bytes done so far
#pragma unroll 1
  for (int shift = 24; shift >= 0; shift -= 8) {
    hist[255 - tid] = 0;  // the bin this thread scans below (it read it in the previous pass)
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kSeededCols; ++j)
      if (tid + j * 256 < n_vocab && (key[j] & pmask) == prefix) atomicAdd(&hist[(key[j] >> shift) & 255u], 1u);
    __syncthreads();
    // thread t scans bin 255 - t: an inclusive prefix sum over t counts the ids whose byte is >= 255 - t
    const int c = (int)hist[255 - tid];
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    for (int w = 0; w < warp; ++w) incl += wsum[w];
    if (incl >= krem && incl - c < krem) {  // exactly one thread: the byte of the k-th largest
      s_digit = 255u - (uint32_t)tid;
      s_krem = krem - (incl - c);
    }
    __syncthreads();
    prefix |= s_digit << shift;
    pmask |= 0xffu << shift;
    krem = s_krem;
  }
  return prefix;
}

// Gumbel noise -log(-log(u)), u = (h + 0.5) 2^-24 with h the top 24 bits of mix64(seed, step, id).  -log(u) is taken
// from the exact fp32 value of u (h < 2^23) or of 1 - u (h >= 2^23), so u never rounds to 1.
__device__ __forceinline__ float gumbel_log_e(uint64_t seed, uint64_t step, int id) {
  const uint32_t h = (uint32_t)(mix64(seed, step, (uint64_t)id) >> 40);
  const float e = h < (1u << 23) ? -logf(((float)h + 0.5f) * 0x1p-24f)
                                 : -log1pf(-(((float)((1u << 24) - 1u - h) + 0.5f) * 0x1p-24f));
  return logf(e);  // key = z - log(e)
}

// this thread's best (key, id) of the seeded draw over its ids; the caller reduces over the CTA
__device__ __forceinline__ ArgMax seeded_draw(const float (&zr)[kSeededCols], int n_vocab, uint64_t seed,
                                              uint64_t step, int top_k, float temperature) {
  const int tid = threadIdx.x;
  float z[kSeededCols];
#pragma unroll
  for (int j = 0; j < kSeededCols; ++j) z[j] = __fdiv_rn(zr[j], temperature);
  float thr = -CUDART_INF_F;
  if (top_k > 0 && top_k < n_vocab) {  // uniform per CTA
    uint32_t key[kSeededCols];
#pragma unroll
    for (int j = 0; j < kSeededCols; ++j) key[j] = float_order_key(z[j]);
    thr = order_key_float(block_kth_largest(key, n_vocab, top_k));
  }
  ArgMax g{-CUDART_INF_F, 0x7fffffff};
#pragma unroll
  for (int j = 0; j < kSeededCols; ++j) {
    const int i = tid + j * 256;
    if (i < n_vocab && z[j] >= thr) g = better(g, ArgMax{__fsub_rn(z[j], gumbel_log_e(seed, step, i)), i});
  }
  return g;
}

__global__ void __launch_bounds__(256)
ar_sample_kernel(float *__restrict__ logits, int64_t ld_logits, const float *__restrict__ partials, int splits,
                 int ldp, int n_vocab, int eos_id,
                 const float *__restrict__ audio_emb, const float *__restrict__ alpha,
                 const float *__restrict__ pe, int pe_rows, const int32_t *__restrict__ text_len,
                 const int32_t *__restrict__ prompt_len, const int32_t *__restrict__ max_new,
                 int32_t *__restrict__ n_gen, int32_t *__restrict__ finished,
                 int32_t *__restrict__ tokens, int tok_stride, float *__restrict__ x_cur, int d,
                 const int64_t *__restrict__ forced, int reduce_only, LnFoldStats fold, const float *__restrict__ fold_d,
                 SeededDraw sd) {
  __shared__ ArgMax wbest[8], wsamp[8];
  __shared__ int s_tok, s_pos;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  pdl_launch_dependents();
  pdl_wait();
  vb_trace(TR_SAMPLE * 2);
  if (finished[b] != 0 && !reduce_only) {  // uniform per CTA
    // a stopped utterance still rides through the batched step: give it a fixed, bounded input row (its residual
    // stream is updated in place by the layer chain and would otherwise drift step over step); the scatter and
    // attention kernels skip its KV cache
    float *xo = x_cur + (int64_t)b * d;
    for (int c = tid * 4; c < d; c += 1024) *reinterpret_cast<float4 *>(xo + c) = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  // scalars of the stop rule: in flight together with the logits instead of after the argmax
  const int n_new = n_gen[b], p_len = prompt_len[b], cap_new = max_new[b];
  const int forced_tok = forced ? (int)forced[b] : -1;
  const bool seeded = sd.seed != nullptr && !reduce_only;  // uniform per launch
  uint64_t s_seed = 0;
  int s_topk = 0;
  float s_temp = 1.f;
  if (seeded) {
    s_seed = sd.seed[b];
    s_topk = sd.top_k[b];
    s_temp = sd.temperature[b];
  }
  float *row = logits + (int64_t)b * ld_logits;
  ArgMax best{-CUDART_INF_F, 0x7fffffff};
  float zr[kSeededCols];  // seeded mode: the logits of ids tid + 256 j (n_vocab <= 256 * kSeededCols)
  // final LayerNorm folded into ar_predict_layer (gemm_decode_x_kernel): logit = rstd (acc - mean c[i]) + (beta W^T)[i]
  float f_mean = 0.f, f_rstd = 1.f;
  const bool folded = fold.stats != nullptr && partials != nullptr;
  if (folded) ln_fold_moments(fold, b, b, f_mean, f_rstd);
  if (partials && n_vocab <= 5 * 256 && splits <= 8) {
    // head projection split-K partials, summed in fixed order; all loads of the row issued at once
    float v[5][8];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      const int i = tid + j * 256;
      const float *p = partials + (int64_t)b * ldp + min(i, n_vocab - 1);
#pragma unroll
      for (int s = 0; s < 8; ++s) v[j][s] = s < splits ? __ldcg(p + (int64_t)s * 64 * ldp) : 0.f;
    }
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      const int i = tid + j * 256;
      float a = v[j][0];
#pragma unroll
      for (int s = 1; s < 8; ++s)
        if (s < splits) a += v[j][s];
      if (i < n_vocab) {
        if (folded) a = f_rstd * (a - f_mean * fold.c[i]) + fold_d[i];
        row[i] = a;
        zr[j] = a;
        best = better(best, ArgMax{a, i});
      }
    }
  } else {
    for (int i = tid; i < n_vocab; i += 256) {
      float v;
      if (partials) {
        const float *p = partials + (int64_t)b * ldp + i;
        v = __ldcg(p);
#pragma unroll 8
        for (int s = 1; s < splits; ++s) v += __ldcg(p + (int64_t)s * 64 * ldp);
        if (folded) v = f_rstd * (v - f_mean * fold.c[i]) + fold_d[i];
        row[i] = v;
      } else {
        v = row[i];
      }
      best = better(best, ArgMax{v, i});
    }
    if (seeded) {  // this thread wrote (or read) exactly these ids above: no barrier needed
#pragma unroll
      for (int j = 0; j < kSeededCols; ++j) zr[j] = tid + j * 256 < n_vocab ? row[tid + j * 256] : 0.f;
    }
  }
  if (reduce_only) return;
  ArgMax drawn{-CUDART_INF_F, 0x7fffffff};
  if (seeded) drawn = seeded_draw(zr, n_vocab, s_seed, (uint64_t)n_new, s_topk, s_temp);
  best = warp_argmax(best);
  if (lane == 0) wbest[warp] = best;
  if (seeded) {
    drawn = warp_argmax(drawn);
    if (lane == 0) wsamp[warp] = drawn;
  }
  __syncthreads();
  if (tid == 0) {
    ArgMax a = wbest[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) a = better(a, wbest[w]);
    int samp = forced ? forced_tok : a.i;
    if (seeded) {
      ArgMax g = wsamp[0];
#pragma unroll
      for (int w = 1; w < 8; ++w) g = better(g, wsamp[w]);
      samp = g.i;
    }
    const bool stop = (a.i == eos_id) || (samp == eos_id) || (n_new > cap_new) || (n_new >= tok_stride);
    if (stop) {
      finished[b] = (n_new == 0) ? 2 : 1;
      s_tok = -1;
    } else {
      tokens[(int64_t)b * tok_stride + n_new] = samp;
      n_gen[b] = n_new + 1;
      s_tok = samp;
      s_pos = min(p_len + n_new, pe_rows - 1);
    }
  }
  __syncthreads();
  const int tok = s_tok;
  if (tok < 0) {  // stopped at this step: same fixed input row as above
    float *xo = x_cur + (int64_t)b * d;
    for (int c = tid * 4; c < d; c += 1024) *reinterpret_cast<float4 *>(xo + c) = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  const float a = alpha[0];
  const float *e = audio_emb + (int64_t)tok * d;
  const float *p = pe + (int64_t)s_pos * d;
  float *xo = x_cur + (int64_t)b * d;
  for (int c = tid * 4; c < d; c += 1024) {
    const float4 ev = *reinterpret_cast<const float4 *>(e + c);
    const float4 pv = *reinterpret_cast<const float4 *>(p + c);
    float4 o;
    o.x = __fadd_rn(ev.x, __fmul_rn(a, pv.x));
    o.y = __fadd_rn(ev.y, __fmul_rn(a, pv.y));
    o.z = __fadd_rn(ev.z, __fmul_rn(a, pv.z));
    o.w = __fadd_rn(ev.w, __fmul_rn(a, pv.w));
    *reinterpret_cast<float4 *>(xo + c) = o;
  }
}

int launch_ar_sample(float *logits, int64_t ld_logits, const float *partials, int splits, int ldp,
                     const vb_ar_head *head, vb_ar_state *st, int d, const int64_t *forced, int reduce_only, bool pdl,
                     cudaStream_t s, const LnFoldStats *fold) {
  LnFoldStats f{};
  if (fold) f = *fold;
  const float *fold_d = fold ? head->fold.dvec : nullptr;
  SeededDraw sd{};
  if (head->greedy == 2 && forced == nullptr && !reduce_only) {
    VB_CHECK_ARG(st->seed && st->top_k && st->temperature,
                 "seeded sampling (vb_ar_head.greedy == 2) needs vb_ar_state.seed, top_k and temperature");
    VB_CHECK_ARG(head->n_vocab <= kSeededCols * 256, "seeded sampling: n_vocab %d > %d", head->n_vocab,
                 kSeededCols * 256);
    sd = SeededDraw{st->seed, st->top_k, st->temperature};
  }
  VB_CUDA(launch_kernel(ar_sample_kernel, dim3(st->B), dim3(256), 0, s, pdl, logits, ld_logits, partials, splits, ldp,
                        head->n_vocab, head->eos_id, head->audio_emb, head->alpha, head->pe, head->pe_rows,
                        (const int32_t *)st->text_len, (const int32_t *)st->prompt_len, (const int32_t *)st->max_new,
                        st->n_gen, st->finished, st->tokens, st->tok_stride, st->x_cur, d, forced, reduce_only, f,
                        fold_d, sd));
  count_launch();
  return VB_OK;
}

__global__ void nar_argmax_accumulate_kernel(const float *__restrict__ logits, int64_t n_rows, int n_vocab,
                                             int64_t ld_logits, int64_t *__restrict__ codes,
                                             int64_t code_row_stride, const float *__restrict__ next_emb,
                                             float *__restrict__ y_emb, int64_t y_row_stride,
                                             const int32_t *__restrict__ y_rows, int d) {
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const int lane = threadIdx.x & 31;
  const float *row = logits + r * ld_logits;
  ArgMax best{-CUDART_INF_F, 0x7fffffff};
  for (int i = lane; i < n_vocab; i += 32) best = better(best, ArgMax{row[i], i});
  best = warp_argmax(best);
  if (lane == 0) codes[r * code_row_stride] = best.i;
  if (next_emb != nullptr) {
    const float *e = next_emb + (int64_t)best.i * d;
    float *y = y_emb + (y_rows ? (int64_t)y_rows[r] : r) * y_row_stride;
    for (int c = lane * 4; c < d; c += 128) {
      float4 yv = *reinterpret_cast<float4 *>(y + c);
      const float4 ev = *reinterpret_cast<const float4 *>(e + c);
      yv.x = __fadd_rn(yv.x, ev.x);
      yv.y = __fadd_rn(yv.y, ev.y);
      yv.z = __fadd_rn(yv.z, ev.z);
      yv.w = __fadd_rn(yv.w, ev.w);
      *reinterpret_cast<float4 *>(y + c) = yv;
    }
  }
}

}  // namespace vb

using namespace vb;

VB_API int vb_nar_argmax_accumulate(const float *logits, int64_t n_rows, int n_vocab, int64_t ld_logits,
                                        int64_t *codes, int64_t code_row_stride, const float *next_emb,
                                        float *y_emb, int64_t y_row_stride, const int32_t *y_rows, int d,
                                        vb_stream_t stream) {
  VB_CHECK_ARG(d % 4 == 0, "vb_nar_argmax_accumulate: d %% 4 != 0");
  if (n_rows == 0) return VB_OK;
  const int wpb = 4;
  nar_argmax_accumulate_kernel<<<(unsigned)((n_rows + wpb - 1) / wpb), wpb * 32, 0, (cudaStream_t)stream>>>(
      logits, n_rows, n_vocab, ld_logits, codes, code_row_stride, next_emb, y_emb, y_row_stride, y_rows, d);
  VB_LAUNCH_CHECK();
  return VB_OK;
}

// F.cross_entropy per row (valle/models/valle.py:877,936-941): loss[r] = logsumexp(logits[r,:]) -
// logits[r, target[r]]; rows whose target == ignore_index contribute 0.  One warp per row, fp32.
namespace vb {
__global__ void cross_entropy_kernel(const float *__restrict__ logits, int64_t ld, const int64_t *__restrict__ targets,
                                     int64_t n_rows, int n_vocab, int64_t ignore_index, float *__restrict__ loss) {
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const int lane = threadIdx.x & 31;
  const float *row = logits + r * ld;
  const int64_t tg = targets[r];
  float mx = -CUDART_INF_F;
  for (int i = lane; i < n_vocab; i += 32) mx = fmaxf(mx, row[i]);
  mx = warp_max(mx);
  float s = 0.f;
  for (int i = lane; i < n_vocab; i += 32) s += expf(row[i] - mx);
  s = warp_sum(s);
  if (lane == 0) loss[r] = (tg == ignore_index || tg < 0 || tg >= n_vocab) ? 0.f : (logf(s) + mx - row[tg]);
}
}  // namespace vb

VB_API int vb_cross_entropy(const float *logits, int64_t ld_logits, const int64_t *targets, int64_t n_rows,
                            int n_vocab, int64_t ignore_index, float *loss, vb_stream_t stream) {
  if (n_rows == 0) return VB_OK;
  const int wpb = 4;
  vb::cross_entropy_kernel<<<(unsigned)((n_rows + wpb - 1) / wpb), wpb * 32, 0, (cudaStream_t)stream>>>(
      logits, ld_logits, targets, n_rows, n_vocab, ignore_index, loss);
  VB_LAUNCH_CHECK();
  return VB_OK;
}
