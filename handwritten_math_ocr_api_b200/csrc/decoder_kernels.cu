// Non-GEMM kernels of the Transformer decoder (sm_100a): token+position embedding, teacher-forced attention,
// the on-device bookkeeping before and after a greedy decode, and the merge of the scoring partials.
// Follows /root/reference/src/model_swin.py:72-88 and torch.nn.TransformerDecoderLayer
// (post-LN; MultiheadAttention: 8 heads x 32, scores scaled by 1/sqrt(32), causal -inf mask).
#include "gemm.cuh"
#include "kernels.cuh"

namespace hmocr {
namespace {

constexpr int HD = 32;
constexpr float ATT_SCALE = 0.17677669529663687f;   // 1/sqrt(32)

__device__ __forceinline__ void load_row32(const h16* p, float (&out)[HD]) {
  const uint4* p4 = reinterpret_cast<const uint4*>(p);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const uint4 u = p4[c];
    float2 a = unpack16(u.x), b = unpack16(u.y), cc = unpack16(u.z), d = unpack16(u.w);
    out[8 * c] = a.x; out[8 * c + 1] = a.y; out[8 * c + 2] = b.x; out[8 * c + 3] = b.y;
    out[8 * c + 4] = cc.x; out[8 * c + 5] = cc.y; out[8 * c + 6] = d.x; out[8 * c + 7] = d.y;
  }
}

// Warp-cooperative single-query attention over `n` keys (n <= 32*MAXK).
//   q      : the query (already scaled), replicated in every lane
//   K(j)/V(j): pointer to the 32 fp16 of key/value j
// Lane l scores keys l, l+32, ...; softmax by warp shuffles; lane d then accumulates output
// channel d (coalesced 64-byte V rows).  Returns out[d] in lane d.
constexpr int MAXK = 8;   // up to 256 keys
template <class KF, class VF>
__device__ __forceinline__ float warp_attend(const float (&q)[HD], int n, KF K, VF V, int lane) {
  float sc[MAXK];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < MAXK; ++i) {
    const int j = lane + 32 * i;
    sc[i] = -INFINITY;
    if (j < n) {
      float kr[HD];
      load_row32(K(j), kr);
      float a = 0.f;
#pragma unroll
      for (int d = 0; d < HD; ++d) a = fmaf(q[d], kr[d], a);
      sc[i] = a;
      mx = fmaxf(mx, a);
    }
  }
  mx = warp_max(mx);
  float den = 0.f;
#pragma unroll
  for (int i = 0; i < MAXK; ++i) {
    const int j = lane + 32 * i;
    sc[i] = (j < n) ? __expf(sc[i] - mx) : 0.f;
    den += sc[i];
  }
  den = warp_sum(den);
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < MAXK; ++i) {
    const int base = 32 * i;
    if (base < n) {                      // warp-uniform
      const int cnt = min(32, n - base);
      for (int jj = 0; jj < cnt; ++jj) {
        const float p = __shfl_sync(0xffffffffu, sc[i], jj);
        acc = fmaf(p, __half2float(V(base + jj)[lane]), acc);
      }
    }
  }
  return acc / den;
}

__global__ void __launch_bounds__(256) embed_kernel(const int64_t* __restrict__ tok, int ld_tok, int rows, int T,
                                                    const float* __restrict__ emb, const float* __restrict__ pos,
                                                    int d, int vocab, float* __restrict__ x32,
                                                    h16* __restrict__ x16) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  const int b = r / T, t = r % T;
  long long id = tok[(size_t)b * ld_tok + t];
  if (id < 0 || id >= vocab) id = 0;     // torch would raise; the Python wrapper validates first
  for (int c = lane * 4; c < d; c += 128) {
    const float4 e = *reinterpret_cast<const float4*>(emb + (size_t)id * d + c);
    const float4 p = *reinterpret_cast<const float4*>(pos + (size_t)t * d + c);
    const float4 y = make_float4(e.x + p.x, e.y + p.y, e.z + p.z, e.w + p.w);
    *reinterpret_cast<float4*>(x32 + (size_t)r * d + c) = y;
    *reinterpret_cast<uint2*>(x16 + (size_t)r * d + c) = make_uint2(pack16(y.x, y.y), pack16(y.z, y.w));
  }
}

// ---- teacher-forced attention ----------------------------------------------------------------
__global__ void __launch_bounds__(256) prefill_self_kernel(const h16* __restrict__ qkv, int B, int T,
                                                           int nhead, int causal, h16* __restrict__ ctx) {
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= B * T * nhead) return;
  const int lane = threadIdx.x & 31;
  const int h = w % nhead, t = (w / nhead) % T, b = w / (nhead * T);
  const int d = nhead * HD, pitch = 3 * d;
  float q[HD];
  load_row32(qkv + (size_t)(b * T + t) * pitch + h * HD, q);
#pragma unroll
  for (int i = 0; i < HD; ++i) q[i] *= ATT_SCALE;
  const h16* kb = qkv + (size_t)b * T * pitch + d + h * HD;
  const h16* vb = kb + d;
  const float o = warp_attend(
      q, causal ? t + 1 : T, [&](int j) { return kb + (size_t)j * pitch; }, [&](int j) { return vb + (size_t)j * pitch; }, lane);
  ctx[(size_t)(b * T + t) * d + h * HD + lane] = to_h16(o);
}

__global__ void __launch_bounds__(256) cross_kernel(const h16* __restrict__ q16,
                                                    const h16* __restrict__ memkv, int ld_mem, int koff,
                                                    int voff, int rows, int T, int S, int nhead, h16* __restrict__ ctx) {
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= rows * nhead) return;
  const int lane = threadIdx.x & 31;
  const int h = w % nhead, r = w / nhead;       // r = b*T + t
  const int d = nhead * HD;
  const int img = r / T;
  float q[HD];
  load_row32(q16 + (size_t)r * d + h * HD, q);
#pragma unroll
  for (int i = 0; i < HD; ++i) q[i] *= ATT_SCALE;
  const h16* kb = memkv + (size_t)img * S * ld_mem + koff + h * HD;
  const h16* vb = memkv + (size_t)img * S * ld_mem + voff + h * HD;
  const float o = warp_attend(
      q, S, [&](int j) { return kb + (size_t)j * ld_mem; }, [&](int j) { return vb + (size_t)j * ld_mem; }, lane);
  ctx[(size_t)r * d + h * HD + lane] = to_h16(o);
}

__global__ void init_decode_kernel(DecodeState* state, int64_t* tokens, int ld_tok, int rows, int sos, int pad,
                                   uint8_t* finished, float* logprob, int max_len) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) { state->step = 0; state->finished_count = 0; state->steps_executed = 0; state->last_eos = 0; }
  if (i < rows) finished[i] = 0;
  const int total = rows * ld_tok;
  for (int k = i; k < total; k += gridDim.x * blockDim.x) tokens[k] = (k % ld_tok == 0) ? sos : pad;
  if (logprob != nullptr)
    for (int k = i; k < rows * max_len; k += gridDim.x * blockDim.x) logprob[k] = 0.f;
}

__global__ void finalize_decode_kernel(const DecodeState* state, int64_t* tokens, int ld_tok, int rows, int max_len,
                                       int pad, float* logprob, int32_t* steps_out) {
  const int steps = state->steps_executed > 0 ? state->steps_executed : min(state->step, max_len);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0 && steps_out != nullptr) *steps_out = steps;
  const int total = rows * ld_tok;
  for (int k = i; k < total; k += gridDim.x * blockDim.x) {
    const int c = k % ld_tok;
    if (c > steps) tokens[k] = pad;
  }
  if (logprob != nullptr)
    for (int k = i; k < rows * max_len; k += gridDim.x * blockDim.x)
      if (k % max_len >= steps) logprob[k] = 0.f;
}

__global__ void copy_logits_kernel(const float* __restrict__ src, int ld, size_t total, int n_valid,
                                   float* __restrict__ dst) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / n_valid;
    const int c = (int)(i - r * n_valid);
    dst[i] = src[r * ld + c];
  }
}

__global__ void f32_to_f16_kernel(const float* __restrict__ src, size_t n, h16* __restrict__ dst) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    dst[i] = to_h16(src[i]);
}

// ---- detokenise / pack ---------------------------------------------------------------------------------
// What src/inference.py:29-40 does per sequence in Python (skip sos and pad wherever they occur, stop at the first
// eos) as one warp per row: the ids that survive are written, in order, to packed[row, 0..len) and their count to
// lengths[row]; the host then does ONE join per sequence instead of B x T dictionary look-ups behind .item() syncs.
__global__ void __launch_bounds__(256) pack_tokens_kernel(const int64_t* __restrict__ tok, int rows, int ld_tok, int sos,
                                                          int eos, int pad, int32_t* __restrict__ lengths,
                                                          int32_t* __restrict__ packed) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  const int64_t* row = tok + (size_t)r * ld_tok;
  int32_t* out = packed + (size_t)r * ld_tok;
  int n = 0;
  for (int base = 0; base < ld_tok; base += 32) {
    const int i = base + lane;
    const long long id = i < ld_tok ? row[i] : (long long)eos;          // past the end behaves like eos
    const unsigned is_eos = __ballot_sync(0xffffffffu, id == eos);
    const int stop = is_eos ? __ffs(is_eos) - 1 : 32;                   // first eos of this chunk
    const bool keep = lane < stop && id != sos && id != pad;
    const unsigned km = __ballot_sync(0xffffffffu, keep);
    if (keep) out[n + __popc(km & ((1u << lane) - 1u))] = (int32_t)id;
    n += __popc(km);
    if (is_eos) break;
  }
  for (int i = n + lane; i < ld_tok; i += 32) out[i] = pad;
  if (lane == 0) lengths[r] = n;
}

// ---- teacher-forced scoring: merge the log-sum-exp partials of gemm_f16_lse -----------------------
struct LseAcc {
  float m, s, tv, bv;
  int bi;
};

__device__ __forceinline__ void lse_merge(LseAcc& a, const LseAcc& b) {
  const float mn = fmaxf(a.m, b.m);
  if (mn != -INFINITY) a.s = a.s * expf(a.m - mn) + b.s * expf(b.m - mn);
  a.m = mn;
  a.tv = fmaxf(a.tv, b.tv);                                     // only one partial holds the target
  if (b.bv > a.bv || (b.bv == a.bv && b.bi < a.bi)) { a.bv = b.bv; a.bi = b.bi; }
}

constexpr int SCORE_THREADS = 512;
constexpr int SCORE_MAX_T = 256;

// One block per sequence b, one warp per position t (strided).  Lane i merges partials i, i + 32, ... in that order,
// then a fixed shuffle tree merges the lanes.  Position t scores tokens[b, t+1]; positions after the first eos among
// columns 1..T are 0 / pad and are not merged at all.  Thread 0 sums the row in position order.
__global__ void __launch_bounds__(SCORE_THREADS) score_combine_kernel(const LsePartial* __restrict__ parts, int num_parts,
                                                                      const int64_t* __restrict__ tokens, int ld_tok,
                                                                      int T, int eos, int pad,
                                                                      float* __restrict__ logprob,
                                                                      float* __restrict__ score,
                                                                      int32_t* __restrict__ argmax) {
  __shared__ float s_lp[SCORE_MAX_T];
  __shared__ int s_last;                                         // last scored position
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_last = T - 1;
  __syncthreads();
  if (tid < T && tokens[(size_t)b * ld_tok + tid + 1] == eos) atomicMin(&s_last, tid);
  __syncthreads();
  const int last = s_last;
  for (int t = warp; t < T; t += SCORE_THREADS / 32) {
    const size_t o = (size_t)b * T + t;
    if (t > last) {
      if (lane == 0) {
        s_lp[t] = 0.f;
        if (logprob != nullptr) logprob[o] = 0.f;
        if (argmax != nullptr) argmax[o] = pad;
      }
      continue;
    }
    LseAcc a{-INFINITY, 0.f, -INFINITY, -INFINITY, 0x7fffffff};
    const LsePartial* pr = parts + o * num_parts;
    for (int p = lane; p < num_parts; p += 32) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(pr + p));
      const int bi = __ldg(&pr[p].best_idx);
      lse_merge(a, LseAcc{x.x, x.y, x.z, x.w, bi});
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      LseAcc other;
      other.m = __shfl_down_sync(0xffffffffu, a.m, off);
      other.s = __shfl_down_sync(0xffffffffu, a.s, off);
      other.tv = __shfl_down_sync(0xffffffffu, a.tv, off);
      other.bv = __shfl_down_sync(0xffffffffu, a.bv, off);
      other.bi = __shfl_down_sync(0xffffffffu, a.bi, off);
      if (lane < off) lse_merge(a, other);
    }
    if (lane == 0) {
      const float lp = a.tv - (a.m + logf(a.s));
      s_lp[t] = lp;
      if (logprob != nullptr) logprob[o] = lp;
      if (argmax != nullptr) argmax[o] = a.bi;
    }
  }
  __syncthreads();
  if (tid == 0 && score != nullptr) {
    float acc = 0.f;
    for (int t = 0; t < T; ++t) acc += s_lp[t];
    score[b] = acc;
  }
}

inline int grid_for(size_t n, int block) {
  size_t g = (n + block - 1) / block;
  if (g > 148 * 16) g = 148 * 16;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

int embed_tokens(cudaStream_t st, const int64_t* tok, int ld_tok, int B, int T, const float* emb, const float* pos,
                 int d, int vocab, float* x32, h16* x16) {
  HM_CHECK(d % 4 == 0, "embed: d_model must be a multiple of 4");
  const int rows = B * T;
  embed_kernel<<<ceil_div(rows, 8), 256, 0, st>>>(tok, ld_tok, rows, T, emb, pos, d, vocab, x32, x16);
  HM_LAUNCHED();
  return 0;
}

int mha_prefill_self(cudaStream_t st, const h16* qkv16, int B, int T, int nhead, h16* ctx16, bool causal) {
  HM_CHECK(T <= 32 * MAXK, "attention: T=%d exceeds %d", T, 32 * MAXK);
  if (!causal) return mha_full_mma(st, qkv16, B, T, nhead, ctx16);
  prefill_self_kernel<<<ceil_div(B * T * nhead, 8), 256, 0, st>>>(qkv16, B, T, nhead, causal ? 1 : 0, ctx16);
  HM_LAUNCHED();
  return 0;
}

int mha_prefill_cross(cudaStream_t st, const h16* q16, const h16* memkv, int ld_mem, int koff,
                      int voff, int B, int T, int S, int nhead, h16* ctx16) {
  HM_CHECK(S <= 32 * MAXK, "attention: S=%d exceeds %d", S, 32 * MAXK);
  cross_kernel<<<ceil_div(B * T * nhead, 8), 256, 0, st>>>(q16, memkv, ld_mem, koff, voff, B * T, T, S, nhead, ctx16);
  HM_LAUNCHED();
  return 0;
}

int init_decode(cudaStream_t st, DecodeState* state, int64_t* tokens, int ld_tok, int rows, int sos, int pad,
                uint8_t* finished, float* logprob, int max_len) {
  init_decode_kernel<<<grid_for((size_t)rows * ld_tok, 256), 256, 0, st>>>(state, tokens, ld_tok, rows, sos, pad,
                                                                          finished, logprob, max_len);
  HM_LAUNCHED();
  return 0;
}

int finalize_decode(cudaStream_t st, const DecodeState* state, int64_t* tokens, int ld_tok, int rows, int max_len,
                    int pad, float* logprob, int32_t* steps_out) {
  finalize_decode_kernel<<<grid_for((size_t)rows * ld_tok, 256), 256, 0, st>>>(state, tokens, ld_tok, rows, max_len,
                                                                              pad, logprob, steps_out);
  HM_LAUNCHED();
  return 0;
}

int copy_logits(cudaStream_t st, const float* src, int ld, int rows, int n_valid, float* dst) {
  const size_t total = (size_t)rows * n_valid;
  copy_logits_kernel<<<grid_for(total, 256), 256, 0, st>>>(src, ld, total, n_valid, dst);
  HM_LAUNCHED();
  return 0;
}

int score_combine(cudaStream_t st, const LsePartial* parts, int num_parts, const int64_t* tokens, int ld_tok, int B,
                  int T, int eos, int pad, float* logprob, float* score, int32_t* argmax) {
  HM_CHECK(T >= 1 && T <= SCORE_MAX_T, "score: T=%d outside [1, %d]", T, SCORE_MAX_T);
  score_combine_kernel<<<B, SCORE_THREADS, 0, st>>>(parts, num_parts, tokens, ld_tok, T, eos, pad, logprob, score,
                                                    argmax);
  HM_LAUNCHED();
  return 0;
}

int f32_to_f16(cudaStream_t st, const float* src, size_t n, h16* dst) {
  f32_to_f16_kernel<<<grid_for(n, 256), 256, 0, st>>>(src, n, dst);
  HM_LAUNCHED();
  return 0;
}

int pack_tokens(cudaStream_t st, const int64_t* tokens, int rows, int ld_tok, int sos, int eos, int pad, int32_t* lengths,
                int32_t* packed) {
  pack_tokens_kernel<<<ceil_div(rows, 8), 256, 0, st>>>(tokens, rows, ld_tok, sos, eos, pad, lengths, packed);
  HM_LAUNCHED();
  return 0;
}

}  // namespace hmocr
