// Internal launchers of the non-GEMM kernels (all enqueue on `st`, return 0 / negative).
#pragma once
#include "common.cuh"

namespace hmocr {

// ---- Swin encoder ------------------------------------------------------------------------------
int layernorm(cudaStream_t st, const float* x, int rows, int C, const float* gamma, const float* beta,
              h16* out16, float* out32);
int patch_merge_ln(cudaStream_t st, const float* x, int B, int H, int W, int Cin, const float* gamma,
                   const float* beta, h16* out16);
int patch_embed(cudaStream_t st, const float* images, int B, const float* w, const float* b, const float* g,
                const float* beta, float* x);
int window_attention(cudaStream_t st, const h16* qkv, const float* qkv_bias, const float* rel_bias, int B,
                     int H, int W, int C, int heads, int shift, h16* ctx);       // tensor-core (swin_attention.cu)

// fused MLP of a Swin block (swin_mlp.cu): x <- x + fc2(GELU(fc1(xn) + b1)) + b2, hidden tile kept in TMEM / shared
// memory.  xn fp16 [M, C] (= LayerNorm2(x)), w1 fp16 [4C, C], w2 fp16 [C, 4C], x fp32 [M, C] in place.  C in {96, 192}.
bool swin_mlp_supported(int C);
int swin_mlp(cudaStream_t st, const h16* xn, int M, int C, const h16* w1, const float* b1, const h16* w2,
             const float* b2, float* x);

// ---- decoder -------------------------------------------------------------------------------------
struct DecodeState {      // device-resident control block of one generate call
  int step;               // current decode step t (position of the token being fed)
  int finished_count;     // rows that have emitted eos at least once
  int steps_executed;     // ys.shape[1]-1 of the reference once every row has finished, else 0
  int last_eos;           // max over the finished rows (beam: clusters) of (step of the first eos) + 1.  Clusters of the
                          // persistent kernel run their step range independently (and in waves), so the row that
                          // finishes LAST in time is not the row that finishes at the LATEST step: steps_executed is
                          // published from this maximum, never from the publishing thread's own step.
};

// x[r] = embedding[tok[b, t]] + pos[t]  for r = b*T + t   (src/model_swin.py:73-75)
int embed_tokens(cudaStream_t st, const int64_t* tok, int ld_tok, int B, int T, const float* emb, const float* pos,
                 int d, int vocab, float* x32, h16* x16);

// teacher-forced attention over a [B*T, ...] activation buffer: one warp per (b, head, query)
//   self : q,k,v = columns [0,d),[d,2d),[2d,3d) of qkv16 (row pitch 3d), causal
//   cross: q from q16 (pitch d); k,v from memkv (row (b*S+s), pitch ld_mem, column offsets koff/voff)
int mha_prefill_self(cudaStream_t st, const h16* qkv16, int B, int T, int nhead, h16* ctx16, bool causal = true);
// non-causal, T <= 256: tensor-core kernel (swin_attention.cu); used by mha_prefill_self(causal = false)
int mha_full_mma(cudaStream_t st, const h16* qkv, int B, int T, int nhead, h16* ctx);
int mha_prefill_cross(cudaStream_t st, const h16* q16, const h16* memkv, int ld_mem, int koff,
                      int voff, int B, int T, int S, int nhead, h16* ctx16);

// one decode step, one warp per (row, head).  `mem_row` maps a decode row to its image (beam search:
// several hypotheses share one image's memory K/V); nullptr = identity.
int self_attn_step(cudaStream_t st, const DecodeState* state, const h16* qkv16, h16* kcache,
                   h16* vcache, int rows, int nhead, int tmax, h16* ctx16);
int cross_attn_step(cudaStream_t st, const h16* q16, const h16* memkv, int ld_mem, int koff,
                    int voff, const int* mem_row, int rows, int S, int nhead, h16* ctx16);

// greedy head: argmax (first max) + log-softmax of the winner over logits[rows, ld] (n_valid
// columns), append to tokens[:, t+1], update finished bookkeeping, and embed the chosen token
// for step t+1 (src/inference.py:20-24 + src/model_swin.py:73-75).
int greedy_select(cudaStream_t st, DecodeState* state, const float* logits, int ld, int n_valid, int rows,
                  int64_t* tokens, int ld_tok, float* logprob, int max_len, int eos, uint8_t* finished,
                  const float* emb, const float* pos, int d, int max_pos, float* x32, h16* x16);
int advance_step(cudaStream_t st, DecodeState* state);
// teacher-forced scoring: merge the gemm_f16_lse partials (parts [B*T][num_parts]) into logprob f32 [B, T], score f32
// [B] and argmax int32 [B, T] (each may be nullptr), masked after the first eos among tokens[b, 1..T]
struct LsePartial;
int score_combine(cudaStream_t st, const LsePartial* parts, int num_parts, const int64_t* tokens, int ld_tok, int B,
                  int T, int eos, int pad, float* logprob, float* score, int32_t* argmax);
int pack_tokens(cudaStream_t st, const int64_t* tokens, int rows, int ld_tok, int sos, int eos, int pad, int32_t* lengths,
                int32_t* packed);
int init_decode(cudaStream_t st, DecodeState* state, int64_t* tokens, int ld_tok, int rows, int sos, int pad,
                uint8_t* finished, float* logprob, int max_len);
// after the loop: columns past steps_executed -> pad / 0, steps -> int32 out
int finalize_decode(cudaStream_t st, const DecodeState* state, int64_t* tokens, int ld_tok, int rows, int max_len,
                    int pad, float* logprob, int32_t* steps_out);

// ---- ResNet-18 + TransformerEncoder encoder (resnet_kernels.cu; BASELINE.json config 4) ----------------------
int conv7x7_bn_relu(cudaStream_t st, const float* images, int B, const float* w, const float* bias, h16* out);
int maxpool3x3s2(cudaStream_t st, const h16* in, int B, int H, int W, int C, h16* out16, float* out32);
int im2col(cudaStream_t st, const h16* in, int B, int H, int W, int C, int k, int stride, int pad, h16* out);
int avgpool_h(cudaStream_t st, const float* in, int B, int H, int W, int C, h16* out);
int add_pos_permute(cudaStream_t st, const float* x, const float* pos, int B, int S, int d, float* o32, h16* o16);
int permute_back(cudaStream_t st, const float* x, int B, int S, int d, float* o32, h16* o16);

// uint8 grayscale 96x320 images -> normalised f32 (ToTensor + Normalize(0.5, 0.5)), bit-identical to torchvision
int preprocess_u8(cudaStream_t st, const uint8_t* in, size_t pixels, float* out);
// full reference transform (grayscale + PIL bilinear resize + ToTensor + Normalize), preprocess_kernels.cu
int preprocess_gray_cv2(cudaStream_t st, const uint8_t* src_dev, int H, int W, int out_h, int out_w, int* tables_dev,
                        float* out_dev);      // the loader's cv2.resize route
size_t preprocess_table_ints(int H, int W, int out_h, int out_w);
int preprocess_image(cudaStream_t st, const uint8_t* src_dev, int channels, int H, int W, int out_h, int out_w,
                     int* tables_dev, uint8_t* mid_dev, float* out_dev);

// misc
int copy_logits(cudaStream_t st, const float* src, int ld, int rows, int n_valid, float* dst);
int f32_to_f16(cudaStream_t st, const float* src, size_t n, h16* dst);

}  // namespace hmocr
