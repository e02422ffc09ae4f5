// Interface of the persistent cluster decode kernel (decode_persistent.cu).
#pragma once
#include <cuda_fp16.h>

#include "kernels.cuh"

namespace hmocr {

// Packed weight stream (fp16: same bytes as fp16, 3 more mantissa bits; values are saturated to +-65504).  One chunk = one mma m-tile of a projection: 16 weight rows (output
// features) x 256 input columns, rows padded to 264 elements so ldmatrix is bank-conflict free.
// Every chunk is one cp.async.bulk copy of DP_CHUNK bytes.
//
// wstream[cta c][chunk]: per layer (DP_LAYER_CHUNKS chunks)
//    0,1    self_attn.in_proj  q rows of head c          [c*32 + 16m ..]
//    2,3    self_attn.in_proj  k rows of head c
//    4,5    self_attn.in_proj  v rows of head c
//    6,7    self_attn.out_proj rows                      [c*32 + 16m ..]
//    8,9    multihead_attn.in_proj q rows of head c
//   10,11   multihead_attn.out_proj rows                 [c*32 + 16m ..]
//   12..15  linear1 rows                                 [c*64 + 16m ..]
//   16..19  linear2 rows [c*32 + 16m ..], input columns [256*kh .. 256*kh+255]; order (m,kh) = 00,01,10,11
// then fc_tiles chunks of fc_out: rows [c*16*fc_tiles + 16m ..] (zero rows past the vocabulary).
constexpr int DP_CH_ROWS = 16;
constexpr int DP_CHUNK = DP_CH_ROWS * 264 * 2;   // 8448 B
constexpr int DP_LAYER_CHUNKS = 20;

// The fp32 bias of every weight row travels in the padding of that row (halves 256, 257 of 264); the second
// input-half chunks of linear2 carry zeros.
constexpr int DP_ROWS = 8;          // sequences owned by one cluster (= the N of mma.m16n8k16)

struct DecPersistParams {
  const uint8_t* wstream;     // [8][chunks_per_step][DP_CHUNK]
  const float* lnparams;      // [L][6][256]: norm1.weight, norm1.bias, norm2.weight, ... norm3.bias
  const float* emb;           // [vocab][256]
  const float* pos;           // [max_pos][256]
  // fp16 caches in mma-fragment-major blocks of 32 keys x 32 dims (2048 bytes, layout in decode_persistent.cu)
  __half* kcache;             // [L][rows][8][cache_blocks][1024]
  __half* vcache;             // [L][rows][8][cache_blocks][1024]
  const __half* memk;         // [L][images][8][1024]   (mem_len <= 32 memory tokens, the other slots zero)
  const __half* memv;         // [L][images][8][1024]
  int cache_blocks;           // ceil(max_seq_len / 32)
  int mem_len;                // memory tokens per image: 30 (Swin-T) or 10 (ResNet-18 variant)
  int64_t* tokens;            // [rows][ld_tok]
  float* logprob;             // [rows][max_len] or nullptr
  uint8_t* finished;          // [rows]
  DecodeState* state;
  int rows, images, beam;     // rows = images * beam; row r reads the memory of image r / beam
  // ---- beam search (beam > 1; the reference has none - definition in oracle/decode.py::beam_search) ----
  // A cluster owns floor(8 / beam) images = rows_per_cluster rows.  The K/V caches exist twice: step t reads the
  // history of hypothesis j from set (t & 1), row bm_src[j] (its parent's row), and writes history + this step's
  // key/value to set ((t + 1) & 1), row j - the parent gather rides on the attention loads, nothing is copied
  // separately.  Per step the chosen (parent, token) of every row is recorded for the final back-track.
  int rows_per_cluster;       // 8 (greedy) or beam * (8 / beam)
  int num_clusters;
  size_t cache_set_stride;    // halves between the two cache sets (0 in greedy mode)
  float* bm_score;            // [rows] summed log-probability of each live hypothesis
  int* bm_fin;                // [rows] hypothesis has emitted eos
  int* bm_src;                // [rows] cluster-local row that holds the hypothesis' history in the current set
  int* bm_tok;                // [rows] token fed at the next step
  int* bp_parent;             // [max_len][rows] beam index (within the image) of the parent chosen at step t
  int* bp_token;              // [max_len][rows] token chosen at step t
  float* bp_logp;             // [max_len][rows] log-probability of that token (0 once frozen), or nullptr
  int num_layers, fc_tiles, chunks_per_step, vocab;
  int tmax, max_pos, max_len, ld_tok, eos, pad;
  long long* trace;           // optional: clock64() of cluster 0 / CTA 0 / thread 0 at every phase boundary
  int trace_step;             //           of decode step `trace_step`
};

int decode_persistent_init();
int decode_persistent_launch(cudaStream_t st, DecPersistParams p, int t_begin, int t_end);
int decode_persistent_max_clusters(int* out);   // co-resident clusters on this device
// memkv f32 [img*mem_len+s][l*512 + kv*256 + h*32 + d] -> the fp16 memk / memv layouts above
int repack_memkv(cudaStream_t st, const float* memkv, int images, int L, int mem_len, void* memk, void* memv);
constexpr int DP_MAX_BEAM = 5;
// beam search bookkeeping around the persistent kernel
int beam_init(cudaStream_t st, DecodeState* state, float* bm_score, int* bm_fin, int* bm_src, int* bm_tok, int rows,
              int beam, int rows_per_cluster, int sos);
// n_best best hypotheses per image (score descending, ties -> lower beam index), back-tracked through bp_parent /
// bp_token: tokens [images][n_best][1+max_len] (column 0 sos, pad past the steps executed), score_out [images][n_best],
// logprob [images][n_best][max_len] from bp_logp (0 past the steps executed).  score_out, logprob, steps_out may be null.
int beam_finalize(cudaStream_t st, const DecodeState* state, const float* bm_score, const int* bp_parent,
                  const int* bp_token, const float* bp_logp, int images, int beam, int n_best, int rows, int max_len,
                  int sos, int pad, int64_t* tokens, float* logprob, float* score_out, int32_t* steps_out);

}  // namespace hmocr
