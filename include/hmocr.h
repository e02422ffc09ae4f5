/*
 * libhmocr - C ABI of the B200-native image-to-LaTeX engine (sm_100a only, no CPU fallback).
 *
 * The reference (PTD504/handwritten-math-ocr-api) is pure Python and has no FFI; the boundary it
 * offers for this path is the nn.Module surface of `FormulaRecognitionModel`
 * (/root/reference/src/model_swin.py:91-101) and the three greedy drivers built on it.  Each entry
 * point below names the reference interface it replaces; the Python mirror that binds them with
 * ctypes is `handwritten_math_ocr_api_b200/` (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, a negative code on failure; the message is available
 *     from hmocr_last_error() (thread local).  Nothing falls back to another implementation.
 *   - pointers named *_dev are CUDA device pointers owned by the caller (torch tensors on the
 *     Python side); *_host are host pointers.  `stream` is a cudaStream_t passed as void*.
 *     All work is enqueued on that stream; only the *_host entry points synchronise.
 *   - the engine owns its weights (one arena, allocated by hmocr_finalize_weights).  Scratch memory is the CALLER's
 *     when hmocr_set_workspace has been called (one buffer sized by hmocr_workspace_bytes - a torch tensor on the
 *     Python side - inside which the engine places its named buffers; it then allocates nothing); otherwise the
 *     engine takes scratch from the CUDA stream-ordered allocator on the caller's stream (no device-wide sync).
 *   - one engine = one CUDA device (current device at hmocr_create); not thread-safe per handle.
 */
#ifndef HMOCR_H_
#define HMOCR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hmocr_engine hmocr_engine;

/* Hyper-parameters read from the reference's `config` singleton
 * (/root/reference/src/config.py:16-47, /root/reference/app/src/config.py:22-57). */
typedef struct hmocr_config {
  int32_t vocab_size;      /* len(vocab); 5075 in the reference's MLflow run                   */
  int32_t d_model;         /* config.d_model          = 256                                    */
  int32_t nhead;           /* config.nhead            = 8   (head_dim must be 32)              */
  int32_t dim_feedforward; /* config.dim_feedforward  = 512                                    */
  int32_t num_layers;      /* config.swin_num_decoder_layers / num_decoder_layers = 8          */
  int32_t max_seq_len;     /* config.max_seq_len      = 150 (size of pos_encoder / tgt_mask)   */
  int32_t sos_id, eos_id, pad_id; /* vocab['<sos>'], vocab['<eos>'], vocab['<pad>'] = 1, 2, 0  */
  int32_t encoder_arch;    /* 0 = Swin-T (src/model_swin.py, 30 memory tokens);
                              1 = ResNet-18 + TransformerEncoder (src/model_res18trans.py, 10 memory tokens) */
  int32_t enc_num_layers;  /* encoder_arch 1: config.res18trans_num_encoder_layers (src/config.py:28);
                              0 = same as num_layers                                              */
} hmocr_config;

enum { HMOCR_F32 = 0, HMOCR_I64 = 1 };

const char* hmocr_last_error(void);
const char* hmocr_version(void);
/* kernels launched by this library on the calling thread since load (bench.py "gpu_launches") */
int64_t hmocr_launch_count(void);

/* FormulaRecognitionModel(vocab_size)            /root/reference/src/model_swin.py:91-95 */
int hmocr_create(const hmocr_config* cfg, hmocr_engine** out);
void hmocr_destroy(hmocr_engine* e);

/* model.load_state_dict(sd): one call per state-dict entry, reference key names and shapes
 * (/root/reference/src/predict.py:28-29; layout in SURVEY.md section 8b).  `data_host` is fp32 or int64
 * host memory; the engine converts / repacks and uploads.  Unknown or unused keys
 * (encoder.swin.norm.*, encoder.swin.head.*, decoder.tgt_mask, the encoder.swin.features.*
 * aliases) are accepted and ignored.  hmocr_finalize_weights fails if a needed entry is missing. */
int hmocr_load_weight(hmocr_engine* e, const char* key, const void* data_host, const int64_t* shape, int ndim,
                      int dtype);
int hmocr_finalize_weights(hmocr_engine* e);

/* Engine options (all have working defaults):
 *   "steps_per_launch"  decode steps per persistent-kernel launch; 0 (default) = automatic: one launch for the whole
 *                       decode when all clusters of the batch are co-resident (the kernel stops by itself once every
 *                       row has emitted eos), 16-step launches with a host poll in between for multi-wave batches
 *   "encoder_graph"     1 (default) = hmocr_generate* replay the encoder's ~95 kernels as one captured CUDA graph for
 *                       batches of up to 1024 images (GPU-side gain in the launch-bound regime of <= 32 images, host-side
 *                       gain beyond; first call at a batch size runs eagerly, the second captures); 0 = always launch
 *                       kernel by kernel
 *   "conv_impl"         ResNet-18 variant: 0 = convolutions as implicit GEMMs, the patches built by 4-D TMA
 *                       loads (default); 1 = explicit im2col matrix + GEMM (kept for A/B tests)
 *   "mlp_fused"         Swin stages 1 / 2: 1 (default) = fc1 + GELU + fc2 + residual in one kernel, the hidden tile in
 *                       TMEM / shared memory (hmocr_swin_mlp); 0 = two GEMM launches with the hidden tensor in HBM
 *                       (kept for A/B tests) */
int hmocr_set_option(hmocr_engine* e, const char* name, int value);
/* Developer aid: with option "trace_step" = t >= 0 the persistent decode kernel records clock64()
 * of (cluster 0, CTA 0, thread 0) at every phase boundary of decode step t; this copies the first
 * n (<= 1024) stamps to the host (profiles/ phase breakdowns come from here). */
int hmocr_read_trace(hmocr_engine* e, int64_t* out_host, int n);

/* ResNet-18 variant only: the positional table added to the 10 pooled tokens.  The reference creates a fresh
 * N(0,1)-initialised nn.Embedding(10, d_model) on EVERY encoder call (src/model_res18trans.py:57-59), so the
 * table is an input here: pos_host f32 [10, d_model].  Used by the following hmocr_encode / hmocr_generate calls. */
int hmocr_set_pos_table(hmocr_engine* e, const float* pos_host, int rows, int d, void* stream);

/* Scratch memory owned by the caller (SURVEY.md section 8b "Ownership"; the reference has no counterpart - its
 * activations live in torch's caching allocator, which is where this buffer comes from on the Python side).
 *   hmocr_workspace_bytes: bytes of scratch that hmocr_encode + hmocr_generate* (device and host-buffer forms) need
 *     for `batch` images, `max_len` steps and `beam` hypotheses with the engine's current options; beam == 0 asks for
 *     the teacher-forced hmocr_decoder_forward(batch, T = max_len) instead, beam < 0 for hmocr_generate_nbest with
 *     -beam hypotheses.  The engine remembers the per-buffer
 *     maximum over all shapes asked so far, and *bytes covers ALL of them (ask once per shape you will use, pass the
 *     last answer to hmocr_set_workspace).
 *   hmocr_set_workspace: hand the engine one device buffer (256-byte aligned).  It stays the caller's; it must
 *     outlive every call that uses it; calling again (larger buffer) or with NULL (back to engine-owned scratch)
 *     drops all placements - stream-ordered on `stream`.  A call whose buffers do not fit fails with a message
 *     naming the buffer; nothing is allocated behind the caller's back.  The image staging of
 *     hmocr_preprocess_image_u8 / _cv2_u8 is sized by the image, not by (batch, max_len, beam): always engine-owned. */
int hmocr_workspace_bytes(hmocr_engine* e, int batch, int max_len, int beam, size_t* bytes);
int hmocr_set_workspace(hmocr_engine* e, void* workspace_dev, size_t bytes, void* stream);

/* How many 8-CTA decode clusters (16 sequences each) can be co-resident on the current device. */
int hmocr_decode_max_clusters(int* out);

/* model.encoder(images)                          /root/reference/src/model_swin.py:39-46
 * images_dev f32 [B,1,96,320] -> enc_out_dev f32 [B,30,d_model] */
int hmocr_encode(hmocr_engine* e, const float* images_dev, int batch, float* enc_out_dev, void* stream);

/* model.decoder(encoder_out, tgt)                /root/reference/src/model_swin.py:72-88
 * enc_out_dev f32 [B,30,d], tgt_dev int64 [B,T] -> logits_dev f32 [B,T,V] (all T positions) */
int hmocr_decoder_forward(hmocr_engine* e, const float* enc_out_dev, const int64_t* tgt_dev, int batch, int T,
                          float* logits_dev, void* stream);

/* The greedy loops of /root/reference/src/inference.py:15-25, src/predict.py:56-65 and
 * app/src/im2latex.py:20-45 as ONE call: encoder once, KV-cached decode, argmax / beam top-k and
 * the winner's log-softmax on device.
 *   tokens_dev   int64 [B, 1+max_len]  column 0 = sos; columns past *steps are pad
 *   logprob_dev  f32   [B, max_len]    log_softmax(logits)[token] per emitted position (may be NULL)
 *   steps_dev    int32 [1]             number of decode steps executed = ys.shape[1]-1 of the
 *                                      reference (stops when every row has emitted eos)
 * beam == 1: greedy, finished rows keep decoding exactly as the reference does.
 * beam  > 1: beam search (2..5 hypotheses per image) as defined in DESIGN.md section 4.5 - the reference
 *            has none, `beam_size` is an unused parameter of src/inference.py:7; tokens are the best
 *            hypothesis per image (finished hypotheses are padded), score_dev f32 [B] its summed
 *            log-probability (may be NULL); logprob_dev is zero-filled.  beam must not exceed vocab_size (a
 *            step keeps `beam` distinct tokens per hypothesis); a larger beam fails with a message. */
int hmocr_generate(hmocr_engine* e, const float* images_dev, int batch, int max_len, int beam, int64_t* tokens_dev,
                   float* logprob_dev, int32_t* steps_dev, float* score_dev, void* stream);

/* Same, starting from encoder output already in HBM (src/inference.py:13 split from :15-25). */
int hmocr_generate_from_memory(hmocr_engine* e, const float* enc_out_dev, int batch, int max_len, int beam,
                               int64_t* tokens_dev, float* logprob_dev, int32_t* steps_dev, float* score_dev,
                               void* stream);

/* The n best hypotheses of a beam search, ranked, with per-token log-probabilities ("did you mean ..." alternatives).
 * Always runs the beam-search machinery, 1 <= beam <= 5 (beam == 1 runs it with one hypothesis: the greedy sequence,
 * padded after eos, with its score and per-token log-probabilities), beam <= vocab_size; 1 <= n_best <= beam,
 * otherwise the call fails with a message.
 *   input_dev     images f32 [B,1,96,320] (input_is_memory == 0) or encoder output f32 [B,mem_tokens,d_model] (!= 0)
 *   tokens_dev    int64 [B, n_best, 1+max_len]  hypotheses by score, highest first (ties -> lower beam index, so rank 0
 *                                               is exactly what hmocr_generate returns); column 0 = sos, pad after a
 *                                               hypothesis' eos and past *steps
 *   logprob_dev   f32   [B, n_best, max_len]    log_softmax of each emitted token, 0 after eos and past *steps
 *                                               (may be NULL)
 *   score_dev     f32   [B, n_best]             summed log-probability = the fp32 sum of the row of logprob_dev in step
 *                                               order (may be NULL)
 *   steps_dev     int32 [1]                     decode steps executed (may be NULL)
 * The workspace of a call with `beam` hypotheses is sized by hmocr_workspace_bytes(batch, max_len, -beam). */
int hmocr_generate_nbest(hmocr_engine* e, const float* input_dev, int input_is_memory, int batch, int max_len, int beam,
                         int n_best, int64_t* tokens_dev, float* logprob_dev, float* score_dev, int32_t* steps_dev,
                         void* stream);

/* Teacher-forced scoring of given token sequences ("how likely is this formula for this image").
 *   input_dev   images f32 [B,1,96,320] (input_is_memory == 0) or encoder output f32 [B,mem_tokens,d_model] (!= 0)
 *   tokens_dev  int64 [B, 1+T], 1 <= T <= max_seq_len, ids in [0, vocab_size).  Column 0 is the first decoder input
 *               (sos in normal use); columns 1..T are the scored tokens, the same layout hmocr_generate returns.
 *   logprob_dev f32   [B, T]  log_softmax(logits at position t)[tokens[b, t+1]] up to and including the row's first
 *                             eos among columns 1..T; 0 after it.  A row without eos is scored over all T.  (may be NULL)
 *   score_dev   f32   [B]     fp32 sum of the row of logprob in position order, the same definition as
 *                             hmocr_generate_nbest's score (may be NULL)
 *   argmax_dev  int32 [B, T]  the model's most likely token at each position given the row's prefix, ties -> lowest
 *                             index (the greedy rule); pad_id after the first eos (may be NULL)
 * At least one output is non-NULL.  Ids after a row's first eos do not affect that row's outputs.
 * The images form runs the encoder as hmocr_generate does (ResNet-18 variant: with the hmocr_set_pos_table table).
 * The logits are never stored: fc_out runs with a log-sum-exp epilogue that keeps per-row partials of 128 columns,
 * so a row's results do not depend on the batch it is scored in (DESIGN.md section 4.9). */
int hmocr_score(hmocr_engine* e, const float* input_dev, int input_is_memory, int batch, int T,
                const int64_t* tokens_dev, float* logprob_dev, float* score_dev, int32_t* argmax_dev, void* stream);

/* Workspace of hmocr_score(batch, T), both input forms.  It shares the per-buffer maximum with
 * hmocr_workspace_bytes, so the last answer of either function covers every shape asked of both. */
int hmocr_score_workspace_bytes(hmocr_engine* e, int batch, int T, size_t* bytes);

/* End-to-end form with HOST buffers (what `predict(images, model, vocab, idx2char, device)` does
 * around the model: images.to(device) ... ids back on the host): pinned or pageable host memory
 * in, host memory out, H2D and D2H inside, synchronises before returning. */
int hmocr_generate_host(hmocr_engine* e, const float* images_host, int batch, int max_len, int beam,
                        int64_t* tokens_host, float* logprob_host, int32_t* steps_host, float* score_host,
                        void* stream);

/* The reference's whole image transform on the GPU, bit-identical to PIL + torchvision
 * (/root/reference/app/src/preprocess.py:6-16: Grayscale(1) -> Resize((96,320)) -> ToTensor -> Normalize(0.5,0.5)):
 * image_host uint8 [height, width, channels] dense, channels 1 (PIL mode "L") or 3 (mode "RGB", converted with
 * Pillow's integer luma); PIL's antialiased bilinear resample (two passes, 22-bit fixed-point coefficients, uint8
 * intermediate) -> image_dev f32 [1,96,320] (one slot of a [B,1,96,320] batch).  Any image size up to 16384^2.
 * The copy of the pixels is stream-ordered; image_host may be pageable (then the call returns after staging it). */
int hmocr_preprocess_image_u8(hmocr_engine* e, const uint8_t* image_host, int channels, int height, int width,
                              float* image_dev, void* stream);

/* The training / evaluation loader's preprocessing on the GPU, bit-identical to OpenCV + torchvision
 * (/root/reference/src/data_loader.py:31-35: cv2.resize(gray, (320, 96)) [INTER_LINEAR] -> ToTensor -> Normalize):
 * gray_host uint8 [height, width] (what cv2.imread(IMREAD_GRAYSCALE) returns) -> image_dev f32 [1,96,320]. */
int hmocr_preprocess_cv2_u8(hmocr_engine* e, const uint8_t* gray_host, int height, int width, float* image_dev,
                            void* stream);

/* Detokenise on the device (the Python loop of /root/reference/src/inference.py:29-40): for every row of
 * tokens int64 [rows, ld_tok] drop sos and pad ids wherever they occur, stop at the first eos, and write the
 * surviving ids in order to packed int32 [rows, ld_tok] (tail filled with pad) and their count to lengths int32 [rows].
 * The host then needs one D2H copy and one join per sequence. */
int hmocr_pack_tokens(hmocr_engine* e, const int64_t* tokens_dev, int rows, int ld_tok, int32_t* lengths_dev,
                      int32_t* packed_dev, void* stream);

/* The tail of the reference's preprocessing on the device: ToTensor + Normalize(0.5, 0.5)
 * (/root/reference/app/src/preprocess.py:7-12, src/predict.py:36-41) of grayscale uint8 images that are already
 * 96 x 320: images_u8_dev uint8 [B,96,320] -> images_dev f32 [B,1,96,320] = (u/255 - 0.5)/0.5, bit-identical to
 * torchvision (the PIL resize stays on the host). */
int hmocr_preprocess_u8(hmocr_engine* e, const uint8_t* images_u8_dev, int batch, float* images_dev, void* stream);

/* hmocr_generate_host with uint8 images (4x less host-to-device traffic): H2D, preprocess, generate, D2H, sync. */
int hmocr_generate_host_u8(hmocr_engine* e, const uint8_t* images_u8_host, int batch, int max_len, int beam,
                           int64_t* tokens_host, float* logprob_host, int32_t* steps_host, float* score_host,
                           void* stream);

/* Decode steps the persistent kernel actually EXECUTED in the last hmocr_generate* call on this engine (valid after the
 * stream has been synchronised).  The reference's loop breaks right after the step at which the last row emits its
 * first eos (src/inference.py:23-25); the kernel leaves its step loop on the device - one step after that, not at the
 * end of the launch - so this is `steps` + 1 or 2, not `steps` rounded up to two launches. */
int hmocr_last_decode_steps(hmocr_engine* e, int32_t* steps_run);

/* Phase timings of the last hmocr_generate* call on this engine, measured with CUDA events on
 * the caller's stream (valid after the stream has been synchronised): encoder ms, decode ms. */
int hmocr_last_timings(hmocr_engine* e, float* encoder_ms, float* decode_ms);

/* ---- individual kernels, exported for the unit tests ------------------------------------- */

/* nn.Linear (+ fused epilogue): out = LN?( act(A W^T + bias) + residual )
 * A fp16 [M,K] pitch lda, W fp16 [N,K]; act 0 none / 1 GELU(erf) / 2 ReLU; any of bias, residual,
 * out_f32, out_f16, ln_gamma/ln_beta may be NULL.  force_bn 0 = automatic tile width. */
int hmocr_gemm_f16(const void* a_dev, int lda, int M, int K, const void* w_dev, int N, const float* bias_dev,
                    int act, const float* residual_dev, int ldr, float* out_f32_dev, int ld32, void* out_f16_dev,
                    int ld16, const float* ln_gamma_dev, const float* ln_beta_dev, int force_bn, void* stream);

/* MLP of a Swin block fused with its residual add (torchvision swin_transformer.py:444, 455):
 * x <- x + fc2(GELU(fc1(xn))), xn fp16 [M,C] (= norm2(x)), w1 fp16 [4C,C], w2 fp16 [C,4C], x f32 [M,C] in place.
 * C in {96, 192} (Swin-T stages 1 and 2); the hidden tile stays in TMEM / shared memory. */
int hmocr_swin_mlp(const void* xn_dev, int M, int C, const void* w1_dev, const float* b1_dev, const void* w2_dev,
                   const float* b2_dev, float* x_dev, void* stream);

/* nn.LayerNorm over the last axis: x f32 [rows, C] -> fp16 and/or f32 */
int hmocr_layernorm(const float* x_dev, int rows, int C, const float* gamma_dev, const float* beta_dev,
                    void* out_f16_dev, float* out_f32_dev, void* stream);

/* features[0]: Conv2d(1,96,4,4) + Permute + LayerNorm(96)   (swin_transformer.py:556-562)
 * images f32 [B,1,96,320] -> x f32 [B,24,80,96] */
int hmocr_patch_embed(const float* images_dev, int batch, const float* conv_w_dev, const float* conv_b_dev,
                      const float* ln_g_dev, const float* ln_b_dev, float* x_dev, void* stream);

/* PatchMerging gather + LayerNorm(4C)            (swin_transformer.py:35-43, 84)
 * x f32 [B,H,W,C] -> fp16 [B,H/2,W/2,4C] (ready for the bias-free reduction GEMM) */
int hmocr_patch_merge_ln(const float* x_dev, int batch, int H, int W, int C, const float* gamma_dev,
                         const float* beta_dev, void* out_f16_dev, void* stream);

/* torch.nn.MultiheadAttention core (head_dim 32, scale 32^-0.5) on a packed in-projection:
 *   qkv fp16 [B*T, 3*nhead*32] (row = b*T + t; q | k | v) -> ctx fp16 [B*T, nhead*32] (input of out_proj).
 * causal != 0: the teacher-forced decoder self-attention (generate_square_subsequent_mask,
 * /root/reference/src/model_swin.py:75-77); causal == 0: nn.TransformerEncoderLayer.self_attn of the ResNet-18
 * variant (/root/reference/src/model_res18trans.py:62-64), tensor-core kernel.  T <= 256. */
int hmocr_self_attention(const void* qkv_dev, int B, int T, int nhead, int causal, void* ctx_f16_dev, void* stream);

/* shifted_window_attention core (swin_transformer.py:151-214, 219-227) on a qkv buffer computed
 * for the real (un-padded, un-shifted) tokens:
 *   qkv fp16 [B*H*W, 3C] (bias included), qkv_bias f32 [3C] (value of padded tokens),
 *   rel_bias f32 [heads,49,49] (table gathered by relative_position_index), shift 0 or 3
 *   -> ctx fp16 [B*H*W, C] in original token order (input of attn.proj) */
int hmocr_window_attention(const void* qkv_dev, const float* qkv_bias_dev, const float* rel_bias_dev, int batch,
                           int H, int W, int C, int heads, int shift, void* ctx_f16_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HMOCR_H_ */
