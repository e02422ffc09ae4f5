// tcgen05 GEMM with fused epilogues:  C[M,N] = epi( A[M,K] (fp16, K-major) x W[N,K]^T (fp16) )
#pragma once
#include "common.cuh"

namespace hmocr {

struct GemmEpilogue {
  const float* bias = nullptr;        // [N] fp32
  int act = 0;                   // 0 none, 1 GELU(erf), 2 ReLU, 3 ReLU applied AFTER the residual add (ResNet BasicBlock)
  const float* residual = nullptr;    // fp32 [M, ldr]; may alias out_f32 (in-place residual add)
  int ldr = 0;
  float* out_f32 = nullptr;           // fp32 [M, ld32]
  int ld32 = 0;
  h16* out_f16 = nullptr;  // fp16 [M, ld16]
  int ld16 = 0;
  // LayerNorm over the N axis applied after bias/act/residual; needs N == tile width
  // (N in {64,96,128,192,256}).  Outputs then hold the normalised rows.
  const float* ln_gamma = nullptr;
  const float* ln_beta = nullptr;
};

// A: fp16 [M, K] with row pitch lda (elements); W: fp16 [N, K] contiguous.
// Requirements: N % 32 == 0 (pad the weight), lda % 8 == 0, K % 8 == 0, 16-byte aligned pointers.
int gemm_f16(cudaStream_t stream, const h16* A, int lda, int M, int K, const h16* W,
              int N, const GemmEpilogue& epi, int force_bn = 0);

// Convolution as an implicit GEMM on the same kernel: x fp16 NHWC [B, H, W, Cin] (Cin % 64 == 0), Wt fp16
// [N, ksize*ksize*Cin] with K ordered (kh, kw, c); the epilogue's row index is the NHWC output pixel.
// conv_tiling() says whether the output plane can be cut into <=128-pixel boxes (else: explicit im2col + gemm_f16).
bool conv_tiling(int Ho, int Wo, int* tw, int* th, int* tn);
int gemm_conv_f16(cudaStream_t stream, const h16* x, int B, int H, int W, int Cin, int ksize, int stride, int pad,
                  const h16* Wt, int N, const GemmEpilogue& epi);

// Vocabulary projection with a log-sum-exp epilogue (teacher-forced scoring): logits = A W^T + bias are folded in the
// epilogue into per-row partials and never stored.  The tile width is always LSE_BN, so a row's partials do not depend
// on M.  Partial p of a row covers the 32-column chunks of 256-column tile p / 2 with chunk index % 2 == p % 2, folded
// in column order; columns >= n_valid count as -inf (the padded fc_out rows would otherwise be exact zero logits).
constexpr int LSE_BN = 256;
constexpr int LSE_COLS_PER_PART = 128;
struct LsePartial {       // 32 bytes, written as two 16-byte stores
  float max;              // running maximum (-inf when every column of the partial is masked)
  float sum;              // sum of exp(x - max)
  float target;           // logit of the target column if this partial holds it, else -inf
  float best;             // largest logit; best_idx is its lowest column
  int best_idx;           // INT_MAX when every column is masked
  int pad_[3];
};
struct GemmLse {
  const int64_t* tokens = nullptr;   // target of GEMM row r = b*T + t is tokens[b*ld_tok + t + 1] (compared, never an address)
  int ld_tok = 0, T = 0, n_valid = 0;
  LsePartial* partials = nullptr;    // [M][N / LSE_COLS_PER_PART]
};
// N % LSE_BN == 0; same operand requirements as gemm_f16.
int gemm_f16_lse(cudaStream_t stream, const h16* A, int lda, int M, int K, const h16* W, int N, const float* bias,
                 const GemmLse& lse);

int gemm_init();
// 2-D fp16 tensor map (K-major rows, 128B swizzle, box = 64 columns x box_rows rows), cached per (ptr, shape); for the
// other tcgen05 kernels of the library (swin_mlp.cu).  gemm_init() must have run on this device.
int gemm_tensor_map(const void* ptr, int rows, int cols, int ld, int box_rows, CUtensorMap* out);
int gemm_num_sms();
void gemm_set_debug(int v);   // timing experiments only (see gemm.cu)   // resolves cuTensorMapEncodeTiled, sets kernel attributes; idempotent

}  // namespace hmocr
