// Persistent warp-specialised tcgen05 GEMM for sm_100a.
//
//   C[M,N] = epilogue( A[M,K] x W[N,K]^T )      A, W fp16 (K contiguous), fp32 accumulation in TMEM
//
// Replaces every nn.Linear on the hot path (torchvision swin_transformer.py:179,215,444,85;
// /root/reference/src/model_swin.py:45,64,87; torch MultiheadAttention in/out projections,
// TransformerDecoderLayer.linear1/linear2).
//
// Structure (one CTA per SM, 576 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor 128B-swizzled A (128x64) and W (BNx64) tiles
//               into a STAGES-deep shared-memory ring, completion on "full" mbarriers
//   warp 1      MMA issuer: one elected lane issues tcgen05.mma (M=128, N=BN, K=16) x4 per stage,
//               tcgen05.commit releases the ring slot ("empty") and publishes the accumulator
//   warps 2-17  epilogue, two groups of eight.  The Swin GEMMs have K = 96..768: their main loop is a few
//               hundred cycles per tile and the time goes into reading 128 x BN accumulators out of TMEM,
//               applying bias / GELU / residual and writing them coalesced.  So there are two TMEM
//               accumulators, group g owns accumulator g and takes every second tile of the CTA (two tiles
//               are in the epilogue at once while the main loop of the following ones runs), and inside a
//               group two warps share each TMEM lane quarter (a warp may only touch lanes
//               [32*(warp%4), +32)) and take alternate 32-column chunks.
#include "gemm.cuh"

#include <map>
#include <mutex>
#include <tuple>

namespace hmocr {
namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int EPI_WARPS = 16;                 // two groups of eight
constexpr int GROUP_WARPS = 8;
constexpr int NUM_THREADS = 32 * (2 + EPI_WARPS);
constexpr int EPI_WARP_BYTES = 4096 + 128;    // one 32 x 32 fp32 transpose tile + 32 bias values per epilogue warp

template <int BN>
struct Cfg {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int EPI_STAGE_BYTES = EPI_WARPS * EPI_WARP_BYTES;
  static constexpr int STAGES_RAW = (156 * 1024) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
  static constexpr int TMEM_COLS = (2 * BN <= 128) ? 128 : ((2 * BN <= 256) ? 256 : 512);
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + BAR_BYTES + EPI_STAGE_BYTES;
};

enum EpiMode { EPI_GENERAL = 0, EPI_F16 = 1, EPI_LN = 2 };

// Implicit-GEMM convolution (NHWC fp16 activations): an m-tile is a tw x th x tn box of output pixels
// (w fastest, then h, then image), rows_valid = tw*th*tn <= 128 rows of the MMA tile; k-block kb is filter tap
// kb / cin_blocks and input channels 64 * (kb % cin_blocks), fetched by ONE 4-D tiled TMA load at the tap's
// offset - out-of-bounds coordinates are the zero padding, elementStrides are the convolution stride.
struct ConvGeom {
  int tw, th, tn, tiles_w, tiles_h, Ho, Wo, B, stride, pad, ksize, cin_blocks, rows_valid;
};
// output pixel (row of the NHWC output matrix) of row r of m-tile mi; -1 if the row is padding
__device__ __forceinline__ int conv_pixel(const ConvGeom& g, int mi, int r) {
  if (r >= g.rows_valid) return -1;
  const int tile_w = mi % g.tiles_w, t2 = mi / g.tiles_w, tile_h = t2 % g.tiles_h, tile_n = t2 / g.tiles_h;
  const int w = r % g.tw, r2 = r / g.tw, h = r2 % g.th, n = tile_n * g.tn + r2 / g.th;
  if (n >= g.B) return -1;
  return (n * g.Ho + tile_h * g.th + h) * g.Wo + tile_w * g.tw + w;
}

struct GemmParams {
  int M, N, K;
  int num_n_tiles, num_tiles;
  int mode;           // EpiMode, chosen on the host from the epilogue description
  ConvGeom cg;        // CONV kernels only
  int dbg;            // timing experiments only: 1 = skip output stores, 2 = skip residual loads, 4 = skip the epilogue math
  GemmEpilogue epi;
  GemmLse lse;        // LSE kernels only
};
int g_gemm_dbg = 0;

// K-major, 128B-swizzled shared-memory matrix descriptor (8-row x 128B atoms, 1024B apart).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);   // start address        bits [0,14)
  d |= static_cast<uint64_t>(1) << 16;                  // leading byte offset  (unused, K-major swizzled)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;          // stride byte offset   bits [32,46)
  d |= static_cast<uint64_t>(1) << 46;                  // descriptor version 1 (sm_100)
  d |= static_cast<uint64_t>(2) << 61;                  // SWIZZLE_128B
  return d;
}

template <int BN>
__device__ __forceinline__ constexpr uint32_t make_idesc() {
  return (1u << 4)                 // D format  = F32
         | (0u << 7)               // A format  = F16
         | (0u << 10)              // B format  = F16
         | (uint32_t(BN >> 3) << 17)   // N
         | (uint32_t(BM >> 4) << 24);  // M
}

// Epilogue warps hand their TMEM accumulator back as soon as its last chunk has been loaded into registers
// (the bias/activation/store work of that chunk then overlaps the next main loop).  The __syncwarp doubles as
// the "bias slot is written" fence of the fp16 path.
__device__ __forceinline__ void release_accumulator(bool last_chunk, uint32_t release_bar) {   // shared::cluster address
  tc_fence_before();
  __syncwarp();
  if (last_chunk && (threadIdx.x & 31) == 0) mbar_arrive_cluster(release_bar);
}

// fp16-output epilogue (qkv, fc1 + GELU, linear1 + ReLU: no residual, no fp32 copy) of one 32-row x BN-column
// slab, 32 columns at a time.  tcgen05.ld hands every thread one ROW (32 consecutive fp32 of it); bias and
// activation are applied right there, as 32 independent chains per thread (the bias values of the chunk are
// broadcast from a 128-byte shared slot), and the row is packed to 64 bytes of fp16.  Global memory wants the
// opposite of one-row-per-thread: a warp instruction that covers whole rows.  So the packed rows go through a
// 2 KB per-warp shared tile (16-byte pieces XOR-swizzled by row: conflict-free both ways) and leave as four
// 16-byte stores per thread, each warp store covering 8 rows x 64 contiguous bytes.
template <int BN, int ACT, bool CONV>
__device__ __forceinline__ void epilogue_f16(const GemmEpilogue& e, uint32_t taddr, uint32_t st_addr, int m_base,
                                             int M, int n0, int c_first, int dbg, uint32_t release_bar,
                                             const ConvGeom& cg, int mi, int rq) {
  const int lane = threadIdx.x & 31;
  const uint32_t bias_addr = st_addr + 4096;
  const int srow = lane >> 2, sq = lane & 3;              // store layout: rows it*8 + srow, 16-byte piece sq
  const uint32_t wr_addr = st_addr + lane * 64, wr_sw = (lane >> 1) & 3;
  const uint32_t rd_addr = st_addr + srow * 64 + ((sq ^ ((srow >> 1) & 3)) << 4);
  h16* out = e.out_f16 + (size_t)(m_base + srow) * e.ld16 + n0 + sq * 8;
  const size_t out_step = (size_t)8 * e.ld16;
  const int rows_left = (dbg & 1) ? 0 : M - m_base - srow;       // row it*8 + srow exists iff it*8 < rows_left
  int pix[4];                                                    // CONV: output pixel of row it*8 + srow, -1 if none
  if (CONV) {
#pragma unroll
    for (int it = 0; it < 4; ++it) pix[it] = (dbg & 1) ? -1 : conv_pixel(cg, mi, rq + it * 8 + srow);
  }
#pragma unroll 1
  for (int c = c_first; c < BN / 32; c += 2) {
    const float b = e.bias != nullptr ? __ldg(e.bias + n0 + c * 32 + lane) : 0.0f;
    __syncwarp();                                        // the previous chunk has been read out of tile and bias slot
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(bias_addr + lane * 4), "f"(b) : "memory");
    uint32_t r[32];
    tmem_ld32(taddr + c * 32, r);
    release_accumulator(c + 2 >= BN / 32, release_bar);  // the last chunk is in registers: the MMA warp may reuse the columns
    if ((dbg & 4) && r[0] != 0x12345678u) continue;      // timing experiment: main loop + TMEM load only
    uint32_t h[16];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      uint64_t b01, b23;
      asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(b01), "=l"(b23) : "r"(bias_addr + q * 16));
      float v0, v1, v2, v3;
      upk2(add2(pk2(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1])), b01), v0, v1);
      upk2(add2(pk2(__uint_as_float(r[4 * q + 2]), __uint_as_float(r[4 * q + 3])), b23), v2, v3);
      if (ACT == 1) { gelu_erf2(v0, v1); gelu_erf2(v2, v3); }
      if (ACT == 2) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f); }
      h[2 * q] = pack16(v0, v1);
      h[2 * q + 1] = pack16(v2, v3);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(wr_addr + ((q ^ wr_sw) << 4)), "r"(h[4 * q]),
                   "r"(h[4 * q + 1]), "r"(h[4 * q + 2]), "r"(h[4 * q + 3])
                   : "memory");
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      uint4 v;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                   : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                   : "r"(rd_addr + it * 512));
      if (CONV) {
        if (pix[it] >= 0) *reinterpret_cast<uint4*>(e.out_f16 + (size_t)pix[it] * e.ld16 + n0 + sq * 8 + c * 32) = v;
      } else {
        if (it * 8 < rows_left) *reinterpret_cast<uint4*>(out + it * out_step + c * 32) = v;
      }
    }
  }
}

// General epilogue (fp32 output and/or fp32 residual; ReLU before or after the residual add): the raw
// accumulators go through a 4 KB per-warp shared tile (16-byte chunks XOR-swizzled by row) and come back with
// lane = (row % 4, 4-column group), so every load of the fp32 residual and every store is 4 rows x 128
// contiguous bytes (fp16 copy: x 64) instead of 32 scattered 16-byte pieces.  Bias, activation and residual are
// applied in that second layout, where a lane owns the same 4 columns for all 32 rows (one bias load per
// chunk).  The residual loads are issued before the TMEM load so their latency overlaps it.
template <int BN, bool RES, bool CONV>
__device__ __forceinline__ void epilogue_general(const GemmEpilogue& e, uint32_t taddr, uint32_t st_addr, int m_base,
                                                 int M, int n0, int c_first, int dbg, uint32_t release_bar,
                                                 const ConvGeom& cg, int mi, int rq) {
  const int lane = threadIdx.x & 31;
  const int rr = lane >> 3, cg4 = lane & 7;            // second layout: row (it*4 + rr), columns 4*cg .. 4*cg+3
  const float lo_pre = e.act == 2 ? 0.0f : -INFINITY, lo_post = e.act == 3 ? 0.0f : -INFINITY;
  const int rows_left = M - m_base - rr;              // row it*4 + rr exists iff it*4 < rows_left
  const int rows_store = (dbg & 1) ? 0 : rows_left;
  const uint32_t wr_addr = st_addr + lane * 128, wr_sw = lane & 7;
  const uint32_t rd_addr = st_addr + rr * 128;        // + it*512 + ((cg4 ^ ((it*4 + rr) & 7)) << 4)
  int pix[8];                                         // CONV: output pixel of row it*4 + rr, -1 if none
  if (CONV) {
#pragma unroll
    for (int it = 0; it < 8; ++it) pix[it] = conv_pixel(cg, mi, rq + it * 4 + rr);
  }
#pragma unroll 1
  for (int c = c_first; c < BN / 32; c += 2) {
    const int col = n0 + c * 32 + cg4 * 4;
    float4 res[8];
    if (RES) {
      const float* rp = e.residual + (size_t)(m_base + rr) * e.ldr + col;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        if (CONV)
          res[it] = pix[it] >= 0 ? __ldcs(reinterpret_cast<const float4*>(e.residual + (size_t)pix[it] * e.ldr + col))
                                 : make_float4(0.f, 0.f, 0.f, 0.f);
        else
          res[it] = (it * 4 < rows_left) ? __ldcs(reinterpret_cast<const float4*>(rp + (size_t)it * 4 * e.ldr))
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
    if (e.bias != nullptr) bias = __ldg(reinterpret_cast<const float4*>(e.bias + col));
    uint32_t r[32];
    tmem_ld32(taddr + c * 32, r);
    release_accumulator(c + 2 >= BN / 32, release_bar);   // also: the previous chunk has been read out of the tile
    if ((dbg & 4) && r[0] != 0x12345678u) continue;    // timing experiment: main loop + TMEM load only
#pragma unroll
    for (int q = 0; q < 8; ++q)                        // thread = row `lane`: chunk q -> physical chunk q ^ (lane & 7)
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(wr_addr + ((q ^ wr_sw) << 4)), "r"(r[4 * q]),
                   "r"(r[4 * q + 1]), "r"(r[4 * q + 2]), "r"(r[4 * q + 3])
                   : "memory");
    __syncwarp();
    float* o32 = e.out_f32 != nullptr ? e.out_f32 + (size_t)(m_base + rr) * e.ld32 + col : nullptr;
    h16* o16 = e.out_f16 != nullptr ? e.out_f16 + (size_t)(m_base + rr) * e.ld16 + col : nullptr;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      float4 v;
      asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                   : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                   : "r"(rd_addr + it * 512 + ((cg4 ^ ((it * 4 + rr) & 7)) << 4)));
      v.x += bias.x; v.y += bias.y; v.z += bias.z; v.w += bias.w;
      if (e.act == 1) { v.x = gelu_erf(v.x); v.y = gelu_erf(v.y); v.z = gelu_erf(v.z); v.w = gelu_erf(v.w); }
      v.x = fmaxf(v.x, lo_pre); v.y = fmaxf(v.y, lo_pre); v.z = fmaxf(v.z, lo_pre); v.w = fmaxf(v.w, lo_pre);
      if (RES) { v.x += res[it].x; v.y += res[it].y; v.z += res[it].z; v.w += res[it].w; }
      v.x = fmaxf(v.x, lo_post); v.y = fmaxf(v.y, lo_post); v.z = fmaxf(v.z, lo_post); v.w = fmaxf(v.w, lo_post);
      if (CONV) {
        if (pix[it] >= 0 && !(dbg & 1)) {
          if (e.out_f32 != nullptr) *reinterpret_cast<float4*>(e.out_f32 + (size_t)pix[it] * e.ld32 + col) = v;
          if (e.out_f16 != nullptr)
            *reinterpret_cast<uint2*>(e.out_f16 + (size_t)pix[it] * e.ld16 + col) = make_uint2(pack16(v.x, v.y), pack16(v.z, v.w));
        }
      } else if (it * 4 < rows_store) {
        if (o32 != nullptr) *reinterpret_cast<float4*>(o32 + (size_t)it * 4 * e.ld32) = v;
        if (o16 != nullptr)
          *reinterpret_cast<uint2*>(o16 + (size_t)it * 4 * e.ld16) = make_uint2(pack16(v.x, v.y), pack16(v.z, v.w));
      }
    }
  }
}

// LayerNorm epilogue: the whole output row lives in this thread's TMEM lane (N == BN).
// Pass 1 writes v = acc + bias (+act) + residual back to TMEM and sums it; pass 2 sums the
// squared deviations (two-pass variance, as torch does); pass 3 normalises and stores.
template <int BN>
__device__ __forceinline__ void epilogue_ln(const GemmEpilogue& e, uint32_t taddr, int row, bool row_ok, int n0) {
  float sum = 0.0f;
#pragma unroll 1
  for (int c = 0; c < BN / 32; ++c) {
    uint32_t r[32];
    tmem_ld32(taddr + c * 32, r);
    const int col = n0 + c * 32;
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
    if (e.bias != nullptr) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] += __ldg(e.bias + col + j);
    }
    if (e.act == 1) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
    } else if (e.act == 2) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.0f);
    }
    if (row_ok && e.residual != nullptr) {
      const float4* r4 = reinterpret_cast<const float4*>(e.residual + (size_t)row * e.ldr + col);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        float4 x = r4[q];
        v[4 * q + 0] += x.x; v[4 * q + 1] += x.y; v[4 * q + 2] += x.z; v[4 * q + 3] += x.w;
      }
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) { sum += v[j]; r[j] = __float_as_uint(v[j]); }
    tmem_st32(taddr + c * 32, r);
  }
  const float mean = sum * (1.0f / BN);
  float sq = 0.0f;
#pragma unroll 1
  for (int c = 0; c < BN / 32; ++c) {
    uint32_t r[32];
    tmem_ld32(taddr + c * 32, r);
#pragma unroll
    for (int j = 0; j < 32; ++j) { float d = __uint_as_float(r[j]) - mean; sq += d * d; }
  }
  const float rstd = rsqrtf(sq * (1.0f / BN) + 1e-5f);
#pragma unroll 1
  for (int c = 0; c < BN / 32; ++c) {
    uint32_t r[32];
    tmem_ld32(taddr + c * 32, r);
    const int col = n0 + c * 32;
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j)
      v[j] = (__uint_as_float(r[j]) - mean) * rstd * __ldg(e.ln_gamma + col + j) + __ldg(e.ln_beta + col + j);
    if (row_ok) {
      if (e.out_f32 != nullptr) {
        float4* o = reinterpret_cast<float4*>(e.out_f32 + (size_t)row * e.ld32 + col);
#pragma unroll
        for (int q = 0; q < 8; ++q) o[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
      }
      if (e.out_f16 != nullptr) {
        uint4* o = reinterpret_cast<uint4*>(e.out_f16 + (size_t)row * e.ld16 + col);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          o[q] = make_uint4(pack16(v[8 * q], v[8 * q + 1]), pack16(v[8 * q + 2], v[8 * q + 3]),
                            pack16(v[8 * q + 4], v[8 * q + 5]), pack16(v[8 * q + 6], v[8 * q + 7]));
      }
    }
  }
}

// Log-sum-exp epilogue (gemm_f16_lse): one thread = one row, as tcgen05.ld hands it over.  Each thread folds its
// chunks (c = c_first, c_first + 2, ...) in column order into one LsePartial and writes only that: the logits never
// leave the SM.  Inside a chunk the exponentials are summed as a fixed binary tree.
template <int BN>
__device__ __forceinline__ void epilogue_lse(const GemmEpilogue& e, const GemmLse& l, uint32_t taddr, int m_base, int M,
                                             int n0, int c_first, uint32_t release_bar, int n_tile,
                                             int num_n_tiles) {
  const int lane = threadIdx.x & 31;
  const int row = m_base + lane;
  int target = -1;
  if (row < M) {
    const int b = row / l.T, t = row - b * l.T;
    const long long id = l.tokens[(size_t)b * l.ld_tok + t + 1];
    target = (id >= 0 && id < l.n_valid) ? (int)id : -1;
  }
  float m = -INFINITY, s = 0.f, tv = -INFINITY, bv = -INFINITY;
  int bi = 0x7fffffff;
#pragma unroll 1
  for (int c = c_first; c < BN / 32; c += 2) {
    const int col0 = n0 + c * 32;
    uint32_t r[32];
    tmem_ld32(taddr + c * 32, r);
    release_accumulator(c + 2 >= BN / 32, release_bar);
    float v[32];
    const float4* b4 = reinterpret_cast<const float4*>(e.bias + col0);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 bq = __ldg(b4 + q);
      v[4 * q] = __uint_as_float(r[4 * q]) + bq.x;
      v[4 * q + 1] = __uint_as_float(r[4 * q + 1]) + bq.y;
      v[4 * q + 2] = __uint_as_float(r[4 * q + 2]) + bq.z;
      v[4 * q + 3] = __uint_as_float(r[4 * q + 3]) + bq.w;
    }
    float cm = -INFINITY;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (col0 + j >= l.n_valid) v[j] = -INFINITY;
      if (col0 + j == target) tv = v[j];
      cm = fmaxf(cm, v[j]);
    }
    int ci = 0;
#pragma unroll
    for (int j = 31; j >= 0; --j) ci = (v[j] == cm) ? j : ci;       // lowest column holding the chunk maximum
    if (cm > bv) { bv = cm; bi = col0 + ci; }                      // strict: an earlier chunk keeps a tie
    const float mn = fmaxf(m, cm);
    if (mn != -INFINITY) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = expf(v[j] - mn);
#pragma unroll
      for (int w = 16; w >= 1; w >>= 1)
#pragma unroll
        for (int j = 0; j < w; ++j) v[j] += v[j + w];
      s = s * expf(m - mn) + v[0];
      m = mn;
    }
  }
  if (row < M) {
    float4* o = reinterpret_cast<float4*>(l.partials + (size_t)row * (2 * num_n_tiles) + 2 * n_tile + c_first);
    o[0] = make_float4(m, s, tv, bv);
    o[1] = make_float4(__int_as_float(bi), 0.f, 0.f, 0.f);
  }
}

template <int BN, bool CONV, bool LSE = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const GemmParams p) {
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);

  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tfull_bar = empty_bar + C::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  const uint32_t epi_stage = smem_u32(smem + C::STAGES * C::STAGE_BYTES + C::BAR_BYTES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  pdl_launch_dependents();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], GROUP_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, C::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int num_kb = (p.K + BK - 1) / BK;
  pdl_wait();              // A, the residual and the output buffers belong to earlier kernels up to here

  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int t = blockIdx.x; t < p.num_tiles; t += gridDim.x) {
        const int m0 = (t / p.num_n_tiles) * BM;
        const int n0 = (t % p.num_n_tiles) * BN;
        int cw = 0, chh = 0, cn = 0;                   // CONV: input coordinates of the tile's first pixel at tap (0,0)
        if (CONV) {
          const int mi = t / p.num_n_tiles;
          const int tile_w = mi % p.cg.tiles_w, t2 = mi / p.cg.tiles_w;
          cw = tile_w * p.cg.tw * p.cg.stride - p.cg.pad;
          chh = (t2 % p.cg.tiles_h) * p.cg.th * p.cg.stride - p.cg.pad;
          cn = (t2 / p.cg.tiles_h) * p.cg.tn;
        }
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[s], ph ^ 1u);
          uint8_t* st = smem + s * C::STAGE_BYTES;
          if (CONV) {
            mbar_expect_tx(&full_bar[s], p.cg.rows_valid * (BK * 2) + C::B_BYTES);
            const int tap = kb / p.cg.cin_blocks, cb = kb - tap * p.cg.cin_blocks;
            const int kh = tap / p.cg.ksize, kw = tap - kh * p.cg.ksize;
            tma_load_4d(st, &tmA, &full_bar[s], cb * BK, cw + kw, chh + kh, cn);
          } else {
            mbar_expect_tx(&full_bar[s], C::STAGE_BYTES);
            tma_load_2d(st, &tmA, &full_bar[s], kb * BK, m0);
          }
          tma_load_2d(st + C::A_BYTES, &tmB, &full_bar[s], kb * BK, n0);
          if (++s == C::STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc<BN>();
      int s = 0;
      uint32_t ph = 0;
      int it = 0;
      for (int t = blockIdx.x; t < p.num_tiles; t += gridDim.x, ++it) {
        const int a = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        mbar_wait_backoff(&tempty_bar[a], aph ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + a * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t abase = smem_u32(smem + s * C::STAGE_BYTES);
          const uint32_t bbase = abase + C::A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            umma_f16(d_tmem, make_smem_desc(abase + k * 32), make_smem_desc(bbase + k * 32), idesc,
                      (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(&empty_bar[s]);
          if (++s == C::STAGES) { s = 0; ph ^= 1u; }
        }
        umma_commit(&tfull_bar[a]);
      }
    }
  } else {
    const int quarter = warp & 3;          // TMEM lanes [32*quarter, 32*quarter+32) belong to this warp
    const int ew = warp - 2;
    const int group = ew >> 3;             // accumulator / tile parity this warp serves
    const int half = (ew >> 2) & 1;        // which of the two warps of this lane quarter inside the group
    const uint32_t st_addr = epi_stage + ew * EPI_WARP_BYTES;
    const uint32_t taddr = tmem_base + (uint32_t(quarter * 32) << 16) + group * BN;
    const bool has_res = p.epi.residual != nullptr && !(p.dbg & 2);
    int it = group;
    for (int t = blockIdx.x + group * gridDim.x; t < p.num_tiles; t += 2 * gridDim.x, it += 2) {
      const uint32_t aph = (it >> 1) & 1;
      const int m0 = (t / p.num_n_tiles) * BM;
      const int n0 = (t % p.num_n_tiles) * BN;
      mbar_wait_backoff(&tfull_bar[group], aph);
      tc_fence_after();
      const int mb = m0 + quarter * 32;
      const int mi = t / p.num_n_tiles, rq = quarter * 32;
      if constexpr (LSE) {
        epilogue_lse<BN>(p.epi, p.lse, taddr, mb, p.M, n0, half, smem_u32(&tempty_bar[group]), t % p.num_n_tiles,
                         p.num_n_tiles);
        continue;
      }
      if (p.mode == EPI_LN) {
        const int row = mb + lane;
        if (half == 0) epilogue_ln<BN>(p.epi, taddr, row, row < p.M, n0);   // row statistics: one thread per row
      } else if (p.mode == EPI_F16) {
        if (p.epi.act == 1) epilogue_f16<BN, 1, CONV>(p.epi, taddr, st_addr, mb, p.M, n0, half, p.dbg, smem_u32(&tempty_bar[group]), p.cg, mi, rq);
        else if (p.epi.act == 2) epilogue_f16<BN, 2, CONV>(p.epi, taddr, st_addr, mb, p.M, n0, half, p.dbg, smem_u32(&tempty_bar[group]), p.cg, mi, rq);
        else epilogue_f16<BN, 0, CONV>(p.epi, taddr, st_addr, mb, p.M, n0, half, p.dbg, smem_u32(&tempty_bar[group]), p.cg, mi, rq);
      } else {
        if (has_res) epilogue_general<BN, true, CONV>(p.epi, taddr, st_addr, mb, p.M, n0, half, p.dbg, smem_u32(&tempty_bar[group]), p.cg, mi, rq);
        else epilogue_general<BN, false, CONV>(p.epi, taddr, st_addr, mb, p.M, n0, half, p.dbg, smem_u32(&tempty_bar[group]), p.cg, mi, rq);
      }
      if (p.mode == EPI_LN) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[group]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// CTA-pair variant (cta_group::2) for the K-heavy shapes (Swin stages 3/4): their main loop is bound by the
// L2 -> SM operand traffic, not by the tensor pipe.  Two CTAs of a cluster (one TPC) share a 256 x BN tile: each
// loads ITS 128 rows of A and HALF of the W tile (BN/2 rows) per k-block - (128 + BN/2) x 128 B instead of
// (128 + BN) x 128 B per 128 output rows - and the leader CTA's elected thread issues one M = 256 MMA that reads
// both CTAs' shared memory and writes both CTAs' TMEM.  Protocol: "full" barriers live in the leader and count
// the TMA bytes of both CTAs (the peer's loads name the leader's barrier); tcgen05.commit multicasts the
// "slot free" and "accumulator ready" arrivals to both CTAs; the peer's epilogue warps release the accumulator
// with a remote arrive on the leader's barrier.  Epilogues, groups and staging are those of the 1-CTA kernel.
template <int BN>
struct Cfg2 {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = (BN / 2) * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int EPI_STAGE_BYTES = EPI_WARPS * EPI_WARP_BYTES;
  static constexpr int STAGES_RAW = (156 * 1024) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
  static constexpr int TMEM_COLS = (2 * BN <= 128) ? 128 : ((2 * BN <= 256) ? 256 : 512);
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + BAR_BYTES + EPI_STAGE_BYTES;
};

template <int BN>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm2_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const GemmParams p) {
  using C = Cfg2<BN>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);

  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tfull_bar = empty_bar + C::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  const uint32_t epi_stage = smem_u32(smem + C::STAGES * C::STAGE_BYTES + C::BAR_BYTES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cta_rank_in_cluster();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  pdl_launch_dependents();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(&full_bar[s], 1);              // used in the leader only
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 2 * GROUP_WARPS);   // leader only: the epilogue warps of both CTAs
    }
    fence_barrier_init();
  }
  cluster_barrier();                            // both CTAs' barriers exist before any remote arrive / TMA completion
  if (warp == 1) tmem_alloc2(tmem_slot, C::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  cluster_barrier();                            // both allocations done: the leader's MMA writes the peer's TMEM too
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int num_kb = (p.K + BK - 1) / BK;
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int t = pair; t < p.num_tiles; t += npairs) {
        const int m0 = (t / p.num_n_tiles) * (2 * BM) + rank * BM;
        const int n0 = (t % p.num_n_tiles) * BN + rank * (BN / 2);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[s], ph ^ 1u);
          if (rank == 0) mbar_expect_tx(&full_bar[s], 2 * C::STAGE_BYTES);
          uint8_t* st = smem + s * C::STAGE_BYTES;
          tma2_load_2d(st, &tmA, &full_bar[s], kb * BK, m0);
          tma2_load_2d(st + C::A_BYTES, &tmB, &full_bar[s], kb * BK, n0);
          if (++s == C::STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc = (1u << 4) | (uint32_t(BN >> 3) << 17) | (uint32_t((2 * BM) >> 4) << 24);   // F16 in, F32 out, M = 256
      int s = 0;
      uint32_t ph = 0;
      int it = 0;
      for (int t = pair; t < p.num_tiles; t += npairs, ++it) {
        const int a = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        mbar_wait_backoff(&tempty_bar[a], aph ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + a * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t abase = smem_u32(smem + s * C::STAGE_BYTES);
          const uint32_t bbase = abase + C::A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            umma2_f16(d_tmem, make_smem_desc(abase + k * 32), make_smem_desc(bbase + k * 32), idesc,
                      (kb | k) != 0 ? 1u : 0u);
          }
          umma2_commit(&empty_bar[s]);
          if (++s == C::STAGES) { s = 0; ph ^= 1u; }
        }
        umma2_commit(&tfull_bar[a]);
      }
    }
  } else {
    const int quarter = warp & 3;
    const int ew = warp - 2;
    const int group = ew >> 3;
    const int half = (ew >> 2) & 1;
    const uint32_t st_addr = epi_stage + ew * EPI_WARP_BYTES;
    const uint32_t taddr = tmem_base + (uint32_t(quarter * 32) << 16) + group * BN;
    const bool has_res = p.epi.residual != nullptr && !(p.dbg & 2);
    const uint32_t release = smem_u32(&tempty_bar[group]) & PEER_BIT_MASK;      // the leader's barrier
    int it = group;
    for (int t = pair + group * npairs; t < p.num_tiles; t += 2 * npairs, it += 2) {
      const uint32_t aph = (it >> 1) & 1;
      const int m0 = (t / p.num_n_tiles) * (2 * BM) + rank * BM;
      const int n0 = (t % p.num_n_tiles) * BN;
      mbar_wait_backoff(&tfull_bar[group], aph);
      tc_fence_after();
      const int mb = m0 + quarter * 32;
      if (p.mode == EPI_F16) {
        if (p.epi.act == 1) epilogue_f16<BN, 1, false>(p.epi, taddr, st_addr, mb, p.M, n0, half, p.dbg, release, p.cg, 0, 0);
        else if (p.epi.act == 2) epilogue_f16<BN, 2, false>(p.epi, taddr, st_addr, mb, p.M, n0, half, p.dbg, release, p.cg, 0, 0);
        else epilogue_f16<BN, 0, false>(p.epi, taddr, st_addr, mb, p.M, n0, half, p.dbg, release, p.cg, 0, 0);
      } else {
        if (has_res) epilogue_general<BN, true, false>(p.epi, taddr, st_addr, mb, p.M, n0, half, p.dbg, release, p.cg, 0, 0);
        else epilogue_general<BN, false, false>(p.epi, taddr, st_addr, mb, p.M, n0, half, p.dbg, release, p.cg, 0, 0);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_barrier();                            // the peer may still be reading operands / TMEM this CTA's MMA touches
  if (warp == 1) {
    __syncwarp();
    tmem_dealloc2(tmem_base, C::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
int g_sms[HM_MAX_DEVICES] = {};      // per device: filled by gemm_init() on that device (0 = not initialised)
int num_sms() {
  int dev = 0;
  cudaGetDevice(&dev);
  return (dev >= 0 && dev < HM_MAX_DEVICES && g_sms[dev] > 0) ? g_sms[dev] : 148;
}
std::mutex g_mu;
std::map<std::tuple<const void*, int, int, int, int>, CUtensorMap> g_maps;

int get_tensor_map(const void* ptr, int rows, int cols, int ld, int box_rows, CUtensorMap* out) {
  auto key = std::make_tuple(ptr, rows, cols, ld, box_rows);
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_maps.find(key);
  if (it != g_maps.end()) {
    *out = it->second;
    return 0;
  }
  alignas(64) CUtensorMap m;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  HM_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) ptr=%p rows=%d cols=%d ld=%d box_rows=%d", (int)r,
           ptr, rows, cols, ld, box_rows);
  if (g_maps.size() > 4096) g_maps.clear();
  g_maps[key] = m;
  *out = m;
  return 0;
}

template <int BN>
int launch(cudaStream_t stream, const h16* A, int lda, int M, int K, const h16* W, int N,
           const GemmEpilogue& epi) {
  using C = Cfg<BN>;
  alignas(64) CUtensorMap tmA, tmB;
  HM_TRY(get_tensor_map(A, M, K, lda, BM, &tmA));
  HM_TRY(get_tensor_map(W, N, K, K, BN, &tmB));
  GemmParams p;
  p.M = M; p.N = N; p.K = K;
  p.num_n_tiles = N / BN;
  p.num_tiles = ceil_div(M, BM) * p.num_n_tiles;
  p.epi = epi;
  p.dbg = g_gemm_dbg;
  p.mode = epi.ln_gamma != nullptr ? EPI_LN
           : (epi.out_f32 == nullptr && epi.residual == nullptr && epi.act != 3) ? EPI_F16 : EPI_GENERAL;
  const int grid = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  HM_CUDA(launch_pdl(gemm_tcgen05_kernel<BN, false>, dim3(grid), dim3(NUM_THREADS), C::SMEM_BYTES, stream, tmA, tmB, p));
  HM_LAUNCHED();
  return 0;
}

int launch_lse(cudaStream_t stream, const h16* A, int lda, int M, int K, const h16* W, int N, const float* bias,
               const GemmLse& lse) {
  using C = Cfg<LSE_BN>;
  alignas(64) CUtensorMap tmA, tmB;
  HM_TRY(get_tensor_map(A, M, K, lda, BM, &tmA));
  HM_TRY(get_tensor_map(W, N, K, K, LSE_BN, &tmB));
  GemmParams p;
  p.M = M; p.N = N; p.K = K;
  p.num_n_tiles = N / LSE_BN;
  p.num_tiles = ceil_div(M, BM) * p.num_n_tiles;
  p.epi = GemmEpilogue{};
  p.epi.bias = bias;
  p.mode = EPI_GENERAL;
  p.dbg = 0;
  p.cg = ConvGeom{};
  p.lse = lse;
  const int grid = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  HM_CUDA(launch_pdl(gemm_tcgen05_kernel<LSE_BN, false, true>, dim3(grid), dim3(NUM_THREADS), C::SMEM_BYTES, stream, tmA,
                     tmB, p));
  HM_LAUNCHED();
  return 0;
}

// NHWC fp16 activation [B, H, W, C] as a 4-D tensor (C, W, H, B); box = 64 channels x (tw, th, tn) output pixels
// visited with the convolution stride.
std::map<std::tuple<const void*, int, int, int, int, int, int, int, int>, CUtensorMap> g_maps4;
int get_tensor_map_nhwc(const void* ptr, int B, int H, int W, int C, int tw, int th, int tn, int stride, CUtensorMap* out) {
  auto key = std::make_tuple(ptr, B, H, W, C, tw, th, tn, stride);
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_maps4.find(key);
  if (it != g_maps4.end()) {
    *out = it->second;
    return 0;
  }
  alignas(64) CUtensorMap m;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)BK, (cuuint32_t)(tw * stride), (cuuint32_t)(th * stride), (cuuint32_t)tn};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  CUresult r = g_encode(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  HM_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (NHWC) failed (%d) B=%d H=%d W=%d C=%d box=%dx%dx%d stride=%d", (int)r,
           B, H, W, C, tw, th, tn, stride);
  if (g_maps4.size() > 1024) g_maps4.clear();
  g_maps4[key] = m;
  *out = m;
  return 0;
}

template <int BN>
int launch_conv(cudaStream_t stream, const CUtensorMap& tmA, const h16* Wt, int N, int K, const ConvGeom& cg, int m_tiles,
                const GemmEpilogue& epi) {
  using C = Cfg<BN>;
  alignas(64) CUtensorMap tmB;
  HM_TRY(get_tensor_map(Wt, N, K, K, BN, &tmB));
  GemmParams p;
  p.M = m_tiles * BM; p.N = N; p.K = K;
  p.num_n_tiles = N / BN;
  p.num_tiles = m_tiles * p.num_n_tiles;
  p.epi = epi;
  p.dbg = g_gemm_dbg;
  p.mode = (epi.out_f32 == nullptr && epi.residual == nullptr && epi.act != 3) ? EPI_F16 : EPI_GENERAL;
  p.cg = cg;
  const int grid = p.num_tiles < num_sms() ? p.num_tiles : num_sms();
  HM_CUDA(launch_pdl(gemm_tcgen05_kernel<BN, true>, dim3(grid), dim3(NUM_THREADS), C::SMEM_BYTES, stream, tmA, tmB, p));
  HM_LAUNCHED();
  return 0;
}

template <int BN>
int launch2(cudaStream_t stream, const h16* A, int lda, int M, int K, const h16* W, int N, const GemmEpilogue& epi) {
  using C = Cfg2<BN>;
  alignas(64) CUtensorMap tmA, tmB;
  HM_TRY(get_tensor_map(A, M, K, lda, BM, &tmA));
  HM_TRY(get_tensor_map(W, N, K, K, BN / 2, &tmB));
  GemmParams p;
  p.M = M; p.N = N; p.K = K;
  p.num_n_tiles = N / BN;
  p.num_tiles = ceil_div(M, 2 * BM) * p.num_n_tiles;
  p.epi = epi;
  p.dbg = g_gemm_dbg;
  p.mode = (epi.out_f32 == nullptr && epi.residual == nullptr && epi.act != 3) ? EPI_F16 : EPI_GENERAL;
  p.cg = ConvGeom{};
  int pairs = num_sms() / 2;
  if (p.num_tiles < pairs) pairs = p.num_tiles;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  HM_CUDA(cudaLaunchKernelEx(&cfg, gemm2_tcgen05_kernel<BN>, tmA, tmB, p));
  HM_LAUNCHED();
  return 0;
}

}  // namespace

bool conv_tiling(int Ho, int Wo, int* tw, int* th, int* tn) {
  if (Ho * Wo <= BM) {                        // whole images per tile
    *tw = Wo; *th = Ho; *tn = BM / (Ho * Wo);
    if (*tn > 256) *tn = 256;
    return (*tw) * (*th) * (*tn) * 4 >= BM * 3;
  }
  *tn = 1;
  int best_tw = 0, best_th = 0;
  for (int w = 1; w <= Wo && w <= BM; ++w) {  // the fullest tw x th box that tiles the image exactly
    if (Wo % w != 0) continue;
    for (int h = 1; h <= Ho && w * h <= BM; ++h) {
      if (Ho % h != 0) continue;
      if (w * h > best_tw * best_th) { best_tw = w; best_th = h; }
    }
  }
  *tw = best_tw; *th = best_th;
  return best_tw * best_th * 4 >= BM * 3 && best_tw <= 256 && best_th <= 256;
}

int gemm_conv_f16(cudaStream_t stream, const h16* x, int B, int H, int W, int Cin, int ksize, int stride, int pad,
                  const h16* Wt, int N, const GemmEpilogue& epi) {
  HM_TRY(gemm_init());
  const int Ho = (H + 2 * pad - ksize) / stride + 1, Wo = (W + 2 * pad - ksize) / stride + 1;
  ConvGeom cg;
  HM_CHECK(conv_tiling(Ho, Wo, &cg.tw, &cg.th, &cg.tn), "conv: no tile box for a %dx%d output", Ho, Wo);
  HM_CHECK(Cin % BK == 0, "conv: input channels %d must be a multiple of %d", Cin, BK);
  HM_CHECK(cg.tw * stride <= 256 && cg.th * stride <= 256, "conv: tile box too large for TMA");
  HM_CHECK(epi.ln_gamma == nullptr, "conv: fused LayerNorm is not supported");
  HM_CHECK(epi.out_f32 != nullptr || epi.out_f16 != nullptr, "conv: no output");
  cg.tiles_w = Wo / cg.tw; cg.tiles_h = Ho / cg.th;
  cg.Ho = Ho; cg.Wo = Wo; cg.B = B; cg.stride = stride; cg.pad = pad; cg.ksize = ksize;
  cg.cin_blocks = Cin / BK; cg.rows_valid = cg.tw * cg.th * cg.tn;
  const int m_tiles = cg.tiles_w * cg.tiles_h * ceil_div(B, cg.tn);
  const int K = ksize * ksize * Cin;
  alignas(64) CUtensorMap tmA;
  HM_TRY(get_tensor_map_nhwc(x, B, H, W, Cin, cg.tw, cg.th, cg.tn, stride, &tmA));
  int bn = 0;
  const int cands[3] = {256, 128, 64};
  for (int i = 0; i < 3; ++i) {
    if (N % cands[i] != 0) continue;
    bn = cands[i];
    if (m_tiles * (N / cands[i]) >= num_sms()) break;
  }
  HM_CHECK(bn != 0, "conv: output channels %d must be a multiple of 64", N);
  switch (bn) {
    case 64: return launch_conv<64>(stream, tmA, Wt, N, K, cg, m_tiles, epi);
    case 128: return launch_conv<128>(stream, tmA, Wt, N, K, cg, m_tiles, epi);
    default: return launch_conv<256>(stream, tmA, Wt, N, K, cg, m_tiles, epi);
  }
}

void gemm_set_debug(int v) { g_gemm_dbg = v; }
int gemm_tensor_map(const void* ptr, int rows, int cols, int ld, int box_rows, CUtensorMap* out) {
  return get_tensor_map(ptr, rows, cols, ld, box_rows, out);
}
int gemm_num_sms() { return num_sms(); }

int gemm_init() {
  // per DEVICE: the shared-memory opt-in of a kernel is an attribute of the function on one device
  std::lock_guard<std::mutex> lk(g_mu);
  int cur = 0;
  HM_CUDA(cudaGetDevice(&cur));
  HM_CHECK(cur >= 0 && cur < HM_MAX_DEVICES, "device index %d", cur);
  if (g_sms[cur] > 0) return 0;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  HM_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
  HM_CHECK(fn != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available in this driver");
  const int dev = cur;
  cudaDeviceProp prop;
  HM_CUDA(cudaGetDeviceProperties(&prop, dev));
  HM_CHECK(prop.major == 10, "libhmocr is built for sm_100a only; device is sm_%d%d (no fallback path)", prop.major,
           prop.minor);
  // set once, up front: nothing but launches may happen while a step graph is being captured
  HM_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel<64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<64>::SMEM_BYTES));
  HM_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel<96, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<96>::SMEM_BYTES));
  HM_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel<128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<128>::SMEM_BYTES));
  HM_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel<192, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<192>::SMEM_BYTES));
  HM_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel<256, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<256>::SMEM_BYTES));
  HM_CUDA(cudaFuncSetAttribute(gemm2_tcgen05_kernel<192>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg2<192>::SMEM_BYTES));
  HM_CUDA(cudaFuncSetAttribute(gemm2_tcgen05_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg2<256>::SMEM_BYTES));
  HM_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel<64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<64>::SMEM_BYTES));
  HM_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel<128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<128>::SMEM_BYTES));
  HM_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel<256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<256>::SMEM_BYTES));
  HM_CUDA(cudaFuncSetAttribute(gemm_tcgen05_kernel<LSE_BN, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               Cfg<LSE_BN>::SMEM_BYTES));
  g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  g_sms[dev] = prop.multiProcessorCount;
  return 0;
}

int gemm_f16(cudaStream_t stream, const h16* A, int lda, int M, int K, const h16* W, int N,
              const GemmEpilogue& epi, int force_bn) {
  HM_TRY(gemm_init());
  HM_CHECK(M > 0 && N > 0 && K > 0, "gemm: empty problem M=%d N=%d K=%d", M, N, K);
  HM_CHECK(N % 32 == 0, "gemm: N=%d must be a multiple of 32 (pad the weight)", N);
  HM_CHECK(K % 8 == 0 && lda % 8 == 0, "gemm: K=%d and lda=%d must be multiples of 8", K, lda);
  HM_CHECK((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0,
           "gemm: operands must be 16-byte aligned");
  HM_CHECK(epi.out_f32 != nullptr || epi.out_f16 != nullptr, "gemm: no output");
  HM_CHECK(epi.out_f32 == nullptr || epi.ld32 % 4 == 0, "gemm: ld32 must be a multiple of 4");
  HM_CHECK(epi.out_f16 == nullptr || epi.ld16 % 8 == 0, "gemm: ld16 must be a multiple of 8");
  HM_CHECK(epi.residual == nullptr || epi.ldr % 4 == 0, "gemm: ldr must be a multiple of 4");
  int bn = force_bn;
  if (epi.ln_gamma != nullptr) {
    HM_CHECK(N == 64 || N == 96 || N == 128 || N == 192 || N == 256,
             "gemm: fused LayerNorm needs N in {64,96,128,192,256}, got %d", N);
    HM_CHECK(epi.ln_beta != nullptr, "gemm: ln_beta missing");
    bn = N;
  }
  if (bn == 0) {
    const int cands[5] = {256, 192, 128, 96, 64};
    const int mt = ceil_div(M, BM);
    int smallest = 0;
    for (int i = 0; i < 5; ++i) {
      if (N % cands[i] != 0) continue;
      smallest = cands[i];
      if (bn == 0 && mt * (N / cands[i]) >= num_sms()) bn = cands[i];
    }
    if (bn == 0) bn = smallest;
    HM_CHECK(bn != 0, "gemm: N=%d is not a multiple of 64 or 96", N);
  }
  // K-heavy shapes (fc2 of Swin stages 3/4, the last patch-merging reduction): the CTA-pair kernel's halved W-tile
  // traffic is worth 8-15 % there (profiles/README.md); everything else stays on the 1-CTA kernel
  if (force_bn == 0 && epi.ln_gamma == nullptr && K >= 1024 && N % 192 == 0 && M >= 4 * BM)
    return launch2<192>(stream, A, lda, M, K, W, N, epi);
  if (force_bn == 2192 || force_bn == 2256) {            // CTA-pair kernel, explicit (tests / timing)
    bn = force_bn - 2000;
    HM_CHECK(N % bn == 0 && epi.ln_gamma == nullptr, "gemm: pair kernel needs N %% %d == 0 and no fused LayerNorm", bn);
    return bn == 192 ? launch2<192>(stream, A, lda, M, K, W, N, epi) : launch2<256>(stream, A, lda, M, K, W, N, epi);
  }
  HM_CHECK(N % bn == 0, "gemm: N=%d not divisible by tile width %d", N, bn);
  switch (bn) {
    case 64: return launch<64>(stream, A, lda, M, K, W, N, epi);
    case 96: return launch<96>(stream, A, lda, M, K, W, N, epi);
    case 128: return launch<128>(stream, A, lda, M, K, W, N, epi);
    case 192: return launch<192>(stream, A, lda, M, K, W, N, epi);
    case 256: return launch<256>(stream, A, lda, M, K, W, N, epi);
  }
  HM_CHECK(false, "gemm: unsupported tile width %d", bn);
  return -2;
}

int gemm_f16_lse(cudaStream_t stream, const h16* A, int lda, int M, int K, const h16* W, int N, const float* bias,
                 const GemmLse& lse) {
  HM_TRY(gemm_init());
  HM_CHECK(M > 0 && K > 0 && N > 0 && N % LSE_BN == 0, "gemm_lse: M=%d K=%d, N=%d must be a multiple of %d", M, K, N,
           LSE_BN);
  HM_CHECK(K % 8 == 0 && lda % 8 == 0, "gemm_lse: K=%d and lda=%d must be multiples of 8", K, lda);
  HM_CHECK((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(bias) & 15) == 0,
           "gemm_lse: operands and bias must be 16-byte aligned");
  HM_CHECK(bias != nullptr && lse.tokens != nullptr && lse.partials != nullptr, "gemm_lse: null buffer");
  HM_CHECK(lse.T >= 1 && lse.ld_tok > lse.T && M % lse.T == 0 && lse.n_valid >= 1 && lse.n_valid <= N,
           "gemm_lse: bad target geometry M=%d T=%d ld_tok=%d n_valid=%d N=%d", M, lse.T, lse.ld_tok, lse.n_valid, N);
  return launch_lse(stream, A, lda, M, K, W, N, bias, lse);
}

}  // namespace hmocr
