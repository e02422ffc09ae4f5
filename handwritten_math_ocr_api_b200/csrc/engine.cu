// Engine: weights, scratch memory, the encoder / decoder / generate schedules and the C ABI
// declared in include/hmocr.h.
#include <stdarg.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "decode_persistent.cuh"
#include "gemm.cuh"
#include "hmocr.h"
#include "kernels.cuh"

#include <nvtx3/nvToolsExt.h>      // header-only; ranges are no-ops unless a profiler injects the NVTX library

#define HM_API extern "C" __attribute__((visibility("default")))

namespace hmocr {

thread_local long g_launch_count = 0;
static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

namespace {

// NVTX ranges around the phases of a generate call (SURVEY.md section 5): encode / cross-KV / decode launch k
inline void nvtx_push(const char* name) { nvtxRangePushA(name); }
inline void nvtx_pop() { nvtxRangePop(); }

constexpr int IMG_H = 96, IMG_W = 320, SWIN_OUT = 768;
constexpr int RES18_MEM = 10, SWIN_MEM = 30;
constexpr int RES18_C[4] = {64, 128, 256, 512};
constexpr int RES18_STRIDE[4] = {1, 2, 2, 2};
constexpr int DEPTHS[4] = {2, 2, 6, 2};
constexpr int HEADS[4] = {3, 6, 12, 24};
constexpr int STEP_CHUNK = 8;     // decode steps between early-exit polls

struct HostTensor {
  std::vector<float> f;
  std::vector<int64_t> i;
  std::vector<int64_t> shape;
};

struct Lin {
  h16* w = nullptr;   // [n, k] fp16 (n padded to a multiple of 32 with zero rows)
  float* b = nullptr;           // [n] fp32 or nullptr
  int n = 0, k = 0;
};
struct Norm { float* g = nullptr; float* b = nullptr; };
struct SwinBlock { Norm n1, n2; Lin qkv, proj, fc1, fc2; float* rel_bias = nullptr; };
struct Merge { Norm norm; Lin red; };
struct DecLayer { Lin sa_in, sa_out, ca_q, ca_out, l1, l2; Norm n1, n2, n3; };
struct EncLayer { Lin in_proj, out_proj, l1, l2; Norm n1, n2; };        // ResNet variant: nn.TransformerEncoderLayer
struct ResBlock { Lin conv1, conv2, down; bool has_down = false; };      // BasicBlock, BatchNorm folded

struct Buf {
  void* p = nullptr;
  size_t cap = 0;
};

}  // namespace
}  // namespace hmocr

using namespace hmocr;

struct hmocr_engine {
  hmocr_config cfg;
  int device = 0;
  int vpad = 0;                       // vocab padded to a multiple of 256
  std::map<std::string, HostTensor> host;
  bool finalized = false;

  // device weights (one arena)
  uint8_t* arena = nullptr;
  size_t arena_cap = 0, arena_used = 0;
  float *pe_w = nullptr, *pe_b = nullptr;
  Norm pe_norm;
  SwinBlock blocks[12];
  Merge merges[3];
  Lin proj;
  float *emb = nullptr, *pos = nullptr;
  std::vector<DecLayer> layers;
  // ResNet-18 + TransformerEncoder variant (cfg.encoder_arch == 1)
  int mem_len = SWIN_MEM;             // memory tokens per image: 30 (Swin-T) / 10 (ResNet-18 variant)
  float *r18_w1 = nullptr, *r18_b1 = nullptr;     // conv1 7x7 with bn1 folded: [64][49], [64]
  ResBlock r18_blocks[8];
  Lin r18_proj;
  std::vector<EncLayer> enc_layers;
  float* pos_table = nullptr;         // [10][d] device copy of the positional table given by hmocr_set_pos_table
  bool pos_table_set = false;
  Lin ca_kv;                          // stacked cross-attention K/V projection of all layers [L*2d, d]
  Lin fc;
  // packed operands of the persistent cluster decode kernel (decode_persistent.cuh)
  uint8_t* dp_wstream = nullptr;
  float* dp_lnparams = nullptr;
  int dp_fc_tiles = 0, dp_chunks_per_step = 0;
  int decode_impl = 0;                // 0 = persistent cluster kernel, 1 = per-kernel step graph
  int steps_per_launch = 0;           // 0 = automatic (see generate_persistent)
  int trace_step = -1;                // >= 0: record phase-boundary clocks of that decode step
  int conv_impl = 0;                  // ResNet trunk: 0 = implicit GEMM (TMA patches), 1 = explicit im2col + GEMM
  int mlp_fused = 1;                  // Swin stages 1/2: fc1 + GELU + fc2 + residual in one kernel (0 = two GEMM launches)

  // Scratch buffers, addressed by name; any (re)placement invalidates the captured graphs (ws_epoch).
  //  * caller-owned (SURVEY.md 8b "Ownership"): hmocr_set_workspace hands the engine ONE buffer (a torch tensor on the
  //    Python side, sized by hmocr_workspace_bytes); names are bump-allocated inside it and the engine allocates nothing.
  //  * engine-owned (no hmocr_set_workspace call): stream-ordered cudaMallocAsync / cudaFreeAsync on the caller's
  //    stream - no cudaDeviceSynchronize, no device-wide stall on growth.
  std::map<std::string, Buf> ws;
  uint64_t ws_epoch = 0;
  uint8_t* ext_ws = nullptr;          // caller-owned pool
  size_t ext_cap = 0, ext_used = 0;
  cudaStream_t cur_stream = nullptr;  // stream of the API call in progress (engine-owned allocations are ordered on it)
  bool planning = false;              // hmocr_workspace_bytes: the schedules only record their buffer sizes
  std::map<std::string, size_t> plan;
  std::map<std::string, size_t> planned;   // per-buffer maximum over every hmocr_workspace_bytes call: placements use it,
                                           // so a small call followed by a large one never places a buffer twice

  struct StepGraph { cudaGraphExec_t exec = nullptr; uint64_t epoch = 0; };
  std::map<long long, StepGraph> graphs;   // key: rows
  // small batches: the ~95 encoder kernels are launch-bound, so generate() replays them as one captured graph
  struct EncGraph { cudaGraphExec_t exec = nullptr; uint64_t epoch = 0; bool warm = false; long launches = 0; };
  std::map<int, EncGraph> enc_graphs;      // key: batch
  int encoder_graph = 1;                   // option "encoder_graph": 0 disables (falls back by itself if capture fails)
  cudaStream_t cap_stream = nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};   // enc start, enc end, dec end, poll
  cudaEvent_t poll_ev[2] = {nullptr, nullptr};
  DecodeState* pinned_state = nullptr;   // [2]
  int last_poll_slot = -1;               // pinned_state slot that receives the state after the LAST persistent-kernel launch
  float last_enc_ms = 0.f, last_dec_ms = 0.f;
  bool timings_pending = false;
};

namespace hmocr {
namespace {

constexpr size_t WS_ALIGN = 256;
inline size_t ws_round(size_t b) { return (b + WS_ALIGN - 1) / WS_ALIGN * WS_ALIGN; }
// image staging of the preprocessing entry points: sized by the caller's IMAGE, not by (batch, max_len, beam), so it
// is not part of hmocr_workspace_bytes and always engine-owned (stream-ordered)
inline bool ws_pool_exempt(const char* name) { return name[0] == 'p' && name[1] == 'p' && name[2] == '.'; }

template <class T>
int ws_get(hmocr_engine* e, const char* name, size_t count, T** out) {
  const size_t bytes = ws_round(count * sizeof(T) + 1);
  if (e->planning) {
    size_t& need = e->plan[name];
    if (need < bytes) need = bytes;
    *out = reinterpret_cast<T*>(WS_ALIGN);      // never dereferenced: every schedule returns right after its ws_get calls
    return 0;
  }
  Buf& b = e->ws[name];
  if (b.cap < bytes) {
    if (e->ext_ws != nullptr && !ws_pool_exempt(name)) {
      const size_t off = ws_round(e->ext_used);
      auto pl = e->planned.find(name);
      const size_t bytes_now = bytes;
      const size_t bytes = (pl != e->planned.end() && pl->second > bytes_now) ? pl->second : bytes_now;
      HM_CHECK(off + bytes <= e->ext_cap,
               "caller-owned workspace too small for '%s' (%zu + %zu > %zu bytes): size it with hmocr_workspace_bytes for "
               "the largest (batch, max_len, beam) you call with", name, off, bytes, e->ext_cap);
      b.p = e->ext_ws + off;
      b.cap = bytes;
      e->ext_used = off + bytes;
    } else {
      if (b.p != nullptr) {
        HM_CUDA(cudaFreeAsync(b.p, e->cur_stream));      // ordered after the kernels already enqueued on this stream
        b.p = nullptr;
        b.cap = 0;
      }
      const size_t want = ws_round(bytes + bytes / 8);
      HM_CUDA(cudaMallocAsync(&b.p, want, e->cur_stream));
      b.cap = want;
    }
    ++e->ws_epoch;
  }
  *out = reinterpret_cast<T*>(b.p);
  return 0;
}

int arena_alloc(hmocr_engine* e, size_t bytes, void** out) {
  const size_t off = (e->arena_used + 255) & ~size_t(255);
  HM_CHECK(off + bytes <= e->arena_cap, "weight arena overflow (%zu + %zu > %zu)", off, bytes, e->arena_cap);
  *out = e->arena + off;
  e->arena_used = off + bytes;
  return 0;
}

const HostTensor* find(hmocr_engine* e, const std::string& key) {
  auto it = e->host.find(key);
  return it == e->host.end() ? nullptr : &it->second;
}

int need(hmocr_engine* e, const std::string& key, std::vector<int64_t> shape, const HostTensor** out) {
  const HostTensor* t = find(e, key);
  HM_CHECK(t != nullptr, "missing state-dict entry '%s'", key.c_str());
  HM_CHECK(t->shape == shape, "state-dict entry '%s' has the wrong shape", key.c_str());
  HM_CHECK(!t->f.empty(), "state-dict entry '%s' must be float32", key.c_str());
  *out = t;
  return 0;
}

// host-side fp32 -> fp16, saturating like the device conversions
inline h16 host_to_h16(float v) { return __float2half(v > 65504.f ? 65504.f : (v < -65504.f ? -65504.f : v)); }

int upload_f32(hmocr_engine* e, const float* src, size_t n, float** out) {
  void* p;
  HM_TRY(arena_alloc(e, n * sizeof(float), &p));
  HM_CUDA(cudaMemcpy(p, src, n * sizeof(float), cudaMemcpyHostToDevice));
  *out = reinterpret_cast<float*>(p);
  return 0;
}

int upload_vec(hmocr_engine* e, const std::string& key, int64_t n, float** out) {
  const HostTensor* t;
  HM_TRY(need(e, key, {n}, &t));
  return upload_f32(e, t->f.data(), (size_t)n, out);
}

int upload_norm(hmocr_engine* e, const std::string& prefix, int64_t n, Norm* out) {
  HM_TRY(upload_vec(e, prefix + ".weight", n, &out->g));
  return upload_vec(e, prefix + ".bias", n, &out->b);
}

// rows [r0, r0+rows) of a [*, k] fp32 matrix -> fp16 [npad, k] (zero padded), bias likewise
int upload_lin_rows(hmocr_engine* e, const float* w, const float* b, int rows, int k, Lin* out) {
  const int npad = (rows + 31) / 32 * 32;
  std::vector<h16> tmp((size_t)npad * k, host_to_h16(0.f));
  for (size_t i = 0; i < (size_t)rows * k; ++i) tmp[i] = host_to_h16(w[i]);
  void* p;
  HM_TRY(arena_alloc(e, tmp.size() * 2, &p));
  HM_CUDA(cudaMemcpy(p, tmp.data(), tmp.size() * 2, cudaMemcpyHostToDevice));
  out->w = reinterpret_cast<h16*>(p);
  out->n = npad;
  out->k = k;
  out->b = nullptr;
  if (b != nullptr) {
    std::vector<float> bt(npad, 0.f);
    memcpy(bt.data(), b, sizeof(float) * rows);
    HM_TRY(upload_f32(e, bt.data(), npad, &out->b));
  }
  return 0;
}

int upload_lin(hmocr_engine* e, const std::string& prefix, int n, int k, bool bias, Lin* out) {
  const HostTensor *w, *b = nullptr;
  HM_TRY(need(e, prefix + ".weight", {n, k}, &w));
  if (bias) HM_TRY(need(e, prefix + ".bias", {n}, &b));
  return upload_lin_rows(e, w->f.data(), b ? b->f.data() : nullptr, n, k, out);
}

// eval-mode BatchNorm folded into the preceding bias-free convolution: y = conv(x) * g / sqrt(var + eps) + (b - mean * g / sqrt(var + eps))
int fold_bn(hmocr_engine* e, const std::string& bn, int cout, std::vector<float>* scale, std::vector<float>* shift) {
  const HostTensor *g, *b, *m, *v;
  HM_TRY(need(e, bn + ".weight", {cout}, &g));
  HM_TRY(need(e, bn + ".bias", {cout}, &b));
  HM_TRY(need(e, bn + ".running_mean", {cout}, &m));
  HM_TRY(need(e, bn + ".running_var", {cout}, &v));
  scale->resize(cout); shift->resize(cout);
  for (int i = 0; i < cout; ++i) {
    const float sc = g->f[i] / sqrtf(v->f[i] + 1e-5f);
    (*scale)[i] = sc;
    (*shift)[i] = b->f[i] - m->f[i] * sc;
  }
  return 0;
}

// conv weight [cout, cin, k, k] (+ folded BN) -> GEMM weight [cout, (ky, kx, cin)] matching im2col's column order
int upload_conv(hmocr_engine* e, const std::string& conv, const std::string& bn, int cout, int cin, int k, Lin* out) {
  const HostTensor* w;
  HM_TRY(need(e, conv + ".weight", {cout, cin, k, k}, &w));
  std::vector<float> scale, shift;
  HM_TRY(fold_bn(e, bn, cout, &scale, &shift));
  std::vector<float> m((size_t)cout * k * k * cin);
  for (int o = 0; o < cout; ++o)
    for (int ci = 0; ci < cin; ++ci)
      for (int ky = 0; ky < k; ++ky)
        for (int kx = 0; kx < k; ++kx)
          m[(size_t)o * k * k * cin + (size_t)(ky * k + kx) * cin + ci] =
              w->f[(((size_t)o * cin + ci) * k + ky) * k + kx] * scale[o];
  return upload_lin_rows(e, m.data(), shift.data(), cout, k * k * cin, out);
}

int load_res18_weights(hmocr_engine* e) {
  const hmocr_config& c = e->cfg;
  const int d = c.d_model, ff = c.dim_feedforward;
  const std::string f = "encoder.features.";
  {
    const HostTensor* w;
    HM_TRY(need(e, f + "0.weight", {64, 1, 7, 7}, &w));
    std::vector<float> scale, shift;
    HM_TRY(fold_bn(e, f + "1", 64, &scale, &shift));
    std::vector<float> w1(64 * 49);
    for (int o = 0; o < 64; ++o)
      for (int i = 0; i < 49; ++i) w1[o * 49 + i] = w->f[o * 49 + i] * scale[o];
    HM_TRY(upload_f32(e, w1.data(), w1.size(), &e->r18_w1));
    HM_TRY(upload_f32(e, shift.data(), shift.size(), &e->r18_b1));
  }
  int cin = 64;
  for (int sidx = 0; sidx < 4; ++sidx) {
    const int cout = RES18_C[sidx];
    for (int j = 0; j < 2; ++j) {
      const std::string p = f + std::to_string(4 + sidx) + "." + std::to_string(j) + ".";
      ResBlock& rb = e->r18_blocks[sidx * 2 + j];
      HM_TRY(upload_conv(e, p + "conv1", p + "bn1", cout, j == 0 ? cin : cout, 3, &rb.conv1));
      HM_TRY(upload_conv(e, p + "conv2", p + "bn2", cout, cout, 3, &rb.conv2));
      rb.has_down = find(e, p + "downsample.0.weight") != nullptr;
      if (rb.has_down) HM_TRY(upload_conv(e, p + "downsample.0", p + "downsample.1", cout, cin, 1, &rb.down));
    }
    cin = cout;
  }
  HM_TRY(upload_lin(e, "encoder.projection", d, 512, true, &e->r18_proj));
  // config.res18trans_num_encoder_layers is independent of the decoder depth (src/config.py:28-29)
  const int enc_layers = c.enc_num_layers > 0 ? c.enc_num_layers : c.num_layers;
  HM_CHECK(find(e, "encoder.transformer_encoder.layers." + std::to_string(enc_layers) + ".linear1.weight") == nullptr,
           "checkpoint has more than %d TransformerEncoder layers: set hmocr_config.enc_num_layers "
           "(config.res18trans_num_encoder_layers)", enc_layers);
  e->enc_layers.resize(enc_layers);
  for (int l = 0; l < enc_layers; ++l) {
    const std::string p = "encoder.transformer_encoder.layers." + std::to_string(l) + ".";
    EncLayer& L = e->enc_layers[l];
    const HostTensor *w, *b;
    HM_TRY(need(e, p + "self_attn.in_proj_weight", {3 * d, d}, &w));
    HM_TRY(need(e, p + "self_attn.in_proj_bias", {3 * d}, &b));
    HM_TRY(upload_lin_rows(e, w->f.data(), b->f.data(), 3 * d, d, &L.in_proj));
    HM_TRY(upload_lin(e, p + "self_attn.out_proj", d, d, true, &L.out_proj));
    HM_TRY(upload_lin(e, p + "linear1", ff, d, true, &L.l1));
    HM_TRY(upload_lin(e, p + "linear2", d, ff, true, &L.l2));
    HM_TRY(upload_norm(e, p + "norm1", d, &L.n1));
    HM_TRY(upload_norm(e, p + "norm2", d, &L.n2));
  }
  void* pt;
  HM_TRY(arena_alloc(e, sizeof(float) * RES18_MEM * d, &pt));
  e->pos_table = static_cast<float*>(pt);
  return 0;
}

int run_lin(cudaStream_t st, const h16* a, int lda, int M, const Lin& l, GemmEpilogue epi) {
  epi.bias = l.b;
  return gemm_f16(st, a, lda, M, l.k, l.w, l.n, epi);
}

// ------------------------------------------------------------------------------------------------
// encoder schedule            /root/reference/src/model_swin.py:39-46 over swin_t.features
// ------------------------------------------------------------------------------------------------
int encode_impl(hmocr_engine* e, const float* images, int B, float* enc32, h16* enc16, cudaStream_t st) {
  const size_t tok1 = (size_t)B * 24 * 80;
  float *xa, *xb;
  h16 *xn, *qkv, *ctx, *hid;
  HM_TRY(ws_get(e, "enc.xa", tok1 * 96, &xa));
  HM_TRY(ws_get(e, "enc.xb", tok1 * 96 / 2, &xb));
  HM_TRY(ws_get(e, "enc.xn", tok1 * 96, &xn));
  HM_TRY(ws_get(e, "enc.qkv", tok1 * 288, &qkv));
  HM_TRY(ws_get(e, "enc.ctx", tok1 * 96, &ctx));
  HM_TRY(ws_get(e, "enc.hid", tok1 * 384, &hid));
  if (e->planning) return 0;

  HM_TRY(patch_embed(st, images, B, e->pe_w, e->pe_b, e->pe_norm.g, e->pe_norm.b, xa));
  int H = 24, W = 80, C = 96, blk = 0;
  float* x = xa;
  float* other = xb;
  for (int s = 0; s < 4; ++s) {
    const int rows = B * H * W;
    for (int j = 0; j < DEPTHS[s]; ++j, ++blk) {
      const SwinBlock& sb = e->blocks[blk];
      HM_TRY(layernorm(st, x, rows, C, sb.n1.g, sb.n1.b, xn, nullptr));
      GemmEpilogue eq;
      eq.out_f16 = qkv; eq.ld16 = 3 * C;
      HM_TRY(run_lin(st, xn, C, rows, sb.qkv, eq));
      HM_TRY(window_attention(st, qkv, sb.qkv.b, sb.rel_bias, B, H, W, C, HEADS[s], (j & 1) ? 3 : 0, ctx));
      GemmEpilogue ep;
      ep.residual = x; ep.ldr = C; ep.out_f32 = x; ep.ld32 = C;
      HM_TRY(run_lin(st, ctx, C, rows, sb.proj, ep));
      HM_TRY(layernorm(st, x, rows, C, sb.n2.g, sb.n2.b, xn, nullptr));
      if (e->mlp_fused && swin_mlp_supported(C)) {       // the [rows, 4C] hidden tensor never reaches HBM
        HM_TRY(swin_mlp(st, xn, rows, C, sb.fc1.w, sb.fc1.b, sb.fc2.w, sb.fc2.b, x));
      } else {
        GemmEpilogue e1;
        e1.act = 1; e1.out_f16 = hid; e1.ld16 = 4 * C;
        HM_TRY(run_lin(st, xn, C, rows, sb.fc1, e1));
        GemmEpilogue e2;
        e2.residual = x; e2.ldr = C; e2.out_f32 = x; e2.ld32 = C;
        HM_TRY(run_lin(st, hid, 4 * C, rows, sb.fc2, e2));
      }
    }
    if (s < 3) {
      const Merge& m = e->merges[s];
      HM_TRY(patch_merge_ln(st, x, B, H, W, C, m.norm.g, m.norm.b, xn));
      GemmEpilogue em;
      em.out_f32 = other; em.ld32 = 2 * C;
      HM_TRY(run_lin(st, xn, 4 * C, rows / 4, m.red, em));
      float* t = x; x = other; other = t;
      // the smaller buffer (xb) can hold every later stage; keep ping-ponging between xa and xb
      H /= 2; W /= 2; C *= 2;
    }
  }
  const int rows = B * e->mem_len;
  HM_TRY(f32_to_f16(st, x, (size_t)rows * SWIN_OUT, xn));
  GemmEpilogue eo;
  eo.out_f32 = enc32; eo.ld32 = e->cfg.d_model;
  eo.out_f16 = enc16; eo.ld16 = e->cfg.d_model;
  HM_TRY(run_lin(st, xn, SWIN_OUT, rows, e->proj, eo));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// ResNet-18 + TransformerEncoder encoder      /root/reference/src/model_res18trans.py:48-64
// ------------------------------------------------------------------------------------------------
int conv_gemm(hmocr_engine* e, cudaStream_t st, const h16* x16, int B, int H, int W, int C, int k, int stride,
              const Lin& w, h16* col, GemmEpilogue epi) {
  const int pad = (k == 3) ? 1 : 0;
  const int Ho = (H + 2 * pad - k) / stride + 1, Wo = (W + 2 * pad - k) / stride + 1;
  int tw, th, tn;
  if (e->conv_impl == 0 && C % 64 == 0 && w.n % 64 == 0 && conv_tiling(Ho, Wo, &tw, &th, &tn)) {
    epi.bias = w.b;
    return gemm_conv_f16(st, x16, B, H, W, C, k, stride, pad, w.w, w.n, epi);       // implicit GEMM: TMA builds the patches
  }
  HM_TRY(im2col(st, x16, B, H, W, C, k, stride, pad, col));
  return run_lin(st, col, k * k * C, B * Ho * Wo, w, epi);
}

int encode_res18_impl(hmocr_engine* e, const float* images, int B, float* enc32, h16* enc16, cudaStream_t st) {
  const int d = e->cfg.d_model, ff = e->cfg.dim_feedforward, nh = e->cfg.nhead;
  HM_CHECK(e->planning || e->pos_table_set, "ResNet-18 variant: call hmocr_set_pos_table first - the reference draws a fresh "
                             "nn.Embedding(10, d_model) table on every encoder call (src/model_res18trans.py:57-59)");
  HM_CHECK(B <= 256, "ResNet-18 variant: the encoder attends ACROSS the batch (SURVEY.md D7); batch %d > 256 unsupported", B);
  const size_t m1 = (size_t)B * 24 * 80;                       // pixels after the stem
  h16 *stem, *xa16, *xb16, *h16b, *col;
  float *xa32, *xb32, *ds32;
  HM_TRY(ws_get(e, "r18.stem", (size_t)B * 48 * 160 * 64, &stem));
  HM_TRY(ws_get(e, "r18.xa16", m1 * 64, &xa16));
  HM_TRY(ws_get(e, "r18.xb16", m1 * 64, &xb16));
  HM_TRY(ws_get(e, "r18.h16", m1 * 64, &h16b));
  HM_TRY(ws_get(e, "r18.xa32", m1 * 64, &xa32));
  HM_TRY(ws_get(e, "r18.xb32", m1 * 64, &xb32));
  HM_TRY(ws_get(e, "r18.ds32", m1 * 64 / 2, &ds32));
  HM_TRY(ws_get(e, "r18.col", m1 * 576, &col));
  const int S = RES18_MEM, rows = B * S;
  h16 *pool16, *z16, *qkv, *ctx, *hid;
  float *q32, *z32;
  HM_TRY(ws_get(e, "r18.pool16", (size_t)rows * 512, &pool16));
  HM_TRY(ws_get(e, "r18.q32", (size_t)rows * d, &q32));
  HM_TRY(ws_get(e, "r18.z32", (size_t)rows * d, &z32));
  HM_TRY(ws_get(e, "r18.z16", (size_t)rows * d, &z16));
  HM_TRY(ws_get(e, "r18.qkv", (size_t)rows * 3 * d, &qkv));
  HM_TRY(ws_get(e, "r18.ctx", (size_t)rows * d, &ctx));
  HM_TRY(ws_get(e, "r18.hid", (size_t)rows * ff, &hid));
  if (e->planning) return 0;
  HM_TRY(conv7x7_bn_relu(st, images, B, e->r18_w1, e->r18_b1, stem));
  HM_TRY(maxpool3x3s2(st, stem, B, 48, 160, 64, xa16, xa32));
  int H = 24, W = 80, C = 64;
  h16 *x16 = xa16, *y16 = xb16;
  float *x32 = xa32, *y32 = xb32;
  for (int sidx = 0; sidx < 4; ++sidx) {
    for (int j = 0; j < 2; ++j) {
      const ResBlock& rb = e->r18_blocks[sidx * 2 + j];
      const int cout = RES18_C[sidx], stride = (j == 0) ? RES18_STRIDE[sidx] : 1;
      const int Ho = H / stride, Wo = W / stride, M = B * Ho * Wo;
      GemmEpilogue e1;                                         // relu(bn1(conv1(x)))
      e1.act = 2; e1.out_f16 = h16b; e1.ld16 = cout;
      HM_TRY(conv_gemm(e, st, x16, B, H, W, C, 3, stride, rb.conv1, col, e1));
      const float* identity = x32;
      if (rb.has_down) {                                       // bn(conv1x1(x)), stride 2
        GemmEpilogue ed;
        ed.out_f32 = ds32; ed.ld32 = cout;
        HM_TRY(conv_gemm(e, st, x16, B, H, W, C, 1, stride, rb.down, col, ed));
        identity = ds32;
      }
      GemmEpilogue e2;                                         // relu(bn2(conv2(.)) + identity)
      e2.act = 3; e2.residual = identity; e2.ldr = cout; e2.out_f32 = y32; e2.ld32 = cout; e2.out_f16 = y16; e2.ld16 = cout;
      HM_TRY(conv_gemm(e, st, h16b, B, Ho, Wo, cout, 3, 1, rb.conv2, col, e2));
      (void)M;
      h16* t16 = x16; x16 = y16; y16 = t16;
      float* t32 = x32; x32 = y32; y32 = t32;
      H = Ho; W = Wo; C = cout;
    }
  }
  // AdaptiveAvgPool2d((1, None)) -> Linear 512 -> d -> + positional table -> [10, B, d] -> 8 encoder layers over B
  HM_TRY(avgpool_h(st, x32, B, H, W, C, pool16));
  GemmEpilogue ep;
  ep.out_f32 = q32; ep.ld32 = d;
  HM_TRY(run_lin(st, pool16, 512, rows, e->r18_proj, ep));
  HM_TRY(add_pos_permute(st, q32, e->pos_table, B, S, d, z32, z16));
  for (size_t l = 0; l < e->enc_layers.size(); ++l) {
    const EncLayer& L = e->enc_layers[l];
    GemmEpilogue ei;
    ei.out_f16 = qkv; ei.ld16 = 3 * d;
    HM_TRY(run_lin(st, z16, d, rows, L.in_proj, ei));
    HM_TRY(mha_prefill_self(st, qkv, S, B, nh, ctx, /*causal=*/false));      // batch = 10 positions, sequence = B images
    GemmEpilogue e1;                                                          // x = LN1(x + out_proj(ctx))
    e1.residual = z32; e1.ldr = d; e1.out_f32 = z32; e1.ld32 = d; e1.out_f16 = z16; e1.ld16 = d;
    e1.ln_gamma = L.n1.g; e1.ln_beta = L.n1.b;
    HM_TRY(run_lin(st, ctx, d, rows, L.out_proj, e1));
    GemmEpilogue ef;
    ef.act = 2; ef.out_f16 = hid; ef.ld16 = ff;
    HM_TRY(run_lin(st, z16, d, rows, L.l1, ef));
    GemmEpilogue e2;                                                          // x = LN2(x + linear2(relu(linear1 x)))
    e2.residual = z32; e2.ldr = d; e2.out_f32 = z32; e2.ld32 = d; e2.out_f16 = z16; e2.ld16 = d;
    e2.ln_gamma = L.n2.g; e2.ln_beta = L.n2.b;
    HM_TRY(run_lin(st, hid, ff, rows, L.l2, e2));
  }
  return permute_back(st, z32, B, S, d, enc32, enc16);
}

// memory K/V of all layers in one GEMM: memkv[b*S+s, l*2d + {0..d-1: K, d..2d-1: V}]
int project_memory(hmocr_engine* e, const h16* enc16, int B, h16* memkv, cudaStream_t st) {
  GemmEpilogue ek;
  ek.out_f16 = memkv; ek.ld16 = e->ca_kv.n;
  return run_lin(st, enc16, e->cfg.d_model, B * e->mem_len, e->ca_kv, ek);
}

struct DecBufs {
  float* x32;
  h16 *x16, *qkv, *q, *ctx, *hid;
  float* logits;
};

// the activations of the layer stack; logits stays nullptr (hmocr_score keeps no logits)
int dec_layer_bufs(hmocr_engine* e, const char* tag, size_t rows, DecBufs* b) {
  const int d = e->cfg.d_model, ff = e->cfg.dim_feedforward;
  std::string t(tag);
  HM_TRY(ws_get(e, (t + ".x32").c_str(), rows * d, &b->x32));
  HM_TRY(ws_get(e, (t + ".x16").c_str(), rows * d, &b->x16));
  HM_TRY(ws_get(e, (t + ".qkv").c_str(), rows * 3 * d, &b->qkv));
  HM_TRY(ws_get(e, (t + ".q").c_str(), rows * d, &b->q));
  HM_TRY(ws_get(e, (t + ".ctx").c_str(), rows * d, &b->ctx));
  HM_TRY(ws_get(e, (t + ".hid").c_str(), rows * ff, &b->hid));
  b->logits = nullptr;
  return 0;
}

// the layer-stack activations plus the rows x vpad fp32 logits
int dec_bufs(hmocr_engine* e, const char* tag, size_t rows, DecBufs* b) {
  HM_TRY(dec_layer_bufs(e, tag, rows, b));
  return ws_get(e, (std::string(tag) + ".logits").c_str(), rows * e->vpad, &b->logits);
}

// everything of one decoder layer after the self-attention context is in b.ctx
int layer_tail(hmocr_engine* e, const DecLayer& L, int l, const DecBufs& b, int rows, const h16* memkv,
               const int* mem_row, int T, cudaStream_t st) {
  const int d = e->cfg.d_model, ff = e->cfg.dim_feedforward, nh = e->cfg.nhead;
  GemmEpilogue e1;                       // x = LN1(x + out_proj(ctx))
  e1.residual = b.x32; e1.ldr = d; e1.out_f32 = b.x32; e1.ld32 = d; e1.out_f16 = b.x16; e1.ld16 = d;
  e1.ln_gamma = L.n1.g; e1.ln_beta = L.n1.b;
  HM_TRY(run_lin(st, b.ctx, d, rows, L.sa_out, e1));
  GemmEpilogue eq;
  eq.out_f16 = b.q; eq.ld16 = d;
  HM_TRY(run_lin(st, b.x16, d, rows, L.ca_q, eq));
  if (T > 0)
    HM_TRY(mha_prefill_cross(st, b.q, memkv, e->ca_kv.n, l * 2 * d, l * 2 * d + d, rows / T, T, e->mem_len, nh, b.ctx));
  else
    HM_TRY(cross_attn_step(st, b.q, memkv, e->ca_kv.n, l * 2 * d, l * 2 * d + d, mem_row, rows, e->mem_len, nh, b.ctx));
  GemmEpilogue e2;                       // x = LN2(x + out_proj(ctx))
  e2.residual = b.x32; e2.ldr = d; e2.out_f32 = b.x32; e2.ld32 = d; e2.out_f16 = b.x16; e2.ld16 = d;
  e2.ln_gamma = L.n2.g; e2.ln_beta = L.n2.b;
  HM_TRY(run_lin(st, b.ctx, d, rows, L.ca_out, e2));
  GemmEpilogue ef;
  ef.act = 2; ef.out_f16 = b.hid; ef.ld16 = ff;
  HM_TRY(run_lin(st, b.x16, d, rows, L.l1, ef));
  GemmEpilogue e3;                       // x = LN3(x + linear2(relu(linear1 x)))
  e3.residual = b.x32; e3.ldr = d; e3.out_f32 = b.x32; e3.ld32 = d; e3.out_f16 = b.x16; e3.ld16 = d;
  e3.ln_gamma = L.n3.g; e3.ln_beta = L.n3.b;
  HM_TRY(run_lin(st, b.hid, ff, rows, L.l2, e3));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// teacher-forced decoder       /root/reference/src/model_swin.py:72-88
// ------------------------------------------------------------------------------------------------
// The layer stack of the teacher-forced paths: memory K/V of all layers, x = embedding[tok[b, t]] + pos[t] for t < T
// (tok row pitch ld_tok), then the L layers; the last hidden state is in b.x16.  enc32 != nullptr: the memory is the
// caller's fp32 encoder output and is converted into enc16 first; enc32 == nullptr: enc16 already holds it.
int decoder_layers(hmocr_engine* e, const float* enc32, h16* enc16, h16* memkv, const int64_t* tok, int ld_tok, int B,
                   int T, const DecBufs& b, cudaStream_t st) {
  const int d = e->cfg.d_model, nh = e->cfg.nhead;
  const int rows = B * T;
  if (enc32 != nullptr) HM_TRY(f32_to_f16(st, enc32, (size_t)B * e->mem_len * d, enc16));
  HM_TRY(project_memory(e, enc16, B, memkv, st));
  HM_TRY(embed_tokens(st, tok, ld_tok, B, T, e->emb, e->pos, d, e->cfg.vocab_size, b.x32, b.x16));
  for (int l = 0; l < e->cfg.num_layers; ++l) {
    const DecLayer& L = e->layers[l];
    GemmEpilogue ei;
    ei.out_f16 = b.qkv; ei.ld16 = 3 * d;
    HM_TRY(run_lin(st, b.x16, d, rows, L.sa_in, ei));
    HM_TRY(mha_prefill_self(st, b.qkv, B, T, nh, b.ctx));
    HM_TRY(layer_tail(e, L, l, b, rows, memkv, nullptr, T, st));
  }
  return 0;
}

int decoder_forward_impl(hmocr_engine* e, const float* enc32, const int64_t* tgt, int B, int T, float* logits,
                         cudaStream_t st) {
  const int d = e->cfg.d_model;
  const int rows = B * T;
  h16 *enc16, *memkv;
  HM_TRY(ws_get(e, "tf.enc16", (size_t)B * e->mem_len * d, &enc16));
  HM_TRY(ws_get(e, "tf.memkv", (size_t)B * e->mem_len * e->ca_kv.n, &memkv));
  DecBufs b;
  HM_TRY(dec_bufs(e, "tf", rows, &b));
  if (e->planning) return 0;
  HM_TRY(decoder_layers(e, enc32, enc16, memkv, tgt, T, B, T, b, st));
  GemmEpilogue eo;
  eo.out_f32 = b.logits; eo.ld32 = e->vpad;
  HM_TRY(run_lin(st, b.x16, d, rows, e->fc, eo));
  HM_TRY(copy_logits(st, b.logits, e->vpad, rows, e->cfg.vocab_size, logits));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// greedy generate              /root/reference/src/inference.py:15-25 with a KV cache
// ------------------------------------------------------------------------------------------------
struct GenBufs {
  DecBufs b;
  h16 *kcache, *vcache;   // [L][rows][nhead][tmax][32]
  DecodeState* state;
  uint8_t* finished;
  int tmax;
};

int enqueue_step(hmocr_engine* e, const GenBufs& g, int rows, const h16* memkv, int64_t* tokens,
                 float* logprob, int max_len, cudaStream_t st) {
  const int d = e->cfg.d_model, nh = e->cfg.nhead;
  const size_t layer_stride = (size_t)rows * nh * g.tmax * 32;
  for (int l = 0; l < e->cfg.num_layers; ++l) {
    const DecLayer& L = e->layers[l];
    GemmEpilogue ei;
    ei.out_f16 = g.b.qkv; ei.ld16 = 3 * d;
    HM_TRY(run_lin(st, g.b.x16, d, rows, L.sa_in, ei));
    HM_TRY(self_attn_step(st, g.state, g.b.qkv, g.kcache + l * layer_stride, g.vcache + l * layer_stride, rows, nh,
                          g.tmax, g.b.ctx));
    HM_TRY(layer_tail(e, L, l, g.b, rows, memkv, nullptr, 0, st));
  }
  GemmEpilogue eo;
  eo.out_f32 = g.b.logits; eo.ld32 = e->vpad;
  HM_TRY(run_lin(st, g.b.x16, d, rows, e->fc, eo));
  HM_TRY(greedy_select(st, g.state, g.b.logits, e->vpad, e->cfg.vocab_size, rows, tokens, max_len + 1, logprob,
                       max_len, e->cfg.eos_id, g.finished, e->emb, e->pos, d, e->cfg.max_seq_len, g.b.x32, g.b.x16));
  HM_TRY(advance_step(st, g.state));
  return 0;
}

int generate_persistent(hmocr_engine* e, const h16* enc16, int B, int max_len, int beam, int64_t* tokens,
                        float* logprob, int32_t* steps, float* score, cudaStream_t st, int n_best);

// n_best == 0: the hmocr_generate contract (best hypothesis only; logprob zero-filled in beam mode).
// n_best >= 1: the hmocr_generate_nbest contract (beam machinery always; tokens / logprob / score hold n_best
// hypotheses per image).  The step-graph decode is greedy only, so n-best always takes the persistent kernel.
int generate_from_memory_impl(hmocr_engine* e, const h16* enc16, int B, int max_len, int beam,
                              int64_t* tokens, float* logprob, int32_t* steps, float* score, cudaStream_t st,
                              int n_best = 0) {
  HM_CHECK(max_len >= 1 && max_len <= e->cfg.max_seq_len,
           "max_len=%d outside [1, %d] (size of pos_encoder, src/model_swin.py:54)", max_len, e->cfg.max_seq_len);
  HM_CHECK(beam >= 1 && beam <= DP_MAX_BEAM, "beam=%d outside [1, %d]", beam, DP_MAX_BEAM);
  // The beam kernel merges per-hypothesis top-`beam` token lists; with fewer tokens than hypotheses a list has empty
  // slots, and the candidate built from one (hyp * vocab + 0x7fffffff) overflows into a negative parent index.
  HM_CHECK(beam <= e->cfg.vocab_size, "beam=%d exceeds vocab_size=%d", beam, e->cfg.vocab_size);
  if (e->decode_impl == 0 || n_best > 0)
    return generate_persistent(e, enc16, B, max_len, beam, tokens, logprob, steps, score, st, n_best);
  HM_CHECK(beam == 1, "the step-graph decode (decode_impl=1) is greedy only; beam=%d needs decode_impl=0", beam);
  const int d = e->cfg.d_model, nh = e->cfg.nhead, L = e->cfg.num_layers;
  const int rows = B;
  h16* memkv;
  HM_TRY(ws_get(e, "gen.memkv", (size_t)B * e->mem_len * e->ca_kv.n, &memkv));
  GenBufs g;
  g.tmax = e->cfg.max_seq_len;
  HM_TRY(dec_bufs(e, "gen", rows, &g.b));
  const size_t cache_elems = (size_t)L * rows * nh * g.tmax * 32;
  HM_TRY(ws_get(e, "gen.kcache", cache_elems, &g.kcache));
  HM_TRY(ws_get(e, "gen.vcache", cache_elems, &g.vcache));
  HM_TRY(ws_get(e, "gen.state", 1, &g.state));
  HM_TRY(ws_get(e, "gen.finished", rows, &g.finished));
  // per-call output pointers are baked into the step graph: stage them in engine-owned buffers
  int64_t* tok_ws;
  float* lp_ws;
  HM_TRY(ws_get(e, "gen.tokens", (size_t)rows * (g.tmax + 1), &tok_ws));
  HM_TRY(ws_get(e, "gen.logprob", (size_t)rows * g.tmax, &lp_ws));
  if (e->planning) return 0;

  HM_TRY(project_memory(e, enc16, B, memkv, st));
  HM_TRY(init_decode(st, g.state, tok_ws, max_len + 1, rows, e->cfg.sos_id, e->cfg.pad_id, g.finished, lp_ws, max_len));
  HM_TRY(embed_tokens(st, tok_ws, max_len + 1, rows, 1, e->emb, e->pos, d, e->cfg.vocab_size, g.b.x32, g.b.x16));

  // one decode step captured once per (rows, max_len) and replayed: the step index lives in HBM
  const long long key = (long long)rows * 1024 + max_len;
  hmocr_engine::StepGraph& sg = e->graphs[key];
  if (sg.exec == nullptr || sg.epoch != e->ws_epoch) {
    if (sg.exec != nullptr) { cudaGraphExecDestroy(sg.exec); sg.exec = nullptr; }
    cudaGraph_t graph = nullptr;
    HM_CUDA(cudaStreamBeginCapture(e->cap_stream, cudaStreamCaptureModeThreadLocal));
    const long launches_before = g_launch_count;
    int rc = enqueue_step(e, g, rows, memkv, tok_ws, lp_ws, max_len, e->cap_stream);
    g_launch_count = launches_before;            // captured, not launched
    cudaError_t ce = cudaStreamEndCapture(e->cap_stream, &graph);
    if (rc != 0) { if (graph) cudaGraphDestroy(graph); return rc; }
    HM_CUDA(ce);
    ce = cudaGraphInstantiate(&sg.exec, graph, 0);
    cudaGraphDestroy(graph);
    HM_CUDA(ce);
    sg.epoch = e->ws_epoch;
  }
  size_t nodes_per_step = 8 * (size_t)L + 3;
  int launched_steps = 0, poll_idx = 0;
  bool done = false;
  for (int s0 = 0; s0 < max_len && !done; s0 += STEP_CHUNK, ++poll_idx) {
    const int n = (max_len - s0 < STEP_CHUNK) ? (max_len - s0) : STEP_CHUNK;
    for (int i = 0; i < n; ++i) {
      HM_CUDA(cudaGraphLaunch(sg.exec, st));
      g_launch_count += (long)nodes_per_step;
    }
    launched_steps += n;
    const int slot = poll_idx & 1;
    HM_CUDA(cudaMemcpyAsync(&e->pinned_state[slot], g.state, sizeof(DecodeState), cudaMemcpyDeviceToHost, st));
    HM_CUDA(cudaEventRecord(e->poll_ev[slot], st));
    if (poll_idx >= 1) {                         // look at the chunk before: the GPU never idles
      const int prev = (poll_idx - 1) & 1;
      HM_CUDA(cudaEventSynchronize(e->poll_ev[prev]));
      if (e->pinned_state[prev].steps_executed > 0) done = true;   // every row has emitted eos
    }
  }
  (void)launched_steps;
  HM_TRY(finalize_decode(st, g.state, tok_ws, max_len + 1, rows, max_len, e->cfg.pad_id, lp_ws, steps));
  HM_CUDA(cudaMemcpyAsync(tokens, tok_ws, sizeof(int64_t) * rows * (max_len + 1), cudaMemcpyDeviceToDevice, st));
  if (logprob != nullptr)
    HM_CUDA(cudaMemcpyAsync(logprob, lp_ws, sizeof(float) * rows * max_len, cudaMemcpyDeviceToDevice, st));
  return 0;
}


// ------------------------------------------------------------------------------------------------
// operand packing for decode_persistent.cu (host side, once at load)
// ------------------------------------------------------------------------------------------------
// 16 weight rows [row0, row0+16) x 256 input columns [col0, col0+256) of a [valid_rows, K] fp32 matrix -> one
// stream chunk (fp16 [16][264], zero padded)
// `bias` (may be null): fp32 bias of the same rows, stored in the padding of each row (halves 256, 257)
void pack_chunk(std::vector<__half>& dst, size_t off, const float* w, const float* bias, int row0, int col0, int K,
                int valid_rows) {
  for (int r = 0; r < DP_CH_ROWS; ++r) {
    for (int k = 0; k < 264; ++k) {
      const bool ok = (k < 256) && (row0 + r < valid_rows);
      dst[off + (size_t)r * 264 + k] = host_to_h16(ok ? w[(size_t)(row0 + r) * K + col0 + k] : 0.f);
    }
    const float b = (bias != nullptr && row0 + r < valid_rows) ? bias[row0 + r] : 0.f;
    memcpy(&dst[off + (size_t)r * 264 + 256], &b, sizeof(float));
  }
}

int pack_decode_operands(hmocr_engine* e) {
  const hmocr_config& c = e->cfg;
  const int d = c.d_model, ff = c.dim_feedforward, V = c.vocab_size, L = c.num_layers;
  HM_CHECK(d == 256 && ff == 512 && c.nhead == 8,
           "the persistent decode kernel is specialised for d_model=256, nhead=8, dim_feedforward=512 "
           "(reference config.py:19-21); got %d/%d/%d", d, c.nhead, ff);
  e->dp_fc_tiles = ((V + 127) / 128 + 7) / 8 * 8;      // 16-row tiles per CTA, a multiple of the 8 warps
  e->dp_chunks_per_step = DP_LAYER_CHUNKS * L + e->dp_fc_tiles;
  const size_t S = (size_t)e->dp_chunks_per_step, CE = DP_CHUNK / 2;        // chunk size in elements
  std::vector<__half> stream(8 * S * CE);
  std::vector<float> lnpar((size_t)L * 6 * d);
  for (int l = 0; l < L; ++l) {
    const std::string p = "decoder.decoder.layers." + std::to_string(l) + ".";
    const HostTensor *sin, *sinb, *so, *sob, *cin, *cinb, *co, *cob, *w1, *b1, *w2, *b2;
    HM_TRY(need(e, p + "self_attn.in_proj_weight", {3 * d, d}, &sin));
    HM_TRY(need(e, p + "self_attn.in_proj_bias", {3 * d}, &sinb));
    HM_TRY(need(e, p + "self_attn.out_proj.weight", {d, d}, &so));
    HM_TRY(need(e, p + "self_attn.out_proj.bias", {d}, &sob));
    HM_TRY(need(e, p + "multihead_attn.in_proj_weight", {3 * d, d}, &cin));
    HM_TRY(need(e, p + "multihead_attn.in_proj_bias", {3 * d}, &cinb));
    HM_TRY(need(e, p + "multihead_attn.out_proj.weight", {d, d}, &co));
    HM_TRY(need(e, p + "multihead_attn.out_proj.bias", {d}, &cob));
    HM_TRY(need(e, p + "linear1.weight", {ff, d}, &w1));
    HM_TRY(need(e, p + "linear1.bias", {ff}, &b1));
    HM_TRY(need(e, p + "linear2.weight", {d, ff}, &w2));
    HM_TRY(need(e, p + "linear2.bias", {d}, &b2));
    for (int ct = 0; ct < 8; ++ct) {
      size_t off = ((size_t)ct * S + (size_t)l * DP_LAYER_CHUNKS) * CE;
      for (int part = 0; part < 3; ++part)             // q, k, v rows of head ct
        for (int m = 0; m < 2; ++m, off += CE) pack_chunk(stream, off, sin->f.data(), sinb->f.data(), part * d + ct * 32 + 16 * m, 0, d, 3 * d);
      for (int m = 0; m < 2; ++m, off += CE) pack_chunk(stream, off, so->f.data(), sob->f.data(), ct * 32 + 16 * m, 0, d, d);
      for (int m = 0; m < 2; ++m, off += CE) pack_chunk(stream, off, cin->f.data(), cinb->f.data(), ct * 32 + 16 * m, 0, d, 3 * d);
      for (int m = 0; m < 2; ++m, off += CE) pack_chunk(stream, off, co->f.data(), cob->f.data(), ct * 32 + 16 * m, 0, d, d);
      for (int m = 0; m < 4; ++m, off += CE) pack_chunk(stream, off, w1->f.data(), b1->f.data(), ct * 64 + 16 * m, 0, d, ff);
      for (int m = 0; m < 2; ++m)
        for (int kh = 0; kh < 2; ++kh, off += CE) pack_chunk(stream, off, w2->f.data(), kh == 0 ? b2->f.data() : nullptr, ct * 32 + 16 * m, 256 * kh, ff, d);
    }
    const char* ln[3] = {"norm1", "norm2", "norm3"};
    for (int i = 0; i < 3; ++i) {
      const HostTensor *lg, *lb;
      HM_TRY(need(e, p + ln[i] + ".weight", {d}, &lg));
      HM_TRY(need(e, p + ln[i] + ".bias", {d}, &lb));
      memcpy(&lnpar[((size_t)l * 6 + 2 * i) * d], lg->f.data(), sizeof(float) * d);
      memcpy(&lnpar[((size_t)l * 6 + 2 * i + 1) * d], lb->f.data(), sizeof(float) * d);
    }
  }
  const int cols_per_cta = e->dp_fc_tiles * 16;
  {
    const HostTensor *w, *b;
    HM_TRY(need(e, "decoder.fc_out.weight", {V, d}, &w));
    HM_TRY(need(e, "decoder.fc_out.bias", {V}, &b));
    for (int ct = 0; ct < 8; ++ct)
      for (int m = 0; m < e->dp_fc_tiles; ++m)
        pack_chunk(stream, ((size_t)ct * S + (size_t)L * DP_LAYER_CHUNKS + m) * CE, w->f.data(), b->f.data(),
                   ct * cols_per_cta + 16 * m, 0, d, V);
  }
  void* q;
  HM_TRY(arena_alloc(e, stream.size() * 2, &q));
  HM_CUDA(cudaMemcpy(q, stream.data(), stream.size() * 2, cudaMemcpyHostToDevice));
  e->dp_wstream = static_cast<uint8_t*>(q);
  HM_TRY(upload_f32(e, lnpar.data(), lnpar.size(), &e->dp_lnparams));
  return 0;
}

// decode with the persistent cluster kernel: a few launches of `steps_per_launch` steps, the host only polls
// the all-finished flag of the PREVIOUS launch (the GPU never idles).  beam == 1: greedy
// (src/inference.py:15-25).  beam > 1 (or n_best > 0, at any beam): beam search as defined in
// oracle/decode.py::beam_search - rows = images x beam hypotheses, two K/V cache sets, back-track at the end.
int generate_persistent(hmocr_engine* e, const h16* enc16, int B, int max_len, int beam, int64_t* tokens,
                        float* logprob, int32_t* steps, float* score, cudaStream_t st, int n_best) {
  const int nh = e->cfg.nhead, L = e->cfg.num_layers, rows = B * beam;
  const bool beam_mode = beam > 1 || n_best > 0;
  HM_CHECK(beam >= 1 && beam <= DP_MAX_BEAM, "beam=%d outside [1, %d]", beam, DP_MAX_BEAM);
  float* memkv;                       // memory K/V of all layers, fp32 out of the GEMM, fp16 after the repack
  __half *memk, *memv, *kcache, *vcache;
  DecodeState* state;
  uint8_t* finished;
  const int tmax = e->cfg.max_seq_len, cache_blocks = (tmax + 31) / 32;
  HM_TRY(ws_get(e, "dp.memkv32", (size_t)B * e->mem_len * e->ca_kv.n, &memkv));
  HM_TRY(ws_get(e, "dp.memk", (size_t)L * B * nh * 1024, &memk));
  HM_TRY(ws_get(e, "dp.memv", (size_t)L * B * nh * 1024, &memv));
  const size_t set_elems = (size_t)L * rows * nh * cache_blocks * 1024;
  {
    // whole 32-key blocks are read: the unwritten tail of a block must always hold finite numbers
    const size_t elems = set_elems * (beam_mode ? 2 : 1);
    uint64_t epoch = e->ws_epoch;
    HM_TRY(ws_get(e, "dp.kcache", elems, &kcache));
    if (!e->planning && e->ws_epoch != epoch) HM_CUDA(cudaMemsetAsync(kcache, 0, e->ws["dp.kcache"].cap, st));
    epoch = e->ws_epoch;
    HM_TRY(ws_get(e, "dp.vcache", elems, &vcache));
    if (!e->planning && e->ws_epoch != epoch) HM_CUDA(cudaMemsetAsync(vcache, 0, e->ws["dp.vcache"].cap, st));
  }
  HM_TRY(ws_get(e, "gen.state", 1, &state));
  HM_TRY(ws_get(e, "gen.finished", rows, &finished));
  DecPersistParams p;
  memset(&p, 0, sizeof(p));
  if (beam_mode) {
    HM_TRY(ws_get(e, "bm.score", rows, &p.bm_score));
    HM_TRY(ws_get(e, "bm.fin", rows, &p.bm_fin));
    HM_TRY(ws_get(e, "bm.src", rows, &p.bm_src));
    HM_TRY(ws_get(e, "bm.tok", rows, &p.bm_tok));
    HM_TRY(ws_get(e, "bm.parent", (size_t)max_len * rows, &p.bp_parent));
    HM_TRY(ws_get(e, "bm.token", (size_t)max_len * rows, &p.bp_token));
    if (n_best > 0) HM_TRY(ws_get(e, "bm.logp", (size_t)max_len * rows, &p.bp_logp));
  }
  if (e->trace_step >= 0) HM_TRY(ws_get(e, "gen.trace", 1024, &p.trace));
  if (e->planning) return 0;
  nvtx_push("hmocr.cross_kv");
  {
    GemmEpilogue ek;
    ek.out_f32 = memkv; ek.ld32 = e->ca_kv.n;
    const int rc = run_lin(st, enc16, e->cfg.d_model, B * e->mem_len, e->ca_kv, ek);
    if (rc != 0) { nvtx_pop(); return rc; }
  }
  {
    const int rc = repack_memkv(st, memkv, B, L, e->mem_len, memk, memv);
    nvtx_pop();
    HM_TRY(rc);
  }
  p.wstream = e->dp_wstream;
  p.lnparams = e->dp_lnparams;
  p.emb = e->emb; p.pos = e->pos; p.kcache = kcache; p.vcache = vcache; p.memk = memk; p.memv = memv;
  p.tokens = tokens; p.logprob = logprob; p.finished = finished; p.state = state;
  p.rows = rows; p.images = B; p.beam = beam; p.num_layers = L; p.fc_tiles = e->dp_fc_tiles;
  p.chunks_per_step = e->dp_chunks_per_step;
  p.vocab = e->cfg.vocab_size; p.tmax = tmax; p.max_pos = e->cfg.max_seq_len; p.max_len = max_len;
  p.ld_tok = max_len + 1; p.eos = e->cfg.eos_id; p.pad = e->cfg.pad_id; p.cache_blocks = cache_blocks; p.mem_len = e->mem_len;
  p.trace_step = e->trace_step;
  p.rows_per_cluster = DP_ROWS;
  if (beam_mode) {
    p.rows_per_cluster = beam * (DP_ROWS / beam);
    p.cache_set_stride = set_elems;
    HM_TRY(beam_init(st, state, p.bm_score, p.bm_fin, p.bm_src, p.bm_tok, rows, beam, p.rows_per_cluster, e->cfg.sos_id));
  } else {
    HM_TRY(init_decode(st, state, tokens, max_len + 1, rows, e->cfg.sos_id, e->cfg.pad_id, finished, logprob, max_len));
  }
  if (p.trace != nullptr) HM_CUDA(cudaMemsetAsync(p.trace, 0, 1024 * sizeof(long long), st));
  // Steps per launch.  The kernel leaves its step loop by itself once every row has finished, so a batch whose clusters
  // are all co-resident runs as ONE launch (no launch boundaries, no host polling).  A batch that needs several waves
  // is cut into 16-step launches: a first-wave cluster cannot stop before the rows of the later waves have finished,
  // so with one long launch it would run all max_len steps before the second wave even starts.
  int chunk = e->steps_per_launch;
  if (chunk <= 0) {
    int max_clusters = 0;
    HM_TRY(decode_persistent_max_clusters(&max_clusters));
    chunk = ceil_div(rows, p.rows_per_cluster) <= max_clusters ? max_len : 16;
  }
  bool done = false;
  int poll_idx = 0;
  for (int s0 = 0; s0 < max_len && !done; s0 += chunk, ++poll_idx) {
    const int s1 = (s0 + chunk < max_len) ? s0 + chunk : max_len;
    {
      char tag[48];
      snprintf(tag, sizeof(tag), "hmocr.decode launch %d [%d,%d)", poll_idx, s0, s1);
      nvtx_push(tag);
      const int rc = decode_persistent_launch(st, p, s0, s1);
      nvtx_pop();
      HM_TRY(rc);
    }
    const int slot = poll_idx & 1;
    e->last_poll_slot = slot;
    HM_CUDA(cudaMemcpyAsync(&e->pinned_state[slot], state, sizeof(DecodeState), cudaMemcpyDeviceToHost, st));
    HM_CUDA(cudaEventRecord(e->poll_ev[slot], st));
    if (poll_idx >= 1) {
      const int prev = (poll_idx - 1) & 1;
      HM_CUDA(cudaEventSynchronize(e->poll_ev[prev]));
      if (e->pinned_state[prev].steps_executed > 0) done = true;
    }
  }
  if (n_best > 0) {
    HM_TRY(beam_finalize(st, state, p.bm_score, p.bp_parent, p.bp_token, p.bp_logp, B, beam, n_best, rows, max_len,
                         e->cfg.sos_id, e->cfg.pad_id, tokens, logprob, score, steps));
  } else if (beam_mode) {
    HM_TRY(beam_finalize(st, state, p.bm_score, p.bp_parent, p.bp_token, nullptr, B, beam, 1, rows, max_len,
                         e->cfg.sos_id, e->cfg.pad_id, tokens, nullptr, score, steps));
    if (logprob != nullptr) HM_CUDA(cudaMemsetAsync(logprob, 0, sizeof(float) * B * max_len, st));
  } else {
    HM_TRY(finalize_decode(st, state, tokens, max_len + 1, rows, max_len, e->cfg.pad_id, logprob, steps));
  }
  return 0;
}

constexpr int ENC_GRAPH_MAX_BATCH = 1024;

int encode_any(hmocr_engine* e, const float* images, int B, float* enc32, h16* enc16, cudaStream_t st) {
  return e->cfg.encoder_arch == 1 ? encode_res18_impl(e, images, B, enc32, enc16, st) : encode_impl(e, images, B, enc32, enc16, st);
}

// Encoder of a generate() call.  Up to 32 images the encoder's ~95 kernels take a few microseconds each and the
// time is the launches; at large batches the GPU time does not care, but the HOST does: one cudaGraphLaunch instead of
// ~95 launches per batch is what keeps eight ranks on one 16-core host from queueing behind each other (end-to-end
// figure at 8 GPUs).  The first call at a batch size runs the kernels eagerly (allocations, function attributes), the
// second captures them - reading from a staging copy of the images, so the graph has no caller pointers in it -
// and every later call is one cudaGraphLaunch.  A workspace reallocation (ws_epoch) re-captures; a capture failure
// turns the feature off for this engine.
int encode_for_generate(hmocr_engine* e, const float* images, int B, float* enc32, h16* enc16, cudaStream_t st) {
  if (!e->encoder_graph || B > ENC_GRAPH_MAX_BATCH) return encode_any(e, images, B, enc32, enc16, st);
  const size_t img_n = (size_t)B * IMG_H * IMG_W;
  float* stage;
  HM_TRY(ws_get(e, "gen.img_stage", img_n, &stage));
  if (e->planning) return encode_any(e, images, B, enc32, enc16, st);
  hmocr_engine::EncGraph& eg = e->enc_graphs[B];
  if (!eg.warm) {                                   // first call: eager (everything gets allocated and initialised)
    eg.warm = true;
    return encode_any(e, images, B, enc32, enc16, st);
  }
  if (eg.exec == nullptr || eg.epoch != e->ws_epoch) {
    if (eg.exec != nullptr) { cudaGraphExecDestroy(eg.exec); eg.exec = nullptr; }
    const uint64_t epoch_before = e->ws_epoch;
    cudaGraph_t graph = nullptr;
    HM_CUDA(cudaStreamBeginCapture(e->cap_stream, cudaStreamCaptureModeThreadLocal));
    const long launches_before = g_launch_count;
    const int rc = encode_any(e, stage, B, enc32, enc16, e->cap_stream);
    eg.launches = g_launch_count - launches_before;
    g_launch_count = launches_before;               // captured, not launched
    cudaError_t ce = cudaStreamEndCapture(e->cap_stream, &graph);
    if (rc == 0 && ce == cudaSuccess && e->ws_epoch == epoch_before) ce = cudaGraphInstantiate(&eg.exec, graph, 0);
    if (graph) cudaGraphDestroy(graph);
    if (rc != 0 || ce != cudaSuccess || e->ws_epoch != epoch_before || eg.exec == nullptr) {
      (void)cudaGetLastError();
      eg.exec = nullptr;
      e->encoder_graph = 0;                         // never again on this engine; the eager path is always correct
      return encode_any(e, images, B, enc32, enc16, st);
    }
    eg.epoch = e->ws_epoch;
  }
  HM_CUDA(cudaMemcpyAsync(stage, images, img_n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  HM_CUDA(cudaGraphLaunch(eg.exec, st));
  g_launch_count += eg.launches;
  return 0;
}

int generate_impl(hmocr_engine* e, const float* images, int B, int max_len, int beam, int64_t* tokens, float* logprob,
                  int32_t* steps, float* score, cudaStream_t st, int n_best = 0) {
  float* enc32;
  h16* enc16;
  HM_TRY(ws_get(e, "gen.enc32", (size_t)B * e->mem_len * e->cfg.d_model, &enc32));
  HM_TRY(ws_get(e, "gen.enc16", (size_t)B * e->mem_len * e->cfg.d_model, &enc16));
  if (e->planning) {
    HM_TRY(encode_for_generate(e, images, B, enc32, enc16, st));
    return generate_from_memory_impl(e, enc16, B, max_len, beam, tokens, logprob, steps, score, st, n_best);
  }
  HM_CUDA(cudaEventRecord(e->ev[0], st));
  nvtx_push("hmocr.encode");
  const int rc_enc = encode_for_generate(e, images, B, enc32, enc16, st);
  nvtx_pop();
  HM_TRY(rc_enc);
  HM_CUDA(cudaEventRecord(e->ev[1], st));
  HM_TRY(generate_from_memory_impl(e, enc16, B, max_len, beam, tokens, logprob, steps, score, st, n_best));
  HM_CUDA(cudaEventRecord(e->ev[2], st));
  e->timings_pending = true;
  return 0;
}

// generate from encoder output already in HBM (f32 [B, mem_len, d_model])
int generate_from_enc32(hmocr_engine* e, const float* enc_out, int B, int max_len, int beam, int64_t* tokens,
                        float* logprob, int32_t* steps, float* score, cudaStream_t st, int n_best) {
  h16* enc16;
  HM_TRY(ws_get(e, "gen.enc16", (size_t)B * e->mem_len * e->cfg.d_model, &enc16));
  HM_TRY(f32_to_f16(st, enc_out, (size_t)B * e->mem_len * e->cfg.d_model, enc16));
  HM_CUDA(cudaEventRecord(e->ev[0], st));
  HM_CUDA(cudaEventRecord(e->ev[1], st));
  HM_TRY(generate_from_memory_impl(e, enc16, B, max_len, beam, tokens, logprob, steps, score, st, n_best));
  HM_CUDA(cudaEventRecord(e->ev[2], st));
  e->timings_pending = true;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// teacher-forced scoring of given sequences (hmocr_score): the layer stack of decoder_forward, then fc_out with the
// log-sum-exp epilogue (per-row partials, no logits buffer) and one combine kernel
// ------------------------------------------------------------------------------------------------
int score_impl(hmocr_engine* e, const float* input, int input_is_memory, int B, int T, const int64_t* tokens,
               float* logprob, float* score, int32_t* argmax, cudaStream_t st) {
  const int d = e->cfg.d_model;
  const int rows = B * T, num_parts = e->vpad / LSE_COLS_PER_PART;
  const size_t mem_n = (size_t)B * e->mem_len * d;
  h16 *enc16, *memkv;
  LsePartial* parts;
  DecBufs b;
  HM_TRY(ws_get(e, "tf.memkv", (size_t)B * e->mem_len * e->ca_kv.n, &memkv));
  HM_TRY(dec_layer_bufs(e, "tf", rows, &b));
  HM_TRY(ws_get(e, "score.partials", (size_t)rows * num_parts, &parts));
  const float* enc32 = nullptr;
  if (input_is_memory) {
    HM_TRY(ws_get(e, "tf.enc16", mem_n, &enc16));
    enc32 = input;
  } else {
    float* enc_out;
    HM_TRY(ws_get(e, "gen.enc32", mem_n, &enc_out));
    HM_TRY(ws_get(e, "gen.enc16", mem_n, &enc16));
    HM_TRY(encode_for_generate(e, input, B, enc_out, enc16, st));     // records the encoder's buffers when planning
  }
  if (e->planning) return 0;
  HM_TRY(decoder_layers(e, enc32, enc16, memkv, tokens, T + 1, B, T, b, st));
  GemmLse lse;
  lse.tokens = tokens; lse.ld_tok = T + 1; lse.T = T; lse.n_valid = e->cfg.vocab_size; lse.partials = parts;
  HM_TRY(gemm_f16_lse(st, b.x16, d, rows, d, e->fc.w, e->fc.n, e->fc.b, lse));
  return score_combine(st, parts, num_parts, tokens, T + 1, B, T, e->cfg.eos_id, e->cfg.pad_id, logprob, score, argmax);
}

int check_ready(hmocr_engine* e, int B, void* stream) {
  HM_CHECK(e != nullptr, "null engine");
  HM_CHECK(e->finalized, "weights not loaded: call hmocr_load_weight for every entry, then hmocr_finalize_weights");
  HM_CHECK(B >= 1, "batch must be >= 1 (got %d)", B);
  HM_CUDA(cudaSetDevice(e->device));
  e->cur_stream = static_cast<cudaStream_t>(stream);
  return 0;
}

// every scratch buffer a call with this shape asks for (the schedules run in planning mode: ws_get records, nothing launches)
// records the per-buffer maximum of the plan just made and answers the bytes that cover every shape asked so far
int finish_plan(hmocr_engine* e, size_t* bytes) {
  e->planning = false;
  for (auto& kv : e->plan) {
    size_t& m = e->planned[kv.first];
    if (m < kv.second) m = kv.second;
  }
  e->plan.clear();
  size_t total = 0;
  for (auto& kv : e->planned) total += kv.second;    // every entry is already rounded to WS_ALIGN
  *bytes = total + WS_ALIGN;
  return 0;
}

int plan_workspace(hmocr_engine* e, int B, int max_len, int beam, size_t* bytes) {
  e->plan.clear();
  e->planning = true;
  int rc = 0;
  float* fdummy = reinterpret_cast<float*>(WS_ALIGN);
  int64_t* tdummy = reinterpret_cast<int64_t*>(WS_ALIGN);
  if (beam == 0) {                                   // teacher-forced hmocr_decoder_forward(B, T = max_len)
    rc = decoder_forward_impl(e, fdummy, tdummy, B, max_len, fdummy, nullptr);
  } else if (beam < 0) {                             // hmocr_generate_nbest with -beam hypotheses (either input form)
    rc = generate_impl(e, fdummy, B, max_len, -beam, tdummy, fdummy, nullptr, fdummy, nullptr, 1);
  } else {                                           // hmocr_encode + hmocr_generate* (device and host-buffer forms)
    h16* d16;
    uint8_t* u8;
    float* f32;
    int64_t* i64;
    int32_t* i32;
    const size_t img_n = (size_t)B * IMG_H * IMG_W;
    rc = ws_get(e, "enc.out16", (size_t)B * e->mem_len * e->cfg.d_model, &d16);
    if (rc == 0) rc = ws_get(e, "host.images_u8", img_n, &u8);
    if (rc == 0) rc = ws_get(e, "host.images", img_n, &f32);
    if (rc == 0) rc = ws_get(e, "host.tokens", (size_t)B * (max_len + 1), &i64);
    if (rc == 0) rc = ws_get(e, "host.logprob", (size_t)B * max_len, &f32);
    if (rc == 0) rc = ws_get(e, "host.steps", 1, &i32);
    if (rc == 0) rc = ws_get(e, "host.score", B, &f32);
    if (rc == 0) rc = generate_impl(e, fdummy, B, max_len, beam, tdummy, fdummy, nullptr, fdummy, nullptr);
  }
  finish_plan(e, bytes);
  return rc;
}

// hmocr_score(B, T) in both input forms
int plan_score_workspace(hmocr_engine* e, int B, int T, size_t* bytes) {
  e->plan.clear();
  e->planning = true;
  float* fdummy = reinterpret_cast<float*>(WS_ALIGN);
  int64_t* tdummy = reinterpret_cast<int64_t*>(WS_ALIGN);
  int rc = score_impl(e, fdummy, 1, B, T, tdummy, fdummy, fdummy, nullptr, nullptr);
  if (rc == 0) rc = score_impl(e, fdummy, 0, B, T, tdummy, fdummy, fdummy, nullptr, nullptr);
  finish_plan(e, bytes);
  return rc;
}

}  // namespace
}  // namespace hmocr

// ====================================================================================================
// C ABI
// ====================================================================================================
HM_API const char* hmocr_last_error(void) { return g_err; }
HM_API const char* hmocr_version(void) { return "hmocr 0.1 (sm_100a, tcgen05/TMA)"; }
HM_API int64_t hmocr_launch_count(void) { return g_launch_count; }

HM_API int hmocr_create(const hmocr_config* cfg, hmocr_engine** out) {
  HM_CHECK(cfg != nullptr && out != nullptr, "hmocr_create: null argument");
  HM_CHECK(cfg->d_model == 256 && cfg->nhead == 8,
           "this build supports d_model=256, nhead=8 (head_dim 32) as in the reference config; got %d/%d",
           cfg->d_model, cfg->nhead);
  HM_CHECK(cfg->dim_feedforward % 64 == 0 && cfg->dim_feedforward > 0, "dim_feedforward must be a multiple of 64");
  HM_CHECK(cfg->num_layers >= 1 && cfg->num_layers <= 32, "num_layers out of range");
  HM_CHECK(cfg->enc_num_layers >= 0 && cfg->enc_num_layers <= 32, "enc_num_layers out of range");
  HM_CHECK(cfg->max_seq_len >= 2 && cfg->max_seq_len <= 256, "max_seq_len must be in [2,256]");
  HM_CHECK(cfg->vocab_size >= 4, "vocab_size too small");
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  HM_CHECK(ce == cudaSuccess && ndev > 0, "no CUDA device: libhmocr has no CPU fallback (%s)", cudaGetErrorString(ce));
  HM_TRY(gemm_init());
  hmocr_engine* e = new hmocr_engine();
  e->cfg = *cfg;
  HM_CUDA(cudaGetDevice(&e->device));
  HM_CHECK(cfg->encoder_arch == 0 || cfg->encoder_arch == 1, "encoder_arch must be 0 (Swin-T) or 1 (ResNet-18 + TransformerEncoder)");
  e->mem_len = cfg->encoder_arch == 1 ? RES18_MEM : SWIN_MEM;
  e->vpad = (cfg->vocab_size + 255) / 256 * 256;
  e->layers.resize(cfg->num_layers);
  HM_CUDA(cudaStreamCreateWithFlags(&e->cap_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 4; ++i) HM_CUDA(cudaEventCreate(&e->ev[i]));
  for (int i = 0; i < 2; ++i) HM_CUDA(cudaEventCreateWithFlags(&e->poll_ev[i], cudaEventDisableTiming));
  HM_CUDA(cudaMallocHost(reinterpret_cast<void**>(&e->pinned_state), 2 * sizeof(DecodeState)));
  *out = e;
  return 0;
}

HM_API void hmocr_destroy(hmocr_engine* e) {
  if (e == nullptr) return;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  for (auto& kv : e->graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  for (auto& kv : e->enc_graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  for (auto& kv : e->ws) {
    uint8_t* p = static_cast<uint8_t*>(kv.second.p);
    const bool in_pool = e->ext_ws != nullptr && p >= e->ext_ws && p < e->ext_ws + e->ext_cap;   // the caller's memory
    if (p != nullptr && !in_pool) cudaFree(p);
  }
  if (e->arena) cudaFree(e->arena);
  if (e->cap_stream) cudaStreamDestroy(e->cap_stream);
  for (int i = 0; i < 4; ++i)
    if (e->ev[i]) cudaEventDestroy(e->ev[i]);
  for (int i = 0; i < 2; ++i)
    if (e->poll_ev[i]) cudaEventDestroy(e->poll_ev[i]);
  if (e->pinned_state) cudaFreeHost(e->pinned_state);
  delete e;
}

HM_API int hmocr_load_weight(hmocr_engine* e, const char* key, const void* data, const int64_t* shape, int ndim,
                             int dtype) {
  HM_CHECK(e != nullptr && key != nullptr && data != nullptr, "hmocr_load_weight: null argument");
  HM_CHECK(!e->finalized, "weights already finalized");
  HM_CHECK(dtype == HMOCR_F32 || dtype == HMOCR_I64, "unsupported dtype %d for '%s'", dtype, key);
  std::string k(key);
  // the reference registers the Swin trunk twice (encoder.swin.features.* and encoder.features.*
  // share storage, src/model_swin.py:35); keep one canonical name
  const std::string alias = "encoder.swin.features.";
  if (k.compare(0, alias.size(), alias) == 0) k = "encoder.features." + k.substr(alias.size());
  // src/model_res18trans.py names the same decoder module `transformer_decoder`
  const std::string dec2 = "decoder.transformer_decoder.";
  if (k.compare(0, dec2.size(), dec2) == 0) k = "decoder.decoder." + k.substr(dec2.size());
  HostTensor t;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
  if (dtype == HMOCR_F32) t.f.assign(static_cast<const float*>(data), static_cast<const float*>(data) + n);
  else t.i.assign(static_cast<const int64_t*>(data), static_cast<const int64_t*>(data) + n);
  e->host[k] = std::move(t);
  return 0;
}

static int finalize_weights_impl(hmocr_engine* e);

HM_API int hmocr_finalize_weights(hmocr_engine* e) {
  HM_CHECK(e != nullptr, "null engine");
  HM_CHECK(!e->finalized, "weights already finalized");
  HM_CUDA(cudaSetDevice(e->device));
  const int rc = finalize_weights_impl(e);
  if (rc != 0 && e->arena != nullptr) {       // a failed load (missing / mis-shaped entry) must not leak the arena on retry
    cudaFree(e->arena);
    e->arena = nullptr;
    e->arena_cap = e->arena_used = 0;
  }
  return rc;
}

static int finalize_weights_impl(hmocr_engine* e) {
  const hmocr_config& c = e->cfg;
  const int d = c.d_model, ff = c.dim_feedforward, V = c.vocab_size;
  size_t total = 0;
  for (auto& kv : e->host) total += kv.second.f.size() * 4 + 1024;
  e->arena_cap = total + (size_t)e->vpad * d * 4 + (size_t)c.num_layers * 2 * d * (d + 1) * 4 + (64u << 20) +
                 (size_t)8 * (DP_LAYER_CHUNKS * c.num_layers + V / 128 + 16) * DP_CHUNK + (size_t)c.num_layers * 8192 * 4;
  HM_CUDA(cudaMalloc(&e->arena, e->arena_cap));
  e->arena_used = 0;

  const std::string f = "encoder.features.";
  const HostTensor* t;
  if (c.encoder_arch == 1) {
    HM_TRY(load_res18_weights(e));
  } else {
  HM_TRY(need(e, f + "0.0.weight", {96, 1, 4, 4}, &t));
  HM_TRY(upload_f32(e, t->f.data(), 96 * 16, &e->pe_w));
  HM_TRY(upload_vec(e, f + "0.0.bias", 96, &e->pe_b));
  HM_TRY(upload_norm(e, f + "0.2", 96, &e->pe_norm));
  int C = 96, blk = 0;
  for (int s = 0; s < 4; ++s) {
    const int fi = 1 + 2 * s, heads = HEADS[s];
    for (int j = 0; j < DEPTHS[s]; ++j, ++blk) {
      const std::string p = f + std::to_string(fi) + "." + std::to_string(j) + ".";
      SwinBlock& sb = e->blocks[blk];
      HM_TRY(upload_norm(e, p + "norm1", C, &sb.n1));
      HM_TRY(upload_norm(e, p + "norm2", C, &sb.n2));
      HM_TRY(upload_lin(e, p + "attn.qkv", 3 * C, C, true, &sb.qkv));
      HM_TRY(upload_lin(e, p + "attn.proj", C, C, true, &sb.proj));
      HM_TRY(upload_lin(e, p + "mlp.0", 4 * C, C, true, &sb.fc1));
      HM_TRY(upload_lin(e, p + "mlp.3", C, 4 * C, true, &sb.fc2));
      // relative position bias gathered to [heads,49,49]  (swin_transformer.py:49-56)
      const HostTensor* tab;
      HM_TRY(need(e, p + "attn.relative_position_bias_table", {169, heads}, &tab));
      const HostTensor* idx = find(e, p + "attn.relative_position_index");
      HM_CHECK(idx != nullptr && idx->i.size() == 2401, "missing/invalid '%sattn.relative_position_index'", p.c_str());
      std::vector<float> rb((size_t)heads * 2401);
      for (int q = 0; q < 2401; ++q) {
        const int64_t r = idx->i[q];
        HM_CHECK(r >= 0 && r < 169, "relative_position_index out of range");
        for (int h = 0; h < heads; ++h) rb[(size_t)h * 2401 + q] = tab->f[(size_t)r * heads + h];
      }
      HM_TRY(upload_f32(e, rb.data(), rb.size(), &sb.rel_bias));
    }
    if (s < 3) {
      const std::string p = f + std::to_string(fi + 1) + ".";
      HM_TRY(upload_norm(e, p + "norm", 4 * C, &e->merges[s].norm));
      HM_TRY(upload_lin(e, p + "reduction", 2 * C, 4 * C, false, &e->merges[s].red));
      C *= 2;
    }
  }
  HM_TRY(upload_lin(e, "encoder.projection", d, SWIN_OUT, true, &e->proj));
  }

  HM_TRY(need(e, "decoder.embedding.weight", {V, d}, &t));
  HM_TRY(upload_f32(e, t->f.data(), (size_t)V * d, &e->emb));
  HM_TRY(need(e, "decoder.pos_encoder.weight", {c.max_seq_len, d}, &t));
  HM_TRY(upload_f32(e, t->f.data(), (size_t)c.max_seq_len * d, &e->pos));
  std::vector<float> kvw((size_t)c.num_layers * 2 * d * d), kvb((size_t)c.num_layers * 2 * d);
  for (int l = 0; l < c.num_layers; ++l) {
    const std::string p = "decoder.decoder.layers." + std::to_string(l) + ".";
    DecLayer& L = e->layers[l];
    const HostTensor *w, *b;
    HM_TRY(need(e, p + "self_attn.in_proj_weight", {3 * d, d}, &w));
    HM_TRY(need(e, p + "self_attn.in_proj_bias", {3 * d}, &b));
    HM_TRY(upload_lin_rows(e, w->f.data(), b->f.data(), 3 * d, d, &L.sa_in));
    HM_TRY(upload_lin(e, p + "self_attn.out_proj", d, d, true, &L.sa_out));
    HM_TRY(need(e, p + "multihead_attn.in_proj_weight", {3 * d, d}, &w));
    HM_TRY(need(e, p + "multihead_attn.in_proj_bias", {3 * d}, &b));
    HM_TRY(upload_lin_rows(e, w->f.data(), b->f.data(), d, d, &L.ca_q));          // rows [0,d) = Wq
    memcpy(&kvw[(size_t)l * 2 * d * d], w->f.data() + (size_t)d * d, sizeof(float) * 2 * d * d);   // Wk | Wv
    memcpy(&kvb[(size_t)l * 2 * d], b->f.data() + d, sizeof(float) * 2 * d);
    HM_TRY(upload_lin(e, p + "multihead_attn.out_proj", d, d, true, &L.ca_out));
    HM_TRY(upload_lin(e, p + "linear1", ff, d, true, &L.l1));
    HM_TRY(upload_lin(e, p + "linear2", d, ff, true, &L.l2));
    HM_TRY(upload_norm(e, p + "norm1", d, &L.n1));
    HM_TRY(upload_norm(e, p + "norm2", d, &L.n2));
    HM_TRY(upload_norm(e, p + "norm3", d, &L.n3));
  }
  HM_TRY(upload_lin_rows(e, kvw.data(), kvb.data(), c.num_layers * 2 * d, d, &e->ca_kv));
  {
    const HostTensor *w, *b;
    HM_TRY(need(e, "decoder.fc_out.weight", {V, d}, &w));
    HM_TRY(need(e, "decoder.fc_out.bias", {V}, &b));
    std::vector<float> wp((size_t)e->vpad * d, 0.f), bp(e->vpad, 0.f);
    memcpy(wp.data(), w->f.data(), sizeof(float) * (size_t)V * d);
    memcpy(bp.data(), b->f.data(), sizeof(float) * V);
    HM_TRY(upload_lin_rows(e, wp.data(), bp.data(), e->vpad, d, &e->fc));
  }
  HM_TRY(pack_decode_operands(e));
  HM_TRY(decode_persistent_init());
  e->host.clear();
  e->finalized = true;
  return 0;
}

HM_API int hmocr_set_pos_table(hmocr_engine* e, const float* pos_host, int rows, int d, void* stream) {
  HM_CHECK(e != nullptr && pos_host != nullptr, "hmocr_set_pos_table: null argument");
  HM_CHECK(e->finalized && e->cfg.encoder_arch == 1, "hmocr_set_pos_table: only for a loaded ResNet-18 variant engine");
  HM_CHECK(rows == RES18_MEM && d == e->cfg.d_model, "positional table must be [%d, %d]", RES18_MEM, e->cfg.d_model);
  HM_CUDA(cudaSetDevice(e->device));
  // stream-ordered: an encoder still running on this stream keeps reading the old table until it is done
  HM_CUDA(cudaMemcpyAsync(e->pos_table, pos_host, sizeof(float) * rows * d, cudaMemcpyHostToDevice,
                          static_cast<cudaStream_t>(stream)));
  e->pos_table_set = true;
  return 0;
}

HM_API int hmocr_workspace_bytes(hmocr_engine* e, int batch, int max_len, int beam, size_t* bytes) {
  HM_CHECK(e != nullptr && bytes != nullptr, "hmocr_workspace_bytes: null argument");
  HM_CHECK(e->finalized, "hmocr_workspace_bytes: load the weights first (buffer sizes depend on the checkpoint's vocabulary)");
  HM_CHECK(batch >= 1 && max_len >= 1 && beam >= -DP_MAX_BEAM, "hmocr_workspace_bytes: bad shape batch=%d max_len=%d beam=%d", batch, max_len, beam);
  return plan_workspace(e, batch, max_len, beam, bytes);
}

HM_API int hmocr_score_workspace_bytes(hmocr_engine* e, int batch, int T, size_t* bytes) {
  HM_CHECK(e != nullptr && bytes != nullptr, "hmocr_score_workspace_bytes: null argument");
  HM_CHECK(e->finalized, "hmocr_score_workspace_bytes: load the weights first (buffer sizes depend on the checkpoint's vocabulary)");
  HM_CHECK(batch >= 1 && T >= 1 && T <= e->cfg.max_seq_len, "hmocr_score_workspace_bytes: bad shape batch=%d T=%d", batch, T);
  return plan_score_workspace(e, batch, T, bytes);
}

HM_API int hmocr_set_workspace(hmocr_engine* e, void* workspace_dev, size_t bytes, void* stream) {
  HM_CHECK(e != nullptr, "hmocr_set_workspace: null engine");
  HM_CHECK(workspace_dev == nullptr || (reinterpret_cast<uintptr_t>(workspace_dev) % WS_ALIGN == 0 && bytes >= WS_ALIGN),
           "hmocr_set_workspace: the buffer must be %zu-byte aligned and non-empty", WS_ALIGN);
  HM_CUDA(cudaSetDevice(e->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (auto& kv : e->ws) {                     // engine-owned buffers go back to the pool, stream-ordered
    uint8_t* p = static_cast<uint8_t*>(kv.second.p);
    const bool in_pool = e->ext_ws != nullptr && p >= e->ext_ws && p < e->ext_ws + e->ext_cap;
    if (p != nullptr && !in_pool) HM_CUDA(cudaFreeAsync(p, st));
  }
  e->ws.clear();
  e->ext_ws = static_cast<uint8_t*>(workspace_dev);
  e->ext_cap = workspace_dev ? bytes : 0;
  e->ext_used = 0;
  ++e->ws_epoch;                               // captured graphs hold the old addresses
  return 0;
}

HM_API int hmocr_decode_max_clusters(int* out) {
  HM_CHECK(out != nullptr, "null argument");
  return decode_persistent_max_clusters(out);
}

HM_API int hmocr_set_option(hmocr_engine* e, const char* name, int value) {
  HM_CHECK(e != nullptr && name != nullptr, "hmocr_set_option: null argument");
  const std::string n(name);
  if (n == "decode_impl") {
    HM_CHECK(value == 0 || value == 1, "decode_impl must be 0 (persistent cluster kernel) or 1 (step graph)");
    e->decode_impl = value;
  } else if (n == "steps_per_launch") {
    HM_CHECK(value >= 0 && value <= 256, "steps_per_launch must be in [0,256] (0 = automatic)");
    e->steps_per_launch = value;
  } else if (n == "trace_step") {
    e->trace_step = value;
  } else if (n == "encoder_graph") {
    HM_CHECK(value == 0 || value == 1, "encoder_graph must be 0 or 1");
    e->encoder_graph = value;
  } else if (n == "conv_impl") {
    HM_CHECK(value == 0 || value == 1, "conv_impl must be 0 (implicit GEMM) or 1 (im2col)");
    e->conv_impl = value;
  } else if (n == "gemm_dbg") {
    gemm_set_debug(value);
  } else if (n == "mlp_fused") {
    HM_CHECK(value == 0 || value == 1, "mlp_fused must be 0 (fc1 and fc2 as two GEMM launches) or 1 (one kernel)");
    if (e->mlp_fused != value) ++e->ws_epoch;            // captured encoder graphs hold the other schedule
    e->mlp_fused = value;
  } else {
    HM_CHECK(false, "unknown option '%s'", name);
  }
  return 0;
}

HM_API int hmocr_read_trace(hmocr_engine* e, int64_t* out_host, int n) {
  HM_CHECK(e != nullptr && out_host != nullptr && n >= 1 && n <= 1024, "hmocr_read_trace: bad argument");
  auto it = e->ws.find("gen.trace");
  HM_CHECK(it != e->ws.end() && it->second.p != nullptr, "no trace recorded (set option trace_step first)");
  HM_CUDA(cudaMemcpy(out_host, it->second.p, sizeof(int64_t) * n, cudaMemcpyDeviceToHost));
  return 0;
}

HM_API int hmocr_encode(hmocr_engine* e, const float* images, int B, float* enc_out, void* stream) {
  HM_TRY(check_ready(e, B, stream));
  HM_CHECK(images != nullptr && enc_out != nullptr, "hmocr_encode: null buffer");
  h16* enc16;
  HM_TRY(ws_get(e, "enc.out16", (size_t)B * e->mem_len * e->cfg.d_model, &enc16));
  return e->cfg.encoder_arch == 1 ? encode_res18_impl(e, images, B, enc_out, enc16, static_cast<cudaStream_t>(stream))
                                  : encode_impl(e, images, B, enc_out, enc16, static_cast<cudaStream_t>(stream));
}

HM_API int hmocr_decoder_forward(hmocr_engine* e, const float* enc_out, const int64_t* tgt, int B, int T,
                                 float* logits, void* stream) {
  HM_TRY(check_ready(e, B, stream));
  HM_CHECK(enc_out != nullptr && tgt != nullptr && logits != nullptr, "hmocr_decoder_forward: null buffer");
  HM_CHECK(T >= 1 && T <= e->cfg.max_seq_len, "T=%d outside [1,%d] (tgt_mask / pos_encoder size)", T,
           e->cfg.max_seq_len);
  return decoder_forward_impl(e, enc_out, tgt, B, T, logits, static_cast<cudaStream_t>(stream));
}

HM_API int hmocr_score(hmocr_engine* e, const float* input, int input_is_memory, int B, int T, const int64_t* tokens,
                       float* logprob, float* score, int32_t* argmax, void* stream) {
  HM_TRY(check_ready(e, B, stream));
  HM_CHECK(input != nullptr && tokens != nullptr, "hmocr_score: null buffer");
  HM_CHECK(logprob != nullptr || score != nullptr || argmax != nullptr, "hmocr_score: every output is NULL");
  HM_CHECK(T >= 1 && T <= e->cfg.max_seq_len, "hmocr_score: T=%d outside [1,%d] (tgt_mask / pos_encoder size)", T,
           e->cfg.max_seq_len);
  return score_impl(e, input, input_is_memory, B, T, tokens, logprob, score, argmax, static_cast<cudaStream_t>(stream));
}

HM_API int hmocr_generate(hmocr_engine* e, const float* images, int B, int max_len, int beam, int64_t* tokens,
                          float* logprob, int32_t* steps, float* score, void* stream) {
  HM_TRY(check_ready(e, B, stream));
  HM_CHECK(images != nullptr && tokens != nullptr, "hmocr_generate: null buffer");
  return generate_impl(e, images, B, max_len, beam, tokens, logprob, steps, score, static_cast<cudaStream_t>(stream));
}

HM_API int hmocr_generate_from_memory(hmocr_engine* e, const float* enc_out, int B, int max_len, int beam,
                                      int64_t* tokens, float* logprob, int32_t* steps, float* score, void* stream) {
  HM_TRY(check_ready(e, B, stream));
  HM_CHECK(enc_out != nullptr && tokens != nullptr, "hmocr_generate_from_memory: null buffer");
  return generate_from_enc32(e, enc_out, B, max_len, beam, tokens, logprob, steps, score,
                             static_cast<cudaStream_t>(stream), 0);
}

HM_API int hmocr_generate_nbest(hmocr_engine* e, const float* input, int input_is_memory, int B, int max_len, int beam,
                                int n_best, int64_t* tokens, float* logprob, float* score, int32_t* steps, void* stream) {
  HM_TRY(check_ready(e, B, stream));
  HM_CHECK(beam >= 1 && beam <= DP_MAX_BEAM, "hmocr_generate_nbest: beam=%d outside [1, %d]", beam, DP_MAX_BEAM);
  HM_CHECK(n_best >= 1 && n_best <= beam, "hmocr_generate_nbest: n_best=%d outside [1, beam=%d]", n_best, beam);
  HM_CHECK(input != nullptr && tokens != nullptr, "hmocr_generate_nbest: null buffer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (input_is_memory) return generate_from_enc32(e, input, B, max_len, beam, tokens, logprob, steps, score, st, n_best);
  return generate_impl(e, input, B, max_len, beam, tokens, logprob, steps, score, st, n_best);
}

HM_API int hmocr_generate_host(hmocr_engine* e, const float* images_host, int B, int max_len, int beam,
                               int64_t* tokens_host, float* logprob_host, int32_t* steps_host, float* score_host,
                               void* stream) {
  HM_TRY(check_ready(e, B, stream));
  HM_CHECK(images_host != nullptr && tokens_host != nullptr, "hmocr_generate_host: null buffer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float *img_d, *lp_d, *score_d;
  int64_t* tok_d;
  int32_t* steps_d;
  const size_t img_n = (size_t)B * IMG_H * IMG_W;
  HM_TRY(ws_get(e, "host.images", img_n, &img_d));
  HM_TRY(ws_get(e, "host.tokens", (size_t)B * (max_len + 1), &tok_d));
  HM_TRY(ws_get(e, "host.logprob", (size_t)B * max_len, &lp_d));
  HM_TRY(ws_get(e, "host.steps", 1, &steps_d));
  HM_TRY(ws_get(e, "host.score", B, &score_d));
  HM_CUDA(cudaMemcpyAsync(img_d, images_host, img_n * sizeof(float), cudaMemcpyHostToDevice, st));
  HM_TRY(generate_impl(e, img_d, B, max_len, beam, tok_d, logprob_host ? lp_d : nullptr, steps_d,
                       score_host ? score_d : nullptr, st));
  HM_CUDA(cudaMemcpyAsync(tokens_host, tok_d, sizeof(int64_t) * B * (max_len + 1), cudaMemcpyDeviceToHost, st));
  if (logprob_host) HM_CUDA(cudaMemcpyAsync(logprob_host, lp_d, sizeof(float) * B * max_len, cudaMemcpyDeviceToHost, st));
  if (steps_host) HM_CUDA(cudaMemcpyAsync(steps_host, steps_d, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (score_host) HM_CUDA(cudaMemcpyAsync(score_host, score_d, sizeof(float) * B, cudaMemcpyDeviceToHost, st));
  HM_CUDA(cudaStreamSynchronize(st));
  return 0;
}

HM_API int hmocr_preprocess_image_u8(hmocr_engine* e, const uint8_t* image_host, int channels, int height, int width,
                                     float* image_dev, void* stream) {
  HM_CHECK(e != nullptr && image_host != nullptr && image_dev != nullptr, "hmocr_preprocess_image_u8: null argument");
  HM_CHECK(channels == 1 || channels == 3, "hmocr_preprocess_image_u8: channels must be 1 (mode L) or 3 (mode RGB), got %d", channels);
  HM_CHECK(height >= 1 && width >= 1 && height <= 16384 && width <= 16384, "hmocr_preprocess_image_u8: bad size %dx%d", height, width);
  HM_CUDA(cudaSetDevice(e->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  e->cur_stream = st;
  uint8_t *src, *mid;
  int* tables;
  const size_t bytes = (size_t)height * width * channels;
  HM_TRY(ws_get(e, "pp.src", bytes, &src));
  HM_TRY(ws_get(e, "pp.mid", (size_t)height * IMG_W, &mid));
  HM_TRY(ws_get(e, "pp.tables", preprocess_table_ints(height, width, IMG_H, IMG_W), &tables));
  HM_CUDA(cudaMemcpyAsync(src, image_host, bytes, cudaMemcpyHostToDevice, st));
  return preprocess_image(st, src, channels, height, width, IMG_H, IMG_W, tables, mid, image_dev);
}

HM_API int hmocr_preprocess_cv2_u8(hmocr_engine* e, const uint8_t* gray_host, int height, int width, float* image_dev,
                                   void* stream) {
  HM_CHECK(e != nullptr && gray_host != nullptr && image_dev != nullptr, "hmocr_preprocess_cv2_u8: null argument");
  HM_CHECK(height >= 1 && width >= 1 && height <= 16384 && width <= 16384, "hmocr_preprocess_cv2_u8: bad size %dx%d", height, width);
  HM_CUDA(cudaSetDevice(e->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  e->cur_stream = st;
  uint8_t* src;
  int* tables;
  const size_t bytes = (size_t)height * width;
  HM_TRY(ws_get(e, "pp.src", bytes, &src));
  HM_TRY(ws_get(e, "pp.tables", (size_t)4 * (IMG_H + IMG_W) + preprocess_table_ints(height, width, IMG_H, IMG_W), &tables));
  HM_CUDA(cudaMemcpyAsync(src, gray_host, bytes, cudaMemcpyHostToDevice, st));
  return preprocess_gray_cv2(st, src, height, width, IMG_H, IMG_W, tables, image_dev);
}

HM_API int hmocr_pack_tokens(hmocr_engine* e, const int64_t* tokens_dev, int rows, int ld_tok, int32_t* lengths_dev,
                             int32_t* packed_dev, void* stream) {
  HM_CHECK(e != nullptr && tokens_dev != nullptr && lengths_dev != nullptr && packed_dev != nullptr, "hmocr_pack_tokens: null argument");
  HM_CHECK(rows >= 1 && ld_tok >= 1, "hmocr_pack_tokens: bad shape rows=%d ld=%d", rows, ld_tok);
  HM_CUDA(cudaSetDevice(e->device));
  return pack_tokens(static_cast<cudaStream_t>(stream), tokens_dev, rows, ld_tok, e->cfg.sos_id, e->cfg.eos_id, e->cfg.pad_id,
                     lengths_dev, packed_dev);
}

HM_API int hmocr_preprocess_u8(hmocr_engine* e, const uint8_t* images_u8_dev, int B, float* images_dev, void* stream) {
  HM_CHECK(e != nullptr && images_u8_dev != nullptr && images_dev != nullptr && B >= 1, "hmocr_preprocess_u8: bad argument");
  HM_CUDA(cudaSetDevice(e->device));
  return preprocess_u8(static_cast<cudaStream_t>(stream), images_u8_dev, (size_t)B * IMG_H * IMG_W, images_dev);
}

HM_API int hmocr_generate_host_u8(hmocr_engine* e, const uint8_t* images_u8_host, int B, int max_len, int beam,
                                  int64_t* tokens_host, float* logprob_host, int32_t* steps_host, float* score_host,
                                  void* stream) {
  HM_TRY(check_ready(e, B, stream));
  HM_CHECK(images_u8_host != nullptr && tokens_host != nullptr, "hmocr_generate_host_u8: null buffer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* u8_d;
  float *img_d, *lp_d, *score_d;
  int64_t* tok_d;
  int32_t* steps_d;
  const size_t img_n = (size_t)B * IMG_H * IMG_W;
  HM_TRY(ws_get(e, "host.images_u8", img_n, &u8_d));
  HM_TRY(ws_get(e, "host.images", img_n, &img_d));
  HM_TRY(ws_get(e, "host.tokens", (size_t)B * (max_len + 1), &tok_d));
  HM_TRY(ws_get(e, "host.logprob", (size_t)B * max_len, &lp_d));
  HM_TRY(ws_get(e, "host.steps", 1, &steps_d));
  HM_TRY(ws_get(e, "host.score", B, &score_d));
  HM_CUDA(cudaMemcpyAsync(u8_d, images_u8_host, img_n, cudaMemcpyHostToDevice, st));
  HM_TRY(preprocess_u8(st, u8_d, img_n, img_d));
  HM_TRY(generate_impl(e, img_d, B, max_len, beam, tok_d, logprob_host ? lp_d : nullptr, steps_d,
                       score_host ? score_d : nullptr, st));
  HM_CUDA(cudaMemcpyAsync(tokens_host, tok_d, sizeof(int64_t) * B * (max_len + 1), cudaMemcpyDeviceToHost, st));
  if (logprob_host) HM_CUDA(cudaMemcpyAsync(logprob_host, lp_d, sizeof(float) * B * max_len, cudaMemcpyDeviceToHost, st));
  if (steps_host) HM_CUDA(cudaMemcpyAsync(steps_host, steps_d, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (score_host) HM_CUDA(cudaMemcpyAsync(score_host, score_d, sizeof(float) * B, cudaMemcpyDeviceToHost, st));
  HM_CUDA(cudaStreamSynchronize(st));
  return 0;
}

HM_API int hmocr_last_decode_steps(hmocr_engine* e, int32_t* steps_run) {
  HM_CHECK(e != nullptr && steps_run != nullptr, "hmocr_last_decode_steps: null argument");
  HM_CHECK(e->last_poll_slot >= 0 && e->pinned_state != nullptr, "no persistent-kernel decode has run on this engine");
  *steps_run = e->pinned_state[e->last_poll_slot].step;
  return 0;
}

HM_API int hmocr_last_timings(hmocr_engine* e, float* encoder_ms, float* decode_ms) {
  HM_CHECK(e != nullptr, "null engine");
  if (e->timings_pending) {
    HM_CUDA(cudaEventSynchronize(e->ev[2]));
    HM_CUDA(cudaEventElapsedTime(&e->last_enc_ms, e->ev[0], e->ev[1]));
    HM_CUDA(cudaEventElapsedTime(&e->last_dec_ms, e->ev[1], e->ev[2]));
    e->timings_pending = false;
  }
  if (encoder_ms) *encoder_ms = e->last_enc_ms;
  if (decode_ms) *decode_ms = e->last_dec_ms;
  return 0;
}

// ---- kernel-level exports ----------------------------------------------------------------------------
HM_API int hmocr_gemm_f16(const void* a, int lda, int M, int K, const void* w, int N, const float* bias, int act,
                           const float* residual, int ldr, float* out_f32, int ld32, void* out_f16, int ld16,
                           const float* ln_gamma, const float* ln_beta, int force_bn, void* stream) {
  GemmEpilogue epi;
  epi.bias = bias; epi.act = act; epi.residual = residual; epi.ldr = ldr;
  epi.out_f32 = out_f32; epi.ld32 = ld32;
  epi.out_f16 = static_cast<h16*>(out_f16); epi.ld16 = ld16;
  epi.ln_gamma = ln_gamma; epi.ln_beta = ln_beta;
  return gemm_f16(static_cast<cudaStream_t>(stream), static_cast<const h16*>(a), lda, M, K,
                   static_cast<const h16*>(w), N, epi, force_bn);
}

HM_API int hmocr_swin_mlp(const void* xn, int M, int C, const void* w1, const float* b1, const void* w2, const float* b2,
                          float* x, void* stream) {
  HM_CHECK(xn != nullptr && w1 != nullptr && w2 != nullptr && x != nullptr, "null buffer");
  return swin_mlp(static_cast<cudaStream_t>(stream), static_cast<const h16*>(xn), M, C, static_cast<const h16*>(w1), b1,
                  static_cast<const h16*>(w2), b2, x);
}

HM_API int hmocr_layernorm(const float* x, int rows, int C, const float* gamma, const float* beta, void* out_f16,
                           float* out_f32, void* stream) {
  return layernorm(static_cast<cudaStream_t>(stream), x, rows, C, gamma, beta, static_cast<h16*>(out_f16),
                   out_f32);
}

HM_API int hmocr_patch_embed(const float* images, int B, const float* w, const float* b, const float* g,
                             const float* beta, float* x, void* stream) {
  return patch_embed(static_cast<cudaStream_t>(stream), images, B, w, b, g, beta, x);
}

HM_API int hmocr_patch_merge_ln(const float* x, int B, int H, int W, int C, const float* gamma, const float* beta,
                                void* out_f16, void* stream) {
  return patch_merge_ln(static_cast<cudaStream_t>(stream), x, B, H, W, C, gamma, beta,
                        static_cast<h16*>(out_f16));
}

HM_API int hmocr_self_attention(const void* qkv, int B, int T, int nhead, int causal, void* ctx, void* stream) {
  HM_CHECK(qkv != nullptr && ctx != nullptr, "null buffer");
  HM_CHECK(B >= 1 && T >= 1 && nhead >= 1, "bad shape B=%d T=%d nhead=%d", B, T, nhead);
  return mha_prefill_self(static_cast<cudaStream_t>(stream), static_cast<const h16*>(qkv), B, T, nhead,
                          static_cast<h16*>(ctx), causal != 0);
}

HM_API int hmocr_window_attention(const void* qkv, const float* qkv_bias, const float* rel_bias, int B, int H, int W,
                                  int C, int heads, int shift, void* ctx, void* stream) {
  return window_attention(static_cast<cudaStream_t>(stream), static_cast<const h16*>(qkv), qkv_bias,
                          rel_bias, B, H, W, C, heads, shift, static_cast<h16*>(ctx));
}
