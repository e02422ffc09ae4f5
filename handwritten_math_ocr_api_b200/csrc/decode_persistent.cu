// Persistent cluster decode kernel (sm_100a).
//
// Replaces the whole greedy loop body of /root/reference/src/inference.py:18-25 — i.e. one
// DecoderTransformer.forward step (src/model_swin.py:72-88, 8 x torch TransformerDecoderLayer,
// post-LN) + fc_out + argmax — for a range of steps [t_begin, t_end) in ONE launch.
//
// Mapping.  A thread-block CLUSTER of 8 CTAs owns 8 sequences end to end.  CTA rank c is
//   * attention head c (self- and cross-attention of the cluster's 8 rows for that head; warp w = row w), and
//   * the c-th 1/8 slice of the output features of every projection (q/k/v of head c, 32 features of
//     each out_proj and of linear2, 64 of linear1, V/8 vocabulary rows of fc_out).
// So each SM streams only 1/8 of the decoder weights per step.
//
// Math.  Projections run as  C^T[16 features x 8 rows] = W[16 x K] . X^T  with mma.sync.m16n8k16
// (fp16 in, fp32 accumulate): the WEIGHTS are the M=16 operand and the cluster's 8 rows are exactly
// the N=8 operand, so no tensor-core lane is wasted and one weight fragment is read from shared
// memory exactly once.  tcgen05 needs M >= 64 rows and the step does 13-15 MFLOP per token: this
// kernel is latency/bandwidth bound, not tensor bound.
//
// Weights.  Pre-packed per CTA as a stream of 8448-byte chunks (one m-tile: 16 features x 256 inputs,
// see decode_persistent.cuh).  Chunk i of the stream belongs to warp (i mod 8): every warp owns ONE
// shared-memory slot, waits for its chunk on its own mbarrier, runs its 16 mma, and immediately
// re-arms the slot with its next chunk (cp.async.bulk, 8 chunks ahead in the stream).  Producer and
// consumer of a slot are the same warp, so the ring needs no empty-barriers and no block barrier.
//
// The vocabulary projection (40 chunks per CTA, 5 per warp) is bound by the shared-memory port at two CTAs per SM
// (every weight byte crosses it twice: TMA in, ldmatrix out): its activation fragments are loaded into registers
// once per step, not once per chunk.
//
// Exchange.  The activations of the 8 rows are all-gathered between the 8 CTAs through distributed
// shared memory with st.async (remote store + complete_tx on an mbarrier of the DESTINATION CTA):
// point to point, no fence on the sender, no cluster-wide barrier; a CTA proceeds as soon as ITS
// inputs have arrived.  Six exchanges per layer (context, y, context, y, hidden, y) + one per step
// (arg-max partials).  barrier.cluster is used only at kernel start and end.
//
// Attention.  One warp per (row, head), on tensor cores: S = K q as mma.m16n8k16 with 16 cached keys
// as the M operand, softmax in fp32 on ex2, then O = V^T p with 16 head dims as the M operand.  Both caches are
// fp16 and stored in the REGISTER ORDER of the mma A operand (fragment-major blocks of 32 keys x 32 dims = 2 KB),
// so a fragment is one coalesced 16-byte load per lane.  One pass with an online softmax: the K and the V block of
// the same 32 keys are in flight together (4 KB per warp), the probabilities reach the P operand by two shuffles
// per 16 keys (no shared memory); a last block with <= 16 keys is read as 1 KB.
// The cache rows of the NEXT layer are pulled into L2 (cp.async.bulk.prefetch.L2) one layer ahead; history
// loads carry L2 evict_first, the weight stream and the memory K/V evict_last (they are re-read every step).
//
// Occupancy is part of the design: ~104 KB of shared memory and <= 128 registers, so TWO CTAs (of
// different clusters) share an SM; B=256 runs as 32 clusters in a single wave.
#include <cuda_fp16.h>

#include "decode_persistent.cuh"

namespace hmocr {
namespace {

constexpr int CL = 8, THREADS = 256, NW = 8, R = DP_ROWS;
constexpr int D = 256, FF = 512, HD = 32, NH = 8;
constexpr int PD = D + 8, PF = FF + 8;            // padded operand pitches (elements): conflict-free ldmatrix
constexpr float ATT_SCALE = 0.17677669529663687f * 1.4426950408889634f;   // log2(e) / sqrt(32): softmax on ex2
constexpr float LN_EPS = 1e-5f;

struct __align__(16) Partial { float m; int idx; float s; int pad; };
// beam search: K best (logit, token) of a row, best first; 48 bytes = three 16-byte DSMEM stores
struct __align__(16) TopList { float v[DP_MAX_BEAM]; int i[DP_MAX_BEAM]; int pad[2]; };
struct Cand { float score; int flat; float lp; };           // lp = log_softmax of the candidate's token
struct Sel { float score; int parent; int tok; float lp; };

struct Smem {
  alignas(128) uint8_t slot[NW][DP_CHUNK];  // warp-private weight slots
  alignas(16) float y32[R][D];              // pre-LayerNorm rows gathered from the 8 feature slices
  alignas(16) __half xa[R][PD];             // LayerNorm output (full rows), fp16 operand
  alignas(16) __half ctx[R][PD];            // attention context gathered from the 8 heads
  alignas(16) __half hf[R][PF];             // relu(linear1) gathered from the 8 slices
  alignas(16) float stg[4][16][9];          // staging of GEMM tiles [task][feature][row] (hidden: fp16 [8][72])
  alignas(16) float x32s[R][32];            // fp32 residual stream, this CTA's 32-feature slice only
  alignas(16) __half qh[R][HD];             // this head's scaled query (fp16 mma operand)
  alignas(16) __half knew[R][HD];           // this step's key / value of head c (appended to the caches after use)
  alignas(16) __half vnew[R][HD];
  Partial part[CL][R];                      // per-CTA argmax / sum-exp partials (gathered)
  Partial wpart[NW][R];                     // per-warp partials
  // beam search only
  TopList wtop[NW][R];                      // per-warp top-K logits of every row
  TopList ctop[CL][R];                      // per-CTA top-K, gathered from the 8 CTAs
  Cand cand[R][DP_MAX_BEAM];                // candidate (score, hypothesis * V + token, log-prob) of every row
  Sel sel[R];                               // chosen (score, parent row, token, log-prob) of every new hypothesis
  float bscore[R];
  int bfin[R], bsrc[R];
  alignas(8) uint64_t full[NW];
  alignas(8) uint64_t xbar[5];              // exchange barriers: context, y, hidden, partials, top-K lists
  int stop_flag;                            // rank 0's reading of "every row has finished" at kernel entry
};
enum { X_CTX = 0, X_Y = 1, X_HF = 2, X_PART = 3, X_TOP = 4 };
constexpr uint32_t XB_CTX = R * D * 2, XB_Y = R * D * 4, XB_HF = R * FF * 2, XB_PART = CL * R * sizeof(Partial);
constexpr uint32_t XB_TOP = CL * R * sizeof(TopList);
static_assert(sizeof(Smem) <= 112 * 1024, "two CTAs must fit one SM");
static_assert(sizeof(float) * 4 * 16 * 9 >= sizeof(__half) * R * 72, "hidden staging aliases stg");

// ---- PTX helpers ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// st.async: a remote (DSMEM) store that also performs complete_tx(bytes) on an mbarrier of the
// destination CTA - the sender needs no fence and no barrier, the receiver waits on its own mbarrier.
__device__ __forceinline__ void st_async_v4(uint32_t addr, uint4 v, uint32_t mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
                   addr),
               "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(mbar)
               : "memory");
}
// Wait for a phase whose bytes were written into THIS CTA's shared memory by st.async of other CTAs.
// Plain try_wait, as for TMA multicast: a cluster-scope acquire would make ptxas emit CCTL.IVALL (an
// L1 invalidate, ~400 cycles) after every wait, and shared memory is not cached in L1.
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  long long t0 = 0;
  for (;;) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(a), "r"(parity)
        : "memory");
    if (ok) return;
    if (t0 == 0) t0 = clock64();
    else if (clock64() - t0 > 4000000000LL) {
      __trap();                     // a protocol bug fails the launch instead of hanging the GPU (no printf: code size)
    }
  }
}
__device__ __forceinline__ void mbar_wait_trap(uint64_t* bar, uint32_t parity) {       // common.cuh mbar_wait without the printf
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}
// L2 residency (126 MB, two partitions).  Per decode step at B = 256 the kernel touches three kinds of bytes:
//   * the weight stream (13.5 MB, read by EVERY cluster every step) and the memory K/V of cross-attention (67 MB,
//     read by its cluster every step): reusable -> evict_last, they should stay L2-resident across steps;
//   * the self-attention history (2 MB x t, every byte read exactly once per step, 315 MB at t = 150): streaming ->
//     evict_first, so it does not push the reusable set out.
// Policy operands are the fixed encodings of createpolicy.fractional.L2::evict_{first,last} with fraction 1.0.
constexpr uint64_t L2_EVICT_FIRST = 0x12F0000000000000ull, L2_EVICT_LAST = 0x14F0000000000000ull;
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {     // weights: keep in L2
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                   smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar)), "l"(L2_EVICT_LAST)
               : "memory");
}
template <bool KEEP>
__device__ __forceinline__ void prefetch_l2(const void* src, int bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(reinterpret_cast<uint64_t>(src)), "r"(bytes),
               "l"(KEEP ? L2_EVICT_LAST : L2_EVICT_FIRST)
               : "memory");
}
// 16-byte cache-block load that bypasses L1 (every line is used once per SM) with an L2 eviction priority
template <bool KEEP>
__device__ __forceinline__ uint4 ld_kv(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p), "l"(KEEP ? L2_EVICT_LAST : L2_EVICT_FIRST)
               : "memory");
  return v;
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void mma_f16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                        uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ __half to_half_sat(float x) { return to_h16(x); }                 // saturating (common.cuh)
__device__ __forceinline__ uint32_t pack_half(float a, float b) { return pack16(a, b); }

// C^T[16 features x 8 rows] = W[16 x 256] (one weight chunk, pitch PD) . X[8 rows x 256]^T (smem, pitch PB)
//   c[0]: (feature lane/4, row 2*(lane%4)), c[1]: (same feature, row + 1), c[2], c[3]: feature + 8
// Four independent accumulator chains keep the tensor pipe busy from a single warp.
template <int PB>
__device__ __forceinline__ void gemm16(const uint8_t* W, const __half* X, int lane, float (&c)[4]) {
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
  const uint32_t a_addr = smem_u32(W) + ((lane & 15) * PD + (lane >> 4) * 8) * 2;
  const uint32_t b_addr = smem_u32(X) + ((lane & 7) * PB + (lane >> 3) * 8) * 2;
#pragma unroll
  for (int kk = 0; kk < 8; ++kk) {         // 32 input columns per iteration
    uint32_t b[4], a0[4], a1[4];
    ldsm_x4(b_addr + kk * 64, b);
    ldsm_x4(a_addr + kk * 64, a0);
    ldsm_x4(a_addr + kk * 64 + 32, a1);
    mma_f16(acc[(2 * kk) & 3], a0[0], a0[1], a0[2], a0[3], b[0], b[1]);
    mma_f16(acc[(2 * kk + 1) & 3], a1[0], a1[1], a1[2], a1[3], b[2], b[3]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) c[i] = (acc[0][i] + acc[1][i]) + (acc[2][i] + acc[3][i]);
}

// The same product with the activation (B) fragments already in registers: the vocabulary projection runs five weight
// chunks per warp against the SAME 8 x 256 activations, and at two CTAs per SM that phase is bound by the shared-memory
// port (TMA writes + ldmatrix reads of the weights + the activation re-reads) - loading the 32 fragment registers once
// per step instead of once per chunk takes a fifth of the port traffic away.  Same mma order as gemm16: same bits.
template <int PB>
__device__ __forceinline__ void load_bfrags(const __half* X, int lane, uint32_t (&bf)[8][4]) {
  const uint32_t b_addr = smem_u32(X) + ((lane & 7) * PB + (lane >> 3) * 8) * 2;
#pragma unroll
  for (int kk = 0; kk < 8; ++kk) ldsm_x4(b_addr + kk * 64, bf[kk]);
}
__device__ __forceinline__ void gemm16_pre(const uint8_t* W, const uint32_t (&bf)[8][4], int lane, float (&c)[4]) {
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
  const uint32_t a_addr = smem_u32(W) + ((lane & 15) * PD + (lane >> 4) * 8) * 2;
#pragma unroll
  for (int kk = 0; kk < 8; ++kk) {
    uint32_t a0[4], a1[4];
    ldsm_x4(a_addr + kk * 64, a0);
    ldsm_x4(a_addr + kk * 64 + 32, a1);
    mma_f16(acc[(2 * kk) & 3], a0[0], a0[1], a0[2], a0[3], bf[kk][0], bf[kk][1]);
    mma_f16(acc[(2 * kk + 1) & 3], a1[0], a1[1], a1[2], a1[3], bf[kk][2], bf[kk][3]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) c[i] = (acc[0][i] + acc[1][i]) + (acc[2][i] + acc[3][i]);
}

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---- fragment-major K / V caches ---------------------------------------------------------------------
// Both caches are stored in the register layout of the mma.m16n8k16 A operand, so a cache fragment is ONE
// coalesced 16-byte load per lane (512 contiguous bytes per warp instruction) and needs no address
// arithmetic, no clamping and no register shuffling.  A block = 32 keys x 32 dims = 2048 bytes:
//   K block: [tile 0..1][k-step s 0..1][lane][a0 a1 a2 a3]   tile = 16 keys, lane = (g, t):
//            a0 = key g,   dims 16s+4t+{0,1};  a1 = key g+8, same dims;
//            a2 = key g,   dims 16s+4t+{2,3};  a3 = key g+8, same dims.
//   V block: [k-step ks 0..1][m-tile mt 0..1][lane][a0 a1 a2 a3]   k-step = the 16 keys of K tile ks:
//            a0 = dim 4g+2mt,   slots 2t, 2t+1;   a1 = dim 4g+2mt+1, same slots;
//            a2 = dim 4g+2mt,   slots 2t+8, 2t+9; a3 = dim 4g+2mt+1, same slots,
//            where key r = g' + 8h of the tile sits in slot 8*(g'/4) + 2*(g'%4) + h - so the two scores a
//            lane gets from the K tile (keys g', g'+8) are exactly one packed half2 of the P operand.
// Offsets below are in halves, relative to the start of the (layer, row, head) region.
__device__ __forceinline__ int kfrag_word(int key_in_blk, int i) {     // 32-bit word index of dims (2i, 2i+1), i < 16
  const int tile = key_in_blk >> 4, r = key_in_blk & 15, g = r & 7, h = r >> 3;
  const int sidx = i >> 3, t = (i >> 1) & 3, w = i & 1;
  return tile * 256 + sidx * 128 + (g * 4 + t) * 4 + 2 * w + h;
}
__device__ __forceinline__ int vfrag_half(int key_in_blk, int d) {      // half index of (dim d, key)
  const int ks = key_in_blk >> 4, r = key_in_blk & 15, g = r & 7, h = r >> 3;
  const int gd = d >> 2, mt = (d >> 1) & 1, hd = d & 1;
  return (ks * 2 + mt) * 256 + (gd * 4 + (g & 3)) * 8 + (2 * (g >> 2) + hd) * 2 + h;
}

// One query row of one head against n cached keys, on tensor cores.
//   scores:  S[16 keys x 8] = K[16 keys x 32 dims] . q      (q replicated in all 8 columns; two k-steps)
//   output:  O[16 dims x 8] = Vt[16 dims x 16 keys] . p     (p replicated in all columns; two m-tiles)
// q is pre-scaled by log2(e)/sqrt(32): the softmax runs on ex2.  Keys come in blocks of 32 (2 KB of K and 2 KB of V).
// Result: out[j] = context of dim 4*g4 + j (identical in the 4 lanes that share g4).
// If NEW, one more key/value (this step's own, still in shared memory) is folded in on CUDA cores, so the
// attention never waits for its own cache append to travel through L2.

// Block b of a (layer, row, head) region holding `n` keys in all.  In both layouts the first 1 KB of a block is its
// first 16 keys (K: tile 0, V: k-step 0), so a last block with <= 16 keys is read as 1 KB, not 2 (the other half is
// the unwritten tail: its scores are masked and its probabilities are zero - the registers are zeroed so that 0 x V
// stays finite).  MEM: memory K/V of cross-attention (re-read every step -> evict_last); history -> evict_first.
template <bool MEM>
__device__ __forceinline__ void load_block(const uint4* base, int b, int n, uint4 (&d)[4]) {
  const bool half = n - 32 * b <= 16;                                // warp-uniform
#pragma unroll
  for (int u = 0; u < 2; ++u) d[u] = ld_kv<MEM>(base + 128 * b + 32 * u);
  if (half) {
    d[2] = make_uint4(0u, 0u, 0u, 0u); d[3] = make_uint4(0u, 0u, 0u, 0u);
  } else {
#pragma unroll
    for (int u = 2; u < 4; ++u) d[u] = ld_kv<MEM>(base + 128 * b + 32 * u);
  }
}
// bytes of a region that hold its first `keys` keys at 1 KB granularity (for the L2 prefetch)
__device__ __forceinline__ int region_bytes(int keys) { return ((keys + 15) >> 4) * 1024; }
// If COPY (beam search), every consumed history block is also stored to (Kd, Vd): the destination row of the
// other cache set - the parent gather of the beam reorder rides on the attention loads.
__device__ __forceinline__ void store_block(uint4* base, int b, const uint4 (&d)[4]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) __stcg(base + 128 * b + 32 * u, d[u]);
}
// One pass, online softmax.  (The two-pass form of round 1 - all scores, softmax, then P.V - kept ONE 2 KB block in
// flight per warp: every K block, then every V block, paid a full L2 round trip behind the previous one, and the
// softmax between them overlapped nothing: 7.2k cycles per layer at step 100, now 5.9k.)  The K and the V block
// of the same 32 keys travel TOGETHER (two register slots, 4 KB in flight per warp) and every block is finished
// before the next: scores -> running maximum -> probabilities -> accumulators rescaled -> P.V.  The next K block
// is requested as soon as the scores of this one exist, the next V block as soon as its P.V is issued, so the
// softmax arithmetic of block b hides under the loads of block b+1, and the 4 * NB score registers of the
// two-pass form are gone.  The P operand needs no shared memory: the V cache's key order makes the packed pair
// {p[key g], p[key g+8]} of lane group g exactly the half2 that lanes t = g (b0) and t = g - 4 (b1) feed to the
// mma, so two shuffles per 16 keys replace the store / __syncwarp / load round trip.
struct KvPair { uint4 k[4], v[4]; };
template <bool MEM>
__device__ __forceinline__ void attend_issue2(const __half* Kc, const __half* Vc, int n, int lane, KvPair& kv) {
  if (n > 0) {                                                       // warp-uniform
    load_block<MEM>(reinterpret_cast<const uint4*>(Kc) + lane, 0, n, kv.k);
    load_block<MEM>(reinterpret_cast<const uint4*>(Vc) + lane, 0, n, kv.v);
  }
}
template <int NB, bool NEW, bool COPY, bool MEM>
__device__ __forceinline__ void attend_online(const __half* qh, const __half* Kc, const __half* Vc, int n,
                                              const __half* knew, const __half* vnew, int lane, KvPair& kv,
                                              float (&out)[4], __half* Kd = nullptr, __half* Vd = nullptr) {
  const int g4 = lane >> 2, t4 = lane & 3;
  const uint2 q0 = *reinterpret_cast<const uint2*>(qh + 4 * t4), q1 = *reinterpret_cast<const uint2*>(qh + 16 + 4 * t4);
  const int nb = (n + 31) >> 5;
  const uint4* Kl = reinterpret_cast<const uint4*>(Kc) + lane;
  const uint4* Vl = reinterpret_cast<const uint4*>(Vc) + lane;
  float m = -INFINITY, den = 0.f;                                    // den: this lane's share (its two keys per tile)
  float acc0[4] = {0.f, 0.f, 0.f, 0.f}, acc1[4] = {0.f, 0.f, 0.f, 0.f};
  if (NEW) {                                                         // this step's own key / value start the recurrence
    const uint4 kn = *reinterpret_cast<const uint4*>(knew + t4 * 8), qn = *reinterpret_cast<const uint4*>(qh + t4 * 8);
    const uint32_t qw[4] = {qn.x, qn.y, qn.z, qn.w}, kw[4] = {kn.x, kn.y, kn.z, kn.w};
    float a = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 qf = __half22float2(*reinterpret_cast<const __half2*>(&qw[i]));
      const float2 kf = __half22float2(*reinterpret_cast<const __half2*>(&kw[i]));
      a = fmaf(qf.x, kf.x, a); a = fmaf(qf.y, kf.y, a);
    }
    a += __shfl_xor_sync(0xffffffffu, a, 1);
    a += __shfl_xor_sync(0xffffffffu, a, 2);
    m = a;                                                           // p = 2^0 = 1 exactly
    den = (g4 == 0) ? 1.f : 0.f;                                     // counted once in the reduction over g4
    const uint2 vn = *reinterpret_cast<const uint2*>(vnew + 4 * g4);
    const float2 v01 = __half22float2(*reinterpret_cast<const __half2*>(&vn.x));
    const float2 v23 = __half22float2(*reinterpret_cast<const __half2*>(&vn.y));
    acc0[0] = v01.x; acc0[2] = v01.y; acc1[0] = v23.x; acc1[2] = v23.y;
  }
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    if (b < nb) {                                                    // warp-uniform
      float sc[4];
#pragma unroll
      for (int tile = 0; tile < 2; ++tile) {
        float c[4] = {0.f, 0.f, 0.f, 0.f};
        mma_f16(c, kv.k[2 * tile].x, kv.k[2 * tile].y, kv.k[2 * tile].z, kv.k[2 * tile].w, q0.x, q0.y);
        mma_f16(c, kv.k[2 * tile + 1].x, kv.k[2 * tile + 1].y, kv.k[2 * tile + 1].z, kv.k[2 * tile + 1].w, q1.x, q1.y);
        const int key = 32 * b + 16 * tile + g4;
        sc[2 * tile] = (key < n) ? c[0] : -INFINITY;
        sc[2 * tile + 1] = (key + 8 < n) ? c[2] : -INFINITY;
      }
      if (COPY && Kd != nullptr) store_block(reinterpret_cast<uint4*>(Kd) + lane, b, kv.k);
      if (b + 1 < NB && b + 1 < nb) load_block<MEM>(Kl, b + 1, n, kv.k);
      float bm = fmaxf(fmaxf(sc[0], sc[1]), fmaxf(sc[2], sc[3]));
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) bm = fmaxf(bm, __shfl_xor_sync(0xffffffffu, bm, o));
      const float mn = fmaxf(m, bm);                                 // finite: the block holds at least one key
      const float rs = ex2f(m - mn);                                 // 0 on the first block without NEW (m = -inf)
      m = mn;
      const __half2 ph0 = __floats2half2_rn(ex2f(sc[0] - m), ex2f(sc[1] - m));
      const __half2 ph1 = __floats2half2_rn(ex2f(sc[2] - m), ex2f(sc[3] - m));
      const float2 pf0 = __half22float2(ph0), pf1 = __half22float2(ph1);   // normalise with the rounded weights
      den = fmaf(den, rs, (pf0.x + pf0.y) + (pf1.x + pf1.y));
#pragma unroll
      for (int i = 0; i < 4; ++i) { acc0[i] *= rs; acc1[i] *= rs; }
      const uint32_t w0 = *reinterpret_cast<const uint32_t*>(&ph0), w1 = *reinterpret_cast<const uint32_t*>(&ph1);
      const uint32_t p0x = __shfl_sync(0xffffffffu, w0, t4 << 2), p0y = __shfl_sync(0xffffffffu, w0, (t4 + 4) << 2);
      const uint32_t p1x = __shfl_sync(0xffffffffu, w1, t4 << 2), p1y = __shfl_sync(0xffffffffu, w1, (t4 + 4) << 2);
      mma_f16(acc0, kv.v[0].x, kv.v[0].y, kv.v[0].z, kv.v[0].w, p0x, p0y);
      mma_f16(acc1, kv.v[1].x, kv.v[1].y, kv.v[1].z, kv.v[1].w, p0x, p0y);
      mma_f16(acc0, kv.v[2].x, kv.v[2].y, kv.v[2].z, kv.v[2].w, p1x, p1y);
      mma_f16(acc1, kv.v[3].x, kv.v[3].y, kv.v[3].z, kv.v[3].w, p1x, p1y);
      if (COPY && Vd != nullptr) store_block(reinterpret_cast<uint4*>(Vd) + lane, b, kv.v);
      if (b + 1 < NB && b + 1 < nb) load_block<MEM>(Vl, b + 1, n, kv.v);
    }
  }
#pragma unroll
  for (int o = 4; o < 32; o <<= 1) den += __shfl_xor_sync(0xffffffffu, den, o);
  const float inv = __fdividef(1.0f, den);
  out[0] = acc0[0] * inv; out[1] = acc0[2] * inv; out[2] = acc1[0] * inv; out[3] = acc1[2] * inv;
}

__device__ __forceinline__ void merge_partial(Partial& a, const Partial& b) {
  // combine (max, first-argmax, sum exp(x - max)); ties -> lower index (torch.argmax)
  if (b.m > a.m || (b.m == a.m && b.idx < a.idx)) {
    const float sa = (a.m == -INFINITY) ? 0.f : a.s * __expf(a.m - b.m);
    a.s = sa + b.s; a.m = b.m; a.idx = b.idx;
  } else {
    const float sb = (b.m == -INFINITY) ? 0.f : b.s * __expf(b.m - a.m);
    a.s += sb;
  }
}
__device__ __forceinline__ void update_partial(Partial& a, float v, int idx) {
  if (v > a.m) { a.s = a.s * __expf(a.m - v) + 1.0f; a.m = v; a.idx = idx; }
  else a.s += __expf(v - a.m);
}
__device__ __forceinline__ Partial shfl_partial(const Partial& a, int o) {
  Partial r;
  r.m = __shfl_xor_sync(0xffffffffu, a.m, o);
  r.idx = __shfl_xor_sync(0xffffffffu, a.idx, o);
  r.s = __shfl_xor_sync(0xffffffffu, a.s, o);
  r.pad = 0;
  return r;
}

struct LnRegs { float4 g0, g1, b0, b1; };

// ---- beam search: per-thread / per-warp top-K lists ------------------------------------------------------
// order of candidates: higher value first; equal values: lower index first (torch's stable descending sort)
__device__ __forceinline__ bool cand_before(float v, int i, float w, int j) { return v > w || (v == w && i < j); }
template <int KB>
struct TopK {
  float v[KB];
  int i[KB];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int k = 0; k < KB; ++k) { v[k] = -INFINITY; i[k] = 0x7fffffff; }
  }
  __device__ __forceinline__ void insert(float x, int idx) {
    if (!cand_before(x, idx, v[KB - 1], i[KB - 1])) return;
    v[KB - 1] = x; i[KB - 1] = idx;
#pragma unroll
    for (int k = KB - 1; k > 0; --k) {
      const bool sw = cand_before(v[k], i[k], v[k - 1], i[k - 1]);
      const float tv = v[k]; const int ti = i[k];
      v[k] = sw ? v[k - 1] : v[k]; i[k] = sw ? i[k - 1] : i[k];
      v[k - 1] = sw ? tv : v[k - 1]; i[k - 1] = sw ? ti : i[k - 1];
    }
  }
  __device__ __forceinline__ void merge_xor(int mask) {           // butterfly step: both lanes end with the union's top-K
    float ov[KB]; int oi[KB];
#pragma unroll
    for (int k = 0; k < KB; ++k) { ov[k] = __shfl_xor_sync(0xffffffffu, v[k], mask); oi[k] = __shfl_xor_sync(0xffffffffu, i[k], mask); }
#pragma unroll
    for (int k = 0; k < KB; ++k) insert(ov[k], oi[k]);
  }
  __device__ __forceinline__ void store(TopList& d) const {
#pragma unroll
    for (int k = 0; k < KB; ++k) { d.v[k] = v[k]; d.i[k] = i[k]; }
  }
  __device__ __forceinline__ void load(const TopList& d) {
#pragma unroll
    for (int k = 0; k < KB; ++k) { v[k] = d.v[k]; i[k] = d.i[k]; }
  }
};
template <>
struct TopK<0> {                                                  // greedy instantiation: no state, no work
  __device__ __forceinline__ void init() {}
  __device__ __forceinline__ void insert(float, int) {}
};

// The fp32 bias of weight row r travels in the padding of that row (halves 256, 257 of 264): it arrives with
// the weights, costs no extra copy, barrier or shared memory, and is read before the slot is released.
__device__ __forceinline__ float chunk_bias(const uint8_t* slot, int r) {
  return *reinterpret_cast<const float*>(slot + (r * PD + D) * 2);
}

// KB = 0: greedy.  KB = DP_MAX_BEAM: beam search with p.beam <= KB hypotheses per image (see decode_persistent.cuh).
// DEV = true: the instrumented build (phase tracing); the production instantiations carry none of that code.
template <int NB, int KB, bool DEV>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(THREADS, 2)
decode_persistent_kernel(const DecPersistParams p, int t_begin, int t_end) {
  constexpr bool BEAM = KB > 0;
  extern __shared__ __align__(128) uint8_t smem_raw[];
  Smem& s = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = (int)cluster_ctarank();              // feature slice == attention head
  const int RPC = BEAM ? p.rows_per_cluster : R;     // rows owned by one cluster
  const int row0 = (blockIdx.x / CL) * RPC;
  const int nrows = min(RPC, p.rows - row0);         // valid rows of this cluster (1..8)
  const int g4 = lane >> 2, t4 = lane & 3;           // mma fragment coordinates
  const int L = p.num_layers, S = p.chunks_per_step, FT = p.fc_tiles;
  const int total_chunks = (t_end - t_begin) * S;
  const int cols_per_cta = FT * 16;
  const uint8_t* wst = p.wstream + (size_t)c * S * DP_CHUNK;
  const bool row_ok = warp < nrows;                  // warp w owns row w in the per-row phases
  const int my_row = row0 + min(warp, nrows - 1);    // clamped: padded rows recompute the last valid row

  // ---- distributed shared memory addressing: remote(ptr, rank) = cl0 + rank * stride + offset ------
  const uint32_t s_local = smem_u32(&s);
  const uint32_t cl0 = mapa(s_local, 0);
  const uint32_t cl_stride = mapa(s_local, 1) - cl0;
  if (tid < CL && mapa(s_local, tid) != cl0 + tid * cl_stride) {
    printf("hmocr: non-linear shared::cluster window\n");
    __trap();
  }

  // ---- weight slots: warp w consumes chunks w, w+8, w+16, ... of the stream ------------------------
  int wk = 0;                 // chunks this warp has consumed
  int wgi = warp;             // stream index (this launch) of the chunk in / on its way to the slot
  int wpos = warp % S;        // ... modulo the per-step period
  auto slot_fetch = [&]() {   // lane 0
    if (wgi < total_chunks) {
      mbar_expect_tx(&s.full[warp], DP_CHUNK);
      bulk_g2s(s.slot[warp], wst + (size_t)wpos * DP_CHUNK, DP_CHUNK, &s.full[warp]);
    }
  };
  auto slot_wait = [&]() { mbar_wait_trap(&s.full[warp], wk & 1); };
  auto slot_release = [&]() {
    __syncwarp();
    // The warp has read the slot through the generic proxy (ldmatrix, the bias words); the refill below writes it
    // through the async proxy (TMA).  Without this cross-proxy fence the two are not ordered: under heavy memory
    // traffic (two CTAs per SM) about 1 % of the (image, run) pairs of a B = 256 decode came back with slightly
    // different log-probabilities - a few elements of the NEXT weight tile leaking into the current one
    // (DESIGN.md 4.4; found with scratch/beam_repeat_probe3.py and scratch/poison_probe.py).
    fence_proxy_async();
    ++wk; wgi += NW; wpos += NW;
    if (wpos >= S) wpos -= S;
    if (lane == 0) slot_fetch();
  };
  // ---- exchanges --------------------------------------------------------------------------------------
  // The mbarrier phase parities follow from two counters instead of one per exchange: per layer the context barrier
  // completes twice (parities 0, 1), the y barrier three times (parity (layer + site) & 1), the hidden barrier once
  // (layer & 1); partials / top-K lists once per step.
  uint32_t nlayer = 0, nstep = 0;            // layers / steps done since the launch started
  auto xwait = [&](int X, uint32_t parity, uint32_t bytes) {
    mbar_wait_cluster(&s.xbar[X], parity & 1);
    if (tid == 0) mbar_expect_tx(&s.xbar[X], bytes);      // arm the next phase
  };
  auto send_all = [&](const void* local_dst, uint4 v, int X) {    // the same 16 bytes to all 8 CTAs
    const uint32_t off = smem_u32(local_dst) - s_local, boff = smem_u32(&s.xbar[X]) - s_local;
#pragma unroll
    for (int rk = 0; rk < CL; ++rk) {
      const uint32_t base = cl0 + rk * cl_stride;
      st_async_v4(base + off, v, base + boff);
    }
  };
  // LayerNorm gamma/beta of this lane's 8 columns, fetched (L2) a phase ahead of their use
  auto load_ln = [&](int l, int which) {
    const float* g = p.lnparams + ((size_t)l * 6 + 2 * which) * D + lane * 8;
    LnRegs r;
    r.g0 = __ldg(reinterpret_cast<const float4*>(g));
    r.g1 = __ldg(reinterpret_cast<const float4*>(g + 4));
    r.b0 = __ldg(reinterpret_cast<const float4*>(g + D));
    r.b1 = __ldg(reinterpret_cast<const float4*>(g + D + 4));
    return r;
  };
  // finish a row: fp16 operand row + this CTA's fp32 residual slice
  auto put_row = [&](const float (&v)[8]) {
    if ((lane >> 2) == c) {                              // features c*32 .. c*32+31 live in lanes 4c .. 4c+3
      *reinterpret_cast<float4*>(&s.x32s[warp][(lane & 3) * 8]) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(&s.x32s[warp][(lane & 3) * 8 + 4]) = make_float4(v[4], v[5], v[6], v[7]);
    }
    *reinterpret_cast<uint4*>(&s.xa[warp][lane * 8]) =
        make_uint4(pack_half(v[0], v[1]), pack_half(v[2], v[3]), pack_half(v[4], v[5]), pack_half(v[6], v[7]));
  };
  // LayerNorm of the gathered rows: warp w owns row w; lane owns 8 consecutive columns
  auto layer_norm = [&](const LnRegs& ln) {
    const float4 a = *reinterpret_cast<const float4*>(&s.y32[warp][lane * 8]);
    const float4 b = *reinterpret_cast<const float4*>(&s.y32[warp][lane * 8 + 4]);
    float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    // one pass: sum and sum of squares reduced together (5 shuffle rounds instead of 10).  The rows are
    // residual + projection of normalised activations (|mean| well below the spread), so E[x^2] - mean^2 in
    // fp32 loses nothing that matters; clamped at 0 for safety.
    float sum = 0.f, sq = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) { sum += v[e]; sq = fmaf(v[e], v[e], sq); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sum += __shfl_xor_sync(0xffffffffu, sum, o);
      sq += __shfl_xor_sync(0xffffffffu, sq, o);
    }
    const float mean = sum * (1.0f / D);
    const float rstd = rsqrtf(fmaxf(sq * (1.0f / D) - mean * mean, 0.f) + LN_EPS);
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] -= mean;
    v[0] = v[0] * rstd * ln.g0.x + ln.b0.x; v[1] = v[1] * rstd * ln.g0.y + ln.b0.y;
    v[2] = v[2] * rstd * ln.g0.z + ln.b0.z; v[3] = v[3] * rstd * ln.g0.w + ln.b0.w;
    v[4] = v[4] * rstd * ln.g1.x + ln.b1.x; v[5] = v[5] * rstd * ln.g1.y + ln.b1.y;
    v[6] = v[6] * rstd * ln.g1.z + ln.b1.z; v[7] = v[7] * rstd * ln.g1.w + ln.b1.w;
    put_row(v);
  };
  // x = embedding[token] + pos[t] of row `warp`
  auto embed_row = [&](int t, long long tk) {
    if (tk < 0 || tk >= p.vocab) tk = 0;
    const float4* e = reinterpret_cast<const float4*>(p.emb + (size_t)tk * D + lane * 8);
    const float4* ps = reinterpret_cast<const float4*>(p.pos + (size_t)t * D + lane * 8);
    const float4 e0 = __ldg(e), e1 = __ldg(e + 1), p0 = __ldg(ps), p1 = __ldg(ps + 1);
    const float v[8] = {e0.x + p0.x, e0.y + p0.y, e0.z + p0.z, e0.w + p0.w,
                        e1.x + p1.x, e1.y + p1.y, e1.z + p1.z, e1.w + p1.w};
    put_row(v);
  };
  // attention context of (row `warp`, head c) -> ctx[warp][c*32 ..] of every CTA.  A lane holds dims
  // 4*g4 .. 4*g4+3; with its neighbour (g4 ^ 1) that is one 16-byte piece, sent to CTA (g4 & 1) * 4 + t4.
  auto send_ctx = [&](const float (&o)[4]) {
    const uint32_t u0 = pack_half(o[0], o[1]), u1 = pack_half(o[2], o[3]);
    const uint32_t w0 = __shfl_xor_sync(0xffffffffu, u0, 4), w1 = __shfl_xor_sync(0xffffffffu, u1, 4);
    const uint4 v = (g4 & 1) ? make_uint4(w0, w1, u0, u1) : make_uint4(u0, u1, w0, w1);
    const uint32_t base = cl0 + ((g4 & 1) * 4 + t4) * cl_stride;
    st_async_v4(base + (smem_u32(&s.ctx[warp][c * HD + (g4 >> 1) * 8]) - s_local), v,
                base + (smem_u32(&s.xbar[X_CTX]) - s_local));
  };
  // tile of an out-projection -> staging; then 64 threads add bias + residual and send y (4 features each)
  auto stage_tile = [&](int slot_idx, const float (&acc)[4], float b0, float b1) {     // + the chunk's bias
    s.stg[slot_idx][g4][2 * t4] = acc[0] + b0; s.stg[slot_idx][g4][2 * t4 + 1] = acc[1] + b0;
    s.stg[slot_idx][g4 + 8][2 * t4] = acc[2] + b1; s.stg[slot_idx][g4 + 8][2 * t4 + 1] = acc[3] + b1;
  };
  auto send_y = [&](int u, bool two_partials) {   // u in [0, 64): row u/8, features 4*(u%8) ..
    const int r = u >> 3, fq = u & 7, mt = fq >> 2, f0 = (fq & 3) * 4;
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float a = two_partials ? s.stg[2 * mt][f0 + e][r] + s.stg[2 * mt + 1][f0 + e][r] : s.stg[mt][f0 + e][r];
      v[e] = a + s.x32s[r][fq * 4 + e];
    }
    send_all(&s.y32[r][c * 32 + fq * 4],
             make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3])), X_Y);
  };

  if (tid == 0) {
    for (int i = 0; i < NW; ++i) mbar_init(&s.full[i], 1);
    for (int i = 0; i < 5; ++i) mbar_init(&s.xbar[i], 1);
    fence_barrier_init();
    mbar_expect_tx(&s.xbar[X_CTX], XB_CTX);
    mbar_expect_tx(&s.xbar[X_Y], XB_Y);
    mbar_expect_tx(&s.xbar[X_HF], XB_HF);
    mbar_expect_tx(&s.xbar[X_PART], XB_PART);
    mbar_expect_tx(&s.xbar[X_TOP], XB_TOP);
  }
  if (BEAM && tid < R) {                              // hypothesis state of this cluster's rows (kept in HBM between launches)
    const bool ok = tid < nrows;
    s.bscore[tid] = ok ? p.bm_score[row0 + tid] : -INFINITY;
    s.bfin[tid] = ok ? p.bm_fin[row0 + tid] : 1;
    s.bsrc[tid] = ok ? p.bm_src[row0 + tid] : nrows - 1;
  }
  embed_row(t_begin, BEAM ? (long long)p.bm_tok[my_row] : p.tokens[(size_t)my_row * p.ld_tok + t_begin]);
  __syncthreads();
  bool cluster_done = false;                          // beam search: every hypothesis of this cluster has emitted eos
  if (BEAM && tid == 0) {
    cluster_done = true;
    for (int r = 0; r < nrows; ++r) cluster_done = cluster_done && s.bfin[r] != 0;
  }
  // Device-side early exit (src/inference.py:23-25 breaks as soon as every row has emitted eos; the host only polls
  // between launches, one launch behind).  "Every row has finished" is a global flag that flips at an arbitrary
  // moment, and the 8 CTAs of a cluster must leave the step loop at the SAME step (a CTA that stayed would wait
  // for exchanges forever): CTA rank 0 alone reads the flag - here, and once per step when it composes its arg-max
  // partials - and the others take ITS reading (through the cluster barrier here, through the partials exchange below).
  // What is read is the VALUE steps_executed = the reference's final ys.shape[1] - 1: a cluster that lags behind the
  // one that finished last keeps going until it has run that many steps, so every row's columns up to `steps` hold
  // what the reference's ys holds there (rows that finished early keep decoding in the reference too).
  if (c == 0 && tid == 0) s.stop_flag = *reinterpret_cast<volatile int*>(&p.state->steps_executed);
  cluster_sync_all();      // every CTA of the cluster is resident and its barriers are armed before any DSMEM store
  bool stop;
  {
    uint32_t f;
    asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(f) : "r"(cl0 + (smem_u32(&s.stop_flag) - s_local)) : "memory");
    stop = (int)f > 0 && t_begin >= (int)f;
  }
  const bool fetching = !stop;        // the weight stream was started
  if (lane == 0 && fetching) slot_fetch();
  int t_done = t_begin;               // steps this cluster has completed

  const size_t kv_rh = (size_t)p.cache_blocks * 1024;              // halves per (layer, row, head) region
  const size_t kv_layer = (size_t)p.rows * NH * kv_rh, kv_row = ((size_t)my_row * NH + c) * kv_rh;
  const int my_img = my_row / p.beam;
  const size_t m_layer = (size_t)p.images * NH * 1024, m_row = ((size_t)my_img * NH + c) * 1024;
  int g = 0;     // stream index of the next chunk (chunk g + j belongs to warp (g + j) % 8)
  const bool tracing = DEV && p.trace != nullptr && blockIdx.x == 0 && tid == 0;
  int ti = 0;
#define TR() do { if (tracing && t == p.trace_step && ti < 1024) p.trace[ti++] = clock64(); } while (0)
  for (int t = t_begin; t < t_end && !stop; ++t) {
    // where this step's key / value go inside the (layer, row, head) region of the fragment-major caches
    const int k_app = (t >> 5) * 512 + kfrag_word(t & 31, lane & 15);       // 32-bit word index (lanes 0..15)
    const int v_app = (t >> 5) * 1024 + vfrag_half(t & 31, lane);           // half index (lane = dim)
    // beam search: history is read from the parent's row of set (t & 1) and re-written, with this step's
    // key/value, to this hypothesis' own row of the other set; greedy: one set, one row
    const size_t set_rd = BEAM ? (size_t)(t & 1) * p.cache_set_stride : 0;
    const size_t set_wr = BEAM ? (size_t)((t & 1) ^ 1) * p.cache_set_stride : 0;
    const size_t kv_src = BEAM ? ((size_t)(row0 + s.bsrc[min(warp, nrows - 1)]) * NH + c) * kv_rh : kv_row;
    for (int l = 0; l < L; ++l) {
      const __half* Kc = p.kcache + set_rd + (size_t)l * kv_layer + kv_src;     // history of (row `warp`, head c)
      const __half* Vc = p.vcache + set_rd + (size_t)l * kv_layer + kv_src;
      __half* Kd = p.kcache + set_wr + (size_t)l * kv_layer + kv_row;           // where this step's key / value go
      __half* Vd = p.vcache + set_wr + (size_t)l * kv_layer + kv_row;
      TR();
      // ---- self-attention: q, k, v of head c = 6 tiles ---------------------------------------------
      if (lane < 2) prefetch_l2<true>((lane ? p.memv : p.memk) + (size_t)l * m_layer + m_row, region_bytes(p.mem_len));   // this layer's memory K/V -> L2
      {
        const int j = (warp - g) & 7;
        if (j < 6) {
          float acc[4];
          const int part = j >> 1, f = (j & 1) * 16 + g4;               // 0 = q, 1 = k, 2 = v; feature f, f+8 of the head
          slot_wait();
          TR();
          gemm16<PD>(s.slot[warp], &s.xa[0][0], lane, acc);
          const float b0 = chunk_bias(s.slot[warp], g4), b1 = chunk_bias(s.slot[warp], g4 + 8);
          slot_release();
          const int r0 = 2 * t4;
          if (part == 0) {
            s.qh[r0][f] = to_half_sat((acc[0] + b0) * ATT_SCALE); s.qh[r0 + 1][f] = to_half_sat((acc[1] + b0) * ATT_SCALE);
            s.qh[r0][f + 8] = to_half_sat((acc[2] + b1) * ATT_SCALE); s.qh[r0 + 1][f + 8] = to_half_sat((acc[3] + b1) * ATT_SCALE);
          } else {
            __half(*dst)[HD] = (part == 1) ? s.knew : s.vnew;
            dst[r0][f] = to_half_sat(acc[0] + b0); dst[r0 + 1][f] = to_half_sat(acc[1] + b0);
            dst[r0][f + 8] = to_half_sat(acc[2] + b1); dst[r0 + 1][f + 8] = to_half_sat(acc[3] + b1);
          }
        }
        g += 6;
      }
      KvPair kv;
      attend_issue2<false>(Kc, Vc, t, lane, kv);           // the first K and V block fly across the barrier
      TR();
      __syncthreads();
      TR();
      {
        float o[4];
        attend_online<NB, true, BEAM, false>(&s.qh[warp][0], Kc, Vc, t, &s.knew[warp][0], &s.vnew[warp][0],
                                             lane, kv, o, row_ok ? Kd : nullptr, row_ok ? Vd : nullptr);   // padding warps
        // recompute the last valid row: they must not copy its blocks (a late copy would overwrite the append below)
        TR();
        send_ctx(o);
        if (BEAM) __syncwarp();                                // the block copies above are ordered before the append
        if (row_ok) {                                          // append this step's key / value (fragment-major)
          if (lane < 16) reinterpret_cast<uint32_t*>(Kd)[k_app] = reinterpret_cast<const uint32_t*>(&s.knew[warp][0])[lane];
          Vd[v_app] = s.vnew[warp][lane];
        }
        // self-attention cache of the NEXT layer (next step's layer 0 after the last one) -> L2.  Greedy only: in
        // beam search the parent row is not known a step ahead (the beam kernel is 2 % faster without it).
        const bool last = l + 1 == L;
        const int keys = last ? t + 1 : t;
        if (!BEAM && keys > 0 && lane < 2) {
          const size_t nxt = last ? set_wr + kv_row : set_rd + (size_t)(l + 1) * kv_layer + kv_src;
          prefetch_l2<false>((lane ? p.vcache : p.kcache) + nxt, region_bytes(keys));
        }
      }
      TR();
      // the memory K / V of cross-attention depend on nothing in this step: requested here, they travel under the
      // out-projection, LayerNorm 1 and the cross-query projection
      attend_issue2<true>(p.memk + (size_t)l * m_layer + m_row, p.memv + (size_t)l * m_layer + m_row, p.mem_len, lane, kv);
      // ---- x = LN1(x + out_proj(ctx)) ---------------------------------------------------------------
      xwait(X_CTX, 0u, XB_CTX);
      TR();
      {
        const int j = (warp - g) & 7;
        if (j < 2) {
          float acc[4];
          slot_wait();
          gemm16<PD>(s.slot[warp], &s.ctx[0][0], lane, acc);
          const float b0 = chunk_bias(s.slot[warp], g4), b1 = chunk_bias(s.slot[warp], g4 + 8);
          stage_tile(j, acc, b0, b1);
          named_bar_sync(1, 64);
          send_y(j * 32 + lane, false);
          slot_release();                          // peers wait for y: send first, re-arm the weight slot after
        }
        g += 2;
      }
      TR();
      LnRegs ln = load_ln(l, 0);          // fetched while y is in flight: not live across the GEMM above
      xwait(X_Y, nlayer, XB_Y);
      TR();
      layer_norm(ln);
      __syncthreads();
      TR();
      // ---- cross-attention over the 30 memory tokens ----------------------------------------------
      {
        const int j = (warp - g) & 7;
        if (j < 2) {
          float acc[4];
          const int f = j * 16 + g4, r0 = 2 * t4;
          slot_wait();
          gemm16<PD>(s.slot[warp], &s.xa[0][0], lane, acc);
          const float b0 = chunk_bias(s.slot[warp], g4), b1 = chunk_bias(s.slot[warp], g4 + 8);
          slot_release();
          s.qh[r0][f] = to_half_sat((acc[0] + b0) * ATT_SCALE); s.qh[r0 + 1][f] = to_half_sat((acc[1] + b0) * ATT_SCALE);
          s.qh[r0][f + 8] = to_half_sat((acc[2] + b1) * ATT_SCALE); s.qh[r0 + 1][f + 8] = to_half_sat((acc[3] + b1) * ATT_SCALE);
        }
        g += 2;
      }
      const __half* Mk = p.memk + (size_t)l * m_layer + m_row;       // (not live across the self-attention block)
      const __half* Mv = p.memv + (size_t)l * m_layer + m_row;
      __syncthreads();
      TR();
      {
        float o[4];
        attend_online<1, false, false, true>(&s.qh[warp][0], Mk, Mv, p.mem_len, nullptr, nullptr, lane, kv, o);
        send_ctx(o);
      }
      TR();
      xwait(X_CTX, 1u, XB_CTX);
      TR();
      {
        const int j = (warp - g) & 7;
        if (j < 2) {
          float acc[4];
          slot_wait();
          gemm16<PD>(s.slot[warp], &s.ctx[0][0], lane, acc);
          const float b0 = chunk_bias(s.slot[warp], g4), b1 = chunk_bias(s.slot[warp], g4 + 8);
          stage_tile(j, acc, b0, b1);
          named_bar_sync(1, 64);
          send_y(j * 32 + lane, false);
          slot_release();                          // peers wait for y: send first, re-arm the weight slot after
        }
        g += 2;
      }
      TR();
      ln = load_ln(l, 1);
      xwait(X_Y, nlayer + 1u, XB_Y);
      TR();
      layer_norm(ln);
      __syncthreads();
      TR();
      // ---- feed-forward: 64 features of linear1 (+ReLU) per CTA, then 32 features of linear2 ---------
      {
        const int j = (warp - g) & 7;
        if (j < 4) {
          float acc[4];
          const int f = j * 16 + g4, r0 = 2 * t4;
          slot_wait();
          gemm16<PD>(s.slot[warp], &s.xa[0][0], lane, acc);
          const float b0 = chunk_bias(s.slot[warp], g4), b1 = chunk_bias(s.slot[warp], g4 + 8);
          __half(*hs)[72] = reinterpret_cast<__half(*)[72]>(&s.stg[0][0][0]);
          hs[r0][f] = to_half_sat(fmaxf(acc[0] + b0, 0.f)); hs[r0 + 1][f] = to_half_sat(fmaxf(acc[1] + b0, 0.f));
          hs[r0][f + 8] = to_half_sat(fmaxf(acc[2] + b1, 0.f)); hs[r0 + 1][f + 8] = to_half_sat(fmaxf(acc[3] + b1, 0.f));
          named_bar_sync(2, 128);
          if (j < 2) {
            const int u = j * 32 + lane, r = u >> 3, piece = u & 7;
            send_all(&s.hf[r][c * 64 + piece * 8], *reinterpret_cast<const uint4*>(&hs[r][piece * 8]), X_HF);
          }
          slot_release();
        }
        g += 4;
      }
      TR();
      xwait(X_HF, nlayer, XB_HF);
      TR();
      {
        const int j = (warp - g) & 7;
        if (j < 4) {                                            // tile j / 2, input half j % 2
          float acc[4];
          slot_wait();
          gemm16<PF>(s.slot[warp], &s.hf[0][(j & 1) * 256], lane, acc);
          const float b0 = chunk_bias(s.slot[warp], g4), b1 = chunk_bias(s.slot[warp], g4 + 8);   // zero in the kh = 1 chunk
          stage_tile(j, acc, b0, b1);
          named_bar_sync(3, 128);
          if (j < 2) send_y(j * 32 + lane, true);
          slot_release();
        }
        g += 4;
      }
      TR();
      ln = load_ln(l, 2);
      xwait(X_Y, nlayer, XB_Y);   // third of the layer: (layer + 2) & 1
      ++nlayer;
      TR();
      layer_norm(ln);
      __syncthreads();
      TR();
    }
    // ---- fc_out slice + running (max, argmax, sum-exp): FT tiles of 16 vocabulary rows --------------
    TR();
    Partial pa, pb;        // rows 2*t4 and 2*t4+1 over this thread's features
    pa.m = pb.m = -INFINITY; pa.idx = pb.idx = 0x7fffffff; pa.s = pb.s = 0.f; pa.pad = pb.pad = 0;
    TopK<KB> ta, tb;       // beam search: the K best logits of rows 2*t4 / 2*t4+1 seen by this thread
    ta.init(); tb.init();
    {
      const int j0 = (warp - g) & 7;
      uint32_t bf[8][4];
      load_bfrags<PD>(&s.xa[0][0], lane, bf);
#pragma unroll 1
      for (int m = j0; m < FT; m += NW) {
        float acc[4];
        slot_wait();
        gemm16_pre(s.slot[warp], bf, lane, acc);
        const float b0 = chunk_bias(s.slot[warp], g4), b1 = chunk_bias(s.slot[warp], g4 + 8);
        slot_release();
        const int lf = m * 16 + g4, v0 = c * cols_per_cta + lf;
        if (v0 < p.vocab) {
          update_partial(pa, acc[0] + b0, v0); update_partial(pb, acc[1] + b0, v0);
          ta.insert(acc[0] + b0, v0); tb.insert(acc[1] + b0, v0);
        }
        if (v0 + 8 < p.vocab) {
          update_partial(pa, acc[2] + b1, v0 + 8); update_partial(pb, acc[3] + b1, v0 + 8);
          ta.insert(acc[2] + b1, v0 + 8); tb.insert(acc[3] + b1, v0 + 8);
        }
      }
      g += FT;
    }
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) {       // over the 8 feature lanes that share t4
      Partial oa = shfl_partial(pa, o), ob = shfl_partial(pb, o);
      merge_partial(pa, oa);
      merge_partial(pb, ob);
    }
    if (g4 == 0) { s.wpart[warp][2 * t4] = pa; s.wpart[warp][2 * t4 + 1] = pb; }
    if constexpr (BEAM) {
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) { ta.merge_xor(o); tb.merge_xor(o); }
      if (g4 == 0) { ta.store(s.wtop[warp][2 * t4]); tb.store(s.wtop[warp][2 * t4 + 1]); }
    }
    __syncthreads();
    TR();
    if (warp == 0) {                         // lane = (row, quarter): merge the 8 warps, then send to CTAs 2q, 2q+1
      const int r = lane >> 2, q = lane & 3;
      Partial a = s.wpart[2 * q][r];
      merge_partial(a, s.wpart[2 * q + 1][r]);
      Partial b1 = shfl_partial(a, 1);
      merge_partial(a, b1);
      Partial b2 = shfl_partial(a, 2);
      merge_partial(a, b2);
      // 4th word: rank 0's reading of steps_executed (one load instruction for the whole warp: one value)
      const uint32_t all_done = (c == 0) ? (uint32_t)*reinterpret_cast<volatile int*>(&p.state->steps_executed) : 0u;
      const uint4 v = make_uint4(__float_as_uint(a.m), (uint32_t)a.idx, __float_as_uint(a.s), all_done);
      const uint32_t off = smem_u32(&s.part[c][r]) - s_local, boff = smem_u32(&s.xbar[X_PART]) - s_local;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const uint32_t base = cl0 + (2 * q + k) * cl_stride;
        st_async_v4(base + off, v, base + boff);
      }
    }
    if constexpr (BEAM) {                    // row `warp`: the CTA's K best logits -> every CTA (lane k serves CTA k)
      TopK<KB> tl;
      if (lane < NW) tl.load(s.wtop[lane][warp]); else tl.init();
#pragma unroll
      for (int o = 1; o < NW; o <<= 1) tl.merge_xor(o);
      if (lane < CL) {
        static_assert(KB == 5, "TopList packing below assumes 5 entries");
        const uint4 v0 = make_uint4(__float_as_uint(tl.v[0]), __float_as_uint(tl.v[1]), __float_as_uint(tl.v[2]), __float_as_uint(tl.v[3]));
        const uint4 v1 = make_uint4(__float_as_uint(tl.v[4]), (uint32_t)tl.i[0], (uint32_t)tl.i[1], (uint32_t)tl.i[2]);
        const uint4 v2 = make_uint4((uint32_t)tl.i[3], (uint32_t)tl.i[4], 0u, 0u);
        const uint32_t base = cl0 + lane * cl_stride;
        const uint32_t off = base + (smem_u32(&s.ctop[c][warp]) - s_local), bar = base + (smem_u32(&s.xbar[X_TOP]) - s_local);
        st_async_v4(off, v0, bar);
        st_async_v4(off + 16, v1, bar);
        st_async_v4(off + 32, v2, bar);
      }
    }
    xwait(X_PART, nstep, XB_PART);
    const bool stop_after = s.part[0][0].pad > 0 && t + 1 >= s.part[0][0].pad;      // rank 0's reading: the same value in all 8 CTAs
    TR();
    Partial a;                               // row `warp`: (max, argmax, sum-exp) over the whole vocabulary
    if (lane < CL) a = s.part[lane][warp];
    else { a.m = -INFINITY; a.idx = 0x7fffffff; a.s = 0.f; a.pad = 0; }
#pragma unroll
    for (int o = 1; o < CL; o <<= 1) {
      Partial b = shfl_partial(a, o);
      merge_partial(a, b);
    }
    int tok;
    if constexpr (!BEAM) {
      tok = __shfl_sync(0xffffffffu, a.idx, 0);
      if (c == 0 && lane == 0 && row_ok) {
        const int gr = row0 + warp;
        p.tokens[(size_t)gr * p.ld_tok + t + 1] = tok;
        if (p.logprob != nullptr) p.logprob[(size_t)gr * p.max_len + t] = -logf(a.s);   // log_softmax of the argmax
        if (tok == p.eos && !p.finished[gr]) {
          p.finished[gr] = 1;
          // src/inference.py:23-25 stops after the step at which the LAST row emits its first eos = the maximum of
          // (first-eos step + 1) over the rows.  Clusters are not in lockstep (and run in waves), so the thread that
          // completes the count publishes that maximum, not its own t.
          atomicMax(&p.state->last_eos, t + 1);
          __threadfence();
          const int cnt = atomicAdd(&p.state->finished_count, 1) + 1;
          if (cnt == p.rows) p.state->steps_executed = atomicMax(&p.state->last_eos, 0);
        }
      }
    } else {
      // ---- beam step (oracle/decode.py::beam_search): candidates -> K best per image -> new hypotheses -----
      xwait(X_TOP, nstep, XB_TOP);
      TopK<KB> tl;
      if (lane < CL) tl.load(s.ctop[lane][warp]); else tl.init();
#pragma unroll
      for (int o = 1; o < CL; o <<= 1) tl.merge_xor(o);
      if (lane == 0) {                       // candidates of hypothesis `warp`: score + log_softmax(logit)
        const float lse = a.m + logf(a.s), sc = s.bscore[warp];
        const bool fin = s.bfin[warp] != 0;
        const int hyp = warp % p.beam;
#pragma unroll
        for (int k = 0; k < KB; ++k) {
          Cand cd;
          cd.score = -INFINITY; cd.flat = 0x7fffffff; cd.lp = 0.f;
          if (row_ok && k < p.beam) {
            if (fin) { if (k == 0) { cd.score = sc; cd.flat = hyp * p.vocab + p.pad; } }     // frozen: one candidate
            else { cd.lp = tl.v[k] - lse; cd.score = sc + cd.lp; cd.flat = hyp * p.vocab + tl.i[k]; }
          }
          s.cand[warp][k] = cd;
        }
      }
      __syncthreads();
      if (warp * p.beam < nrows) {           // warp i = image i of this cluster: K rounds of arg-best over K x KB candidates
        const int hyp = lane / KB, k = lane - hyp * KB;
        Cand cd;
        cd.score = -INFINITY; cd.flat = 0x7fffffff; cd.lp = 0.f;
        if (hyp < p.beam) cd = s.cand[warp * p.beam + hyp][k];
        for (int j = 0; j < p.beam; ++j) {
          float bv = cd.score, bl = cd.lp;
          int bf = cd.flat;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int of = __shfl_xor_sync(0xffffffffu, bf, o);
            const float ol = __shfl_xor_sync(0xffffffffu, bl, o);
            if (cand_before(ov, of, bv, bf)) { bv = ov; bf = of; bl = ol; }
          }
          if (lane == 0) {
            Sel se;
            se.score = bv;
            se.parent = (bf == 0x7fffffff) ? warp * p.beam : warp * p.beam + bf / p.vocab;
            se.tok = (bf == 0x7fffffff) ? p.pad : bf % p.vocab;
            se.lp = (bf == 0x7fffffff) ? 0.f : bl;
            s.sel[warp * p.beam + j] = se;
          }
          if (cd.flat == bf) { cd.score = -INFINITY; cd.flat = 0x7fffffff; }      // taken
        }
      }
      __syncthreads();
      const Sel me = s.sel[min(warp, nrows - 1)];
      const int parent_fin = s.bfin[me.parent];
      tok = me.tok;
      __syncthreads();                       // every warp has read the old state
      if (lane == 0 && row_ok) {
        s.bscore[warp] = me.score;
        s.bfin[warp] = parent_fin | (tok == p.eos);
        s.bsrc[warp] = me.parent;
        if (c == 0) {
          p.bp_parent[(size_t)t * p.rows + row0 + warp] = me.parent % p.beam;     // clusters hold whole images
          p.bp_token[(size_t)t * p.rows + row0 + warp] = tok;
          if (p.bp_logp != nullptr) p.bp_logp[(size_t)t * p.rows + row0 + warp] = me.lp;
          p.bm_tok[row0 + warp] = tok;
        }
      }
    }
    // ---- next input: embedding[token] + pos[t+1] ---------------------------------------------------
    ++nstep;
    if (t + 1 < p.max_pos) embed_row(t + 1, tok);
    __syncthreads();
    if (BEAM && tid == 0 && c == 0 && !cluster_done) {
      bool all = true;
      for (int r = 0; r < nrows; ++r) all = all && s.bfin[r] != 0;
      if (all) {
        cluster_done = true;
        atomicMax(&p.state->last_eos, t + 1);          // see the greedy branch: the last cluster in TIME publishes the max
        __threadfence();
        const int cnt = atomicAdd(&p.state->finished_count, 1) + 1;
        if (cnt == p.num_clusters) p.state->steps_executed = atomicMax(&p.state->last_eos, 0);
      }
    }
    TR();
    t_done = t + 1;
    stop = stop_after;
  }
  if (fetching && wgi < total_chunks) {
    // left early: this warp's slot still has a weight chunk on its way (every release re-arms the slot while the
    // stream lasts) - the CTA must not exit under a TMA copy
    slot_wait();
  }
  if (BEAM && c == 0 && tid < nrows) {       // hypothesis state back to HBM for the next launch / the back-track
    p.bm_score[row0 + tid] = s.bscore[tid];
    p.bm_fin[row0 + tid] = s.bfin[tid];
    p.bm_src[row0 + tid] = s.bsrc[tid];
  }
  if (c == 0 && tid == 0 && t_done > t_begin) atomicMax(&p.state->step, t_done);   // steps actually run (finalize: the count when no row ever finished)
  cluster_sync_all();      // no CTA exits while a peer may still address its shared memory
}

// memkv f32 [img*mem_len+s][l*512 + kv*256 + h*32 + d]  ->  one fragment-major block (32 key slots, the slots past
// mem_len zero) of memk and of memv per (l, img, h).  One warp per (l, img, h, kv): lane = key slot; the block is
// assembled in shared memory (fragment order) and written out as 2 KB of coalesced 16-byte stores.
__global__ void __launch_bounds__(256) repack_memkv_kernel(const float* __restrict__ memkv, int images, int L, int MEM_S,
                                                           __half* __restrict__ memk, __half* __restrict__ memv) {
  __shared__ __align__(16) __half tile[8][1024];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const size_t total = (size_t)L * images * NH * 2;
  for (size_t item = blockIdx.x * 8 + wib; item < total; item += (size_t)gridDim.x * 8) {
    const int kv = item & 1, h = (item >> 1) & 7;
    const size_t rest = item >> 4;
    const size_t img = rest % images;
    const int l = (int)(rest / images);
    const int key = lane;
    const bool ok = key < MEM_S;
    const float* src = memkv + (img * MEM_S + min(key, MEM_S - 1)) * (size_t)L * 512 + l * 512 + kv * 256 + h * 32;
    float v[HD];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 x = ok ? __ldg(reinterpret_cast<const float4*>(src) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
      v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
    }
    __half* t = tile[wib];
    if (kv == 0) {
      uint32_t* tw = reinterpret_cast<uint32_t*>(t);
#pragma unroll
      for (int w = 0; w < 16; ++w) tw[kfrag_word(key, w)] = pack16(v[2 * w], v[2 * w + 1]);
    } else {
#pragma unroll
      for (int d = 0; d < HD; ++d) t[vfrag_half(key, d)] = to_h16(v[d]);
    }
    __syncwarp();
    uint4* dst = reinterpret_cast<uint4*>((kv ? memv : memk) + ((((size_t)l * images + img) * NH + h) << 10));
    const uint4* s4 = reinterpret_cast<const uint4*>(t);
#pragma unroll
    for (int q = 0; q < 4; ++q) dst[q * 32 + lane] = s4[q * 32 + lane];
    __syncwarp();
  }
}

__global__ void beam_init_kernel(DecodeState* state, float* bm_score, int* bm_fin, int* bm_src, int* bm_tok, int rows,
                                 int beam, int rows_per_cluster, int sos) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) { state->step = 0; state->finished_count = 0; state->steps_executed = 0; state->last_eos = 0; }
  if (i < rows) {
    bm_score[i] = (i % beam == 0) ? 0.f : -INFINITY;     // all hypotheses start as [sos]: only the first one counts
    bm_fin[i] = 0;
    bm_src[i] = i % rows_per_cluster;
    bm_tok[i] = sos;
  }
}

// One thread per hypothesis: its rank among the image's K hypotheses (score descending, ties -> lower beam index, so
// rank 0 is the first maximum); ranks below n_best are back-tracked into slot [img][rank].
__global__ void beam_finalize_kernel(const DecodeState* state, const float* bm_score, const int* bp_parent,
                                     const int* bp_token, const float* bp_logp, int images, int beam, int n_best,
                                     int rows, int max_len, int sos, int pad, int64_t* tokens, float* logprob,
                                     float* score_out, int32_t* steps_out) {
  const int steps = state->steps_executed > 0 ? state->steps_executed : min(state->step, max_len);
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r == 0 && steps_out != nullptr) *steps_out = steps;
  if (r >= images * beam) return;
  const int img = r / beam, j = r - img * beam;
  const float* sc = bm_score + (size_t)img * beam;
  auto key = [](float v) { return isnan(v) ? -INFINITY : v; };     // a strict total order: ranks are a permutation
  const float mine = key(sc[j]);
  int rank = 0;
  for (int i = 0; i < beam; ++i) rank += key(sc[i]) > mine || (key(sc[i]) == mine && i < j);
  if (rank >= n_best) return;
  const size_t slot = (size_t)img * n_best + rank;
  if (score_out != nullptr) score_out[slot] = sc[j];
  int64_t* out = tokens + slot * (max_len + 1);
  float* lp = logprob != nullptr ? logprob + slot * max_len : nullptr;
  out[0] = sos;
  for (int k = steps + 1; k <= max_len; ++k) out[k] = pad;
  if (lp != nullptr)
    for (int k = steps; k < max_len; ++k) lp[k] = 0.f;
  int b = j;
  for (int t = steps - 1; t >= 0; --t) {     // a frozen hypothesis recorded (itself, pad, 0) after its eos
    const size_t at = (size_t)t * rows + img * beam + b;
    out[t + 1] = bp_token[at];
    if (lp != nullptr) lp[t] = bp_logp[at];
    b = bp_parent[at];
  }
}

int g_max_clusters[HM_MAX_DEVICES] = {};      // co-resident 8-CTA clusters, per device

}  // namespace

// Per DEVICE (function attributes and the occupancy answer belong to a device, not to the process).
int decode_persistent_init() {
  HM_DEVICE_ONCE({
    HM_CUDA(cudaFuncSetAttribute(decode_persistent_kernel<5, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
    HM_CUDA(cudaFuncSetAttribute(decode_persistent_kernel<8, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
    HM_CUDA(cudaFuncSetAttribute(decode_persistent_kernel<5, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
    HM_CUDA(cudaFuncSetAttribute(decode_persistent_kernel<5, DP_MAX_BEAM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
    HM_CUDA(cudaFuncSetAttribute(decode_persistent_kernel<8, DP_MAX_BEAM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(CL * 64);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = sizeof(Smem);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int n = 0;
    HM_CUDA(cudaOccupancyMaxActiveClusters(&n, decode_persistent_kernel<5, 0, false>, &cfg));
    HM_CHECK(n >= 1, "device cannot host an 8-CTA decode cluster");
    g_max_clusters[_dev] = n;
  });
  return 0;
}

int decode_persistent_max_clusters(int* out) {
  HM_TRY(decode_persistent_init());
  int dev = 0;
  HM_CUDA(cudaGetDevice(&dev));
  *out = g_max_clusters[dev];
  return 0;
}

int decode_persistent_launch(cudaStream_t st, DecPersistParams p, int t_begin, int t_end) {
  HM_TRY(decode_persistent_init());
  HM_CHECK(p.tmax <= 256, "decode: max_seq_len %d > 256", p.tmax);
  HM_CHECK(t_begin >= 0 && t_end > t_begin && t_end <= p.tmax, "decode: bad step range [%d,%d)", t_begin, t_end);
  HM_CHECK(p.fc_tiles % NW == 0 && p.fc_tiles > 0, "decode: bad fc_tiles %d", p.fc_tiles);
  HM_CHECK(p.chunks_per_step == DP_LAYER_CHUNKS * p.num_layers + p.fc_tiles, "decode: bad chunks_per_step");
  HM_CHECK(p.cache_blocks * 32 >= p.tmax, "decode: %d cache blocks cannot hold %d positions", p.cache_blocks, p.tmax);
  HM_CHECK(p.mem_len >= 1 && p.mem_len <= 32, "decode: %d memory tokens per image (1..32 supported)", p.mem_len);
  HM_CHECK(p.beam >= 1 && p.beam <= DP_MAX_BEAM, "decode: beam %d outside [1, %d]", p.beam, DP_MAX_BEAM);
  const bool beam = p.beam > 1 || p.bm_score != nullptr;     // beam machinery (n-best runs it at beam = 1 too)
  // Rows per cluster: 8 (greedy) or whole images (beam).  Clusters are independent, so a batch larger than
  // rows_per_cluster x (co-resident clusters) simply runs in several waves.
  if (beam) {
    HM_CHECK(p.rows_per_cluster == p.beam * (R / p.beam) && p.rows % p.beam == 0, "decode: bad beam geometry");
    HM_CHECK(p.bm_score && p.bm_fin && p.bm_src && p.bm_tok && p.bp_parent && p.bp_token, "decode: beam buffers missing");
  } else {
    p.rows_per_cluster = R;
  }
  p.num_clusters = ceil_div(p.rows, p.rows_per_cluster);
  dim3 grid(p.num_clusters * CL);
  if (p.trace != nullptr) {                                  // instrumented build: greedy, <= 160 positions only
    HM_CHECK(!beam && p.tmax <= 160, "decode: tracing needs greedy decoding and max_seq_len <= 160");
    decode_persistent_kernel<5, 0, true><<<grid, THREADS, sizeof(Smem), st>>>(p, t_begin, t_end);
  } else if (p.tmax <= 160) {
    if (beam) decode_persistent_kernel<5, DP_MAX_BEAM, false><<<grid, THREADS, sizeof(Smem), st>>>(p, t_begin, t_end);
    else decode_persistent_kernel<5, 0, false><<<grid, THREADS, sizeof(Smem), st>>>(p, t_begin, t_end);
  } else {
    if (beam) decode_persistent_kernel<8, DP_MAX_BEAM, false><<<grid, THREADS, sizeof(Smem), st>>>(p, t_begin, t_end);
    else decode_persistent_kernel<8, 0, false><<<grid, THREADS, sizeof(Smem), st>>>(p, t_begin, t_end);
  }
  HM_LAUNCHED();
  return 0;
}

int beam_init(cudaStream_t st, DecodeState* state, float* bm_score, int* bm_fin, int* bm_src, int* bm_tok, int rows,
              int beam, int rows_per_cluster, int sos) {
  beam_init_kernel<<<ceil_div(rows, 256), 256, 0, st>>>(state, bm_score, bm_fin, bm_src, bm_tok, rows, beam,
                                                        rows_per_cluster, sos);
  HM_LAUNCHED();
  return 0;
}

int beam_finalize(cudaStream_t st, const DecodeState* state, const float* bm_score, const int* bp_parent,
                  const int* bp_token, const float* bp_logp, int images, int beam, int n_best, int rows, int max_len,
                  int sos, int pad, int64_t* tokens, float* logprob, float* score_out, int32_t* steps_out) {
  HM_CHECK(n_best >= 1 && n_best <= beam, "n_best=%d outside [1, beam=%d]", n_best, beam);
  HM_CHECK(logprob == nullptr || bp_logp != nullptr, "beam_finalize: per-token log-probs were not recorded");
  beam_finalize_kernel<<<ceil_div(images * beam, 128), 128, 0, st>>>(state, bm_score, bp_parent, bp_token, bp_logp, images,
                                                                     beam, n_best, rows, max_len, sos, pad, tokens,
                                                                     logprob, score_out, steps_out);
  HM_LAUNCHED();
  return 0;
}

int repack_memkv(cudaStream_t st, const float* memkv, int images, int L, int mem_len, void* memk, void* memv) {
  HM_CHECK(mem_len >= 1 && mem_len <= 32, "decode: %d memory tokens per image (1..32 supported)", mem_len);
  const size_t total = (size_t)L * images * NH * 2;          // one warp per (l, image, head, K|V)
  size_t blocks = (total + 7) / 8;
  if (blocks > 148 * 16) blocks = 148 * 16;
  repack_memkv_kernel<<<(int)blocks, 256, 0, st>>>(memkv, images, L, mem_len, static_cast<__half*>(memk), static_cast<__half*>(memv));
  HM_LAUNCHED();
  return 0;
}

}  // namespace hmocr
