// Fused pre-LN encoder stack for dim 256 or 128 / 8 heads x 32 (SFormer, fusion head; AU_formers, VA_former): ONE persistent kernel runs
//   x + to_out(softmax(q k^T / sqrt(dh)) v)   and   x + W2 gelu(W1 LN(x) + b1) + b2        (models/heads.py:164-256)
// for `depth` layers on 128-row tiles (floor(128 / n_tok) whole sequences per tile) without touching HBM in between.
//
//   * the fp32 residual stream of the tile lives in TMEM columns [0,D): the out-projection and the second MLP GEMM
//     ACCUMULATE onto it (tcgen05.mma with accumulate=1 on a tile pre-loaded with x + bias), so both residual adds
//     and both bias adds cost nothing;
//   * LayerNorm runs on the row workers (one TMEM lane = one token row, two threads per row) and writes the bf16
//     A operand straight into the 128B-swizzled K-major layout tcgen05.mma reads;
//   * attention is per head on the tensor cores: [Q|K|V]_h = LN(x) Wqkv_h^T (N=96), S = Q K^T over the whole tile
//     (block-diagonal: a row only uses the columns of its own sequence), softmax in registers, P written back as
//     bf16 INTO the S columns of TMEM and used as the A operand of O = P V (V is an MN-major B operand);
//   * the out-projection runs PER HEAD (x += O_h Wout[:, 32h:32h+32]^T, N = 256, K = 32) as soon as O_h is normalised: O_h / l is
//     written back over its own accumulator columns as packed bf16 and is the TMEM A operand of that GEMM (no attention-output
//     buffer, no proxy fence); [Wq_h; Wk_h; Wv_h] arrive through their own ring of 6 x 12 KB (one and a half heads in flight, one
//     "head full" barrier per head), so QKV(h+1) never waits for L2;
//   * the other weights are streamed from L2 by TMA through 16 KB slots (two during attention, nine in the MLP phase, when the
//     Q/K/V staging and the QKV ring are idle; one barrier per group of four), activations enter / leave as whole NCHW frames
//     by bulk copies (SFormer, models/vformer.py:245-259) or as fp32 rows (+ an optional positional table; the fusion head's
//     12 AU logits and decisions can be taken from the last layer's output sweep instead of storing the token rows);
//   * the model width D (256 or 128) is a template parameter.  The shared-memory map, the TMEM map and the per-layer vector
//     block are laid out for D = 256; at D = 128 the A0 operand, the residual columns and the vectors use their first halves,
//     and every GEMM whose K or N is the model width has half the panels (QKV / FF1 K, out-projection / FF2 N);
//   * tiles are handed out by an atomic counter (NCHW form): the weight producer fetches the next index one tile ahead and
//     publishes it to the other roles through a four-entry queue in shared memory (see next_tile).
//
// Warp roles: 0 = TMA producer (out-proj / MLP weights; also the next tile's input frames), 1 = TMEM allocator + MMA issuer
// (one thread), 2 = TMA producer of the QKV ring, 3.. = row workers (warp w owns TMEM lanes 32*(w%4)..+31; the NSPLIT warps
// of a lane quarter split the columns).
#include <cuda.h>

#include "avf_common.cuh"
#include "avf_fused_helpers.cuh"
#include "avf_internal.h"

namespace avf {

int make_tmap_bf16_2d(CUtensorMap* tm, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols = 64);

namespace {
using namespace fused;

// DIM: the widest model (256) — the layouts below are sized for it — and the only width of the NCHW form.  Kernels take the
// model width as the template parameter D (256 or 128).
constexpr int DIM = 256, HEADS = 8, DH = 32;
constexpr int MAX_DEPTH = 3, MAX_MLP = 1024;
constexpr int NSPLIT = 2;                  // threads per token row (each owns D / NSPLIT columns of the residual stream)
constexpr int WORKER_T0 = 96;              // first worker thread
constexpr int NUM_WORKERS = 128 * NSPLIT;
constexpr int NUM_THREADS = WORKER_T0 + NUM_WORKERS;
// Main weight ring, 16 KB slots laid out contiguously from OFF_Q.  Slots 2-3 are free in every phase (out-projection slices
// rotate over them); the MLP weights rotate over all nine: slots 0-1 alias the Q/K/V staging and slots 4-8 the QKV ring (plus the
// 8 KB behind it), all idle in the MLP phase — 144 KB in flight cover the L2 latency at the MLP's consumption rate (16 KB per 256 tensor cycles).
constexpr int RING = 9, RING_LO = 2, RING_HI = 4, SLOT_BYTES = 16384;
// QKV ring: one slot = one 64-wide K panel of [Wq_h; Wk_h; Wv_h] (3 x 32 rows x 128 B); six slots = one and a half heads in
// flight.  With four (one head) every QKV_{h+1} waited ~400 cycles for its first panels, and the chain E1_h -> QKV_{h+1} -> E1_{h+1}
// (D1 is single-buffered in TMEM) is what paces the attention phase.
constexpr int QRING = 6, QSLOT_BYTES = 12288;
// K panels per head in the QKV ring (= K panels of A0) at model width D
template <int D> constexpr int KPH = D / 64;
// "Head full" barriers of the QKV ring: head hq signals barrier hq % NQG, whose phase (hq / NQG) & 1 the MMA thread waits for.
// Head hq + NQG re-arms that barrier (expect_tx) when its first panel is issued, i.e. after the producer's wait for the slot of
// panel KPH * (hq + NQG) - QRING to be consumed.  With NQG = ceil(QRING / KPH) that panel number lies in
// [KPH * hq, KPH * hq + KPH - 1]: it is one of head hq's OWN panels, consumed only after the MMA thread's wait for head hq.  So a
// barrier never completes a second phase before its first one has been waited for.  (D = 256, QRING = 6: KPH = 4, NQG = 2, head
// hq + 2 reuses the slot of head hq's third panel; D = 128: KPH = 2, NQG = 3, head hq + 3 reuses the slot of head hq's first panel.)
template <int D> constexpr int NQG = (QRING + KPH<D> - 1) / KPH<D>;
constexpr int MAX_QG = NQG<128>;
static_assert(KPH<256> * (NQG<256> - 1) < QRING && QRING <= KPH<256> * NQG<256>, "head-full barrier parity (D = 256)");
static_assert(KPH<128> * (NQG<128> - 1) < QRING && QRING <= KPH<128> * NQG<128>, "head-full barrier parity (D = 128)");
// MLP weight slots per "group full" barrier: one barrier per GEMM (four slots at D = 256)
constexpr int MLPG = 4;
// At D = 128 an MLP GEMM (FF1: K = D, FF2: N = D) is two 16 KB slots: one group per GEMM
template <int D> constexpr int GSLOTS = MLPG < D / 64 ? MLPG : D / 64;

// shared memory map (offsets from a 1024-byte aligned base)
constexpr int OFF_A0 = 0;                          // 64 KB  LN output [128 x D] bf16, D / 64 K-panels of 16 KB; also the NCHW input staging
constexpr int OFF_Q = 65536;                       // 8 KB   Q_h [128 x 32] K-major SW64
constexpr int OFF_K = OFF_Q + 8192;                // 8 KB   K_h
constexpr int OFF_V = OFF_K + 8192;                // 2x8 KB V_h [128 tok x 32] MN-major SW64, double buffered
constexpr int OFF_RING = OFF_V + 16384;            // 2 x 16 KB weight ring (slots 2-3; slots 0-1 = the 32 KB of Q/K/V staging above)
constexpr int OFF_QRING = OFF_RING + 2 * SLOT_BYTES;   // QRING x 12 KB QKV weight ring, right behind slot 3; also the NCHW output staging (2 x 64 x 256 bf16 at most)
constexpr int OFF_OUTST = OFF_QRING;
static_assert(QRING * QSLOT_BYTES >= 2 * 64 * 256 * 2, "the NCHW output staging lives in the QKV ring");
constexpr int QRING_END = OFF_QRING + QRING * QSLOT_BYTES;
constexpr int OFF_XCH = QRING_END > OFF_Q + RING * SLOT_BYTES ? QRING_END : OFF_Q + RING * SLOT_BYTES;      // row exchange [2][128][4] floats
static_assert(OFF_XCH - OFF_Q >= RING * SLOT_BYTES, "the nine MLP ring slots fit in [OFF_Q, OFF_XCH)");
static_assert(OFF_RING == OFF_Q + RING_LO * SLOT_BYTES, "ring slots are contiguous from OFF_Q");
__host__ __device__ constexpr int slot_offset(uint32_t s) { return OFF_Q + int(s) * SLOT_BYTES; }
constexpr int OFF_VEC = OFF_XCH + 2 * 128 * 4 * 4;      // per-layer vectors (first D entries of each used)
constexpr int V_BOUT = 0, V_BFF2 = DIM, V_BFF1 = 2 * DIM;   // fp32 biases
constexpr int V_B16 = V_BFF1 + MAX_MLP;             // then bf16 copies of the LayerNorm affine vectors: [ln1_g | ln1_b | ln2_g | ln2_b] x DIM
constexpr int OFF_BAR = OFF_VEC + (V_B16 + 512) * 4;
constexpr int SMEM_USED = OFF_BAR + 512;
constexpr int SMEM_ALLOC = SMEM_USED + 1024;       // slack for the 1024-byte alignment of the base
static_assert(SMEM_ALLOC <= 232448, "shared memory budget");

// K-panel order of the two GEMMs that read a fresh LayerNorm output (QKV, FF1).  The two threads of a row write panels {0,1} and {2,3}
// of A0, so panels 0 and 2 are complete when every thread is half-way through its normalisation sweep (B_A0_HALF): the first GEMM behind
// a LayerNorm starts on them and only then waits for the whole operand (B_A0_READY).  At D = 128 each thread writes ONE panel,
// both at the same time: plain order, one barrier.
template <int D> constexpr bool A0_HALF = D == 256;
template <int D>
__device__ __forceinline__ constexpr int kpanel(int i) { return A0_HALF<D> ? (((i & 1) << 1) | (i >> 1)) : i; }      // 0, 2, 1, 3

// TMEM columns (residual stream: [0, D))
constexpr uint32_t TM_X = 0, TM_D1 = 256, TM_O = 352, TM_S = 384, TM_H0 = 256, TM_H1 = 384;

enum {
  B_RING_FULL = 0, B_RING_EMPTY = RING, B_X0_FULL = 2 * RING, B_A0_FREE, B_A0_READY, B_D1_FULL, B_STAGED, B_S_FULL, B_P_READY, B_O_FULL,
  B_O_DRAINED, B_X1_FULL, B_HACC_FULL, B_HACC_FULL1, B_H_READY, B_H_READY1, B_X2_FULL,
  B_QG_FULL, B_QR_EMPTY = B_QG_FULL + MAX_QG, B_A1_FREE = B_QR_EMPTY + QRING, B_OUT_READ, B_QKV_FREE, B_G_FULL, B_TQ_FULL = B_G_FULL + 8, B_A0_HALF = B_TQ_FULL + 4, NUM_BARS
};
static_assert(NUM_BARS * 8 + 8 + 16 <= 512, "barrier block (+ TMEM slot + tile queue)");

// Tile scheduler.  The first tile of a CTA is blockIdx.x; the following ones come from an atomic counter (DYNAMIC: the persistent grid
// then balances itself — a CTA that starts late because an NCCL kernel or a neighbouring stream holds its SM, or that runs on a
// slower-clocked part of the chip, simply takes fewer tiles instead of finishing a fixed share late) or from static striding.  The
// weight producer fetches the index of tile k+1 while it issues tile k and publishes it through a four-entry queue in shared
// memory (one mbarrier per entry); the other roles read entry k when they get there.  -1 ends the loop.
__device__ __forceinline__ int* tile_queue(uint64_t* bars) { return reinterpret_cast<int*>(bars + NUM_BARS) + 2; }   // behind the TMEM slot word
__device__ __forceinline__ int next_tile(uint64_t* bars, uint32_t k) {
  mbar_wait(&bars[B_TQ_FULL + (k & 3u)], (k >> 2) & 1u);
  return *reinterpret_cast<volatile int*>(tile_queue(bars) + (k & 3u));
}

enum { IO_NCHW_BF16 = 0, IO_ROWS_F32 = 1 };
constexpr int POS_LD = 64;   // row stride of the channel-major positional table

// worker phases
enum { PW_INPUT = 0, PW_VEC, PW_LN1, PW_WAIT_D1, PW_E1, PW_WAIT_O, PW_E3, PW_WAIT_S, PW_E2, PW_WAIT_X1, PW_LN2, PW_WAIT_HACC, PW_GELU, PW_WAIT_X2,
       PW_OUTPUT, PW_TILES, PW_E2_LD, PW_E2_EXP, PW_E2_XCH, PW_E2_ST,
       // MMA thread phases
       PM_WAIT_A0 = 32, PM_QKV, PM_WAIT_STAGED, PM_S, PM_WAIT_P, PM_PV, PM_WAIT_OD7, PM_OUT, PM_WAIT_A0B, PM_FF1, PM_WAIT_H, PM_FF2, PM_RINGWAIT,
       PM_RW_QKV, PM_RW_OUT, PM_RW_FF1, PM_RW_FF2, PM_REFILL_CYC, PM_REFILL_N };

struct LayerArgs {
  CUtensorMap tm_qkv, tm_out, tm_w1, tm_w2;     // tm_out: box [256 rows x 32 cols], 64B swizzle (one head's K slice of Wout)
  const float *ln1_g, *ln1_b, *b_out, *ln2_g, *ln2_b, *b_ff1, *b_ff2;
  uint64_t pad_;
};

// A tile is 128 token rows = `spt` sequences, each padded to a row slot of `slot` rows (the power of two >= n_tok,
// at least 16): row r belongs to sequence r / slot, token r % slot.  With slot >= 32 all rows of a warp belong to ONE
// sequence, so the whole warp reads the same window of score columns.
struct FusedArgs {
  LayerArgs layer[MAX_DEPTH];
  const void* in;
  void* out;                 // IO_ROWS_F32: nullptr = the token rows are not stored (w_last given)
  const float* pos;          // [n_tok, D] or nullptr (IO_ROWS_F32)
  const float* w_last;       // IO_ROWS_F32, n_tok = 12: [12, D] AU weights or nullptr; out21 [n_seq, 21] and decisions [n_seq, 12]
  float* out21;              // (nullable) are then written by the last layer's output sweep
  int* decisions;
  const float* pos_t;        // IO_NCHW_BF16: the same table as [256 / 4][POS_LD tokens][4 channels]: one 16-byte load per 4 channels,
                             // and the lanes of a warp (consecutive tokens) read consecutive 16-byte words
  int ld_in, ld_out;         // IO_ROWS_F32 row strides (elements)
  int* tile_counter;         // dynamic tile scheduler: a zeroed device counter (nullptr = static striding, tile = blockIdx.x + k * gridDim.x)
  int n_seq, n_tok, slot, slot_log2, spt, n_tiles, n_chunks, depth;
};

// Developer aid: a host-mapped word block that the weight producer fills in when its wait for a ring slot times out (a protocol
// bug) before it traps — the trap poisons the context, but pinned host memory stays readable: {block, thread, barrier index,
// parity}.  Set with avf_debug_set_trap_buffer (tools/trap_probe.py).
__device__ unsigned* g_trap_buffer = nullptr;

// ---------------------------------------------------------------------------------------------
// row workers: thread (row, g) owns columns [g*CW, g*CW+CW) of token row `row` (= TMEM lane), CW = D / NSPLIT
// ---------------------------------------------------------------------------------------------
template <int D>
struct Worker {
  static constexpr int CW = D / NSPLIT;

  uint8_t* smem;
  uint64_t* bars;
  const float* vec;     // per-layer vectors in shared memory
  uint32_t tl;          // TMEM address of this warp's lane quarter, column 0
  int lane, q, g, row;
  uint32_t xslot;

  // all-gather of one float between the NSPLIT threads of a row
  __device__ __forceinline__ const float* exchange(float mine) {
    float* s = reinterpret_cast<float*>(smem + OFF_XCH) + xslot * (128 * 4);
    xslot ^= 1;
    s[row * 4 + g] = mine;
    bar_sync(1 + q, 32 * NSPLIT);
    return s + row * 4;
  }
  __device__ __forceinline__ float exchange_sum(float mine) {
    const float* v = exchange(mine);
    return v[0] + v[1];
  }
  __device__ __forceinline__ float exchange_max(float mine) {
    const float* v = exchange(mine);
    return fmaxf(v[0], v[1]);
  }
  __device__ __forceinline__ void arrive(int bar) {             // one arrive per warp, after every lane's fences
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&bars[bar]);
  }
  __device__ __forceinline__ void arrive_tmem_only(int bar) {   // the phase wrote TMEM only (no shared-memory operand for the async proxy)
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&bars[bar]);
  }
  // Statistics are accumulated as shifted sums (shift = the thread's first element) and merged across the row's threads
  // by Chan's formula, so one sweep over the row is enough and nothing cancels catastrophically.
  struct Stats {
    float shift, s, ss;
    __device__ __forceinline__ void add(const float (&x)[32], bool first) {
      if (first) shift = x[0];
      // pairs: d = x - shift, s += d, ss += d * d as three packed instructions per two elements
      const uint64_t nshift = f2_pack(-shift, -shift);
      uint64_t s2 = f2_pack(0.f, 0.f), q2 = s2;
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        const uint64_t d = f2_add(f2_pack(x[j], x[j + 1]), nshift);
        s2 = f2_add(s2, d);
        q2 = f2_fma(d, d, q2);
      }
      float a, b;
      f2_unpack(s2, a, b);
      s += a + b;
      f2_unpack(q2, a, b);
      ss += a + b;
    }
  };
  __device__ __forceinline__ void finish_stats(const Stats& st, float& mean, float& rstd) {
    constexpr float n = float(CW);
    const float mean_g = st.shift + st.s * (1.f / n);
    const float m2_g = fmaxf(st.ss - st.s * st.s * (1.f / n), 0.f);
    mean = exchange_sum(mean_g) * (1.f / NSPLIT);
    const float dm = mean_g - mean;
    const float m2 = exchange_sum(fmaf(dm * dm, n, m2_g));
    rstd = rsqrtf(m2 * (1.f / D) + 1e-5f);
  }
  // Sweep 1 of a LayerNorm whose input already sits in TMEM (x1 after the out-projection, x2 after the MLP).
  __device__ __forceinline__ void stats_from_tmem(float& mean, float& rstd) {
    Stats st{0.f, 0.f, 0.f};
#pragma unroll
    for (int c0 = 0; c0 < CW; c0 += 32) {
      float x[32];
      tmem_ld32(tl + TM_X + g * CW + c0, reinterpret_cast<uint32_t(&)[32]>(x));
      tmem_ld_wait();
      st.add(x, c0 == 0);
    }
    finish_stats(st, mean, rstd);
  }
  // Sweep 2: LN(x) -> A0 (bf16, K-major SW128 panels), x + next_bias -> TMEM; then signal the MMA thread.
  // (x - mean) * rstd in fp32, the affine part on bf16 pairs (gamma / beta pre-rounded to bf16 in shared memory); ln_sel 0 / 1 = LN1 / LN2
  __device__ __forceinline__ void normalize_from_tmem(float mean, float rstd, int ln_sel, int v_next_bias) {
    const int cbase = g * CW;
    const float nmr = -mean * rstd;
    const uint64_t rstd2 = f2_pack(rstd, rstd), nmr2 = f2_pack(nmr, nmr);
#pragma unroll 1
    for (int c0 = 0; c0 < CW; c0 += 32) {
      float x[32];
      tmem_ld32(tl + TM_X + cbase + c0, reinterpret_cast<uint32_t(&)[32]>(x));
      tmem_ld_wait();
      const int col0 = cbase + c0;
      uint8_t* dst = smem + OFF_A0 + (col0 >> 6) * 16384 + row * 128;
      const int chunk0 = (col0 & 63) >> 3;
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const __nv_bfloat16* v16 = reinterpret_cast<const __nv_bfloat16*>(vec + V_B16) + ln_sel * (2 * DIM) + col0 + ch * 8;
        const uint4 gm = *reinterpret_cast<const uint4*>(v16), bt = *reinterpret_cast<const uint4*>(v16 + DIM);
        uint4 pk;
        pk.x = fma_bf16x2(cvt_bf16x2_pair(f2_fma(f2_pack(x[ch * 8], x[ch * 8 + 1]), rstd2, nmr2)), gm.x, bt.x);
        pk.y = fma_bf16x2(cvt_bf16x2_pair(f2_fma(f2_pack(x[ch * 8 + 2], x[ch * 8 + 3]), rstd2, nmr2)), gm.y, bt.y);
        pk.z = fma_bf16x2(cvt_bf16x2_pair(f2_fma(f2_pack(x[ch * 8 + 4], x[ch * 8 + 5]), rstd2, nmr2)), gm.z, bt.z);
        pk.w = fma_bf16x2(cvt_bf16x2_pair(f2_fma(f2_pack(x[ch * 8 + 6], x[ch * 8 + 7]), rstd2, nmr2)), gm.w, bt.w);
        *reinterpret_cast<uint4*>(dst + (((chunk0 + ch) ^ (row & 7)) << 4)) = pk;
      }
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        const ulonglong2 b = *reinterpret_cast<const ulonglong2*>(vec + v_next_bias + col0 + j);      // two fp32 pairs
        f2_unpack(f2_add(f2_pack(x[j], x[j + 1]), b.x), x[j], x[j + 1]);
        f2_unpack(f2_add(f2_pack(x[j + 2], x[j + 3]), b.y), x[j + 2], x[j + 3]);
      }
      tmem_st32(tl + TM_X + col0, reinterpret_cast<const uint32_t(&)[32]>(x));
      if (A0_HALF<D> && c0 == 32) arrive(B_A0_HALF);          // this thread's first panel (0 or 2) is written
    }
    tmem_st_wait();
    arrive(B_A0_READY);
  }
};

// Softmax of one head for a thread that owns NC whole 8-column chunks of its row's window, geometry known at compile time
// (TAILV > 0: only the first TAILV columns of the last chunk exist).  S is read at `ts`, P (bf16 pairs) written at `tp`;
// returns the thread's partial row sum.  Same arithmetic as the general path in worker_main.
template <int NC, int TAILV, class W>
__device__ __forceinline__ float softmax_fixed(W& w, uint32_t ts, uint32_t tp, float sm_scale, Prof& pf) {
  float s[NC][8];
#pragma unroll
  for (int c = 0; c < NC; ++c) tmem_ld8(ts + c * 8, reinterpret_cast<uint32_t(&)[8]>(s[c]));
  tmem_ld_wait();
  pf.mark(PW_E2_LD);
  float mc[NC];                                   // per-chunk maxima as trees (independent chains), then one short chain across chunks
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (TAILV > 0 && c == NC - 1) {
      mc[c] = s[c][0];
#pragma unroll
      for (int j = 1; j < 8; ++j)
        if (j < TAILV) mc[c] = fmaxf(mc[c], s[c][j]);
    } else {
      mc[c] = fmaxf(fmaxf(fmaxf(s[c][0], s[c][1]), fmaxf(s[c][2], s[c][3])), fmaxf(fmaxf(s[c][4], s[c][5]), fmaxf(s[c][6], s[c][7])));
    }
  }
  float mloc = mc[0];
#pragma unroll
  for (int c = 1; c < NC; ++c) mloc = fmaxf(mloc, mc[c]);
  pf.mark(PW_E2_EXP);
  const float mrow = w.exchange_max(mloc);      // also orders every S load of the row before any P store (P overwrites S)
  pf.mark(PW_E2_XCH);
  const float nml = -mrow * sm_scale;
  const uint64_t sc2 = f2_pack(sm_scale, sm_scale), nml2 = f2_pack(nml, nml);
  uint64_t sum2 = f2_pack(0.f, 0.f);             // (sum of the low halves, sum of the high halves) of the exponentiated pairs
  float sum_lo = 0.f;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int nv = (TAILV > 0 && c == NC - 1) ? TAILV : 8;
    uint32_t e[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (2 * j + 1 < nv) {
        e[j] = ex2_bf16x2(cvt_bf16x2_pair(f2_fma(f2_pack(s[c][2 * j], s[c][2 * j + 1]), sc2, nml2)));
        sum2 = f2_add(sum2, f2_pack(__uint_as_float(e[j] << 16), __uint_as_float(e[j] & 0xFFFF0000u)));
      } else if (2 * j < nv) {                   // only the low half of the pair exists
        e[j] = ex2_bf16x2(cvt_bf16x2(fmaf(s[c][2 * j], sm_scale, nml), -INFINITY)) & 0xFFFFu;
        sum_lo += __uint_as_float(e[j] << 16);
      } else {
        e[j] = 0u;
      }
    }
    tmem_st4(tp + c * 4, e[0], e[1], e[2], e[3]);
  }
  float a, b;
  f2_unpack(sum2, a, b);
  return sum_lo + (a + b);
}

__host__ __device__ constexpr int slot_of(int n_tok) { return n_tok <= 16 ? 16 : (n_tok <= 32 ? 32 : 64); }
__host__ __device__ constexpr int log2_of(int v) { return v == 16 ? 4 : (v == 32 ? 5 : 6); }

// NTOK > 0: the sequence length is a compile-time constant (the SFormer's 49): the transposing tile sweeps address the staged
// NCHW frames with immediate offsets and the softmax geometry folds away.  NTOK = 0: everything from FusedArgs.
template <int IO, int NTOK, int D>
__device__ void worker_main(const FusedArgs& a, uint8_t* smem, uint64_t* bars, uint32_t tmem) {
  using W = Worker<D>;
  constexpr int CW = W::CW;
  W w;
  w.smem = smem;
  w.bars = bars;
  w.vec = reinterpret_cast<const float*>(smem + OFF_VEC);
  const int wt = threadIdx.x - WORKER_T0;
  w.lane = wt & 31;
  w.q = (threadIdx.x >> 5) & 3;          // TMEM lane quarter = warp index mod 4
  w.g = wt >> 7;                         // which part of the columns
  w.row = w.q * 32 + w.lane;
  w.tl = tmem + (uint32_t(w.q * 32) << 16);
  w.xslot = 0;
  const int q = w.q, g = w.g, row = w.row;
  const uint32_t tl = w.tl;
  const float* vec = w.vec;
  const int n_tok = NTOK ? NTOK : a.n_tok, slot = NTOK ? slot_of(NTOK) : a.slot, spt = NTOK ? 128 / slot_of(NTOK) : a.spt;
  const int slot_log2 = NTOK ? log2_of(slot_of(NTOK)) : a.slot_log2;
  const int seq_in_tile = row >> slot_log2, t_in_seq = row & (slot - 1);
  // softmax geometry.  This row attends to score columns [lo, lo + n_tok).  The warp's rows cover sequences s0..s1, so
  // the warp sweeps the 8-column chunks [c_lo, c_hi) and the row's threads split them evenly (<= 8 / NSPLIT chunks each).
  const int lo = seq_in_tile * slot, hi = lo + n_tok;
  const int s0 = (q * 32) >> slot_log2, s1 = (q * 32 + 31) >> slot_log2;
  const int c_lo = (s0 * slot) >> 3, c_hi = (s1 * slot + n_tok + 7) >> 3;
  constexpr int MAXC = 8 / NSPLIT;
  const int per = (c_hi - c_lo + NSPLIT - 1) / NSPLIT;
  const int my_c0 = c_lo + g * per;
  const int my_nc = max(0, min(per, c_hi - my_c0));
  // does any chunk of this thread contain a column outside some row's window?  (interior chunks need no mask)
  const bool warp_one_seq = s0 == s1;
  const float sm_scale = 1.4426950408889634f * rsqrtf(float(DH));
  uint32_t n_x0 = 0, n_x1 = 0, n_x2 = 0, n_hacc0 = 0, n_hacc1 = 0;
  bool vec_loaded = false;
  Prof pf;
  pf.start(blockIdx.x == 0 && wt == 0);

  for (uint32_t tk = 0;; ++tk) {
    const int tile = next_tile(bars, tk);
    if (tile < 0) break;
    const int seqs_here = min(spt, a.n_seq - tile * spt);
    const bool valid = seq_in_tile < seqs_here && t_in_seq < n_tok;
    const size_t grow = (size_t(tile) * spt + seq_in_tile) * n_tok + t_in_seq;     // global token row (IO_ROWS_F32)

    // ---- tile input: x (+ pos) -> TMEM, statistics of LN1 on the way --------------------------------------
    float mean, rstd;
    {
      typename W::Stats st{0.f, 0.f, 0.f};
      // Branch-free: padding rows (and sequences beyond the end of the batch) read a valid location, i.e. they carry a copy of a
      // real token.  Nothing ever looks at them: as keys they are outside every row's softmax window, as rows they are not stored.
      const int t_safe = valid ? t_in_seq : 0, seq_safe = valid ? seq_in_tile : 0;
      const float* pp = (IO == IO_ROWS_F32 && a.pos != nullptr) ? a.pos + t_safe * D + g * CW : nullptr;
      const float4* ppt = reinterpret_cast<const float4*>(a.pos_t) + size_t(g * CW / 4) * POS_LD + t_safe;
      if constexpr (IO == IO_NCHW_BF16) mbar_wait(&bars[B_X0_FULL], (n_x0++) & 1);
      const __nv_bfloat16* src16 = reinterpret_cast<const __nv_bfloat16*>(smem + OFF_A0) + size_t(seq_safe * D + g * CW) * n_tok + t_safe;
      const float* src32 = static_cast<const float*>(a.in) + ((size_t(tile) * spt + seq_safe) * n_tok + t_safe) * a.ld_in + g * CW;
#pragma unroll 1
      for (int c0 = 0; c0 < CW; c0 += 32) {
        float x[32];
        if constexpr (IO == IO_NCHW_BF16) {
          // positional values first (coalesced: the lanes of a warp are consecutive tokens of one channel row), the 32
          // shared-memory reads of the staged frame overlap their L1/L2 round trip
          float4 p[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) p[j] = __ldg(ppt + (c0 / 4 + j) * POS_LD);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            f2_unpack(f2_add(f2_pack(__bfloat162float(src16[(c0 + 4 * j) * n_tok]), __bfloat162float(src16[(c0 + 4 * j + 1) * n_tok])),
                             f2_pack(p[j].x, p[j].y)), x[4 * j], x[4 * j + 1]);
            f2_unpack(f2_add(f2_pack(__bfloat162float(src16[(c0 + 4 * j + 2) * n_tok]), __bfloat162float(src16[(c0 + 4 * j + 3) * n_tok])),
                             f2_pack(p[j].z, p[j].w)), x[4 * j + 2], x[4 * j + 3]);
          }
        } else {
          float4 p4[8];
          if (pp != nullptr) {
#pragma unroll
            for (int j = 0; j < 8; ++j) p4[j] = __ldg(reinterpret_cast<const float4*>(pp + c0) + j);
          }
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 x4 = *reinterpret_cast<const float4*>(src32 + c0 + j);
            x[j] = x4.x; x[j + 1] = x4.y; x[j + 2] = x4.z; x[j + 3] = x4.w;
          }
          if (pp != nullptr) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              x[4 * j] += p4[j].x; x[4 * j + 1] += p4[j].y; x[4 * j + 2] += p4[j].z; x[4 * j + 3] += p4[j].w;
            }
          }
        }
        st.add(x, c0 == 0);
        tmem_st32(tl + TM_X + g * CW + c0, reinterpret_cast<const uint32_t(&)[32]>(x));
      }
      tmem_st_wait();
      w.finish_stats(st, mean, rstd);
      if constexpr (IO == IO_NCHW_BF16) {
        // the previous tile's output store must have finished READING A1 before this tile's attention writes it again: waited
        // for here (one thread, ordered for everybody by the barrier below) instead of right after issuing it
        if (threadIdx.x == WORKER_T0) {
          bulk_wait_read0();
          mbar_arrive(&bars[B_OUT_READ]);   // ... and before the QKV ring (which lives in A1) is refilled for this tile
        }
        bar_sync(5, NUM_WORKERS);   // every worker has read its part of the staged frames out of A0
      }
    }
    pf.mark(PW_INPUT);

    for (int l = 0; l < a.depth; ++l) {
      const LayerArgs& L = a.layer[l];
      if (a.depth > 1 || !vec_loaded) {          // per-layer vectors -> shared memory (once per CTA when there is one layer)
        if (vec_loaded) bar_sync(5, NUM_WORKERS);  // previous layer's readers are done
        float* vs = reinterpret_cast<float*>(smem + OFF_VEC);
        for (int i = wt; i < D; i += NUM_WORKERS) {
          vs[V_BOUT + i] = L.b_out[i]; vs[V_BFF2 + i] = L.b_ff2[i];
          __nv_bfloat16* v16 = reinterpret_cast<__nv_bfloat16*>(vs + V_B16);
          v16[i] = __float2bfloat16_rn(L.ln1_g[i]); v16[DIM + i] = __float2bfloat16_rn(L.ln1_b[i]);
          v16[2 * DIM + i] = __float2bfloat16_rn(L.ln2_g[i]); v16[3 * DIM + i] = __float2bfloat16_rn(L.ln2_b[i]);
        }
        for (int i = wt; i < a.n_chunks * 128; i += NUM_WORKERS) vs[V_BFF1 + i] = L.b_ff1[i];
        bar_sync(5, NUM_WORKERS);
        vec_loaded = true;
      }
      pf.mark(PW_VEC);
      w.normalize_from_tmem(mean, rstd, 0, V_BOUT);
      pf.mark(PW_LN1);

      // ---- attention: per head  E1 (QKV -> smem), E3 of the previous head (O / l -> TMEM), E2 (softmax) -------------
      float inv_l = 0.f;
#pragma unroll 1
      for (int h = 0; h <= HEADS; ++h) {
        if (h < HEADS) {         // E1: D1 = [Q|K|V]_h as 12 chunks of 8 columns, 12 / NSPLIT per thread
          mbar_wait(&bars[B_D1_FULL], h & 1);
          tc_fence_after();
          pf.mark(PW_WAIT_D1);
          constexpr int NCH = 12 / NSPLIT;
          const uint32_t sw = uint32_t((row >> 1) & 3);
          uint32_t r[NCH * 8];
          tmem_ld32(tl + TM_D1 + g * 48, reinterpret_cast<uint32_t(&)[32]>(r[0]));
          tmem_ld16(tl + TM_D1 + g * 48 + 32, reinterpret_cast<uint32_t(&)[16]>(r[32]));
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            const int id = g * NCH + c;                    // 0..3 Q, 4..7 K, 8..11 V
            uint8_t* base = id < 4 ? smem + OFF_Q : (id < 8 ? smem + OFF_K : smem + OFF_V + (h & 1) * 8192);
            *reinterpret_cast<uint4*>(base + row * 64 + ((uint32_t(id & 3) ^ sw) << 4)) = pack8u(&r[c * 8]);
          }
          w.arrive(B_STAGED);
          pf.mark(PW_E1);
        }
        if (h > 0) {             // E3 of head h-1: O / l -> bf16 over its own TMEM columns (A operand of the per-head out-projection)
          mbar_wait(&bars[B_O_FULL], (h - 1) & 1);
          tc_fence_after();
          pf.mark(PW_WAIT_O);
          constexpr int OW = DH / NSPLIT;                  // 16 columns
          uint32_t r[OW];
          tmem_ld16(tl + TM_O + g * OW, reinterpret_cast<uint32_t(&)[16]>(r[0]));
          tmem_ld_wait();
          {   // l = own + partner's partial row sum of head h-1 (written before their P_READY arrive, which PV -> O_FULL follows)
            const float* sums = reinterpret_cast<const float*>(smem + OFF_XCH) + ((h - 1) & 1) * (128 * 4) + row * 4 + 2;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv_l) : "f"(sums[0] + sums[1]));
          }
          const uint64_t inv2 = f2_pack(inv_l, inv_l);
          // O_h / l goes back INTO the accumulator's TMEM columns as packed bf16 (like P over S and gelu(H) over H): thread g turns its 16
          // fp32 columns [16g, 16g + 16) into 8 packed columns at [16g, 16g + 8) — columns only it reads — and the out-projection takes
          // its A operand from TMEM, one 16-wide k-step per thread.  No shared-memory staging, no generic->async proxy fence.
          uint32_t pk[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) pk[j] = cvt_bf16x2_pair(f2_mul(f2_pack(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])), inv2));
          tmem_st8(tl + TM_O + g * OW, pk);
          tmem_st_wait();
          w.arrive_tmem_only(B_O_DRAINED);
          pf.mark(PW_E3);
        }
        if (h < HEADS) {         // E2: softmax of this row over its own sequence's columns, P (bf16) over the S columns
          mbar_wait(&bars[B_S_FULL], h & 1);
          tc_fence_after();
          pf.mark(PW_WAIT_S);
          if constexpr (NTOK > 32) {
            // 64-row slots, compile-time window: the row's chunks are [8 seq, 8 seq + NCH_ALL), thread 0 takes the first four, thread 1 the rest
            constexpr int NCH_ALL = (NTOK + 7) / 8, NC1 = NCH_ALL - 4, TAILV = NTOK & 7;
            static_assert(NC1 >= 1 && NC1 <= 4, "softmax split");
            const uint32_t sb = tl + TM_S + uint32_t(seq_in_tile) * 64, pb = tl + TM_S + uint32_t(seq_in_tile) * 32;
            const float sum_g = g == 0 ? softmax_fixed<4, 0>(w, sb, pb, sm_scale, pf) : softmax_fixed<NC1, TAILV>(w, sb + 32, pb + 16, sm_scale, pf);
            reinterpret_cast<float*>(smem + OFF_XCH)[(h & 1) * (128 * 4) + row * 4 + 2 + g] = sum_g;
            // P columns the MMA reads (all 64 = 128 keys) but this row does not own: zeros; thread g takes TMEM columns [32g, 32g + 32)
            if (g == seq_in_tile) {
              zero_p_columns(tl + TM_S, 32 * g + NCH_ALL * 4, 32 * g + 32);
            } else {
              tmem_st16_zero(tl + TM_S + 32 * g);
              tmem_st16_zero(tl + TM_S + 32 * g + 16);
            }
            tmem_st_wait();
            pf.mark(PW_E2_ST);
            w.arrive_tmem_only(B_P_READY);
            pf.mark(PW_E2);
          } else {
          float s[MAXC][8];
#pragma unroll
          for (int c = 0; c < MAXC; ++c)
            if (c < my_nc) tmem_ld8(tl + TM_S + (my_c0 + c) * 8, reinterpret_cast<uint32_t(&)[8]>(s[c]));
          tmem_ld_wait();
          pf.mark(PW_E2_LD);
          float mloc = -INFINITY;
#pragma unroll
          for (int c = 0; c < MAXC; ++c) {
            if (c < my_nc) {
              const int col0 = (my_c0 + c) * 8;
              if (!warp_one_seq || col0 + 8 > hi) {        // boundary chunk (or a warp that spans sequences): mask per column
#pragma unroll
                for (int j = 0; j < 8; ++j) s[c][j] = (col0 + j >= lo && col0 + j < hi) ? s[c][j] : -INFINITY;
              }
              mloc = fmaxf(mloc, fmaxf(fmaxf(fmaxf(s[c][0], s[c][1]), fmaxf(s[c][2], s[c][3])), fmaxf(fmaxf(s[c][4], s[c][5]), fmaxf(s[c][6], s[c][7]))));
            }
          }
          // the row maximum first (one exchange; it also orders every S load of the row before any P store — P is written over
          // the S columns), then 2^(s - max) straight to its final bf16 value, two per MUFU instruction; the partial row sums
          // (fp32, of the rounded values the MMA will see) meet again in E3 through shared memory, no second barrier
          pf.mark(PW_E2_EXP);
          const float mrow = w.exchange_max(mloc);
          pf.mark(PW_E2_XCH);
          const float nml = -mrow * sm_scale;            // every row has at least one valid column: mrow is finite
          float sum_g = 0.f;
#pragma unroll
          for (int c = 0; c < MAXC; ++c) {
            if (c < my_nc) {
              uint32_t e[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                e[j] = ex2_bf16x2(cvt_bf16x2(fmaf(s[c][2 * j], sm_scale, nml), fmaf(s[c][2 * j + 1], sm_scale, nml)));
                sum_g += __uint_as_float(e[j] << 16) + __uint_as_float(e[j] & 0xFFFF0000u);
              }
              tmem_st4(tl + TM_S + (my_c0 + c) * 4, e[0], e[1], e[2], e[3]);
            }
          }
          reinterpret_cast<float*>(smem + OFF_XCH)[(h & 1) * (128 * 4) + row * 4 + 2 + g] = sum_g;
          // P columns the MMA reads (all 128) but this warp's rows never use: zeros; thread g takes TMEM columns [32g, 32g + 32)
          {
            const int z_lo = g * 32, z_hi = z_lo + 32, w_lo = c_lo * 4, w_hi = c_hi * 4;
            zero_p_columns(tl + TM_S, z_lo, min(z_hi, max(z_lo, w_lo)));
            zero_p_columns(tl + TM_S, max(z_lo, min(z_hi, w_hi)), z_hi);
          }
          tmem_st_wait();
          pf.mark(PW_E2_ST);
          w.arrive_tmem_only(B_P_READY);
          pf.mark(PW_E2);
          }
        }
      }

      // ---- LN2 on x1 = x + attention (accumulated in TMEM by the out-projection) ------------------------------
      mbar_wait(&bars[B_X1_FULL], (n_x1++) & 1);
      tc_fence_after();
      pf.mark(PW_WAIT_X1);
      w.stats_from_tmem(mean, rstd);
      w.normalize_from_tmem(mean, rstd, 1, V_BFF2);
      pf.mark(PW_LN2);

      // ---- MLP: per 128-column chunk of the hidden layer, bias + tanh-GELU -> bf16 A operand ---------------------
      // The bf16 result goes back INTO the accumulator's TMEM columns (like P over S): thread g turns its fp32 columns
      // [g*HW, g*HW + HW) of the chunk into HW/2 packed columns at [g*HW, g*HW + HW/2) — columns it has already read — and the
      // second MLP GEMM takes its A operand from TMEM.  No shared-memory buffer, no generic->async proxy fence, and half of the
      // MLP's shared-memory operand traffic is gone (the tensor core re-reads A for every 16-wide k-step).
#pragma unroll 1
      for (int c = 0; c < a.n_chunks; ++c) {
        const int b = c & 1;
        if (b == 0) mbar_wait(&bars[B_HACC_FULL], (n_hacc0++) & 1);
        else mbar_wait(&bars[B_HACC_FULL1], (n_hacc1++) & 1);
        tc_fence_after();
        pf.mark(PW_WAIT_HACC);
        constexpr int HW = 128 / NSPLIT;                   // hidden columns per thread: 64 or 32
        const uint32_t hbase = tl + (b ? TM_H1 : TM_H0) + g * HW;
#pragma unroll
        for (int c0 = 0; c0 < HW; c0 += 32) {
          const float* bias = vec + V_BFF1 + c * 128 + g * HW + c0;
          uint32_t r[32], yk[16];
          tmem_ld32(hbase + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 b4 = *reinterpret_cast<const float4*>(bias + j);
            yk[j / 2] = gelu_bf16x2(cvt_bf16x2_pair(f2_add(f2_pack(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), f2_pack(b4.x, b4.y))));
            yk[j / 2 + 1] = gelu_bf16x2(cvt_bf16x2_pair(f2_add(f2_pack(__uint_as_float(r[j + 2]), __uint_as_float(r[j + 3])), f2_pack(b4.z, b4.w))));
          }
          tmem_st16(hbase + c0 / 2, yk);
        }
        tmem_st_wait();
        w.arrive_tmem_only(B_H_READY + b);
        pf.mark(PW_GELU);
      }

      // ---- x2 = x1 + MLP, accumulated in TMEM by the second MLP GEMM --------------------------------------------
      mbar_wait(&bars[B_X2_FULL], (n_x2++) & 1);
      tc_fence_after();
      pf.mark(PW_WAIT_X2);
      if (l + 1 < a.depth) w.stats_from_tmem(mean, rstd);
    }

    // ---- tile output (+ the AU logits: token t of a clip dotted with w_last[t]) -------------------------------
    {
      __nv_bfloat16* dst16 = reinterpret_cast<__nv_bfloat16*>(smem + OFF_OUTST) + size_t(seq_in_tile * D + g * CW) * n_tok + t_in_seq;
      const bool store = valid && (IO == IO_NCHW_BF16 || a.out != nullptr);
      float* dst32 = static_cast<float*>(a.out) + grow * a.ld_out + g * CW;
      const bool logits = IO == IO_ROWS_F32 && a.w_last != nullptr;
      const float* wl = logits ? a.w_last + (valid ? t_in_seq : 0) * D + g * CW : nullptr;
      float dot = 0.f;
#pragma unroll 1
      for (int c0 = 0; c0 < CW; c0 += 32) {
        float x[32];
        tmem_ld32(tl + TM_X + g * CW + c0, reinterpret_cast<uint32_t(&)[32]>(x));
        tmem_ld_wait();
        if (store) {
          if constexpr (IO == IO_NCHW_BF16) {
#pragma unroll
            for (int j = 0; j < 32; ++j) dst16[(c0 + j) * n_tok] = __float2bfloat16_rn(x[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(dst32 + c0 + j) = make_float4(x[j], x[j + 1], x[j + 2], x[j + 3]);
          }
        }
        if constexpr (IO == IO_ROWS_F32) {
          if (logits) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 w4 = __ldg(reinterpret_cast<const float4*>(wl + c0 + j));
              dot = fmaf(x[j], w4.x, fmaf(x[j + 1], w4.y, fmaf(x[j + 2], w4.z, fmaf(x[j + 3], w4.w, dot))));
            }
          }
        }
      }
      if constexpr (IO == IO_ROWS_F32) {
        if (logits) {      // n_tok = 12 (checked on the host): token t_in_seq of clip `grow / 12` is AU t_in_seq
          const float lg = w.exchange_sum(dot);
          const size_t clip = grow / 12;
          if (valid && g == 0) {
            if (a.out21 != nullptr) a.out21[clip * 21 + t_in_seq] = lg;
            if (a.decisions != nullptr) a.decisions[clip * 12 + t_in_seq] = lg > 0.f ? 1 : 0;     // round(sigmoid(x)) == x > 0
          }
          if (valid && g == 1 && t_in_seq < 9 && a.out21 != nullptr) a.out21[clip * 21 + 12 + t_in_seq] = 0.f;      // zero padding to 21
        }
      }
      if constexpr (IO == IO_NCHW_BF16) {
        fence_proxy_async_smem();
        bar_sync(5, NUM_WORKERS);
        if (threadIdx.x == WORKER_T0) {
          __nv_bfloat16* gdst = static_cast<__nv_bfloat16*>(a.out) + size_t(tile) * spt * n_tok * D;
          bulk_store_1d(gdst, smem + OFF_OUTST, uint32_t(seqs_here) * n_tok * D * 2);   // read completion: see the next tile's input sweep
        }
      }
    }
    pf.mark(PW_OUTPUT);
    pf.count(PW_TILES);
  }
  pf.flush(0, 32);
  if constexpr (IO == IO_NCHW_BF16) {
    if (threadIdx.x == WORKER_T0) bulk_wait_all0();
  }
}

// ---------------------------------------------------------------------------------------------
// weight producer (one thread): must issue slots in exactly the order the MMA thread consumes them
// ---------------------------------------------------------------------------------------------
template <int IO, int D>
__device__ void producer_main(const FusedArgs& a, uint8_t* smem, uint64_t* bars) {
  // (one lane only: this loop polls with try_wait between slots, and a whole-warp version — every lane polling and adopting the
  //  issuing lane's observation — measured 7x slower; the MMA warp, which blocks instead of polling, does run warp-wide)
  uint32_t it = 0;
  // Input frames of the NEXT tile go into A0 as soon as the MMAs of the current tile are done with it (B_A0_FREE, one
  // completion per tile).  Polled between weight slots so that this thread never blocks on it.
  int load_tile = blockIdx.x;                   // tile whose input frames are to be loaded next (-1: none pending)
  uint32_t n_free = 0;
  bool need_free = false;
  auto poll_loader = [&]() {
    if (IO != IO_NCHW_BF16 || load_tile < 0) return;
    if (need_free) {
      if (!mbar_test_wait(&bars[B_A0_FREE], n_free & 1)) return;     // a probe that never suspends: this thread has weight slots to serve
      ++n_free;
    }
    const int seqs_here = min(a.spt, a.n_seq - load_tile * a.spt);
    const uint32_t bytes = uint32_t(seqs_here) * a.n_tok * D * 2;
    mbar_expect_tx(&bars[B_X0_FULL], bytes);
    bulk_load_1d(smem + OFF_A0, static_cast<const __nv_bfloat16*>(a.in) + size_t(load_tile) * a.spt * a.n_tok * D, bytes, &bars[B_X0_FULL]);
    load_tile = -1;
    need_free = true;
  };
  // Slot s is refilled once its previous content has been consumed (per-slot parity bits: the out-projection slices rotate over
  // slots 2-4, the MLP weights over all five — slots 0-1 alias the Q/K/V staging and are only loaded after the attention MMAs).
  uint32_t pbits = 0, n_gate = 0;
  auto poll_wait = [&](uint64_t* bar, uint32_t parity) {
    // Fast path first: in the MLP phase this thread issues a 16 KB slot per ~250 tensor cycles, and every probe (of the slot's
    // barrier or of the input buffer's) costs it ~100 cycles.  The input loader is polled only while the slot is not free yet.
    if (mbar_try_wait(bar, parity)) return;
    poll_loader();
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
      poll_loader();
      if (clock64() - t0 > 4000000000LL) {
        unsigned* tb = g_trap_buffer;
        if (tb != nullptr) {
          tb[0] = blockIdx.x; tb[1] = threadIdx.x; tb[2] = (smem_u32(bar) & 1023u) >> 3; tb[3] = parity;
          __threadfence_system();
        }
        printf("avf: fused encoder producer timed out (block %d item %u)\n", blockIdx.x, it);
        __trap();
      }
    }
  };
  // A wait on an mbarrier costs the waiting thread ~100 cycles even when the phase completed long ago, and the MMA thread is on
  // the critical path of both the attention chain and the MLP.  The four 16 KB slots of one MLP GEMM therefore signal ONE "group
  // full" barrier (armed with the 64 KB of the whole group when its first slot is issued); slots are still released one by one.
  // Out-projection slices (one slot each) keep their per-slot barrier.  Group g uses barrier g % 8: at most five groups (of two
  // slots) fit in the nine slots, and group g + 8 can only be armed after slots of later groups have been released, i.e. after the
  // MMA thread's wait for group g.
  uint32_t gidx = 0;
  auto load = [&](uint32_t s, const CUtensorMap* tm, int c0, int c1, uint64_t* full_bar, uint32_t expect_bytes) {
    poll_wait(&bars[B_RING_EMPTY + s], ((pbits >> s) & 1u) ^ 1u);
    pbits ^= 1u << s;
    if (expect_bytes != 0) mbar_expect_tx(full_bar, expect_bytes);
    tma_load_2d(smem + slot_offset(s), tm, full_bar, c0, c1);
    ++it;
  };
  // tile scheduler (see next_tile): this thread owns the queue
  uint32_t kpub = 0;
  auto publish = [&](int t) {
    tile_queue(bars)[kpub & 3u] = t;
    mbar_arrive(&bars[B_TQ_FULL + (kpub & 3u)]);
    ++kpub;
  };
  int cur = blockIdx.x;
  publish(cur);
  for (;;) {
    int nxt;
    if (a.tile_counter != nullptr) nxt = atomicAdd(a.tile_counter, 1) + int(gridDim.x);
    else nxt = cur + int(gridDim.x);
    if (nxt >= a.n_tiles) nxt = -1;
    publish(nxt);
    if (IO == IO_NCHW_BF16) {
      while (load_tile >= 0) poll_loader();     // the frames of `cur` are on their way (normally long since) before `nxt` becomes the pending load
      load_tile = nxt;
    }
    for (int l = 0; l < a.depth; ++l) {
      const LayerArgs& L = a.layer[l];
      for (int h = 0; h < HEADS; ++h) {                        // Wout[:, 32h .. 32h+32): [D x 32], 64B swizzle
        const uint32_t s = RING_LO + h % (RING_HI - RING_LO);
        load(s, &L.tm_out, h * DH, 0, &bars[B_RING_FULL + s], D * DH * 2);
      }
      poll_wait(&bars[B_QKV_FREE], (n_gate++) & 1);          // the attention MMAs are done with the Q/K/V staging and A1 = slots 0-1, 5-8
      uint32_t m = 0;
      constexpr int G = GSLOTS<D>, NH = D / 128;
      auto ff1 = [&](int c) {                                  // K = D: D / 64 panels of W1[c*128 .. +128, :]
        for (int kp = 0; kp < D / 64; ++kp) {
          if (kp % G == 0) ++gidx;
          load((m++) % RING, &L.tm_w1, kpanel<D>(kp) * 64, c * 128, &bars[B_G_FULL + ((gidx - 1) & 7u)], kp % G == 0 ? G * SLOT_BYTES : 0);
        }
      };
      auto ff2 = [&](int c) {                                  // K = 128 (two panels) x N = D (D / 128 halves)
        for (int i = 0; i < 2 * NH; ++i) {
          const int kp = i / NH, nh = i % NH;
          if (i % G == 0) ++gidx;
          load((m++) % RING, &L.tm_w2, c * 128 + kp * 64, nh * 128, &bars[B_G_FULL + ((gidx - 1) & 7u)], i % G == 0 ? G * SLOT_BYTES : 0);
        }
      };
      ff1(0);
      if (a.n_chunks > 1) ff1(1);
      for (int c = 0; c < a.n_chunks; ++c) {
        ff2(c);
        if (c + 2 < a.n_chunks) ff1(c + 2);
      }
    }
    if (nxt < 0) break;
    cur = nxt;
  }
}

// ---------------------------------------------------------------------------------------------
// QKV weight producer (one thread of its own warp): the QRING x 12 KB ring inside A1
// ---------------------------------------------------------------------------------------------
template <int IO, int D>
__device__ void qkv_producer_main(const FusedArgs& a, uint8_t* smem, uint64_t* bars) {
  uint32_t qit = 0, hq = 0, n_free = 0, n_read = 0;
  bool first = true;
  for (uint32_t tk = 0; next_tile(bars, tk) >= 0; ++tk) {
    // A1 doubles as the NCHW output staging: the previous tile's bulk store must have read it (signalled after this tile's input sweep)
    if constexpr (IO == IO_NCHW_BF16) mbar_wait(&bars[B_OUT_READ], (n_read++) & 1);
    for (int l = 0; l < a.depth; ++l) {
      const LayerArgs& L = a.layer[l];
      if (!first) mbar_wait(&bars[B_A1_FREE], (n_free++) & 1);   // the previous layer's MLP weights (ring slots 5-8 live in A1) are consumed
      first = false;
      for (int h = 0; h < HEADS; ++h, ++hq) {
        // the KPH panels of a head signal ONE barrier (armed with the head's KPH x 12 KB at its first panel): the MMA thread waits
        // once per head.  Barrier hq % NQG is re-armed only after the MMA thread's wait for head hq (see NQG).
        uint64_t* fb = &bars[B_QG_FULL + (hq % uint32_t(NQG<D>))];
        for (int kp = 0; kp < KPH<D>; ++kp) {
          const uint32_t s = qit % QRING, ph = (qit / QRING) & 1;
          mbar_wait(&bars[B_QR_EMPTY + s], ph ^ 1);
          uint8_t* d = smem + OFF_QRING + s * QSLOT_BYTES;
          if (kp == 0) mbar_expect_tx(fb, KPH<D> * QSLOT_BYTES);
          for (int s3 = 0; s3 < 3; ++s3) tma_load_2d(d + s3 * 4096, &L.tm_qkv, fb, kpanel<D>(kp) * 64, s3 * (HEADS * DH) + h * DH);
          ++qit;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// MMA issuer (one thread)
// ---------------------------------------------------------------------------------------------
// Executed by ALL 32 lanes of warp 1 with warp-uniform values (so that descriptors and addresses live in uniform registers and
// the issue loop is a handful of instructions per MMA); only the elected lane issues tcgen05.mma / tcgen05.commit.
template <int D>
__device__ void mma_main(const FusedArgs& a, uint8_t* smem, uint64_t* bars, uint32_t tmem) {
  const bool leader = elect_one();
  const uint32_t a0 = smem_u32(smem + OFF_A0);
  const uint32_t qs = smem_u32(smem + OFF_Q), ks = smem_u32(smem + OFF_K), vs = smem_u32(smem + OFF_V);
  const uint32_t smem0 = smem_u32(smem), qring = smem_u32(smem + OFF_QRING);
  const int kmax = 128;                        // S / P span the whole tile: sequences sit in power-of-two row slots
  const uint32_t id_qkv = make_idesc_bf16(128, 96), id_s = make_idesc_bf16(128, kmax), id_pv = make_idesc_bf16(128, DH, 0, 1),
                 id_128 = make_idesc_bf16(128, 128), id_out = make_idesc_bf16(128, D);
  uint32_t obits = 0, m = 0, qit = 0, hq = 0, gidx = 0, n_a0 = 0, n_hready[2] = {0, 0};
  Prof pf;
  pf.start(blockIdx.x == 0 && leader);
  int ring_phase = PM_QKV;
  auto slot_wait = [&](uint32_t s) -> uint32_t {     // an out-projection slice: its own barrier (same slot sequence as producer_main)
    pf.mark(ring_phase);
    mbar_wait(&bars[B_RING_FULL + s], (obits >> s) & 1u);
    obits ^= 1u << s;
    tc_fence_after();
    pf.mark(PM_RW_OUT);
    return smem0 + uint32_t(slot_offset(s));
  };
  auto group_wait = [&]() {                          // the next MLPG slots of an MLP GEMM: one barrier (see producer_main)
    pf.mark(ring_phase);
    mbar_wait(&bars[B_G_FULL + (gidx & 7u)], (gidx >> 3) & 1u);
    ++gidx;
    tc_fence_after();
    pf.mark(ring_phase == PM_FF1 ? PM_RW_FF1 : PM_RW_FF2);
  };
  auto slot_release = [&](uint32_t s) {
    if (leader) umma_commit(&bars[B_RING_EMPTY + s]);
  };
  // fresh = the first GEMM behind a LayerNorm: its first two panels (0, 2) only need B_A0_HALF, the other two B_A0_READY
  auto a0_wait = [&](int i, bool fresh) {
    if constexpr (A0_HALF<D>) {
      if (!fresh || (i != 0 && i != 2)) return;
      pf.mark(ring_phase);
      if (i == 0) mbar_wait(&bars[B_A0_HALF], n_a0 & 1);
      else mbar_wait(&bars[B_A0_READY], (n_a0++) & 1);
    } else {
      if (!fresh || i != 0) return;
      pf.mark(ring_phase);
      mbar_wait(&bars[B_A0_READY], (n_a0++) & 1);
    }
    tc_fence_after();
    pf.mark(ring_phase == PM_QKV ? PM_WAIT_A0 : PM_WAIT_A0B);
  };
  auto qkv = [&](bool fresh) {                // D1[128 x 96] = LN(x) [Wq_h; Wk_h; Wv_h]^T, weights from the QKV ring
    pf.mark(ring_phase);
    mbar_wait(&bars[B_QG_FULL + (hq % uint32_t(NQG<D>))], (hq / uint32_t(NQG<D>)) & 1u);      // all KPH panels of the head
    ++hq;
    tc_fence_after();
    pf.mark(PM_RW_QKV);
    for (int i = 0; i < KPH<D>; ++i) {
      const int kp = kpanel<D>(i);
      a0_wait(i, fresh);
      const uint32_t s = qit % QRING;
      const uint64_t da = make_desc_sw128_kmajor(a0 + kp * 16384), db = make_desc_sw128_kmajor(qring + s * QSLOT_BYTES);
#pragma unroll
      for (int k = 0; k < 4; ++k) if (leader) umma_bf16(tmem + TM_D1, da + uint64_t(k * 2), db + uint64_t(k * 2), id_qkv, (i | k) != 0 ? 1u : 0u);
      if (leader) umma_commit(&bars[B_QR_EMPTY + s]);
      ++qit;
    }
    if (leader) umma_commit(&bars[B_D1_FULL]);
  };
  auto outproj = [&](int h) {                 // x += (O_h / l) Wout[:, 32h .. 32h+32)^T   (x + b_out was stored by the workers)
    const uint32_t s = RING_LO + h % (RING_HI - RING_LO), sb = slot_wait(s);
    const uint64_t db = desc_sw64(sb);
    if (leader) umma_bf16_ts(tmem + TM_X, tmem + TM_O, db, id_out, 1u);               // k-step 0: thread 0's packed columns
    if (leader) umma_bf16_ts(tmem + TM_X, tmem + TM_O + 16, db + 2, id_out, 1u);      // k-step 1: thread 1's
    slot_release(s);
  };
  bool last_layer = false;
  auto ff1 = [&](int c, bool fresh) {         // H[c&1][128 x 128] = LN2(x) W1[c*128.., :]^T
    const uint32_t d = tmem + ((c & 1) ? TM_H1 : TM_H0);
    for (int i = 0; i < D / 64; ++i) {
      const int kp = kpanel<D>(i);
      if (i % GSLOTS<D> == 0) group_wait();
      a0_wait(i, fresh);
      const uint32_t s = (m++) % RING, sb = smem0 + uint32_t(slot_offset(s));
      const uint64_t da = make_desc_sw128_kmajor(a0 + kp * 16384), db = make_desc_sw128_kmajor(sb);
#pragma unroll
      for (int k = 0; k < 4; ++k) if (leader) umma_bf16(d, da + uint64_t(k * 2), db + uint64_t(k * 2), id_128, (i | k) != 0 ? 1u : 0u);
      slot_release(s);
    }
    if (leader) umma_commit(&bars[B_HACC_FULL + (c & 1)]);
    if (c == a.n_chunks - 1 && last_layer) if (leader) umma_commit(&bars[B_A0_FREE]);
  };

  for (uint32_t tk = 0; next_tile(bars, tk) >= 0; ++tk) {
    for (int l = 0; l < a.depth; ++l) {
      last_layer = l == a.depth - 1;
      ring_phase = PM_QKV;
      qkv(true);                              // (the waits for LayerNorm 1's output are inside)
      pf.mark(PM_QKV);
      for (int h = 0; h < HEADS; ++h) {
        mbar_wait(&bars[B_STAGED], h & 1);
        tc_fence_after();
        pf.mark(PM_WAIT_STAGED);
        {                                     // S[128 x kmax] = Q_h K_h^T
          const uint64_t da = desc_sw64(qs), db = desc_sw64(ks);
          if (leader) umma_bf16(tmem + TM_S, da, db, id_s, 0u);
          if (leader) umma_bf16(tmem + TM_S, da + 2, db + 2, id_s, 1u);
          if (leader) umma_commit(&bars[B_S_FULL]);
        }
        pf.mark(PM_S);
        if (h + 1 < HEADS) qkv(false);
        pf.mark(PM_QKV);
        if (h > 0) {                          // O(h-1) / l is packed in TMEM: its slice of the out-projection
          mbar_wait(&bars[B_O_DRAINED], (h - 1) & 1);
          tc_fence_after();
          pf.mark(PM_WAIT_OD7);
          ring_phase = PM_OUT;
          outproj(h - 1);
          pf.mark(PM_OUT);
          ring_phase = PM_QKV;
        }
        mbar_wait(&bars[B_P_READY], h & 1);
        tc_fence_after();
        pf.mark(PM_WAIT_P);
        for (int k = 0; k < kmax / 16; ++k)   // O[128 x 32] = P V_h   (A from TMEM, B MN-major)
          if (leader) umma_bf16_ts(tmem + TM_O, tmem + TM_S + uint32_t(k * 8), desc_sw64(vs + (h & 1) * 8192 + k * 1024), id_pv, k != 0 ? 1u : 0u);
        if (leader) umma_commit(&bars[B_O_FULL]);
        pf.mark(PM_PV);
      }
      mbar_wait(&bars[B_O_DRAINED], (HEADS - 1) & 1);
      tc_fence_after();
      pf.mark(PM_WAIT_OD7);
      ring_phase = PM_OUT;
      outproj(HEADS - 1);
      if (leader) umma_commit(&bars[B_X1_FULL]);
      if (leader) umma_commit(&bars[B_QKV_FREE]);
      m = 0;
      pf.mark(PM_OUT);

      ring_phase = PM_FF1;
      ff1(0, true);                           // (the waits for LayerNorm 2's output are inside)
      if (a.n_chunks > 1) ff1(1, false);
      for (int c = 0; c < a.n_chunks; ++c) {
        const int b = c & 1;
        pf.mark(PM_FF1);
        mbar_wait(&bars[B_H_READY + b], (n_hready[b]++) & 1);
        tc_fence_after();
        pf.mark(PM_WAIT_H);
        ring_phase = PM_FF2;
        for (int kp = 0; kp < 2; ++kp)        // x += gelu(H_c) W2[:, c*128..]^T
          for (int nh = 0; nh < D / 128; ++nh) {
            if ((kp * (D / 128) + nh) % GSLOTS<D> == 0) group_wait();
            const uint32_t s = (m++) % RING, sb = smem0 + uint32_t(slot_offset(s));
            const uint32_t ta = tmem + (b ? TM_H1 : TM_H0) + uint32_t(kp * 64);       // gelu(H_c) as bf16, 8 columns per 16-wide k-step
            const uint64_t db = make_desc_sw128_kmajor(sb);
#pragma unroll
            for (int k = 0; k < 4; ++k) if (leader) umma_bf16_ts(tmem + TM_X + nh * 128, ta + uint32_t(k * 8), db + uint64_t(k * 2), id_128, 1u);
            slot_release(s);
          }
        pf.mark(PM_FF2);
        ring_phase = PM_FF1;
        if (c + 2 < a.n_chunks) ff1(c + 2, false);     // overwrites H_c: in order behind the MMAs above that read it
      }
      if (leader) umma_commit(&bars[B_X2_FULL]);
      if (leader) umma_commit(&bars[B_A1_FREE]);
    }
  }
  pf.flush(32, 64);
}

template <int IO, int NTOK, int D>
__global__ void __launch_bounds__(NUM_THREADS, 1) encoder_fused_kernel(const __grid_constant__ FusedArgs a) {
  // The kernel has no static shared memory, so the dynamic window starts at the CTA's shared-memory base, which is 1024-byte
  // aligned (checked below).  Using the array itself — not an address rounded up through integer arithmetic — lets the compiler
  // see that every access is to the shared state space: 32-bit LDS / STS with immediate offsets instead of generic LD / ST with
  // 64-bit address arithmetic (IADD3 + IMAD.X per access in the worker sweeps).
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;
  if (threadIdx.x == 0 && (smem_u32(smem_raw) & 1023u) != 0u) {
    printf("avf: encoder_fused_kernel: dynamic shared memory base is not 1024-byte aligned enough\n");
    __trap();
  }
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + NUM_BARS);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int l = 0; l < a.depth; ++l) {
      tma_prefetch_desc(&a.layer[l].tm_qkv);
      tma_prefetch_desc(&a.layer[l].tm_out);
      tma_prefetch_desc(&a.layer[l].tm_w1);
      tma_prefetch_desc(&a.layer[l].tm_w2);
    }
    for (int i = 0; i < NUM_BARS; ++i) {
      const bool by_workers = i == B_A0_READY || i == B_A0_HALF || i == B_STAGED || i == B_P_READY || i == B_O_DRAINED || i == B_H_READY || i == B_H_READY1;
      mbar_init(&bars[i], by_workers ? NUM_WORKERS / 32 : 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  pdl_wait();        // the prologue above overlapped the previous kernel; its results are needed from here on
  pdl_trigger();

  if (warp == 0) {
    if (lane == 0) producer_main<IO, D>(a, smem, bars);
  } else if (warp == 1) {
    mma_main<D>(a, smem, bars, tmem);
  } else if (warp == 2) {
    if (lane == 0) qkv_producer_main<IO, D>(a, smem, bars);
  } else {
    worker_main<IO, NTOK, D>(a, smem, bars, tmem);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
}

// pos [n_tok, 256] -> pos_t [256 / 4][POS_LD][4] (one tiny launch in front of the fused kernel; 64 KB)
__global__ void __launch_bounds__(256) pos_transpose_kernel(const float* __restrict__ pos, float* __restrict__ pos_t, int n_tok, int* tile_counter) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  if (blockIdx.x == 0 && threadIdx.x == 0 && tile_counter != nullptr) *tile_counter = 0;      // the fused kernel's tile scheduler starts from zero
  const int c = blockIdx.x * 4 + (threadIdx.x & 3), t = threadIdx.x >> 2;
  pos_t[(blockIdx.x * POS_LD + t) * 4 + (threadIdx.x & 3)] = t < n_tok ? pos[t * DIM + c] : 0.f;
}

int sm_count_cached() { return sm_count_of_current_device(); }

}  // namespace

int fused_set_trap_buffer(void* host_mapped_words) {
  unsigned* p = static_cast<unsigned*>(host_mapped_words);
  AVF_CUDA(cudaMemcpyToSymbol(g_trap_buffer, &p, sizeof(p)));
  return 0;
}

int fused_prof_read(unsigned long long* out64, int reset) {
#ifdef AVF_FUSED_PROF
  AVF_CUDA(cudaDeviceSynchronize());
  AVF_CUDA(cudaMemcpyFromSymbol(out64, g_prof, sizeof(unsigned long long) * 64));
  if (reset) {
    static unsigned long long zeros[64] = {0};
    AVF_CUDA(cudaMemcpyToSymbol(g_prof, zeros, sizeof(zeros)));
  }
  return 0;
#else
  (void)out64; (void)reset;
  return AVF_EUNSUPPORTED;
#endif
}

bool encoder_fused_supported(const avf_stack_shape* s) {
  return (s->dim == 256 || s->dim == 128) && s->heads == HEADS && s->dim_head == DH && s->mlp_dim % 128 == 0 && s->mlp_dim >= 128 && s->mlp_dim <= MAX_MLP && s->n_tok >= 1 &&
         s->n_tok <= 64 && s->depth >= 1 && s->depth <= MAX_DEPTH;
}

// io_kind 0: in/out are NCHW bf16 maps [n_seq, 256, n_tok] (pos required, dim 256); 1: fp32 token rows with strides ld_in / ld_out,
// pos [n_tok, dim] optional, out == nullptr only with w_last (n_tok 12: AU logits [n_seq, 21] and decisions [n_seq, 12] instead of rows).
size_t encoder_fused_scratch_bytes() { return size_t(DIM) * POS_LD * sizeof(float) + 64; }      // positional table + the tile scheduler's counter

int encoder_fused(int io_kind, const avf_stack_shape* s, const avf_layer_weights* L, const void* in, int ld_in, void* out, int ld_out,
                  const float* pos, void* scratch, const float* w_last, float* out21, int* decisions, cudaStream_t st) {
  AVF_REQUIRE(encoder_fused_supported(s), AVF_EUNSUPPORTED, "fused encoder: unsupported shape dim=%d heads=%d dh=%d mlp=%d n_tok=%d depth=%d",
              s->dim, s->heads, s->dim_head, s->mlp_dim, s->n_tok, s->depth);
  AVF_REQUIRE(io_kind == IO_ROWS_F32 || (pos != nullptr && scratch != nullptr), AVF_EINVAL,
              "fused encoder: NCHW input needs the positional embedding and the scratch buffer");
  AVF_REQUIRE(io_kind == IO_ROWS_F32 || s->dim == DIM, AVF_EUNSUPPORTED, "fused encoder: the NCHW form is dim %d only", DIM);
  AVF_REQUIRE(io_kind == IO_NCHW_BF16 || (ld_in % 4 == 0 && (out == nullptr || ld_out % 4 == 0)), AVF_EINVAL, "fused encoder: row strides must be multiples of 4");
  AVF_REQUIRE(w_last == nullptr || (io_kind == IO_ROWS_F32 && s->n_tok == 12), AVF_EINVAL, "fused encoder: AU logits need 12-token rows");
  AVF_REQUIRE(out != nullptr || w_last != nullptr, AVF_EINVAL, "fused encoder: no output");
  static thread_local FusedArgs a;      // ~2 KB of tensor maps + pointers, passed by value (__grid_constant__) per launch
  static_assert(sizeof(FusedArgs) <= 4000, "kernel parameter space");
  a.in = in; a.out = out; a.pos = pos; a.pos_t = static_cast<const float*>(scratch); a.ld_in = ld_in; a.ld_out = ld_out;
  a.w_last = w_last; a.out21 = out21; a.decisions = decisions;
  a.tile_counter = nullptr;     // fp32 rows: static striding
  if (io_kind == IO_NCHW_BF16) {
    a.tile_counter = reinterpret_cast<int*>(static_cast<uint8_t*>(scratch) + size_t(DIM) * POS_LD * sizeof(float));
    launch_pdl(pos_transpose_kernel, DIM / 4, 256, 0, st, pos, static_cast<float*>(scratch), s->n_tok, a.tile_counter);
    AVF_LAUNCH_CHECK("pos_transpose_kernel");
  }
  a.n_seq = s->n_seq; a.n_tok = s->n_tok;
  a.slot = 16; a.slot_log2 = 4;
  while (a.slot < s->n_tok) { a.slot *= 2; ++a.slot_log2; }
  a.spt = 128 / a.slot;
  a.n_tiles = ceil_div(s->n_seq, a.spt);
  a.n_chunks = s->mlp_dim / 128; a.depth = s->depth;
  const int inner = HEADS * DH, D = s->dim;
  for (int l = 0; l < s->depth; ++l) {
    LayerArgs& A = a.layer[l];
    int e;
    if ((e = make_tmap_bf16_2d(&A.tm_qkv, L[l].w_qkv, 3 * inner, D, D, 32))) return e;
    if ((e = make_tmap_bf16_2d(&A.tm_out, L[l].w_out, D, inner, inner, D, DH))) return e;      // box [D rows x 32 cols]
    if ((e = make_tmap_bf16_2d(&A.tm_w1, L[l].w_ff1, s->mlp_dim, D, D, 128))) return e;
    if ((e = make_tmap_bf16_2d(&A.tm_w2, L[l].w_ff2, D, s->mlp_dim, s->mlp_dim, 128))) return e;
    A.ln1_g = L[l].ln1_gamma; A.ln1_b = L[l].ln1_beta; A.b_out = L[l].b_out;
    A.ln2_g = L[l].ln2_gamma; A.ln2_b = L[l].ln2_beta; A.b_ff1 = L[l].b_ff1; A.b_ff2 = L[l].b_ff2;
  }
  static PerDeviceOnce once;
  if (once.first()) {
    AVF_CUDA(cudaFuncSetAttribute(encoder_fused_kernel<IO_NCHW_BF16, 49, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_ALLOC));
    AVF_CUDA(cudaFuncSetAttribute(encoder_fused_kernel<IO_NCHW_BF16, 0, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_ALLOC));
    AVF_CUDA(cudaFuncSetAttribute(encoder_fused_kernel<IO_ROWS_F32, 0, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_ALLOC));
    AVF_CUDA(cudaFuncSetAttribute(encoder_fused_kernel<IO_ROWS_F32, 0, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_ALLOC));
  }
  const int cap = sm_cap();
  const int grid = min(a.n_tiles, cap > 0 ? min(cap, sm_count_cached()) : sm_count_cached());
  if (io_kind == IO_NCHW_BF16 && a.n_tok == 49)     // the SFormer's 7 x 7 maps: compile-time geometry
    launch_pdl(encoder_fused_kernel<IO_NCHW_BF16, 49, 256>, grid, NUM_THREADS, SMEM_ALLOC, st, a);
  else if (io_kind == IO_NCHW_BF16)
    launch_pdl(encoder_fused_kernel<IO_NCHW_BF16, 0, 256>, grid, NUM_THREADS, SMEM_ALLOC, st, a);
  else if (D == 256)
    launch_pdl(encoder_fused_kernel<IO_ROWS_F32, 0, 256>, grid, NUM_THREADS, SMEM_ALLOC, st, a);
  else
    launch_pdl(encoder_fused_kernel<IO_ROWS_F32, 0, 128>, grid, NUM_THREADS, SMEM_ALLOC, st, a);
  AVF_LAUNCH_CHECK("encoder_fused_kernel");
  return 0;
}

}  // namespace avf
