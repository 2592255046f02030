// Small-sequence attention on the tensor cores (bf16 in/out, fp32 softmax), models/heads.py:221-237.
//
// Sequences on this path are 9..49 tokens with 32- or 64-wide heads: one (sequence, head) problem is a
// handful of 16x8x16 MMAs, far below a 128-row tcgen05 tile, so each WARP owns one problem and keeps the
// whole score matrix in registers (flash-style: S never touches memory).  K and V of the head are staged in
// a per-warp padded shared-memory slab (conflict-free fragment loads / ldmatrix.trans); Q fragments come
// straight from global memory.  qkv [rows, 3*H*dh] with columns q|k|v head-major; out [rows, H*dh].
// (The 49-token SFormer additionally has a fully fused tcgen05 path; this kernel serves every stack.)
// Sequences of 65..256 tokens with 64-wide heads (long TFormer clips) take the CTA-per-problem kernels further down.
#include "avf_common.cuh"
#include "avf_internal.h"

namespace avf {

namespace {

__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void ldmatrix_x2_trans(uint32_t& r0, uint32_t& r1, const void* smem_row_ptr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(smem_u32(smem_row_ptr)));
}

// 4 x 4 transpose of 32-bit words inside every quad of lanes: lane t enters with words 0..3 of ITS 16-byte chunk and leaves
// with word t of the chunks of lanes 0..3 (and back: the transpose is its own inverse).
__device__ __forceinline__ void quad_transpose32(uint32_t (&p)[4], int lane) {
  const bool b0 = lane & 1, b1 = lane & 2;
  uint32_t r;
  r = __shfl_xor_sync(0xffffffffu, b0 ? p[0] : p[1], 1); if (b0) p[0] = r; else p[1] = r;
  r = __shfl_xor_sync(0xffffffffu, b0 ? p[2] : p[3], 1); if (b0) p[2] = r; else p[3] = r;
  r = __shfl_xor_sync(0xffffffffu, b1 ? p[0] : p[2], 2); if (b1) p[0] = r; else p[2] = r;
  r = __shfl_xor_sync(0xffffffffu, b1 ? p[1] : p[3], 2); if (b1) p[1] = r; else p[3] = r;
}

// Keep bits of one sequence (bit j = token j is kept; bits >= n_tok are 0) from its keep row of <= 64 bytes: two ballots of the warp.
__device__ __forceinline__ uint64_t keep_bits(const uint8_t* __restrict__ row, int n_tok, int lane) {
  const uint32_t lo = __ballot_sync(0xffffffffu, lane < n_tok && row[lane] != 0);
  const uint32_t hi = __ballot_sync(0xffffffffu, lane + 32 < n_tok && row[lane + 32] != 0);
  return (uint64_t(hi) << 32) | lo;
}

// Masked score (query kept: row_kept, key column c): a kept query keeps the scores of kept keys and gets -INF on dropped keys, like on
// the padding columns c >= n_tok; a dropped query gets the same score 0 on every real key, i.e. the uniform row that masked_fill with
// -finfo.max gives (and no -INF - (-INF) in the exp).
__device__ __forceinline__ float mask_score(float s, bool row_kept, uint64_t km, int c, int n_tok) {
  if (c >= n_tok) return -INFINITY;
  if (!row_kept) return 0.f;
  return ((km >> c) & 1) ? s : -INFINITY;
}

// MASKED: keep [n_seq, n_tok] uint8 (1 = keep) masks score (i, j) unless tokens i and j are both kept (mask_score).
// PROBS: also write the softmax probabilities exp2(s - m) / l in fp32 (before P is rounded to bf16 for P V) to probs
// [n_seq, heads, n_tok, n_tok]; every query row is computed (the map is full) while O is still stored for the first q_rows rows only.
template <int DH, int NP, bool MASKED, bool PROBS>    // NP = tokens padded to a multiple of 16 (16 / 32 / 48 / 64)
__global__ void __launch_bounds__(DH == 32 ? 128 : 64) attention_mma_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out,
                                                            int n_problems, int n_tok, int heads, float scale_log2e, int q_rows,
                                                            const uint8_t* __restrict__ keep, float* __restrict__ probs) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  // q_rows: only the first q_rows query rows of every sequence are computed and written (compactly: out [n_seq * q_rows, inner]);
  // q_rows = n_tok is plain self-attention, q_rows = 1 is the TFormer's last layer, of which only the cls row is consumed.
  constexpr int PITCH = DH + 8;                       // elements; (DH*2+16) bytes keeps 8 consecutive rows on distinct banks
  constexpr int WARPS = DH == 32 ? 4 : 2;             // keeps the static slab under 48 KB
  __shared__ __align__(16) __nv_bfloat16 smem[WARPS][2][NP][PITCH];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int prob = blockIdx.x * WARPS + warp;         // = seq * heads + head
  if (prob >= n_problems) return;
  const int seq = prob / heads, head = prob - seq * heads;
  const int inner = heads * DH;
  const size_t row0 = size_t(seq) * n_tok;
  const __nv_bfloat16* base = qkv + row0 * (3 * inner) + head * DH;
  __nv_bfloat16 (*Ks)[PITCH] = smem[warp][0];
  __nv_bfloat16 (*Vs)[PITCH] = smem[warp][1];
  uint64_t km = 0;
  if constexpr (MASKED) km = keep_bits(keep + row0, n_tok, lane);

  // stage K and V (zero rows beyond n_tok: 0 * garbage must not become NaN in P*V)
  constexpr int CH = DH / 8;                          // 16-byte chunks per row
  // (all global loads are issued before the first shared-memory store: the warp has nothing else to hide their latency with)
  constexpr int NLD = NP * CH / 32;
  static_assert(NP * CH % 32 == 0, "whole warps of 16-byte chunks");
  uint4 kreg[NLD], vreg[NLD];
#pragma unroll
  for (int u = 0; u < NLD; ++u) {
    const int i = lane + u * 32, r = i / CH, c = i - r * CH;
    kreg[u] = make_uint4(0, 0, 0, 0);
    vreg[u] = make_uint4(0, 0, 0, 0);
    if (r < n_tok) {
      const __nv_bfloat16* p = base + size_t(r) * (3 * inner) + c * 8;
      kreg[u] = *reinterpret_cast<const uint4*>(p + inner);
      vreg[u] = *reinterpret_cast<const uint4*>(p + 2 * inner);
    }
  }
#pragma unroll
  for (int u = 0; u < NLD; ++u) {
    const int i = lane + u * 32, r = i / CH, c = i - r * CH;
    *reinterpret_cast<uint4*>(&Ks[r][c * 8]) = kreg[u];
    *reinterpret_cast<uint4*>(&Vs[r][c * 8]) = vreg[u];
  }
  __syncwarp();

  const int g = lane >> 2, t = lane & 3;
#pragma unroll 1
  for (int mt = 0; mt < NP / 16; ++mt) {
    if (mt * 16 >= (PROBS ? n_tok : q_rows)) break;
    const int r_lo = mt * 16 + g, r_hi = r_lo + 8;
    // Q fragments (A operand, row-major 16x16 per k-step) from global: lane t of a quad fetches the 16-byte chunks t, t+4, ... of
    // its two rows (the quad reads 64 contiguous bytes per row and instruction instead of 4 x 4 bytes), then the quad transposes
    // 4-byte pieces so that every lane holds columns 2t, 2t+1 of each 8-column chunk — the m16n8k16 A layout.
    uint32_t qf[DH / 16][4];
#pragma unroll
    for (int grp = 0; grp < DH / 32; ++grp) {
      uint32_t lo[4] = {0u, 0u, 0u, 0u}, hi[4] = {0u, 0u, 0u, 0u};
      if (r_lo < n_tok) {
        const uint4 v = *reinterpret_cast<const uint4*>(base + size_t(r_lo) * (3 * inner) + (grp * 4 + t) * 8);
        lo[0] = v.x; lo[1] = v.y; lo[2] = v.z; lo[3] = v.w;
      }
      if (r_hi < n_tok) {
        const uint4 v = *reinterpret_cast<const uint4*>(base + size_t(r_hi) * (3 * inner) + (grp * 4 + t) * 8);
        hi[0] = v.x; hi[1] = v.y; hi[2] = v.z; hi[3] = v.w;
      }
      quad_transpose32(lo, lane);
      quad_transpose32(hi, lane);
#pragma unroll
      for (int j = 0; j < 4; ++j) {               // piece t of chunk grp*4 + j = columns (grp*4 + j)*8 + 2t, +1
        const int ks = (grp * 4 + j) >> 1, half = (grp * 4 + j) & 1;
        qf[ks][half * 2] = lo[j];
        qf[ks][half * 2 + 1] = hi[j];
      }
    }
    // S = Q K^T  (B fragment: B[k][n] = K[n][k] -> one 32-bit load per register)
    float s[NP / 8][4];
#pragma unroll
    for (int nt = 0; nt < NP / 8; ++nt) {
      s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) {
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(&Ks[nt * 8 + g][ks * 16 + 2 * t]);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(&Ks[nt * 8 + g][ks * 16 + 8 + 2 * t]);
        mma_bf16_16816(s[nt], qf[ks], b0, b1);
      }
    }
    // softmax over keys, rows r_lo (regs 0,1) and r_hi (regs 2,3); columns >= n_tok masked
    float m_lo = -INFINITY, m_hi = -INFINITY;
    const bool k_lo = (km >> r_lo) & 1, k_hi = (km >> r_hi) & 1;
#pragma unroll
    for (int nt = 0; nt < NP / 8; ++nt) {
      const int c = nt * 8 + 2 * t;
      if constexpr (MASKED) {
        s[nt][0] = mask_score(s[nt][0], k_lo, km, c, n_tok); s[nt][1] = mask_score(s[nt][1], k_lo, km, c + 1, n_tok);
        s[nt][2] = mask_score(s[nt][2], k_hi, km, c, n_tok); s[nt][3] = mask_score(s[nt][3], k_hi, km, c + 1, n_tok);
      } else {
        if (c >= n_tok) { s[nt][0] = -INFINITY; s[nt][2] = -INFINITY; }
        if (c + 1 >= n_tok) { s[nt][1] = -INFINITY; s[nt][3] = -INFINITY; }
      }
      m_lo = fmaxf(m_lo, fmaxf(s[nt][0], s[nt][1]));
      m_hi = fmaxf(m_hi, fmaxf(s[nt][2], s[nt][3]));
    }
    m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 1));
    m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 2));
    m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 1));
    m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 2));
    const float o_lo = m_lo * scale_log2e, o_hi = m_hi * scale_log2e;
    float l_lo = 0.f, l_hi = 0.f;
#pragma unroll
    for (int nt = 0; nt < NP / 8; ++nt) {
      s[nt][0] = exp2f(fmaf(s[nt][0], scale_log2e, -o_lo));
      s[nt][1] = exp2f(fmaf(s[nt][1], scale_log2e, -o_lo));
      s[nt][2] = exp2f(fmaf(s[nt][2], scale_log2e, -o_hi));
      s[nt][3] = exp2f(fmaf(s[nt][3], scale_log2e, -o_hi));
      l_lo += s[nt][0] + s[nt][1];
      l_hi += s[nt][2] + s[nt][3];
    }
    l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 1);
    l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 2);
    l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 1);
    l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 2);
    if constexpr (PROBS) {
      float* p_lo = probs + (size_t(prob) * n_tok + r_lo) * n_tok;
      float* p_hi = p_lo + size_t(8) * n_tok;
#pragma unroll
      for (int nt = 0; nt < NP / 8; ++nt) {
        const int c = nt * 8 + 2 * t;
        if (r_lo < n_tok && c < n_tok) p_lo[c] = s[nt][0] / l_lo;
        if (r_lo < n_tok && c + 1 < n_tok) p_lo[c + 1] = s[nt][1] / l_lo;
        if (r_hi < n_tok && c < n_tok) p_hi[c] = s[nt][2] / l_hi;
        if (r_hi < n_tok && c + 1 < n_tok) p_hi[c + 1] = s[nt][3] / l_hi;
      }
    }
    // O = P V : the C fragments of two adjacent score tiles are exactly one A fragment
    float o[DH / 8][4];
#pragma unroll
    for (int nt = 0; nt < DH / 8; ++nt) o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.f;
#pragma unroll
    for (int kt = 0; kt < NP / 16; ++kt) {
      uint32_t pa[4];
      pa[0] = pack_bf16x2(s[2 * kt][0], s[2 * kt][1]);
      pa[1] = pack_bf16x2(s[2 * kt][2], s[2 * kt][3]);
      pa[2] = pack_bf16x2(s[2 * kt + 1][0], s[2 * kt + 1][1]);
      pa[3] = pack_bf16x2(s[2 * kt + 1][2], s[2 * kt + 1][3]);
#pragma unroll
      for (int nt = 0; nt < DH / 8; ++nt) {
        uint32_t b0, b1;
        ldmatrix_x2_trans(b0, b1, &Vs[kt * 16 + (lane & 15)][nt * 8]);
        mma_bf16_16816(o[nt], pa, b0, b1);
      }
    }
    const float i_lo = 1.f / l_lo, i_hi = 1.f / l_hi;
    __nv_bfloat16* olo = out + (size_t(seq) * q_rows + r_lo) * inner + head * DH;
    __nv_bfloat16* ohi = out + (size_t(seq) * q_rows + r_hi) * inner + head * DH;
#pragma unroll
    for (int grp = 0; grp < DH / 32; ++grp) {     // the same transpose backwards: lane t stores the whole 16-byte chunk grp*4 + t
      uint32_t lo[4], hi[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        lo[j] = pack_bf16x2(o[grp * 4 + j][0] * i_lo, o[grp * 4 + j][1] * i_lo);
        hi[j] = pack_bf16x2(o[grp * 4 + j][2] * i_hi, o[grp * 4 + j][3] * i_hi);
      }
      quad_transpose32(lo, lane);
      quad_transpose32(hi, lane);
      if (r_lo < q_rows) *reinterpret_cast<uint4*>(olo + (grp * 4 + t) * 8) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      if (r_hi < q_rows) *reinterpret_cast<uint4*>(ohi + (grp * 4 + t) * 8) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    }
  }
}

template <int DH, int NP, bool MASKED, bool PROBS>
int launch(const void* qkv, void* out, int n_seq, int n_tok, int heads, int q_rows, const uint8_t* keep, float* probs, cudaStream_t st) {
  const int n_problems = n_seq * heads;
  const float scale_log2e = 1.4426950408889634f / sqrtf(float(DH));
  constexpr int kWarps = DH == 32 ? 4 : 2;
  launch_pdl(attention_mma_kernel<DH, NP, MASKED, PROBS>, ceil_div(n_problems, kWarps), kWarps * 32, 0, st, static_cast<const __nv_bfloat16*>(qkv), static_cast<__nv_bfloat16*>(out),
                                                                      n_problems, n_tok, heads, scale_log2e, q_rows, keep, probs);
  AVF_LAUNCH_CHECK("attention_mma_kernel");
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Backward (training): dQ, dK, dV of one (sequence, head) per warp, all five contractions on mma.sync.
//   pass 1 (rows = queries): S = Q K^T -> P, dP = dO V^T, delta = rowsum(P o dP), dS = P o (dP - delta) / sqrt(dh),
//                            dQ = dS K; the softmax statistics (max, 1/sum) and delta go to shared memory;
//   pass 2 (rows = keys):    S^T = K Q^T -> P^T from the saved statistics, dP^T = V dO^T, dS^T likewise,
//                            dV = P^T dO,  dK = dS^T Q.
// Recomputing the scores in the transposed orientation keeps every A operand a row-major fragment straight out of the
// accumulator registers (no transposes through shared memory).  Q, K, V, dO of the head sit in per-warp padded slabs.
// ---------------------------------------------------------------------------------------------
template <int DH, int NP>
struct BwdCfg {
  static constexpr int PITCH = DH + 8;
  static constexpr int SLAB_BYTES = 4 * NP * PITCH * 2 + 3 * NP * 4;
  static constexpr int WARPS = SLAB_BYTES * 2 <= 46 * 1024 ? 2 : 1;
};

// MASKED: the scores are masked as in the forward (mask_score); dS is 0 wherever a score was filled, and the uniform P of a dropped
// query still carries its dO into dV.
// GMAP: pass 1 also writes the gradient map G = P o dP (fp32 P and fp32-accumulated dP, multiplied once in fp32) to gmap
// [n_seq, heads, n_tok, n_tok]; pass 1 visits every (query, key), and the stores are its only addition.
template <int DH, int NP, bool MASKED, bool GMAP>
__global__ void __launch_bounds__(BwdCfg<DH, NP>::WARPS * 32) attention_bwd_mma_kernel(const __nv_bfloat16* __restrict__ qkv,
                                                                                       const __nv_bfloat16* __restrict__ dout,
                                                                                       __nv_bfloat16* __restrict__ dqkv, int n_problems,
                                                                                       int n_tok, int heads, float scale,
                                                                                       const uint8_t* __restrict__ keep, float* __restrict__ gmap) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  using Cfg = BwdCfg<DH, NP>;
  constexpr int PITCH = Cfg::PITCH, WARPS = Cfg::WARPS;
  __shared__ __align__(16) __nv_bfloat16 smem[WARPS][4][NP][PITCH];
  __shared__ float stats[WARPS][3][NP];               // row max (in exp2 units), 1 / row sum, delta
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int prob = blockIdx.x * WARPS + warp;
  if (prob >= n_problems) return;
  const int seq = prob / heads, head = prob - seq * heads;
  const int inner = heads * DH;
  const size_t row0 = size_t(seq) * n_tok;
  const __nv_bfloat16* base = qkv + row0 * (3 * inner) + head * DH;
  const __nv_bfloat16* dobase = dout + row0 * inner + head * DH;
  __nv_bfloat16* dbase = dqkv + row0 * (3 * inner) + head * DH;
  __nv_bfloat16 (*Qs)[PITCH] = smem[warp][0];
  __nv_bfloat16 (*Ks)[PITCH] = smem[warp][1];
  __nv_bfloat16 (*Vs)[PITCH] = smem[warp][2];
  __nv_bfloat16 (*Os)[PITCH] = smem[warp][3];
  float* st_m = stats[warp][0];
  float* st_il = stats[warp][1];
  float* st_d = stats[warp][2];
  const float scale_log2e = scale * 1.4426950408889634f;
  uint64_t km = 0;
  if constexpr (MASKED) km = keep_bits(keep + row0, n_tok, lane);

  constexpr int CH = DH / 8;
  for (int i = lane; i < NP * CH; i += 32) {
    const int r = i / CH, c = i - r * CH;
    uint4 q = make_uint4(0, 0, 0, 0), k = q, v = q, o = q;
    if (r < n_tok) {
      const __nv_bfloat16* p = base + size_t(r) * (3 * inner) + c * 8;
      q = *reinterpret_cast<const uint4*>(p);
      k = *reinterpret_cast<const uint4*>(p + inner);
      v = *reinterpret_cast<const uint4*>(p + 2 * inner);
      o = *reinterpret_cast<const uint4*>(dobase + size_t(r) * inner + c * 8);
    }
    *reinterpret_cast<uint4*>(&Qs[r][c * 8]) = q;
    *reinterpret_cast<uint4*>(&Ks[r][c * 8]) = k;
    *reinterpret_cast<uint4*>(&Vs[r][c * 8]) = v;
    *reinterpret_cast<uint4*>(&Os[r][c * 8]) = o;
  }
  __syncwarp();

  const int g = lane >> 2, t = lane & 3;
  auto load_a = [&](uint32_t (&f)[DH / 16][4], __nv_bfloat16 (*M)[PITCH], int r_lo) {
#pragma unroll
    for (int ks = 0; ks < DH / 16; ++ks) {
      f[ks][0] = *reinterpret_cast<const uint32_t*>(&M[r_lo][ks * 16 + 2 * t]);
      f[ks][1] = *reinterpret_cast<const uint32_t*>(&M[r_lo + 8][ks * 16 + 2 * t]);
      f[ks][2] = *reinterpret_cast<const uint32_t*>(&M[r_lo][ks * 16 + 8 + 2 * t]);
      f[ks][3] = *reinterpret_cast<const uint32_t*>(&M[r_lo + 8][ks * 16 + 8 + 2 * t]);
    }
  };
  // C[16 x NP] = A (fragments of 16 rows) * M^T  with M [NP x DH] row-major in shared memory
  auto mma_abt = [&](float (&c)[NP / 8][4], const uint32_t (&a)[DH / 16][4], __nv_bfloat16 (*M)[PITCH]) {
#pragma unroll
    for (int nt = 0; nt < NP / 8; ++nt) {
      c[nt][0] = c[nt][1] = c[nt][2] = c[nt][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) {
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(&M[nt * 8 + g][ks * 16 + 2 * t]);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(&M[nt * 8 + g][ks * 16 + 8 + 2 * t]);
        mma_bf16_16816(c[nt], a[ks], b0, b1);
      }
    }
  };
  // D[16 x DH] = X[16 x NP] (fp32 accumulator-layout registers, rounded to bf16) * M [NP x DH]
  auto mma_xm = [&](float (&d)[DH / 8][4], const float (&x)[NP / 8][4], __nv_bfloat16 (*M)[PITCH]) {
#pragma unroll
    for (int nt = 0; nt < DH / 8; ++nt) d[nt][0] = d[nt][1] = d[nt][2] = d[nt][3] = 0.f;
#pragma unroll
    for (int kt = 0; kt < NP / 16; ++kt) {
      uint32_t pa[4];
      pa[0] = pack_bf16x2(x[2 * kt][0], x[2 * kt][1]);
      pa[1] = pack_bf16x2(x[2 * kt][2], x[2 * kt][3]);
      pa[2] = pack_bf16x2(x[2 * kt + 1][0], x[2 * kt + 1][1]);
      pa[3] = pack_bf16x2(x[2 * kt + 1][2], x[2 * kt + 1][3]);
#pragma unroll
      for (int nt = 0; nt < DH / 8; ++nt) {
        uint32_t b0, b1;
        ldmatrix_x2_trans(b0, b1, &M[kt * 16 + (lane & 15)][nt * 8]);
        mma_bf16_16816(d[nt], pa, b0, b1);
      }
    }
  };
  auto store_rows = [&](const float (&d)[DH / 8][4], __nv_bfloat16* dst_col0, int r_lo, float mul) {
    __nv_bfloat16* lo = dst_col0 + size_t(r_lo) * (3 * inner) + 2 * t;
    __nv_bfloat16* hi = lo + size_t(8) * (3 * inner);
#pragma unroll
    for (int nt = 0; nt < DH / 8; ++nt) {
      if (r_lo < n_tok) *reinterpret_cast<uint32_t*>(lo + nt * 8) = pack_bf16x2(d[nt][0] * mul, d[nt][1] * mul);
      if (r_lo + 8 < n_tok) *reinterpret_cast<uint32_t*>(hi + nt * 8) = pack_bf16x2(d[nt][2] * mul, d[nt][3] * mul);
    }
  };

  // ---- pass 1: rows = queries ------------------------------------------------------------------------------
#pragma unroll 1
  for (int mt = 0; mt < NP / 16; ++mt) {
    if (mt * 16 >= n_tok) break;
    const int r_lo = mt * 16 + g;
    uint32_t af[DH / 16][4];
    float s[NP / 8][4], dp[NP / 8][4];
    load_a(af, Qs, r_lo);
    mma_abt(s, af, Ks);
    load_a(af, Os, r_lo);
    mma_abt(dp, af, Vs);
    float m_lo = -INFINITY, m_hi = -INFINITY;
    const bool k_lo = (km >> r_lo) & 1, k_hi = (km >> (r_lo + 8)) & 1;
#pragma unroll
    for (int nt = 0; nt < NP / 8; ++nt) {
      const int c = nt * 8 + 2 * t;
      if constexpr (MASKED) {
        s[nt][0] = mask_score(s[nt][0], k_lo, km, c, n_tok); s[nt][1] = mask_score(s[nt][1], k_lo, km, c + 1, n_tok);
        s[nt][2] = mask_score(s[nt][2], k_hi, km, c, n_tok); s[nt][3] = mask_score(s[nt][3], k_hi, km, c + 1, n_tok);
      } else {
        if (c >= n_tok) { s[nt][0] = -INFINITY; s[nt][2] = -INFINITY; }
        if (c + 1 >= n_tok) { s[nt][1] = -INFINITY; s[nt][3] = -INFINITY; }
      }
      m_lo = fmaxf(m_lo, fmaxf(s[nt][0], s[nt][1]));
      m_hi = fmaxf(m_hi, fmaxf(s[nt][2], s[nt][3]));
    }
    m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 1));
    m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 2));
    m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 1));
    m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 2));
    const float o_lo = m_lo * scale_log2e, o_hi = m_hi * scale_log2e;
    float l_lo = 0.f, l_hi = 0.f;
#pragma unroll
    for (int nt = 0; nt < NP / 8; ++nt) {
      s[nt][0] = exp2f(fmaf(s[nt][0], scale_log2e, -o_lo));
      s[nt][1] = exp2f(fmaf(s[nt][1], scale_log2e, -o_lo));
      s[nt][2] = exp2f(fmaf(s[nt][2], scale_log2e, -o_hi));
      s[nt][3] = exp2f(fmaf(s[nt][3], scale_log2e, -o_hi));
      l_lo += s[nt][0] + s[nt][1];
      l_hi += s[nt][2] + s[nt][3];
    }
    l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 1);
    l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 2);
    l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 1);
    l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 2);
    const float i_lo = 1.f / l_lo, i_hi = 1.f / l_hi;
    float d_lo = 0.f, d_hi = 0.f;
#pragma unroll
    for (int nt = 0; nt < NP / 8; ++nt) {
      s[nt][0] *= i_lo; s[nt][1] *= i_lo; s[nt][2] *= i_hi; s[nt][3] *= i_hi;
      d_lo += s[nt][0] * dp[nt][0] + s[nt][1] * dp[nt][1];
      d_hi += s[nt][2] * dp[nt][2] + s[nt][3] * dp[nt][3];
    }
    d_lo += __shfl_xor_sync(0xffffffffu, d_lo, 1);
    d_lo += __shfl_xor_sync(0xffffffffu, d_lo, 2);
    d_hi += __shfl_xor_sync(0xffffffffu, d_hi, 1);
    d_hi += __shfl_xor_sync(0xffffffffu, d_hi, 2);
    if constexpr (GMAP) {                      // s = P, dp = dP here; __fmul_rn keeps the product out of the FMAs of delta and dS
      float* g_lo = gmap + (size_t(prob) * n_tok + r_lo) * n_tok;
      float* g_hi = g_lo + size_t(8) * n_tok;
#pragma unroll
      for (int nt = 0; nt < NP / 8; ++nt) {
        const int c = nt * 8 + 2 * t;
        if (r_lo < n_tok && c < n_tok) g_lo[c] = __fmul_rn(s[nt][0], dp[nt][0]);
        if (r_lo < n_tok && c + 1 < n_tok) g_lo[c + 1] = __fmul_rn(s[nt][1], dp[nt][1]);
        if (r_lo + 8 < n_tok && c < n_tok) g_hi[c] = __fmul_rn(s[nt][2], dp[nt][2]);
        if (r_lo + 8 < n_tok && c + 1 < n_tok) g_hi[c + 1] = __fmul_rn(s[nt][3], dp[nt][3]);
      }
    }
    if (t == 0) {
      st_m[r_lo] = o_lo; st_il[r_lo] = i_lo; st_d[r_lo] = d_lo;
      st_m[r_lo + 8] = o_hi; st_il[r_lo + 8] = i_hi; st_d[r_lo + 8] = d_hi;
    }
#pragma unroll
    for (int nt = 0; nt < NP / 8; ++nt) {      // dS (the 1/sqrt(dh) is applied once when dQ is stored)
      s[nt][0] *= dp[nt][0] - d_lo; s[nt][1] *= dp[nt][1] - d_lo;
      s[nt][2] *= dp[nt][2] - d_hi; s[nt][3] *= dp[nt][3] - d_hi;
      if constexpr (MASKED) {                  // every score of a dropped query was filled
        if (!k_lo) s[nt][0] = s[nt][1] = 0.f;
        if (!k_hi) s[nt][2] = s[nt][3] = 0.f;
      }
    }
    float dq[DH / 8][4];
    mma_xm(dq, s, Ks);
    store_rows(dq, dbase, r_lo, scale);
  }
  __syncwarp();

  // ---- pass 2: rows = keys ------------------------------------------------------------------------------------
#pragma unroll 1
  for (int mt = 0; mt < NP / 16; ++mt) {
    if (mt * 16 >= n_tok) break;
    const int r_lo = mt * 16 + g;
    uint32_t af[DH / 16][4];
    float p[NP / 8][4], dp[NP / 8][4];
    load_a(af, Ks, r_lo);
    mma_abt(p, af, Qs);                       // S^T[key][query]
    load_a(af, Vs, r_lo);
    mma_abt(dp, af, Os);                      // dP^T[key][query]
    float ds[NP / 8][4];
    const bool k_lo = (km >> r_lo) & 1, k_hi = (km >> (r_lo + 8)) & 1;
#pragma unroll
    for (int nt = 0; nt < NP / 8; ++nt) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int qi = nt * 8 + 2 * t + e;    // query index of elements e (row r_lo) and e + 2 (row r_lo + 8)
        const bool ok = qi < n_tok;
        const float m = ok ? st_m[qi] : 0.f, il = ok ? st_il[qi] : 0.f, dl = ok ? st_d[qi] : 0.f;
        float p0, p1;
        if constexpr (MASKED) {               // dropped query: its uniform row 1 / n_tok (= il of pass 1) and dS = 0
          const bool qk = (km >> qi) & 1;
          p0 = ok ? exp2f(fmaf(qk ? (k_lo ? p[nt][e] : -INFINITY) : 0.f, scale_log2e, -m)) * il : 0.f;       // m = 0 on a dropped row
          p1 = ok ? exp2f(fmaf(qk ? (k_hi ? p[nt][e + 2] : -INFINITY) : 0.f, scale_log2e, -m)) * il : 0.f;
          ds[nt][e] = qk ? p0 * (dp[nt][e] - dl) : 0.f;
          ds[nt][e + 2] = qk ? p1 * (dp[nt][e + 2] - dl) : 0.f;
        } else {
          p0 = ok ? exp2f(fmaf(p[nt][e], scale_log2e, -m)) * il : 0.f;
          p1 = ok ? exp2f(fmaf(p[nt][e + 2], scale_log2e, -m)) * il : 0.f;
          ds[nt][e] = p0 * (dp[nt][e] - dl);
          ds[nt][e + 2] = p1 * (dp[nt][e + 2] - dl);
        }
        p[nt][e] = p0;
        p[nt][e + 2] = p1;
      }
    }
    float acc[DH / 8][4];
    mma_xm(acc, p, Os);                       // dV = P^T dO
    store_rows(acc, dbase + 2 * inner, r_lo, 1.f);
    mma_xm(acc, ds, Qs);                      // dK = dS^T Q / sqrt(dh)
    store_rows(acc, dbase + inner, r_lo, scale);
  }
}

template <int DH, int NP, bool MASKED, bool GMAP>
int launch_bwd(const void* qkv, const void* dout, void* dqkv, int n_seq, int n_tok, int heads, const uint8_t* keep, float* gmap, cudaStream_t st) {
  const int n_problems = n_seq * heads;
  constexpr int kWarps = BwdCfg<DH, NP>::WARPS;
  launch_pdl(attention_bwd_mma_kernel<DH, NP, MASKED, GMAP>, ceil_div(n_problems, kWarps), kWarps * 32, 0, st, static_cast<const __nv_bfloat16*>(qkv), static_cast<const __nv_bfloat16*>(dout), static_cast<__nv_bfloat16*>(dqkv), n_problems, n_tok, heads,
      1.0f / sqrtf(float(DH)), keep, gmap);
  AVF_LAUNCH_CHECK("attention_bwd_mma_kernel");
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Long sequences (65..256 tokens, 64-wide heads: the TFormer of long clips).  A whole score row no longer fits a warp's registers,
// so one CTA takes one (sequence, head): the head's operands sit in padded shared memory ([rows][72] bf16, rows padded to a
// multiple of 64 and zero-filled), warps own 16-row tiles and sweep 64-key blocks, and no warp holds more than a 16 x 64 tile.
// The rounding points are those of the kernels above: exact row max, exp2 against it, fp32 sums, P / dS rounded to bf16 for the
// MMA, O scaled by 1/l before its bf16 store.  Keep bits of up to 256 tokens are four 64-bit words in shared memory.
// ---------------------------------------------------------------------------------------------
constexpr int kLongDH = 64, kLongPitch = kLongDH + 8, kLongWarps = 8, kLongMaxTok = 256;
using LongRow = __nv_bfloat16[kLongPitch];

__host__ __device__ __forceinline__ int long_rows(int n_tok) { return (n_tok + 63) & ~63; }

// Keep bits of one sequence of up to 256 tokens into km[4] (bit j of word w = token 64 w + j is kept); warps 0..3 take a word each.
__device__ __forceinline__ void keep_words(const uint8_t* __restrict__ row, int n_tok, uint64_t* km, int warp, int lane) {
  if (warp < 4) {
    const int b = warp * 64;
    const uint64_t w = keep_bits(row + b, min(max(n_tok - b, 0), 64), lane);
    if (lane == 0) km[warp] = w;
  }
}
__device__ __forceinline__ bool keep_bit(const uint64_t* km, int i) { return (km[i >> 6] >> (i & 63)) & 1; }

// rows [0, n_tok) of the head's 64 columns starting at src (row stride ld elements) -> dst [long_rows(n_tok)][72], zero-filled
__device__ __forceinline__ void stage_rows(LongRow* dst, const __nv_bfloat16* __restrict__ src, size_t ld, int n_tok) {
  const int n = long_rows(n_tok) * (kLongDH / 8);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int r = i >> 3, c = (i & 7) * 8;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (r < n_tok) v = *reinterpret_cast<const uint4*>(src + size_t(r) * ld + c);
    *reinterpret_cast<uint4*>(&dst[r][c]) = v;
  }
}

// A fragments (16 rows from r_lo - g, 64 columns) of a row-major shared-memory matrix
__device__ __forceinline__ void long_load_a(uint32_t (&f)[4][4], const LongRow* M, int r_lo, int t) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    f[ks][0] = *reinterpret_cast<const uint32_t*>(&M[r_lo][ks * 16 + 2 * t]);
    f[ks][1] = *reinterpret_cast<const uint32_t*>(&M[r_lo + 8][ks * 16 + 2 * t]);
    f[ks][2] = *reinterpret_cast<const uint32_t*>(&M[r_lo][ks * 16 + 8 + 2 * t]);
    f[ks][3] = *reinterpret_cast<const uint32_t*>(&M[r_lo + 8][ks * 16 + 8 + 2 * t]);
  }
}
// C[16 x 64] = A * M[0:64]^T  (M: the block's 64 rows, row-major)
__device__ __forceinline__ void long_mma_abt(float (&c)[8][4], const uint32_t (&a)[4][4], const LongRow* M, int g, int t) {
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    c[nt][0] = c[nt][1] = c[nt][2] = c[nt][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint32_t b0 = *reinterpret_cast<const uint32_t*>(&M[nt * 8 + g][ks * 16 + 2 * t]);
      const uint32_t b1 = *reinterpret_cast<const uint32_t*>(&M[nt * 8 + g][ks * 16 + 8 + 2 * t]);
      mma_bf16_16816(c[nt], a[ks], b0, b1);
    }
  }
}
// D[16 x 64] += bf16(X[16 x 64]) * M[0:64]
__device__ __forceinline__ void long_mma_xm(float (&d)[8][4], const float (&x)[8][4], const LongRow* M, int lane) {
#pragma unroll
  for (int kt = 0; kt < 4; ++kt) {
    uint32_t pa[4];
    pa[0] = pack_bf16x2(x[2 * kt][0], x[2 * kt][1]);
    pa[1] = pack_bf16x2(x[2 * kt][2], x[2 * kt][3]);
    pa[2] = pack_bf16x2(x[2 * kt + 1][0], x[2 * kt + 1][1]);
    pa[3] = pack_bf16x2(x[2 * kt + 1][2], x[2 * kt + 1][3]);
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      uint32_t b0, b1;
      ldmatrix_x2_trans(b0, b1, &M[kt * 16 + (lane & 15)][nt * 8]);
      mma_bf16_16816(d[nt], pa, b0, b1);
    }
  }
}
// Scores of key block kb (columns c = kb*64 + local) masked like the short kernels: mask_score on the block's keep word.
template <bool MASKED>
__device__ __forceinline__ void long_mask(float (&s)[8][4], bool k_lo, bool k_hi, uint64_t kw, int n_left, int t) {
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const int c = nt * 8 + 2 * t;
    if constexpr (MASKED) {
      s[nt][0] = mask_score(s[nt][0], k_lo, kw, c, n_left); s[nt][1] = mask_score(s[nt][1], k_lo, kw, c + 1, n_left);
      s[nt][2] = mask_score(s[nt][2], k_hi, kw, c, n_left); s[nt][3] = mask_score(s[nt][3], k_hi, kw, c + 1, n_left);
    } else {
      if (c >= n_left) { s[nt][0] = -INFINITY; s[nt][2] = -INFINITY; }
      if (c + 1 >= n_left) { s[nt][1] = -INFINITY; s[nt][3] = -INFINITY; }
    }
  }
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}
// 16 x 64 fp32 tile * mul -> bf16 rows r_lo, r_lo + 8 (if < n_valid) of dst (row stride ld)
__device__ __forceinline__ void long_store(const float (&d)[8][4], __nv_bfloat16* dst, size_t ld, int r_lo, int n_valid, float mul_lo, float mul_hi,
                                           int t) {
  __nv_bfloat16* lo = dst + size_t(r_lo) * ld + 2 * t;
  __nv_bfloat16* hi = lo + 8 * ld;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    if (r_lo < n_valid) *reinterpret_cast<uint32_t*>(lo + nt * 8) = pack_bf16x2(d[nt][0] * mul_lo, d[nt][1] * mul_lo);
    if (r_lo + 8 < n_valid) *reinterpret_cast<uint32_t*>(hi + nt * 8) = pack_bf16x2(d[nt][2] * mul_hi, d[nt][3] * mul_hi);
  }
}

// Forward: two sweeps over the key blocks per 16-row query tile, the first for the exact row max, the second for exp2, l and P V.
// PROBS: l is known only after the second sweep, so a third sweep recomputes the masked scores and writes exp2(s - m) / l in fp32 to
// probs [n_seq, heads, n_tok, n_tok], each element once; every query row is computed while O is still stored for the first q_rows.
template <bool MASKED, bool PROBS>
__global__ void __launch_bounds__(kLongWarps * 32) attention_long_mma_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out,
                                                                            int n_tok, int heads, float scale_log2e, int q_rows,
                                                                            const uint8_t* __restrict__ keep, float* __restrict__ probs) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  extern __shared__ __align__(16) uint8_t smem_long[];
  const int NR = long_rows(n_tok);
  LongRow* Ks = reinterpret_cast<LongRow*>(smem_long);
  LongRow* Vs = Ks + NR;
  uint64_t* km = reinterpret_cast<uint64_t*>(Vs + NR);
  const int seq = blockIdx.x / heads, head = blockIdx.x - seq * heads;
  const int inner = heads * kLongDH, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t row0 = size_t(seq) * n_tok, ld = size_t(3) * inner;
  const __nv_bfloat16* base = qkv + row0 * ld + head * kLongDH;
  stage_rows(Ks, base + inner, ld, n_tok);
  stage_rows(Vs, base + 2 * inner, ld, n_tok);
  if constexpr (MASKED) keep_words(keep + row0, n_tok, km, warp, lane);
  __syncthreads();

  const int g = lane >> 2, t = lane & 3, nkb = NR / 64;
#pragma unroll 1
  for (int mt = warp; mt * 16 < (PROBS ? n_tok : q_rows); mt += kLongWarps) {
    const int r_lo = mt * 16 + g, r_hi = r_lo + 8;
    uint32_t qf[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c = ks * 16 + h * 8 + 2 * t;
        qf[ks][2 * h] = r_lo < n_tok ? *reinterpret_cast<const uint32_t*>(base + size_t(r_lo) * ld + c) : 0u;
        qf[ks][2 * h + 1] = r_hi < n_tok ? *reinterpret_cast<const uint32_t*>(base + size_t(r_hi) * ld + c) : 0u;
      }
    }
    const bool k_lo = MASKED && keep_bit(km, r_lo), k_hi = MASKED && keep_bit(km, r_hi);
    float s[8][4];
    float m_lo = -INFINITY, m_hi = -INFINITY;
#pragma unroll 1
    for (int kb = 0; kb < nkb; ++kb) {
      long_mma_abt(s, qf, Ks + kb * 64, g, t);
      long_mask<MASKED>(s, k_lo, k_hi, MASKED ? km[kb] : 0, n_tok - kb * 64, t);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        m_lo = fmaxf(m_lo, fmaxf(s[nt][0], s[nt][1]));
        m_hi = fmaxf(m_hi, fmaxf(s[nt][2], s[nt][3]));
      }
    }
    const float o_lo = quad_max(m_lo) * scale_log2e, o_hi = quad_max(m_hi) * scale_log2e;
    float l_lo = 0.f, l_hi = 0.f, o[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.f;
#pragma unroll 1
    for (int kb = 0; kb < nkb; ++kb) {
      long_mma_abt(s, qf, Ks + kb * 64, g, t);
      long_mask<MASKED>(s, k_lo, k_hi, MASKED ? km[kb] : 0, n_tok - kb * 64, t);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = exp2f(fmaf(s[nt][0], scale_log2e, -o_lo));
        s[nt][1] = exp2f(fmaf(s[nt][1], scale_log2e, -o_lo));
        s[nt][2] = exp2f(fmaf(s[nt][2], scale_log2e, -o_hi));
        s[nt][3] = exp2f(fmaf(s[nt][3], scale_log2e, -o_hi));
        l_lo += s[nt][0] + s[nt][1];
        l_hi += s[nt][2] + s[nt][3];
      }
      long_mma_xm(o, s, Vs + kb * 64, lane);
    }
    if constexpr (PROBS) {
      const float L_lo = quad_sum(l_lo), L_hi = quad_sum(l_hi);
      float* p_lo = probs + (size_t(blockIdx.x) * n_tok + r_lo) * n_tok;
      float* p_hi = p_lo + size_t(8) * n_tok;
#pragma unroll 1
      for (int kb = 0; kb < nkb; ++kb) {
        long_mma_abt(s, qf, Ks + kb * 64, g, t);
        long_mask<MASKED>(s, k_lo, k_hi, MASKED ? km[kb] : 0, n_tok - kb * 64, t);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const int c = kb * 64 + nt * 8 + 2 * t;
          if (r_lo < n_tok && c < n_tok) p_lo[c] = exp2f(fmaf(s[nt][0], scale_log2e, -o_lo)) / L_lo;
          if (r_lo < n_tok && c + 1 < n_tok) p_lo[c + 1] = exp2f(fmaf(s[nt][1], scale_log2e, -o_lo)) / L_lo;
          if (r_hi < n_tok && c < n_tok) p_hi[c] = exp2f(fmaf(s[nt][2], scale_log2e, -o_hi)) / L_hi;
          if (r_hi < n_tok && c + 1 < n_tok) p_hi[c + 1] = exp2f(fmaf(s[nt][3], scale_log2e, -o_hi)) / L_hi;
        }
      }
    }
    long_store(o, out + size_t(seq) * q_rows * inner + head * kLongDH, inner, r_lo, q_rows, 1.f / quad_sum(l_lo), 1.f / quad_sum(l_hi), t);
  }
}

// Backward, the two passes of attention_bwd_mma_kernel with Q, K, V, dO of the (sequence, head) in shared memory:
//   pass 1 (rows = queries): sweep 1 the row max, sweep 2 l and sum_j e_j dP_j (delta = that / l), sweep 3 dS and dQ = dS K;
//   pass 2 (rows = keys): one sweep over 64-query blocks, P^T and dS^T from the saved statistics, dV = P^T dO, dK = dS^T Q.
// GMAP: sweep 3 of pass 1, which visits every (query, key) with P and dP in registers, also writes G = P o dP in fp32 to gmap
// [n_seq, heads, n_tok, n_tok].
template <bool MASKED, bool GMAP>
__global__ void __launch_bounds__(kLongWarps * 32) attention_bwd_long_mma_kernel(const __nv_bfloat16* __restrict__ qkv,
                                                                                const __nv_bfloat16* __restrict__ dout,
                                                                                __nv_bfloat16* __restrict__ dqkv, int n_tok, int heads,
                                                                                float scale, const uint8_t* __restrict__ keep,
                                                                                float* __restrict__ gmap) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  extern __shared__ __align__(16) uint8_t smem_long[];
  const int NR = long_rows(n_tok);
  LongRow* Qs = reinterpret_cast<LongRow*>(smem_long);
  LongRow* Ks = Qs + NR;
  LongRow* Vs = Ks + NR;
  LongRow* Os = Vs + NR;
  float* st_m = reinterpret_cast<float*>(Os + NR);      // row max (exp2 units), 1 / row sum, delta
  float* st_il = st_m + NR;
  float* st_d = st_il + NR;
  uint64_t* km = reinterpret_cast<uint64_t*>(st_d + NR);
  const int seq = blockIdx.x / heads, head = blockIdx.x - seq * heads;
  const int inner = heads * kLongDH, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t row0 = size_t(seq) * n_tok, ld = size_t(3) * inner;
  const __nv_bfloat16* base = qkv + row0 * ld + head * kLongDH;
  __nv_bfloat16* dbase = dqkv + row0 * ld + head * kLongDH;
  stage_rows(Qs, base, ld, n_tok);
  stage_rows(Ks, base + inner, ld, n_tok);
  stage_rows(Vs, base + 2 * inner, ld, n_tok);
  stage_rows(Os, dout + row0 * inner + head * kLongDH, inner, n_tok);
  if constexpr (MASKED) keep_words(keep + row0, n_tok, km, warp, lane);
  __syncthreads();
  const float scale_log2e = scale * 1.4426950408889634f;
  const int g = lane >> 2, t = lane & 3, nkb = NR / 64;

  // ---- pass 1: rows = queries ------------------------------------------------------------------------------
#pragma unroll 1
  for (int mt = warp; mt * 16 < n_tok; mt += kLongWarps) {
    const int r_lo = mt * 16 + g, r_hi = r_lo + 8;
    uint32_t qf[4][4], of[4][4];
    long_load_a(qf, Qs, r_lo, t);
    long_load_a(of, Os, r_lo, t);
    const bool k_lo = MASKED && keep_bit(km, r_lo), k_hi = MASKED && keep_bit(km, r_hi);
    float s[8][4], dp[8][4];
    float m_lo = -INFINITY, m_hi = -INFINITY;
#pragma unroll 1
    for (int kb = 0; kb < nkb; ++kb) {
      long_mma_abt(s, qf, Ks + kb * 64, g, t);
      long_mask<MASKED>(s, k_lo, k_hi, MASKED ? km[kb] : 0, n_tok - kb * 64, t);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        m_lo = fmaxf(m_lo, fmaxf(s[nt][0], s[nt][1]));
        m_hi = fmaxf(m_hi, fmaxf(s[nt][2], s[nt][3]));
      }
    }
    const float o_lo = quad_max(m_lo) * scale_log2e, o_hi = quad_max(m_hi) * scale_log2e;
    float l_lo = 0.f, l_hi = 0.f, e_lo = 0.f, e_hi = 0.f;
#pragma unroll 1
    for (int kb = 0; kb < nkb; ++kb) {
      long_mma_abt(s, qf, Ks + kb * 64, g, t);
      long_mask<MASKED>(s, k_lo, k_hi, MASKED ? km[kb] : 0, n_tok - kb * 64, t);
      long_mma_abt(dp, of, Vs + kb * 64, g, t);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const float a0 = exp2f(fmaf(s[nt][0], scale_log2e, -o_lo)), a1 = exp2f(fmaf(s[nt][1], scale_log2e, -o_lo));
        const float a2 = exp2f(fmaf(s[nt][2], scale_log2e, -o_hi)), a3 = exp2f(fmaf(s[nt][3], scale_log2e, -o_hi));
        l_lo += a0 + a1;
        l_hi += a2 + a3;
        e_lo += a0 * dp[nt][0] + a1 * dp[nt][1];
        e_hi += a2 * dp[nt][2] + a3 * dp[nt][3];
      }
    }
    const float i_lo = 1.f / quad_sum(l_lo), i_hi = 1.f / quad_sum(l_hi);
    const float d_lo = quad_sum(e_lo) * i_lo, d_hi = quad_sum(e_hi) * i_hi;
    if (t == 0) {
      st_m[r_lo] = o_lo; st_il[r_lo] = i_lo; st_d[r_lo] = d_lo;
      st_m[r_hi] = o_hi; st_il[r_hi] = i_hi; st_d[r_hi] = d_hi;
    }
    float dq[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) dq[nt][0] = dq[nt][1] = dq[nt][2] = dq[nt][3] = 0.f;
#pragma unroll 1
    for (int kb = 0; kb < nkb; ++kb) {
      long_mma_abt(s, qf, Ks + kb * 64, g, t);
      long_mask<MASKED>(s, k_lo, k_hi, MASKED ? km[kb] : 0, n_tok - kb * 64, t);
      long_mma_abt(dp, of, Vs + kb * 64, g, t);
      if constexpr (GMAP) {                    // the P of the dS below (the same expression), times dP
        float* g_lo = gmap + (size_t(blockIdx.x) * n_tok + r_lo) * n_tok + kb * 64;
        float* g_hi = g_lo + size_t(8) * n_tok;
        const int cols = n_tok - kb * 64;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const int c = nt * 8 + 2 * t;
          const float p0 = exp2f(fmaf(s[nt][0], scale_log2e, -o_lo)) * i_lo, p1 = exp2f(fmaf(s[nt][1], scale_log2e, -o_lo)) * i_lo;
          const float p2 = exp2f(fmaf(s[nt][2], scale_log2e, -o_hi)) * i_hi, p3 = exp2f(fmaf(s[nt][3], scale_log2e, -o_hi)) * i_hi;
          if (r_lo < n_tok && c < cols) g_lo[c] = __fmul_rn(p0, dp[nt][0]);
          if (r_lo < n_tok && c + 1 < cols) g_lo[c + 1] = __fmul_rn(p1, dp[nt][1]);
          if (r_hi < n_tok && c < cols) g_hi[c] = __fmul_rn(p2, dp[nt][2]);
          if (r_hi < n_tok && c + 1 < cols) g_hi[c + 1] = __fmul_rn(p3, dp[nt][3]);
        }
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {        // dS (the 1/sqrt(dh) is applied once when dQ is stored)
        s[nt][0] = exp2f(fmaf(s[nt][0], scale_log2e, -o_lo)) * i_lo * (dp[nt][0] - d_lo);
        s[nt][1] = exp2f(fmaf(s[nt][1], scale_log2e, -o_lo)) * i_lo * (dp[nt][1] - d_lo);
        s[nt][2] = exp2f(fmaf(s[nt][2], scale_log2e, -o_hi)) * i_hi * (dp[nt][2] - d_hi);
        s[nt][3] = exp2f(fmaf(s[nt][3], scale_log2e, -o_hi)) * i_hi * (dp[nt][3] - d_hi);
        if constexpr (MASKED) {                // every score of a dropped query was filled
          if (!k_lo) s[nt][0] = s[nt][1] = 0.f;
          if (!k_hi) s[nt][2] = s[nt][3] = 0.f;
        }
      }
      long_mma_xm(dq, s, Ks + kb * 64, lane);
    }
    long_store(dq, dbase, ld, r_lo, n_tok, scale, scale, t);
  }
  __syncthreads();

  // ---- pass 2: rows = keys ------------------------------------------------------------------------------------
#pragma unroll 1
  for (int mt = warp; mt * 16 < n_tok; mt += kLongWarps) {
    const int r_lo = mt * 16 + g;
    uint32_t kf[4][4], vf[4][4];
    long_load_a(kf, Ks, r_lo, t);
    long_load_a(vf, Vs, r_lo, t);
    const bool k_lo = MASKED && keep_bit(km, r_lo), k_hi = MASKED && keep_bit(km, r_lo + 8);
    float dv[8][4], dk[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) dv[nt][0] = dv[nt][1] = dv[nt][2] = dv[nt][3] = dk[nt][0] = dk[nt][1] = dk[nt][2] = dk[nt][3] = 0.f;
#pragma unroll 1
    for (int qb = 0; qb < nkb; ++qb) {
      float p[8][4], ds[8][4];
      long_mma_abt(p, kf, Qs + qb * 64, g, t);        // S^T[key][query]
      long_mma_abt(ds, vf, Os + qb * 64, g, t);       // dP^T[key][query]
      const uint64_t qw = MASKED ? km[qb] : 0;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int ql = nt * 8 + 2 * t + e, qi = qb * 64 + ql;     // query of elements e (row r_lo) and e + 2 (row r_lo + 8)
          const bool ok = qi < n_tok;
          const float m = ok ? st_m[qi] : 0.f, il = ok ? st_il[qi] : 0.f, dl = ok ? st_d[qi] : 0.f;
          float p0, p1;
          if constexpr (MASKED) {             // dropped query: its uniform row 1 / n_tok (= il of pass 1) and dS = 0
            const bool qk = (qw >> ql) & 1;
            p0 = ok ? exp2f(fmaf(qk ? (k_lo ? p[nt][e] : -INFINITY) : 0.f, scale_log2e, -m)) * il : 0.f;       // m = 0 on a dropped row
            p1 = ok ? exp2f(fmaf(qk ? (k_hi ? p[nt][e + 2] : -INFINITY) : 0.f, scale_log2e, -m)) * il : 0.f;
            ds[nt][e] = qk ? p0 * (ds[nt][e] - dl) : 0.f;
            ds[nt][e + 2] = qk ? p1 * (ds[nt][e + 2] - dl) : 0.f;
          } else {
            p0 = ok ? exp2f(fmaf(p[nt][e], scale_log2e, -m)) * il : 0.f;
            p1 = ok ? exp2f(fmaf(p[nt][e + 2], scale_log2e, -m)) * il : 0.f;
            ds[nt][e] = p0 * (ds[nt][e] - dl);
            ds[nt][e + 2] = p1 * (ds[nt][e + 2] - dl);
          }
          p[nt][e] = p0;
          p[nt][e + 2] = p1;
        }
      }
      long_mma_xm(dv, p, Os + qb * 64, lane);         // dV = P^T dO
      long_mma_xm(dk, ds, Qs + qb * 64, lane);        // dK = dS^T Q / sqrt(dh)
    }
    long_store(dv, dbase + 2 * inner, ld, r_lo, n_tok, 1.f, 1.f, t);
    long_store(dk, dbase + inner, ld, r_lo, n_tok, scale, scale, t);
  }
}

size_t long_fwd_smem(int n_tok) { return size_t(2) * long_rows(n_tok) * kLongPitch * 2 + 4 * sizeof(uint64_t); }
size_t long_bwd_smem(int n_tok) { return size_t(4) * long_rows(n_tok) * kLongPitch * 2 + size_t(3) * long_rows(n_tok) * 4 + 4 * sizeof(uint64_t); }

template <bool MASKED, bool PROBS>
int launch_long(const void* qkv, void* out, int n_seq, int n_tok, int heads, int q_rows, const uint8_t* keep, float* probs, cudaStream_t st) {
  auto kern = attention_long_mma_kernel<MASKED, PROBS>;
  static PerDeviceOnce once;
  if (once.first()) {
    AVF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(long_fwd_smem(kLongMaxTok))));
  }
  launch_pdl(kern, n_seq * heads, kLongWarps * 32, long_fwd_smem(n_tok), st, static_cast<const __nv_bfloat16*>(qkv), static_cast<__nv_bfloat16*>(out), n_tok,
             heads, 1.4426950408889634f / sqrtf(float(kLongDH)), q_rows, keep, probs);
  AVF_LAUNCH_CHECK("attention_long_mma_kernel");
  return 0;
}

template <bool MASKED, bool GMAP>
int launch_bwd_long(const void* qkv, const void* dout, void* dqkv, int n_seq, int n_tok, int heads, const uint8_t* keep, float* gmap, cudaStream_t st) {
  auto kern = attention_bwd_long_mma_kernel<MASKED, GMAP>;
  static PerDeviceOnce once;
  if (once.first()) {
    AVF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(long_bwd_smem(kLongMaxTok))));
  }
  launch_pdl(kern, n_seq * heads, kLongWarps * 32, long_bwd_smem(n_tok), st, static_cast<const __nv_bfloat16*>(qkv), static_cast<const __nv_bfloat16*>(dout),
             static_cast<__nv_bfloat16*>(dqkv), n_tok, heads, 1.0f / sqrtf(float(kLongDH)), keep, gmap);
  AVF_LAUNCH_CHECK("attention_bwd_long_mma_kernel");
  return 0;
}

}  // namespace

int attention_mma_bf16(const void* qkv, void* out, int n_seq, int n_tok, int heads, int dim_head, cudaStream_t st, int q_rows, const uint8_t* keep,
                       float* probs) {
  AVF_REQUIRE(n_tok >= 1 && n_tok <= kLongMaxTok && (n_tok <= 64 || dim_head == kLongDH), AVF_EUNSUPPORTED,
              "attention: n_tok=%d with dim_head=%d (1..64 tokens; 64-wide heads up to 256)", n_tok, dim_head);
  if (q_rows <= 0 || q_rows > n_tok) q_rows = n_tok;
  if (n_tok > 64) {
    if (probs)
      return keep ? launch_long<true, true>(qkv, out, n_seq, n_tok, heads, q_rows, keep, probs, st)
                  : launch_long<false, true>(qkv, out, n_seq, n_tok, heads, q_rows, nullptr, probs, st);
    return keep ? launch_long<true, false>(qkv, out, n_seq, n_tok, heads, q_rows, keep, nullptr, st)
                : launch_long<false, false>(qkv, out, n_seq, n_tok, heads, q_rows, nullptr, nullptr, st);
  }
  const int np = (n_tok + 15) / 16 * 16;
#define AVF_ATT(D, P)                                                                                   \
  if (dim_head == D && np == P) {                                                                       \
    if (probs)                                                                                          \
      return keep ? launch<D, P, true, true>(qkv, out, n_seq, n_tok, heads, q_rows, keep, probs, st)    \
                  : launch<D, P, false, true>(qkv, out, n_seq, n_tok, heads, q_rows, nullptr, probs, st); \
    return keep ? launch<D, P, true, false>(qkv, out, n_seq, n_tok, heads, q_rows, keep, nullptr, st)   \
                : launch<D, P, false, false>(qkv, out, n_seq, n_tok, heads, q_rows, nullptr, nullptr, st); \
  }
  AVF_ATT(32, 16) AVF_ATT(32, 32) AVF_ATT(32, 48) AVF_ATT(32, 64)
  AVF_ATT(64, 16) AVF_ATT(64, 32) AVF_ATT(64, 48) AVF_ATT(64, 64)
#undef AVF_ATT
  AVF_REQUIRE(false, AVF_EUNSUPPORTED, "attention: dim_head=%d (supported: 32, 64)", dim_head);
  return 0;
}

}  // namespace avf

namespace avf {
int attention_bwd_mma_bf16(const void* qkv, const void* dout, void* dqkv, int n_seq, int n_tok, int heads, int dim_head, cudaStream_t st,
                           const uint8_t* keep, float* gmap) {
  AVF_REQUIRE(n_tok >= 1 && n_tok <= kLongMaxTok && (n_tok <= 64 || dim_head == kLongDH), AVF_EUNSUPPORTED,
              "attention_bwd: n_tok=%d with dim_head=%d (1..64 tokens; 64-wide heads up to 256)", n_tok, dim_head);
  if (n_tok > 64) {
    if (gmap)
      return keep ? launch_bwd_long<true, true>(qkv, dout, dqkv, n_seq, n_tok, heads, keep, gmap, st)
                  : launch_bwd_long<false, true>(qkv, dout, dqkv, n_seq, n_tok, heads, nullptr, gmap, st);
    return keep ? launch_bwd_long<true, false>(qkv, dout, dqkv, n_seq, n_tok, heads, keep, nullptr, st)
                : launch_bwd_long<false, false>(qkv, dout, dqkv, n_seq, n_tok, heads, nullptr, nullptr, st);
  }
  const int np = (n_tok + 15) / 16 * 16;
#define AVF_ATT(D, P)                                                                                      \
  if (dim_head == D && np == P) {                                                                          \
    if (gmap)                                                                                              \
      return keep ? launch_bwd<D, P, true, true>(qkv, dout, dqkv, n_seq, n_tok, heads, keep, gmap, st)     \
                  : launch_bwd<D, P, false, true>(qkv, dout, dqkv, n_seq, n_tok, heads, nullptr, gmap, st); \
    return keep ? launch_bwd<D, P, true, false>(qkv, dout, dqkv, n_seq, n_tok, heads, keep, nullptr, st)   \
                : launch_bwd<D, P, false, false>(qkv, dout, dqkv, n_seq, n_tok, heads, nullptr, nullptr, st); \
  }
  AVF_ATT(32, 16) AVF_ATT(32, 32) AVF_ATT(32, 48) AVF_ATT(32, 64)
  AVF_ATT(64, 16) AVF_ATT(64, 32) AVF_ATT(64, 48) AVF_ATT(64, 64)
#undef AVF_ATT
  AVF_REQUIRE(false, AVF_EUNSUPPORTED, "attention_bwd: dim_head=%d (supported: 32, 64)", dim_head);
  return 0;
}
}  // namespace avf
