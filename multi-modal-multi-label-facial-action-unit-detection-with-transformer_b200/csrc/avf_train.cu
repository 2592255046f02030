// Backward / optimiser kernels of the AVFormer hot path (the training step of train.py:206-236 restricted to the
// transformer stack): LayerNorm backward (+ the three column reductions that ride on it), softmax-attention backward,
// column sums (bias / positional-embedding gradients), BatchNorm1d with batch statistics (forward + backward), the
// backward of the 12 per-AU dot products, and Adam / AdamW over a flat parameter bucket.
//
// The dense contractions of the backward pass (dgrad, wgrad) are the tcgen05 GEMM of avf_gemm_umma.cu in its NN / TN
// operand modes; everything here is the memory-bound remainder: one warp per row, 16-byte accesses, fixed-order
// (deterministic) two-stage reductions, no atomics.
#include <algorithm>
#include <cmath>

#include "avf_adam.cuh"
#include "avf_common.cuh"
#include "avf_internal.h"

namespace avf {

namespace {

// ---------------------------------------------------------------------------------------------
// column sums:  out[c] = beta * out[c] + sum_r x[r, c]          (fixed summation order)
// ---------------------------------------------------------------------------------------------
template <typename T> struct RowVec;       // 16-byte row fragment: 8 bf16 / 4 fp32
template <> struct RowVec<__nv_bfloat16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void add(const __nv_bfloat16* p, float (&a)[8]) {
    const uint4 v = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) { a[2 * q] += __uint_as_float(w[q] << 16); a[2 * q + 1] += __uint_as_float(w[q] & 0xffff0000u); }
  }
};
template <> struct RowVec<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ void add(const float* p, float (&a)[4]) {
    const float4 v = *reinterpret_cast<const float4*>(p);
    a[0] += v.x; a[1] += v.y; a[2] += v.z; a[3] += v.w;
  }
};

// Vectorised partial sums: a warp covers 32 * N consecutive columns with one 16-byte load per lane and row; the 8 warps of
// a block take every 8th row of the block's row chunk (two independent accumulator sets for memory-level parallelism).
template <typename T>
__global__ void __launch_bounds__(256) colsum_partial_vec_kernel(const T* __restrict__ x, size_t ld, int rows, int cols, int rows_per_chunk,
                                                                 float* __restrict__ part) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  constexpr int N = RowVec<T>::N;
  __shared__ float red[8][32 * N + 4];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int col = (blockIdx.x * 32 + lane) * N;
  const int r0 = blockIdx.y * rows_per_chunk, r1 = min(rows, r0 + rows_per_chunk);
  float a[N], b[N];
#pragma unroll
  for (int j = 0; j < N; ++j) a[j] = b[j] = 0.f;
  if (col < cols) {
    int r = r0 + warp;
    for (; r + 8 < r1; r += 16) {
      RowVec<T>::add(x + size_t(r) * ld + col, a);
      RowVec<T>::add(x + size_t(r + 8) * ld + col, b);
    }
    if (r < r1) RowVec<T>::add(x + size_t(r) * ld + col, a);
  }
#pragma unroll
  for (int j = 0; j < N; ++j) red[warp][lane * N + j] = a[j] + b[j];
  __syncthreads();
  for (int c = threadIdx.x; c < 32 * N; c += 256) {
    const int gc = blockIdx.x * 32 * N + c;
    if (gc >= cols) continue;
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w][c];
    part[size_t(blockIdx.y) * cols + gc] = s;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) colsum_partial_kernel(const T* __restrict__ x, size_t ld, int rows, int cols, int rows_per_chunk,
                                                             float* __restrict__ part) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  const int r0 = blockIdx.y * rows_per_chunk, r1 = min(rows, r0 + rows_per_chunk);
  float s = 0.f;
  if (col < cols)
    for (int r = r0 + ty; r < r1; r += 8) s += to_f32<T>(x[size_t(r) * ld + col]);
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && col < cols) {
    float a = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) a += red[i][tx];
    part[size_t(blockIdx.y) * cols + col] = a;
  }
}

// out_q[c] = beta * out_q[c] + sum_b part[b, q * cols + c] for up to three outputs packed side by side in `part`.
// 32 columns x 8 partial-row lanes per block: the chunk loop is split 8 ways and unrolled so that the (L2-latency bound)
// loads overlap; the order of the additions is fixed.
__global__ void __launch_bounds__(256) colsum_final_kernel(const float* __restrict__ part, int chunks, int cols, int n_out,
                                                           float* o0, float* o1, float* o2, float beta) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int idx = blockIdx.x * 32 + tx, width = cols * n_out;
  float a = 0.f;
  if (idx < width) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int b = ty;
    for (; b + 24 < chunks; b += 32) {
      a0 += part[size_t(b) * width + idx];
      a1 += part[size_t(b + 8) * width + idx];
      a2 += part[size_t(b + 16) * width + idx];
      a3 += part[size_t(b + 24) * width + idx];
    }
    for (; b < chunks; b += 8) a0 += part[size_t(b) * width + idx];
    a = (a0 + a1) + (a2 + a3);
  }
  red[ty][tx] = a;
  __syncthreads();
  if (ty != 0 || idx >= width) return;
  a = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) a += red[i][tx];
  const int q = idx / cols, c = idx - q * cols;
  float* o = q == 0 ? o0 : (q == 1 ? o1 : o2);
  if (o == nullptr) return;
  o[c] = beta != 0.f ? beta * o[c] + a : a;
}

// ---------------------------------------------------------------------------------------------
// LayerNorm backward of a pre-LN sub-layer  y = x + f(LN(x))   (models/heads.py:169-185)
//   dres  (in)  gradient wrt y  == gradient through the skip connection; also the bias gradient of f's last linear
//   dyn         gradient wrt LN(x) (output of the dgrad GEMM of f's first linear), fp32 dense [rows, DIM]
//   dres  (out) gradient wrt x = dres + rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dyn * gamma
//   dxb         optional bf16 copy of the new dres (operand of the next GEMMs)
//   part        [gridDim.x][3][DIM]: per-block sums of dyn * xhat (dgamma), dyn (dbeta), dres_in (dbias)
// One warp per row, row in registers, per-lane column accumulators, one block-level reduction at the end.
// ---------------------------------------------------------------------------------------------
template <int VEC>   // DIM = 128 * VEC
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const float* __restrict__ x, int ld_x, const float* __restrict__ gamma,
                                                            const float* __restrict__ dyn, float* dres, int ld_d,
                                                            void* __restrict__ dxb, int dxb_bf16, float* __restrict__ part, int rows,
                                                            int rows_per_block, DropSpec drop_in, DropSpec drop_out) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  constexpr int DIM = 128 * VEC;
  __shared__ float red[8][DIM];
  drop_in = drop_resolve(drop_in);
  drop_out = drop_resolve(drop_out);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = blockIdx.x * rows_per_block, r1 = min(rows, r0 + rows_per_block);
  float4 ag[VEC], ab[VEC], ad[VEC], gm[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    ag[i] = ab[i] = ad[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    gm[i] = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32 * i);
  }
  for (int row = r0 + warp; row < r1; row += 8) {
    const float4* xp = reinterpret_cast<const float4*>(x + size_t(row) * ld_x);
    const float4* yp = reinterpret_cast<const float4*>(dyn + size_t(row) * DIM);
    float4* dp = reinterpret_cast<float4*>(dres + size_t(row) * ld_d);
    float4 v[VEC], g[VEC], dy[VEC], rs[VEC];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {          // all three streams of the row are requested before the first reduction
      v[i] = xp[lane + 32 * i];
      dy[i] = yp[lane + 32 * i];
      rs[i] = dp[lane + 32 * i];
    }
#pragma unroll
    for (int i = 0; i < VEC; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    const float mean = warp_sum(s) * (1.0f / DIM);
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
      ss += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
    }
    const float rstd = rsqrtf(warp_sum(ss) * (1.0f / DIM) + 1e-5f);
    float m1 = 0.f, m2 = 0.f;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float4 d = dy[i];
      v[i].x *= rstd; v[i].y *= rstd; v[i].z *= rstd; v[i].w *= rstd;       // xhat
      ag[i].x += d.x * v[i].x; ag[i].y += d.y * v[i].y; ag[i].z += d.z * v[i].z; ag[i].w += d.w * v[i].w;
      ab[i].x += d.x; ab[i].y += d.y; ab[i].z += d.z; ab[i].w += d.w;
      g[i] = make_float4(d.x * gm[i].x, d.y * gm[i].y, d.z * gm[i].z, d.w * gm[i].w);
      m1 += (g[i].x + g[i].y) + (g[i].z + g[i].w);
      m2 += (g[i].x * v[i].x + g[i].y * v[i].y) + (g[i].z * v[i].z + g[i].w * v[i].w);
    }
    m1 = warp_sum(m1) * (1.0f / DIM);
    m2 = warp_sum(m2) * (1.0f / DIM);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float4 r = rs[i];
      if (drop_in.thresh != 0) {      // bias gradient of a sub-layer whose output went through dropout: sum the masked gradient
        const uint32_t i0 = uint32_t(row) * DIM + (lane + 32 * i) * 4;
        ad[i].x += r.x * drop_factor(drop_in, i0); ad[i].y += r.y * drop_factor(drop_in, i0 + 1);
        ad[i].z += r.z * drop_factor(drop_in, i0 + 2); ad[i].w += r.w * drop_factor(drop_in, i0 + 3);
      } else {
        ad[i].x += r.x; ad[i].y += r.y; ad[i].z += r.z; ad[i].w += r.w;
      }
      float4 o;
      o.x = r.x + rstd * (g[i].x - m1 - v[i].x * m2);
      o.y = r.y + rstd * (g[i].y - m1 - v[i].y * m2);
      o.z = r.z + rstd * (g[i].z - m1 - v[i].z * m2);
      o.w = r.w + rstd * (g[i].w - m1 - v[i].w * m2);
      dp[lane + 32 * i] = o;
      if (dxb != nullptr) {
        if (drop_out.thresh != 0) {
          const uint32_t i0 = uint32_t(row) * DIM + (lane + 32 * i) * 4;
          o.x *= drop_factor(drop_out, i0); o.y *= drop_factor(drop_out, i0 + 1);
          o.z *= drop_factor(drop_out, i0 + 2); o.w *= drop_factor(drop_out, i0 + 3);
        }
        const size_t off = size_t(row) * DIM + (lane + 32 * i) * 4;
        if (dxb_bf16) {
          uint2 pk;
          pk.x = pack_bf16x2(o.x, o.y);
          pk.y = pack_bf16x2(o.z, o.w);
          *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(dxb) + off) = pk;
        } else {
          *reinterpret_cast<float4*>(static_cast<float*>(dxb) + off) = o;
        }
      }
    }
  }
  float* pb = part + size_t(blockIdx.x) * 3 * DIM;
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float4 a = q == 0 ? ag[i] : (q == 1 ? ab[i] : ad[i]);
      *reinterpret_cast<float4*>(&red[warp][(lane + 32 * i) * 4]) = a;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < DIM; c += 256) {
      float a = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) a += red[w][c];
      pb[q * DIM + c] = a;
    }
  }
}

template <typename OutT>
__global__ void __launch_bounds__(256) masked_copy_kernel(const float* __restrict__ x, OutT* __restrict__ y, size_t n, DropSpec drop) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  drop = drop_resolve(drop);
  if (i < n) y[i] = from_f32<OutT>(x[i] * drop_factor(drop, uint32_t(i)));
}
__global__ void __launch_bounds__(256) dropout_mask_kernel(float* __restrict__ out, size_t n, DropSpec drop) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  drop = drop_resolve(drop);
  if (i < n) out[i] = drop_factor(drop, uint32_t(i));
}

// ---------------------------------------------------------------------------------------------
// Attention backward (models/heads.py:221-237) for one (sequence, head) per CTA.  P is recomputed from q, k.
//   dV = P^T dO;  dP = dO V^T;  dS = P o (dP - rowsum(P o dP));  dQ = scale dS K;  dK = scale dS^T Q
// Sequences are 12 / 17 / 49 tokens: everything of one head lives in shared memory as fp32.
// MASKED: keep [n_seq, n_tok] uint8 (1 = keep), turned into 64 keep bits by two ballots of every warp.  Scores of a kept query on
// dropped keys are -INF (P = 0); a dropped query's scores are all equal (uniform P); dS = 0 on every filled score.
// ---------------------------------------------------------------------------------------------
template <typename T, int DH, bool MASKED>
__global__ void __launch_bounds__(128) attention_bwd_kernel(const T* __restrict__ qkv, const T* __restrict__ dout, T* __restrict__ dqkv,
                                                            int n_tok, int heads, float scale, const uint8_t* __restrict__ keep) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  extern __shared__ float sm[];
  constexpr int P = DH + 1;
  const int N = n_tok, NP = N + 1;
  float* sq = sm;
  float* sk = sq + N * P;
  float* sv = sk + N * P;
  float* sdo = sv + N * P;
  float* sp = sdo + N * P;      // [N][NP] probabilities
  float* sds = sp + N * NP;     // [N][NP] dS
  const int seq = blockIdx.x / heads, h = blockIdx.x - seq * heads;
  const int inner = heads * DH;
  const size_t row0 = size_t(seq) * N;
  uint64_t km = 0;
  if constexpr (MASKED) {
    const int lane = threadIdx.x & 31;
    const uint32_t lo = __ballot_sync(0xffffffffu, lane < N && keep[row0 + lane] != 0);
    const uint32_t hi = __ballot_sync(0xffffffffu, lane + 32 < N && keep[row0 + lane + 32] != 0);
    km = (uint64_t(hi) << 32) | lo;
  }
  for (int i = threadIdx.x; i < N * DH; i += blockDim.x) {
    const int t = i / DH, d = i - t * DH;
    const T* qp = qkv + (row0 + t) * size_t(3 * inner) + h * DH + d;
    sq[t * P + d] = to_f32<T>(qp[0]);
    sk[t * P + d] = to_f32<T>(qp[inner]);
    sv[t * P + d] = to_f32<T>(qp[2 * inner]);
    sdo[t * P + d] = to_f32<T>(dout[(row0 + t) * size_t(inner) + h * DH + d]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < N * N; i += blockDim.x) {
    const int a = i / N, b = i - a * N;
    float s = 0.f, dp = 0.f;
#pragma unroll 8
    for (int d = 0; d < DH; ++d) {
      s = fmaf(sq[a * P + d], sk[b * P + d], s);
      dp = fmaf(sdo[a * P + d], sv[b * P + d], dp);
    }
    float v = s * scale;
    if constexpr (MASKED) v = !((km >> a) & 1) ? 0.f : ((km >> b) & 1) ? v : -INFINITY;
    sp[a * NP + b] = v;
    sds[a * NP + b] = dp;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int a = warp; a < N; a += 4) {         // row softmax, then dS of that row
    float mx = -INFINITY;
    for (int b = lane; b < N; b += 32) mx = fmaxf(mx, sp[a * NP + b]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int b = lane; b < N; b += 32) {
      const float e = __expf(sp[a * NP + b] - mx);
      sp[a * NP + b] = e;
      sum += e;
    }
    const float inv = 1.0f / warp_sum(sum);
    float delta = 0.f;
    for (int b = lane; b < N; b += 32) {
      const float p = sp[a * NP + b] * inv;
      sp[a * NP + b] = p;
      delta += p * sds[a * NP + b];
    }
    delta = warp_sum(delta);
    const bool filled_row = MASKED && !((km >> a) & 1);
    for (int b = lane; b < N; b += 32) sds[a * NP + b] = filled_row ? 0.f : sp[a * NP + b] * (sds[a * NP + b] - delta) * scale;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < N * DH; i += blockDim.x) {
    const int t = i / DH, d = i - t * DH;
    float dq = 0.f, dk = 0.f, dv = 0.f;
    for (int j = 0; j < N; ++j) {
      dq = fmaf(sds[t * NP + j], sk[j * P + d], dq);
      dk = fmaf(sds[j * NP + t], sq[j * P + d], dk);
      dv = fmaf(sp[j * NP + t], sdo[j * P + d], dv);
    }
    T* op = dqkv + (row0 + t) * size_t(3 * inner) + h * DH + d;
    op[0] = from_f32<T>(dq);
    op[inner] = from_f32<T>(dk);
    op[2 * inner] = from_f32<T>(dv);
  }
}

// ---------------------------------------------------------------------------------------------
// Attention backward of 65..256 tokens with 64-wide heads (fp32), one (sequence, head) per CTA.  Two n_tok x 64 operands fit shared
// memory, four do not, so the CTA runs two passes, each with one warp per row and the lanes over the other side's tokens:
//   pass 1, K | V staged, rows = queries: scores and dP, softmax statistics (max, 1/sum, delta) to shared memory, dQ = scale dS K;
//   pass 2, Q | dO restaged, rows = keys: P and dS again from the statistics, dV = P^T dO, dK = scale dS^T Q.
// The row's own operand pair sits in a per-warp slot (broadcast reads) and its scores in a per-warp line.  Masks as in
// attention_bwd_kernel, with the keep bits in four 64-bit words.
// ---------------------------------------------------------------------------------------------
constexpr int kLongF32Pitch = 64 + 1;
__host__ __device__ constexpr size_t attention_bwd_long_smem(int n_tok) {
  return (size_t(2) * n_tok * kLongF32Pitch + 8 * (2 * 64 + 2 * 256) + 3 * 256) * sizeof(float) + 4 * sizeof(uint64_t);
}

template <bool MASKED>
__global__ void __launch_bounds__(256) attention_bwd_long_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ dout,
                                                                     float* __restrict__ dqkv, int n_tok, int heads, float scale,
                                                                     const uint8_t* __restrict__ keep) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  constexpr int DH = 64, P = kLongF32Pitch;
  extern __shared__ float sm_long[];
  const int N = n_tok;
  float* sa = sm_long;                  // [N][P]  K, then Q
  float* sb = sa + N * P;               // [N][P]  V, then dO
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* own = sb + N * P + warp * (2 * DH + 2 * 256);      // this warp's row pair [2][DH], then its lines [2][256]
  float* l0 = own + 2 * DH;
  float* l1 = l0 + 256;
  float* st_m = sb + N * P + 8 * (2 * DH + 2 * 256);       // [256] row max (exp2 units), 1 / row sum, delta
  float* st_il = st_m + 256;
  float* st_d = st_il + 256;
  uint64_t* km = reinterpret_cast<uint64_t*>(st_d + 256);
  const int seq = blockIdx.x / heads, h = blockIdx.x - seq * heads;
  const int inner = heads * DH;
  const size_t row0 = size_t(seq) * N;
  const float scale_log2e = scale * 1.4426950408889634f;
  auto kept = [&](int i) { return !MASKED || ((km[i >> 6] >> (i & 63)) & 1); };
  auto stage = [&](const float* src_a, size_t ld_a, const float* src_b, size_t ld_b) {
    for (int i = threadIdx.x; i < N * DH; i += blockDim.x) {
      const int t = i / DH, d = i - t * DH;
      sa[t * P + d] = src_a[(row0 + t) * ld_a + d];
      sb[t * P + d] = src_b[(row0 + t) * ld_b + d];
    }
  };
  const float* qbase = qkv + h * DH;
  stage(qbase + inner, 3 * inner, qbase + 2 * inner, 3 * inner);
  if (MASKED && warp < 4) {
    const int b = warp * 64;
    const uint8_t* row = keep + row0 + b;
    const uint32_t lo = __ballot_sync(0xffffffffu, b + lane < N && row[lane] != 0);
    const uint32_t hi = __ballot_sync(0xffffffffu, b + lane + 32 < N && row[lane + 32] != 0);
    if (lane == 0) km[warp] = (uint64_t(hi) << 32) | lo;
  }
  __syncthreads();

  // ---- pass 1: rows = queries, lanes over keys ----
  for (int a = warp; a < N; a += 8) {
    for (int d = lane; d < DH; d += 32) {
      own[d] = qbase[(row0 + a) * (3 * inner) + d];
      own[DH + d] = dout[(row0 + a) * size_t(inner) + h * DH + d];
    }
    __syncwarp();
    const bool row_kept = kept(a);
    float mx = -INFINITY;
    for (int b = lane; b < N; b += 32) {
      float s = 0.f, dp = 0.f;
#pragma unroll 8
      for (int d = 0; d < DH; ++d) {
        s = fmaf(own[d], sa[b * P + d], s);
        dp = fmaf(own[DH + d], sb[b * P + d], dp);
      }
      s = !row_kept ? 0.f : kept(b) ? __fmul_rn(s, scale_log2e) : -INFINITY;      // rounded product in both passes and instantiations
      l0[b] = s;
      l1[b] = dp;
      mx = fmaxf(mx, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int b = lane; b < N; b += 32) sum += exp2f(l0[b] - mx);
    const float il = 1.0f / warp_sum(sum);
    float delta = 0.f;
    for (int b = lane; b < N; b += 32) {
      const float p = exp2f(l0[b] - mx) * il;
      delta += p * l1[b];
      l0[b] = p;
    }
    delta = warp_sum(delta);
    for (int b = lane; b < N; b += 32) l1[b] = row_kept ? l0[b] * (l1[b] - delta) : 0.f;
    if (lane == 0) { st_m[a] = mx; st_il[a] = il; st_d[a] = delta; }
    __syncwarp();
    for (int d = lane; d < DH; d += 32) {
      float dq = 0.f;
      for (int b = 0; b < N; ++b) dq = fmaf(l1[b], sa[b * P + d], dq);
      dqkv[(row0 + a) * (3 * inner) + h * DH + d] = dq * scale;
    }
    __syncwarp();
  }
  __syncthreads();
  stage(qbase, 3 * inner, dout + h * DH, inner);
  __syncthreads();

  // ---- pass 2: rows = keys, lanes over queries ----
  for (int b = warp; b < N; b += 8) {
    for (int d = lane; d < DH; d += 32) {
      own[d] = qbase[(row0 + b) * (3 * inner) + inner + d];
      own[DH + d] = qbase[(row0 + b) * (3 * inner) + 2 * inner + d];
    }
    __syncwarp();
    const bool key_kept = kept(b);
    for (int a = lane; a < N; a += 32) {
      float s = 0.f, dp = 0.f;
#pragma unroll 8
      for (int d = 0; d < DH; ++d) {
        s = fmaf(sa[a * P + d], own[d], s);
        dp = fmaf(sb[a * P + d], own[DH + d], dp);
      }
      const bool qk = kept(a);
      s = !qk ? 0.f : key_kept ? __fmul_rn(s, scale_log2e) : -INFINITY;
      const float p = exp2f(s - st_m[a]) * st_il[a];
      l0[a] = p;
      l1[a] = qk ? p * (dp - st_d[a]) : 0.f;
    }
    __syncwarp();
    for (int d = lane; d < DH; d += 32) {
      float dk = 0.f, dv = 0.f;
      for (int a = 0; a < N; ++a) {
        dv = fmaf(l0[a], sb[a * P + d], dv);
        dk = fmaf(l1[a], sa[a * P + d], dk);
      }
      float* op = dqkv + (row0 + b) * (3 * inner) + h * DH + d;
      op[inner] = dk * scale;
      op[2 * inner] = dv;
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// Backward of the 12 per-AU dots (models/tformer.py:389-401): dx[c*12+i, :] = dl[c,i] w[i,:];  dw[i,:] = sum_c dl[c,i] x[c*12+i,:]
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) au_logits_bwd_dx_kernel(const float* __restrict__ dl, int ld_dl, const float* __restrict__ w_last,
                                                               float* __restrict__ dx, int ld_dx, int n_clips, int dim) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const size_t idx = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= size_t(n_clips) * 12 * dim) return;
  const int c = int(idx % dim);
  const size_t r = idx / dim;
  const int au = int(r % 12);
  dx[r * ld_dx + c] = dl[(r / 12) * ld_dl + au] * __ldg(w_last + size_t(au) * dim + c);
}
__global__ void __launch_bounds__(256) au_logits_bwd_dw_kernel(const float* __restrict__ dl, int ld_dl, const float* __restrict__ x, int ld_x,
                                                               float* __restrict__ dw, int n_clips, int dim) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const int au = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= dim) return;
  float a = 0.f;
  for (int b = 0; b < n_clips; ++b) a = fmaf(dl[size_t(b) * ld_dl + au], x[(size_t(b) * 12 + au) * ld_x + c], a);
  dw[size_t(au) * dim + c] = a;
}

// ---------------------------------------------------------------------------------------------
// BatchNorm1d (AU_BN1, models/heads.py:263,293) with batch statistics: one thread column, 8 row lanes.
// ---------------------------------------------------------------------------------------------
template <typename OutT>
__global__ void __launch_bounds__(256) bn_train_fwd_kernel(const float* __restrict__ x, int ld_x, const float* __restrict__ g,
                                                           const float* __restrict__ b, float* run_mean, float* run_var, float momentum,
                                                           OutT* __restrict__ y, float* __restrict__ save_mean, float* __restrict__ save_rstd,
                                                           int rows, int dim) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  __shared__ float red[8][33];
  __shared__ float stat[2][32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  const bool ok = col < dim;
  float s = 0.f;
  if (ok) for (int r = ty; r < rows; r += 8) s += x[size_t(r) * ld_x + col];
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0) {
    float a = 0.f;
    for (int i = 0; i < 8; ++i) a += red[i][tx];
    stat[0][tx] = a / rows;
  }
  __syncthreads();
  const float mean = stat[0][tx];
  s = 0.f;
  if (ok) for (int r = ty; r < rows; r += 8) { const float d = x[size_t(r) * ld_x + col] - mean; s += d * d; }
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0) {
    float a = 0.f;
    for (int i = 0; i < 8; ++i) a += red[i][tx];
    const float var = a / rows;                       // biased: normalisation
    stat[1][tx] = rsqrtf(var + 1e-5f);
    if (ok) {
      save_mean[col] = mean;
      save_rstd[col] = stat[1][tx];
      if (run_mean != nullptr) {                      // running statistics use the unbiased variance
        run_mean[col] = (1.f - momentum) * run_mean[col] + momentum * mean;
        run_var[col] = (1.f - momentum) * run_var[col] + momentum * (rows > 1 ? a / (rows - 1) : var);
      }
    }
  }
  __syncthreads();
  if (!ok) return;
  const float rstd = stat[1][tx], gg = g[col], bb = b[col];
  for (int r = ty; r < rows; r += 8) y[size_t(r) * dim + col] = from_f32<OutT>((x[size_t(r) * ld_x + col] - mean) * rstd * gg + bb);
}

// batch_stats = 1: full BN backward;  0: statistics are constants (eval mode), dx = dy g rstd.
__global__ void __launch_bounds__(256) bn_bwd_kernel(const float* __restrict__ x, int ld_x, const float* __restrict__ dy,
                                                     const float* __restrict__ g, const float* __restrict__ mean,
                                                     const float* __restrict__ rstd_or_var, int batch_stats, float* __restrict__ dx,
                                                     int ld_dx, float* __restrict__ dgamma, float* __restrict__ dbeta, int rows, int dim) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  __shared__ float red[2][8][33];
  __shared__ float tot[2][32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  const bool ok = col < dim;
  const float mu = ok ? mean[col] : 0.f;
  const float rstd = ok ? (batch_stats ? rstd_or_var[col] : rsqrtf(rstd_or_var[col] + 1e-5f)) : 0.f;
  float s1 = 0.f, s2 = 0.f;
  if (ok)
    for (int r = ty; r < rows; r += 8) {
      const float d = dy[size_t(r) * dim + col];
      s1 += d;
      s2 += d * (x[size_t(r) * ld_x + col] - mu) * rstd;
    }
  red[0][ty][tx] = s1;
  red[1][ty][tx] = s2;
  __syncthreads();
  if (ty == 0) {
    float a = 0.f, c = 0.f;
    for (int i = 0; i < 8; ++i) { a += red[0][i][tx]; c += red[1][i][tx]; }
    tot[0][tx] = a;
    tot[1][tx] = c;
    if (ok) {
      if (dbeta) dbeta[col] = a;
      if (dgamma) dgamma[col] = c;
    }
  }
  __syncthreads();
  if (!ok || dx == nullptr) return;
  const float gg = g[col] * rstd, m1 = batch_stats ? tot[0][tx] / rows : 0.f, m2 = batch_stats ? tot[1][tx] / rows : 0.f;
  for (int r = ty; r < rows; r += 8) {
    const float xh = (x[size_t(r) * ld_x + col] - mu) * rstd;
    dx[size_t(r) * ld_dx + col] = gg * (dy[size_t(r) * dim + col] - m1 - xh * m2);
  }
}

// ---------------------------------------------------------------------------------------------
// Adam (torch.optim.Adam of train.py:334: L2 coupled into the gradient) / AdamW (decoupled) on a flat bucket.
// grad_scale folds the 1/world_size of the data-parallel mean into the update; an optional bf16 shadow of the
// parameters is refreshed in the same pass (GEMM operand copies).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, __nv_bfloat16* __restrict__ shadow, size_t n, float lr, float b1,
                                                   float b2, float eps, float wd, float inv_bc1, float inv_sqrt_bc2, int decoupled,
                                                   float grad_scale) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const size_t i = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  float pv[4], gv[4], mv[4], vv[4];
  const bool full = i + 3 < n;
  const int cnt = full ? 4 : int(n - i);
  if (full) {
    const float4 a = *reinterpret_cast<const float4*>(p + i), b = *reinterpret_cast<const float4*>(g + i);
    const float4 c = *reinterpret_cast<const float4*>(m + i), d = *reinterpret_cast<const float4*>(v + i);
    pv[0] = a.x; pv[1] = a.y; pv[2] = a.z; pv[3] = a.w;
    gv[0] = b.x; gv[1] = b.y; gv[2] = b.z; gv[3] = b.w;
    mv[0] = c.x; mv[1] = c.y; mv[2] = c.z; mv[3] = c.w;
    vv[0] = d.x; vv[1] = d.y; vv[2] = d.z; vv[3] = d.w;
  } else {
    for (int j = 0; j < cnt; ++j) { pv[j] = p[i + j]; gv[j] = g[i + j]; mv[j] = m[i + j]; vv[j] = v[i + j]; }
  }
#pragma unroll
  const AdamParams ap{lr, b1, b2, eps, wd, inv_bc1, inv_sqrt_bc2, grad_scale, decoupled};
  for (int j = 0; j < 4; ++j) {
    if (j >= cnt) break;
    adam_update(pv[j], gv[j], mv[j], vv[j], ap);
  }
  if (full) {
    *reinterpret_cast<float4*>(p + i) = make_float4(pv[0], pv[1], pv[2], pv[3]);
    *reinterpret_cast<float4*>(m + i) = make_float4(mv[0], mv[1], mv[2], mv[3]);
    *reinterpret_cast<float4*>(v + i) = make_float4(vv[0], vv[1], vv[2], vv[3]);
    if (shadow) {
      uint2 o;
      o.x = pack_bf16x2(pv[0], pv[1]);
      o.y = pack_bf16x2(pv[2], pv[3]);
      *reinterpret_cast<uint2*>(shadow + i) = o;
    }
  } else {
    for (int j = 0; j < cnt; ++j) {
      p[i + j] = pv[j]; m[i + j] = mv[j]; v[i + j] = vv[j];
      if (shadow) shadow[i + j] = __float2bfloat16_rn(pv[j]);
    }
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------------
static int colsum_chunks(int rows, int cols) {      // upper bound over both kernel variants (workspace sizing)
  const int col_blocks = ceil_div(cols, 256);
  return std::max(1, std::min(ceil_div(rows, 32), ceil_div(1184, std::max(1, col_blocks))));
}

size_t colsum_workspace_bytes(int rows, int cols) { return size_t(colsum_chunks(rows, cols)) * cols * sizeof(float); }

int colsum(int in_mode, const void* x, size_t ld, int rows, int cols, float* out, float beta, void* ws, size_t ws_bytes, cudaStream_t st) {
  AVF_REQUIRE(rows > 0 && cols > 0 && x && out, AVF_EINVAL, "colsum: rows=%d cols=%d", rows, cols);
  const int vec = in_mode == AVF_BF16 ? 8 : 4, esz = in_mode == AVF_BF16 ? 2 : 4;
  const bool vectorised = cols % vec == 0 && ld % vec == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  const int col_blocks = ceil_div(cols, vectorised ? 32 * vec : 32);
  const int chunks = std::max(1, std::min(colsum_chunks(rows, cols), std::min(ceil_div(rows, 32), ceil_div(1184, col_blocks))));
  AVF_REQUIRE(ws != nullptr && ws_bytes >= size_t(chunks) * cols * 4, AVF_EWORKSPACE, "colsum: workspace too small (%zu < %zu bytes)",
              ws_bytes, size_t(chunks) * cols * 4);
  (void)esz;
  const int rpc = ceil_div(rows, chunks);
  dim3 grid(col_blocks, ceil_div(rows, rpc));
  float* part = static_cast<float*>(ws);
  if (vectorised) {
    if (in_mode == AVF_BF16) launch_pdl(colsum_partial_vec_kernel<__nv_bfloat16>, grid, 256, 0, st, static_cast<const __nv_bfloat16*>(x), ld, rows, cols, rpc, part);
    else launch_pdl(colsum_partial_vec_kernel<float>, grid, 256, 0, st, static_cast<const float*>(x), ld, rows, cols, rpc, part);
  } else {
    if (in_mode == AVF_BF16) launch_pdl(colsum_partial_kernel<__nv_bfloat16>, grid, 256, 0, st, static_cast<const __nv_bfloat16*>(x), ld, rows, cols, rpc, part);
    else launch_pdl(colsum_partial_kernel<float>, grid, 256, 0, st, static_cast<const float*>(x), ld, rows, cols, rpc, part);
  }
  AVF_LAUNCH_CHECK("colsum_partial_kernel");
  launch_pdl(colsum_final_kernel, ceil_div(cols, 32), 256, 0, st, part, int(grid.y), cols, 1, out, nullptr, nullptr, beta);
  AVF_LAUNCH_CHECK("colsum_final_kernel");
  return 0;
}

static int ln_bwd_blocks(int rows) { return std::max(1, std::min(ceil_div(rows, 8), 592)); }
size_t layernorm_bwd_workspace_bytes(int rows, int dim) { return size_t(ln_bwd_blocks(rows)) * 3 * dim * sizeof(float); }

int layernorm_bwd(const float* x, int ld_x, const float* gamma, const float* dyn, float* dres, int ld_d, void* dxb, int dxb_mode, float* dgamma,
                  float* dbeta, float* dbias, float beta_acc, int rows, int dim, void* ws, size_t ws_bytes, cudaStream_t st,
                  DropSpec drop_in, DropSpec drop_out) {
  AVF_REQUIRE(rows > 0 && x && gamma && dyn && dres, AVF_EINVAL, "layernorm_bwd: null pointer / rows=%d", rows);
  AVF_REQUIRE(dim % 128 == 0 && dim <= 512 && ld_x % 4 == 0 && ld_d % 4 == 0, AVF_EUNSUPPORTED,
              "layernorm_bwd: dim=%d must be a multiple of 128, <= 512", dim);
  const int blocks = ln_bwd_blocks(rows);
  AVF_REQUIRE(ws != nullptr && ws_bytes >= size_t(blocks) * 3 * dim * 4, AVF_EWORKSPACE, "layernorm_bwd: workspace too small");
  const int rpb = ceil_div(rows, blocks);
  const int grid = ceil_div(rows, rpb);
  float* part = static_cast<float*>(ws);
  const int xb16 = dxb_mode == AVF_BF16 ? 1 : 0;
  switch (dim / 128) {
    case 1: launch_pdl(layernorm_bwd_kernel<1>, grid, 256, 0, st, x, ld_x, gamma, dyn, dres, ld_d, dxb, xb16, part, rows, rpb, drop_in, drop_out); break;
    case 2: launch_pdl(layernorm_bwd_kernel<2>, grid, 256, 0, st, x, ld_x, gamma, dyn, dres, ld_d, dxb, xb16, part, rows, rpb, drop_in, drop_out); break;
    case 3: launch_pdl(layernorm_bwd_kernel<3>, grid, 256, 0, st, x, ld_x, gamma, dyn, dres, ld_d, dxb, xb16, part, rows, rpb, drop_in, drop_out); break;
    default: launch_pdl(layernorm_bwd_kernel<4>, grid, 256, 0, st, x, ld_x, gamma, dyn, dres, ld_d, dxb, xb16, part, rows, rpb, drop_in, drop_out); break;
  }
  AVF_LAUNCH_CHECK("layernorm_bwd_kernel");
  if (dgamma || dbeta || dbias) {
    launch_pdl(colsum_final_kernel, ceil_div(3 * dim, 32), 256, 0, st, part, grid, dim, 3, dgamma, dbeta, dbias, beta_acc);
    AVF_LAUNCH_CHECK("colsum_final_kernel");
  }
  return 0;
}

int masked_copy(const float* x, void* y, int y_mode, int rows, int dim, DropSpec drop, cudaStream_t st) {
  const size_t n = size_t(rows) * dim;
  AVF_REQUIRE(n > 0 && n < (size_t(1) << 32), AVF_EINVAL, "masked_copy: %zu elements", n);
  if (y_mode == AVF_BF16) launch_pdl(masked_copy_kernel<__nv_bfloat16>, unsigned((n + 255) / 256), 256, 0, st, x, static_cast<__nv_bfloat16*>(y), n, drop);
  else launch_pdl(masked_copy_kernel<float>, unsigned((n + 255) / 256), 256, 0, st, x, static_cast<float*>(y), n, drop);
  AVF_LAUNCH_CHECK("masked_copy_kernel");
  return 0;
}

int dropout_mask(float* out, int rows, int cols, DropSpec drop, cudaStream_t st) {
  const size_t n = size_t(rows) * cols;
  AVF_REQUIRE(out && n > 0 && n < (size_t(1) << 32), AVF_EINVAL, "dropout_mask: %zu elements", n);
  launch_pdl(dropout_mask_kernel, unsigned((n + 255) / 256), 256, 0, st, out, n, drop);
  AVF_LAUNCH_CHECK("dropout_mask_kernel");
  return 0;
}

template <typename T, int DH, bool MASKED>
static int launch_attention_bwd(const void* qkv, const void* dout, void* dqkv, int n_seq, int n_tok, int heads, const uint8_t* keep, cudaStream_t st) {
  const size_t smem = (size_t(4) * n_tok * (DH + 1) + size_t(2) * n_tok * (n_tok + 1)) * sizeof(float);
  AVF_REQUIRE(smem <= 200 * 1024, AVF_EUNSUPPORTED, "attention_bwd: %d tokens x %d do not fit shared memory", n_tok, DH);
  auto kern = attention_bwd_kernel<T, DH, MASKED>;
  static PerDeviceOnce once;
  if (once.first()) {
    AVF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  launch_pdl(kern, n_seq * heads, 128, smem, st, static_cast<const T*>(qkv), static_cast<const T*>(dout), static_cast<T*>(dqkv), n_tok, heads,
                                         rsqrtf(float(DH)), keep);
  AVF_LAUNCH_CHECK("attention_bwd_kernel");
  return 0;
}

int attention_bwd(int io_mode, const void* qkv, const void* dout, void* dqkv, int n_seq, int n_tok, int heads, int dim_head, cudaStream_t st,
                  const uint8_t* keep) {
  AVF_REQUIRE(n_seq > 0 && n_tok > 0 && heads > 0, AVF_EINVAL, "attention_bwd: n_seq=%d n_tok=%d heads=%d", n_seq, n_tok, heads);
  AVF_REQUIRE(dim_head == 32 || dim_head == 64, AVF_EUNSUPPORTED, "attention_bwd: dim_head=%d (supported: 32, 64)", dim_head);
  AVF_REQUIRE(n_tok <= 64 || (dim_head == 64 && n_tok <= 256), AVF_EUNSUPPORTED,
              "attention_bwd: n_tok=%d with dim_head=%d (up to 64 tokens; 64-wide heads up to 256)", n_tok, dim_head);
  if (io_mode == AVF_BF16) return attention_bwd_mma_bf16(qkv, dout, dqkv, n_seq, n_tok, heads, dim_head, st, keep);      // tensor cores
  if (n_tok > 64) {
    auto kern = keep != nullptr ? attention_bwd_long_f32_kernel<true> : attention_bwd_long_f32_kernel<false>;
    static PerDeviceOnce once[2];
    if (once[keep != nullptr].first()) {
      AVF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(attention_bwd_long_smem(256))));
    }
    launch_pdl(kern, n_seq * heads, 256, attention_bwd_long_smem(n_tok), st, static_cast<const float*>(qkv), static_cast<const float*>(dout),
               static_cast<float*>(dqkv), n_tok, heads, rsqrtf(64.f), keep);
    AVF_LAUNCH_CHECK("attention_bwd_long_f32_kernel");
    return 0;
  }
  if (keep != nullptr)
    return dim_head == 32 ? launch_attention_bwd<float, 32, true>(qkv, dout, dqkv, n_seq, n_tok, heads, keep, st)
                          : launch_attention_bwd<float, 64, true>(qkv, dout, dqkv, n_seq, n_tok, heads, keep, st);
  return dim_head == 32 ? launch_attention_bwd<float, 32, false>(qkv, dout, dqkv, n_seq, n_tok, heads, nullptr, st)
                        : launch_attention_bwd<float, 64, false>(qkv, dout, dqkv, n_seq, n_tok, heads, nullptr, st);
}

int au_logits_bwd(const float* dl, int ld_dl, const float* x, int ld_x, const float* w_last, float* dx, int ld_dx, float* dw, int n_clips,
                  int dim, cudaStream_t st) {
  AVF_REQUIRE(n_clips > 0 && dim > 0 && dl && w_last, AVF_EINVAL, "au_logits_bwd: n_clips=%d dim=%d", n_clips, dim);
  if (dx != nullptr) {
    const size_t total = size_t(n_clips) * 12 * dim;
    launch_pdl(au_logits_bwd_dx_kernel, unsigned((total + 255) / 256), 256, 0, st, dl, ld_dl, w_last, dx, ld_dx, n_clips, dim);
    AVF_LAUNCH_CHECK("au_logits_bwd_dx_kernel");
  }
  if (dw != nullptr) {
    AVF_REQUIRE(x != nullptr, AVF_EINVAL, "au_logits_bwd: dw needs the tokens");
    launch_pdl(au_logits_bwd_dw_kernel, dim3(ceil_div(dim, 256), 12), 256, 0, st, dl, ld_dl, x, ld_x, dw, n_clips, dim);
    AVF_LAUNCH_CHECK("au_logits_bwd_dw_kernel");
  }
  return 0;
}

int bn_train_fwd(int out_mode, const float* x, int ld_x, const float* g, const float* b, float* run_mean, float* run_var, float momentum,
                 void* y, float* save_mean, float* save_rstd, int rows, int dim, cudaStream_t st) {
  AVF_REQUIRE(rows > 1, AVF_EINVAL, "batch_norm(train): needs more than one row per channel (rows=%d)", rows);   // like torch
  AVF_REQUIRE(x && g && b && y && save_mean && save_rstd, AVF_EINVAL, "batch_norm(train): null pointer");
  if (out_mode == AVF_BF16)
    launch_pdl(bn_train_fwd_kernel<__nv_bfloat16>, ceil_div(dim, 32), 256, 0, st, x, ld_x, g, b, run_mean, run_var, momentum, static_cast<__nv_bfloat16*>(y), save_mean, save_rstd, rows, dim);
  else
    launch_pdl(bn_train_fwd_kernel<float>, ceil_div(dim, 32), 256, 0, st, x, ld_x, g, b, run_mean, run_var, momentum, static_cast<float*>(y), save_mean, save_rstd, rows, dim);
  AVF_LAUNCH_CHECK("bn_train_fwd_kernel");
  return 0;
}

int bn_bwd(const float* x, int ld_x, const float* dy, const float* g, const float* mean, const float* rstd_or_var, int batch_stats, float* dx,
           int ld_dx, float* dgamma, float* dbeta, int rows, int dim, cudaStream_t st) {
  AVF_REQUIRE(rows > 0 && x && dy && g && mean && rstd_or_var, AVF_EINVAL, "batch_norm_bwd: null pointer / rows=%d", rows);
  launch_pdl(bn_bwd_kernel, ceil_div(dim, 32), 256, 0, st, x, ld_x, dy, g, mean, rstd_or_var, batch_stats, dx, ld_dx, dgamma, dbeta, rows, dim);
  AVF_LAUNCH_CHECK("bn_bwd_kernel");
  return 0;
}

int adam_step(float* p, const float* g, float* m, float* v, void* shadow, size_t n, float lr, float b1, float b2, float eps, float wd, int step,
              int decoupled, float grad_scale, cudaStream_t st) {
  AVF_REQUIRE(p && g && m && v, AVF_EINVAL, "adam_step: null pointer");
  AVF_REQUIRE(step >= 1, AVF_EINVAL, "adam_step: step=%d (1-based)", step);
  if (n == 0) return 0;
  AVF_REQUIRE(((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15) == 0,
              AVF_EINVAL, "adam_step: buckets must be 16-byte aligned");
  const double bc1 = 1.0 - pow(double(b1), step), bc2 = 1.0 - pow(double(b2), step);
  launch_pdl(adam_kernel, unsigned((n / 4 + 256) / 256), 256, 0, st, p, g, m, v, static_cast<__nv_bfloat16*>(shadow), n, lr, b1, b2, eps, wd, float(1.0 / bc1),
                                                               float(1.0 / sqrt(bc2)), decoupled, grad_scale);
  AVF_LAUNCH_CHECK("adam_kernel");
  return 0;
}

}  // namespace avf
