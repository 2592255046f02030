// CUDA-core kernels: the fp32 "parity mode" GEMM (1e-4-relative agreement with the reference needs
// true fp32 products, which the tensor cores do not offer) and the small-sequence attention
// (N <= 64 tokens: 12 / 17 / 49) used by both modes outside the fused tcgen05 layer kernel.
// Masked fp32 attention of 65..256 tokens (64-wide heads) has a kernel of its own.
#include "avf_common.cuh"
#include "avf_internal.h"

namespace avf {

namespace {

// ---------------------------------------------------------------------------------------------
// fp32 GEMM  C[M,N] = epi(A[M,K] W[N,K]^T), 64x64 tile, 16x16 threads x (4x4) micro-tile, BK = 16
// ---------------------------------------------------------------------------------------------
template <typename OutT>
__global__ void __launch_bounds__(256) gemm_f32_kernel(const float* __restrict__ A, int lda, const float* __restrict__ W,
                                                       OutT* __restrict__ C, int ldc, const float* __restrict__ bias,
                                                       const float* __restrict__ res, int ld_res, int M, int N, int K, int flags) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  __shared__ float As[16][64 + 4];
  __shared__ float Ws[16][64 + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  float acc[4][4] = {};
  const int lr = threadIdx.x >> 2, lk = (threadIdx.x & 3) * 4;     // 64 rows x 4 float4 per 16-wide k-slab
  for (int k0 = 0; k0 < K; k0 += 16) {
    float4 a = make_float4(0, 0, 0, 0), w = make_float4(0, 0, 0, 0);
    if (m0 + lr < M) a = *reinterpret_cast<const float4*>(A + size_t(m0 + lr) * lda + k0 + lk);
    if (n0 + lr < N) w = __ldg(reinterpret_cast<const float4*>(W + size_t(n0 + lr) * K + k0 + lk));
    As[lk][lr] = a.x; As[lk + 1][lr] = a.y; As[lk + 2][lr] = a.z; As[lk + 3][lr] = a.w;
    Ws[lk][lr] = w.x; Ws[lk + 1][lr] = w.y; Ws[lk + 2][lr] = w.z; Ws[lk + 3][lr] = w.w;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 wv = *reinterpret_cast<const float4*>(&Ws[k][tx * 4]);
      const float a4[4] = {av.x, av.y, av.z, av.w}, w4[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], w4[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = m0 + ty * 4 + i;
    if (r >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = n0 + tx * 4 + j;
      if (c >= N) continue;
      float v = acc[i][j];
      if (flags & AVF_EPI_BIAS) v += bias[c];
      if (flags & AVF_EPI_GELU) v = gelu_tanh<false>(v);
      if (flags & AVF_EPI_RESIDUAL) v += res[size_t(r) * ld_res + c];
      C[size_t(r) * ldc + c] = from_f32<OutT>(v);
    }
  }
}


// Same tile shape with arbitrary operand orientation (training, parity mode): element (m,k) of A sits at
// A[m*a_rs + k*a_cs], element (n,k) of W at W[n*w_rs + k*w_cs].  Scalar loads: this is the fp32 checking path.
template <typename OutT>
__global__ void __launch_bounds__(256) gemm_f32_generic_kernel(const float* __restrict__ A, long a_rs, long a_cs, const float* __restrict__ W,
                                                               long w_rs, long w_cs, OutT* __restrict__ C, int ldc,
                                                               const float* __restrict__ bias, const float* __restrict__ res, int ld_res,
                                                               float* aux, int ld_aux, int M, int N, int K, int flags, DropSpec drop) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  __shared__ float As[16][64 + 4];
  __shared__ float Ws[16][64 + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  drop = drop_resolve(drop);
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = threadIdx.x + i * 256;
      // make the contiguous index the fast one so that loads coalesce in either orientation
      const int kk_a = a_cs == 1 ? idx & 15 : idx >> 6, mm = a_cs == 1 ? idx >> 4 : idx & 63;
      const int kk_w = w_cs == 1 ? idx & 15 : idx >> 6, nn = w_cs == 1 ? idx >> 4 : idx & 63;
      As[kk_a][mm] = (m0 + mm < M && k0 + kk_a < K) ? A[(m0 + mm) * a_rs + (k0 + kk_a) * a_cs] : 0.f;
      Ws[kk_w][nn] = (n0 + nn < N && k0 + kk_w < K) ? W[(n0 + nn) * w_rs + (k0 + kk_w) * w_cs] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 wv = *reinterpret_cast<const float4*>(&Ws[k][tx * 4]);
      const float a4[4] = {av.x, av.y, av.z, av.w}, w4[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], w4[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = m0 + ty * 4 + i;
    if (r >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = n0 + tx * 4 + j;
      if (c >= N) continue;
      float v = acc[i][j];
      if (flags & AVF_EPI_DGELU) v *= gelu_tanh_grad(aux[size_t(r) * ld_aux + c]);
      if (flags & AVF_EPI_BIAS) v += bias[c];
      if (flags & AVF_EPI_SAVE_PRE) aux[size_t(r) * ld_aux + c] = v;
      if (flags & AVF_EPI_GELU) v = gelu_tanh<false>(v);
      if (flags & AVF_EPI_DROPOUT) v *= drop_factor(drop, uint32_t(r) * uint32_t(N) + uint32_t(c));
      if (flags & AVF_EPI_RESIDUAL) v += res[size_t(r) * ld_res + c];
      if (flags & AVF_EPI_ACCUMULATE) v += to_f32<OutT>(C[size_t(r) * ldc + c]);
      C[size_t(r) * ldc + c] = from_f32<OutT>(v);
    }
  }
}

// 16-byte vectorised row-fragment load (global or shared) with conversion to fp32.
template <typename T, int N>
__device__ __forceinline__ void load_frag(const T* __restrict__ p, float (&dst)[N]) {
  if constexpr (sizeof(T) == 4) {
#pragma unroll
    for (int i = 0; i < N; i += 4) {
      const float4 v = *reinterpret_cast<const float4*>(p + i);
      dst[i] = v.x; dst[i + 1] = v.y; dst[i + 2] = v.z; dst[i + 3] = v.w;
    }
  } else {
#pragma unroll
    for (int i = 0; i < N; i += 8) {
      const uint4 v = *reinterpret_cast<const uint4*>(p + i);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        dst[i + 2 * j] = __uint_as_float(w[j] << 16);
        dst[i + 2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
      }
    }
  }
}
template <typename T, int N>
__device__ __forceinline__ void store_frag(T* __restrict__ p, const float (&src)[N]) {
  if constexpr (sizeof(T) == 4) {
#pragma unroll
    for (int i = 0; i < N; i += 4) *reinterpret_cast<float4*>(p + i) = make_float4(src[i], src[i + 1], src[i + 2], src[i + 3]);
  } else {
#pragma unroll
    for (int i = 0; i < N; i += 8) {
      uint4 o;
      o.x = pack_bf16x2(src[i], src[i + 1]);
      o.y = pack_bf16x2(src[i + 2], src[i + 3]);
      o.z = pack_bf16x2(src[i + 4], src[i + 5]);
      o.w = pack_bf16x2(src[i + 6], src[i + 7]);
      *reinterpret_cast<uint4*>(p + i) = o;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Small-sequence attention, models/heads.py:221-237.  qkv [rows, 3*H*dh] (columns q|k|v, head-major),
// out [rows, H*dh].  A CTA stages K and V of `spb` sequences in shared memory; each thread owns one
// (sequence, head, query) row and runs an online softmax in base 2 over the <= 64 keys.
// MASKED: keep [n_seq, n_tok] uint8 (1 = keep); one warp per staged sequence turns its row into 64 keep bits (behind K|V in shared
// memory).  A kept query skips the dropped keys; a dropped query attends uniformly to all n_tok keys (every score filled alike), so
// its running max starts from a real score and never meets -INF - (-INF).
// ---------------------------------------------------------------------------------------------
template <typename T, int DH, bool MASKED>
__global__ void __launch_bounds__(DH == 32 ? 512 : 256) attention_small_kernel(const T* __restrict__ qkv, T* __restrict__ out, int n_seq, int n_tok,
                                                              int heads, int spb, int hpb, float scale_log2e, const uint8_t* __restrict__ keep) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  extern __shared__ uint8_t smem_attn[];
  T* kv = reinterpret_cast<T*>(smem_attn);                // [spb][n_tok][2][hpb*DH]  (k | v of the block's head group)
  const int inner = heads * DH;
  const int seq0 = blockIdx.x * spb;
  const int nseq_here = min(spb, n_seq - seq0);
  const int h0 = blockIdx.y * hpb, nh = min(hpb, heads - h0), w = hpb * DH;
  // cooperative, 16-byte vectorised copy of the K|V column block of each row
  constexpr int VEC = 16 / sizeof(T);
  const int vec_per_row = 2 * w / VEC;
  const int total_vec = nseq_here * n_tok * vec_per_row;
  for (int i = threadIdx.x; i < total_vec; i += blockDim.x) {
    const int r = i / vec_per_row, c = (i - r * vec_per_row) * VEC;
    const int part = c / w, col = c - part * w;          // 0: k, 1: v
    if (col >= nh * DH) continue;
    const uint4 v = *reinterpret_cast<const uint4*>(qkv + (size_t(seq0) * n_tok + r) * (3 * inner) + size_t(1 + part) * inner + h0 * DH + col);
    *reinterpret_cast<uint4*>(kv + size_t(r) * 2 * w + c) = v;
  }
  uint64_t* kmask = reinterpret_cast<uint64_t*>(kv + size_t(spb) * n_tok * 2 * w);     // [spb] keep bits (MASKED only)
  if constexpr (MASKED) {
    const int lane = threadIdx.x & 31;
    for (int sl = threadIdx.x >> 5; sl < nseq_here; sl += blockDim.x >> 5) {
      const uint8_t* row = keep + size_t(seq0 + sl) * n_tok;
      const uint32_t lo = __ballot_sync(0xffffffffu, lane < n_tok && row[lane] != 0);
      const uint32_t hi = __ballot_sync(0xffffffffu, lane + 32 < n_tok && row[lane + 32] != 0);
      if (lane == 0) kmask[sl] = (uint64_t(hi) << 32) | lo;
    }
  }
  __syncthreads();
  const int items = nseq_here * nh * n_tok;
  for (int it = threadIdx.x; it < items; it += blockDim.x) {
    const int qi = it % n_tok;
    const int hl = (it / n_tok) % nh, h = h0 + hl;
    const int sl = it / (n_tok * nh);
    const size_t row = (size_t(seq0 + sl)) * n_tok + qi;
    float q[DH];
    load_frag<T, DH>(qkv + row * (3 * inner) + h * DH, q);
#pragma unroll
    for (int d = 0; d < DH; ++d) q[d] *= scale_log2e;
    float m = -INFINITY, l = 0.f, acc[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] = 0.f;
    const T* kbase = kv + size_t(sl) * n_tok * 2 * w + hl * DH;
    const uint64_t km = MASKED ? kmask[sl] : 0;
    const bool row_kept = !MASKED || ((km >> qi) & 1);
    for (int j = 0; j < n_tok; ++j) {
      if (MASKED && row_kept && !((km >> j) & 1)) continue;
      const T* kp = kbase + size_t(j) * 2 * w;
      float kf[DH];
      load_frag<T, DH>(kp, kf);
      float s = 0.f;
      if (row_kept) {
#pragma unroll
        for (int d = 0; d < DH; ++d) s = fmaf(q[d], kf[d], s);
      }
      if (s > m) {
        const float corr = exp2f(m - s);
        l *= corr;
#pragma unroll
        for (int d = 0; d < DH; ++d) acc[d] *= corr;
        m = s;
      }
      const float p = exp2f(s - m);
      l += p;
      load_frag<T, DH>(kp + w, kf);
#pragma unroll
      for (int d = 0; d < DH; ++d) acc[d] = fmaf(p, kf[d], acc[d]);
    }
    const float inv = 1.f / l;
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] *= inv;
    store_frag<T, DH>(out + row * inner + h * DH, acc);
  }
}

// Masked fp32 attention of 65..256 tokens with 64-wide heads: one CTA per (sequence, head), K|V of the head in shared memory
// ([n_tok][2][64], the layout of attention_small_kernel with one head per block) and the keep bits as four 64-bit words behind them.
// Every query row runs the per-thread online softmax of attention_small_kernel in the same order, so an all-kept mask gives the
// bits of the unmasked call.
__global__ void __launch_bounds__(256) attention_long_f32_kernel(const float* __restrict__ qkv, float* __restrict__ out, int n_tok, int heads,
                                                                 float scale_log2e, const uint8_t* __restrict__ keep) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  constexpr int DH = 64;
  extern __shared__ __align__(16) uint8_t smem_long_f32[];
  float* kv = reinterpret_cast<float*>(smem_long_f32);
  uint64_t* km = reinterpret_cast<uint64_t*>(kv + size_t(n_tok) * 2 * DH);
  const int seq = blockIdx.x / heads, h = blockIdx.x - seq * heads;
  const int inner = heads * DH, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t row0 = size_t(seq) * n_tok;
  for (int i = threadIdx.x; i < n_tok * 2 * DH / 4; i += blockDim.x) {
    const int r = i / (2 * DH / 4), c = (i - r * (2 * DH / 4)) * 4;
    const int part = c / DH, col = c - part * DH;
    *reinterpret_cast<float4*>(kv + size_t(r) * 2 * DH + c) =
        *reinterpret_cast<const float4*>(qkv + (row0 + r) * (3 * inner) + size_t(1 + part) * inner + h * DH + col);
  }
  if (warp < 4) {
    const int b = warp * 64;
    const uint8_t* row = keep + row0 + b;
    const uint32_t lo = __ballot_sync(0xffffffffu, b + lane < n_tok && row[lane] != 0);
    const uint32_t hi = __ballot_sync(0xffffffffu, b + lane + 32 < n_tok && row[lane + 32] != 0);
    if (lane == 0) km[warp] = (uint64_t(hi) << 32) | lo;
  }
  __syncthreads();
  for (int qi = threadIdx.x; qi < n_tok; qi += blockDim.x) {
    const size_t row = row0 + qi;
    float q[DH];
    load_frag<float, DH>(qkv + row * (3 * inner) + h * DH, q);
#pragma unroll
    for (int d = 0; d < DH; ++d) q[d] *= scale_log2e;
    float m = -INFINITY, l = 0.f, acc[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] = 0.f;
    const bool row_kept = (km[qi >> 6] >> (qi & 63)) & 1;
    for (int j = 0; j < n_tok; ++j) {
      if (row_kept && !((km[j >> 6] >> (j & 63)) & 1)) continue;
      const float* kp = kv + size_t(j) * 2 * DH;
      float kf[DH];
      load_frag<float, DH>(kp, kf);
      float s = 0.f;
      if (row_kept) {
#pragma unroll
        for (int d = 0; d < DH; ++d) s = fmaf(q[d], kf[d], s);
      }
      if (s > m) {
        const float corr = exp2f(m - s);
        l *= corr;
#pragma unroll
        for (int d = 0; d < DH; ++d) acc[d] *= corr;
        m = s;
      }
      const float p = exp2f(s - m);
      l += p;
      load_frag<float, DH>(kp + DH, kf);
#pragma unroll
      for (int d = 0; d < DH; ++d) acc[d] = fmaf(p, kf[d], acc[d]);
    }
    const float inv = 1.f / l;
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] *= inv;
    store_frag<float, DH>(out + row * inner + h * DH, acc);
  }
}

}  // namespace

int linear_f32(const float* a, int lda, const float* w, const float* bias, const float* res, int ld_res, void* c, int ldc,
               int c_mode, int m, int n, int k, int flags, cudaStream_t st) {
  AVF_REQUIRE(m > 0 && n > 0 && k > 0, AVF_EINVAL, "linear: empty problem m=%d n=%d k=%d", m, n, k);
  AVF_REQUIRE(k % 16 == 0 && lda % 4 == 0, AVF_EUNSUPPORTED, "linear(fp32): K=%d must be a multiple of 16 (lda=%d of 4)", k, lda);
  dim3 grid(ceil_div(n, 64), ceil_div(m, 64));
  if (c_mode == AVF_BF16) launch_pdl(gemm_f32_kernel<__nv_bfloat16>, grid, 256, 0, st, a, lda, w, static_cast<__nv_bfloat16*>(c), ldc, bias, res, ld_res, m, n, k, flags);
  else launch_pdl(gemm_f32_kernel<float>, grid, 256, 0, st, a, lda, w, static_cast<float*>(c), ldc, bias, res, ld_res, m, n, k, flags);
  AVF_LAUNCH_CHECK("gemm_f32_kernel");
  return 0;
}

int gemm_f32(int trans_a, int trans_b, const float* a, int lda, const float* w, int ldw, const float* bias, const float* res, int ld_res,
             float* aux, int ld_aux, void* c, int ldc, int c_mode, int m, int n, int k, int flags, cudaStream_t st, DropSpec drop) {
  AVF_REQUIRE(m > 0 && n > 0 && k > 0, AVF_EINVAL, "linear: empty problem m=%d n=%d k=%d", m, n, k);
  AVF_REQUIRE(!(flags & (AVF_EPI_DGELU | AVF_EPI_SAVE_PRE)) || aux != nullptr, AVF_EINVAL, "linear(fp32): DGELU / SAVE_PRE epilogues need the pre-activation buffer");
  if (!trans_a && !trans_b && ldw == k && !(flags & (AVF_EPI_DGELU | AVF_EPI_SAVE_PRE | AVF_EPI_DROPOUT | AVF_EPI_ACCUMULATE)) && k % 16 == 0 && lda % 4 == 0)
    return linear_f32(a, lda, w, bias, res, ld_res, c, ldc, c_mode, m, n, k, flags, st);
  dim3 grid(ceil_div(n, 64), ceil_div(m, 64));
  const long a_rs = trans_a ? 1 : lda, a_cs = trans_a ? lda : 1, w_rs = trans_b ? 1 : ldw, w_cs = trans_b ? ldw : 1;
  if (c_mode == AVF_BF16)
    launch_pdl(gemm_f32_generic_kernel<__nv_bfloat16>, grid, 256, 0, st, a, a_rs, a_cs, w, w_rs, w_cs, static_cast<__nv_bfloat16*>(c), ldc, bias, res, ld_res, aux, ld_aux, m, n, k, flags, drop);
  else
    launch_pdl(gemm_f32_generic_kernel<float>, grid, 256, 0, st, a, a_rs, a_cs, w, w_rs, w_cs, static_cast<float*>(c), ldc, bias, res, ld_res, aux, ld_aux, m, n, k, flags, drop);
  AVF_LAUNCH_CHECK("gemm_f32_generic_kernel");
  return 0;
}

template <typename T, int DH, bool MASKED>
static int launch_attention(const void* qkv, void* out, int n_seq, int n_tok, int heads, const uint8_t* keep, cudaStream_t st) {
  const int inner = heads * DH;
  int hpb = heads;                                        // heads staged per block: all of them unless K|V of a sequence exceed 96 KB
  while (hpb > 1 && size_t(n_tok) * 2 * hpb * DH * sizeof(T) > 96 * 1024) hpb = (hpb + 1) / 2;
  const size_t per_seq = size_t(n_tok) * 2 * hpb * DH * sizeof(T);
  const int threads_per_seq = hpb * n_tok;
  constexpr int kMaxThreads = DH == 32 ? 512 : 256;
  int spb = max(1, min(kMaxThreads / threads_per_seq, int((96 * 1024) / per_seq)));
  spb = min(spb, n_seq);
  const size_t smem = per_seq * spb + (MASKED ? spb * sizeof(uint64_t) : 0);
  AVF_REQUIRE(smem <= 200 * 1024, AVF_EUNSUPPORTED, "attention: %d tokens x %d inner does not fit shared memory", n_tok, inner);
  int threads = min(kMaxThreads, ceil_div(threads_per_seq * spb, 32) * 32);
  auto kern = attention_small_kernel<T, DH, MASKED>;
  static PerDeviceOnce once;
  if (once.first()) {
    AVF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  const float scale_log2e = 1.4426950408889634f / sqrtf(float(DH));
  launch_pdl(kern, dim3(ceil_div(n_seq, spb), ceil_div(heads, hpb)), threads, smem, st, static_cast<const T*>(qkv), static_cast<T*>(out), n_seq, n_tok, heads, spb, hpb,
                                                                               scale_log2e, keep);
  AVF_LAUNCH_CHECK("attention_small_kernel");
  return 0;
}

int attention_small(int io_mode, const void* qkv, void* out, int n_seq, int n_tok, int heads, int dim_head, cudaStream_t st, const uint8_t* keep) {
  AVF_REQUIRE(n_seq > 0 && n_tok > 0 && heads > 0, AVF_EINVAL, "attention: n_seq=%d n_tok=%d heads=%d", n_seq, n_tok, heads);
  AVF_REQUIRE(dim_head == 32 || dim_head == 64, AVF_EUNSUPPORTED, "attention: dim_head=%d (supported: 32, 64)", dim_head);
  AVF_REQUIRE(keep == nullptr || n_tok <= 64 || (dim_head == 64 && n_tok <= 256), AVF_EUNSUPPORTED,
              "attention: a keep mask needs n_tok <= 64, or <= 256 with 64-wide heads (n_tok=%d, dim_head=%d)", n_tok, dim_head);
  if (io_mode == AVF_BF16) return attention_mma_bf16(qkv, out, n_seq, n_tok, heads, dim_head, st, 0, keep);   // tensor cores
  if (keep != nullptr && n_tok > 64) {
    const size_t smem = size_t(n_tok) * 2 * 64 * sizeof(float) + 4 * sizeof(uint64_t);
    static PerDeviceOnce once;
    if (once.first()) {
      AVF_CUDA(cudaFuncSetAttribute(attention_long_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(256 * 2 * 64 * sizeof(float) + 32)));
    }
    launch_pdl(attention_long_f32_kernel, n_seq * heads, 256, smem, st, static_cast<const float*>(qkv), static_cast<float*>(out), n_tok, heads,
               1.4426950408889634f / sqrtf(64.f), keep);
    AVF_LAUNCH_CHECK("attention_long_f32_kernel");
    return 0;
  }
  if (keep != nullptr)
    return dim_head == 32 ? launch_attention<float, 32, true>(qkv, out, n_seq, n_tok, heads, keep, st)
                          : launch_attention<float, 64, true>(qkv, out, n_seq, n_tok, heads, keep, st);
  return dim_head == 32 ? launch_attention<float, 32, false>(qkv, out, n_seq, n_tok, heads, nullptr, st)
                        : launch_attention<float, 64, false>(qkv, out, n_seq, n_tok, heads, nullptr, st);
}

}  // namespace avf
