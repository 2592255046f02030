// Memory-bound pieces of the AVFormer hot path as vectorised, coalesced warp-shuffle kernels:
// LayerNorm, BatchNorm(eval) rows, SFormer NCHW<->token transposes (+pos), TFormer cls/pos embed,
// casts, the 12 per-AU dot products + decisions, and the pos-weighted BCE (+gradient).
#include <algorithm>

#include "avf_common.cuh"

namespace avf {

namespace {

// ---------------------------------------------------------------------------------------------
// LayerNorm: one warp per row, row kept in registers (dim <= 1536, dim % 128 == 0; 1536 = the TFormer of models/tformer.py:301)
// nn.LayerNorm(dim) of PreNorm, models/heads.py:178-185 (biased variance, eps = 1e-5)
// ---------------------------------------------------------------------------------------------
template <typename OutT, int VEC>   // VEC float4 per lane: dim = 128 * VEC
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, int ld_x, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, OutT* __restrict__ y, int rows) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  constexpr int DIM = 128 * VEC;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float4* xp = reinterpret_cast<const float4*>(x + size_t(row) * ld_x);
  float4 v[VEC];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    v[i] = xp[lane + 32 * i];
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mean = warp_sum(s) * (1.0f / DIM);
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
    ss += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
  }
  const float rstd = rsqrtf(warp_sum(ss) * (1.0f / DIM) + 1e-5f);
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const int c = (lane + 32 * i) * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta + c));
    const float o0 = v[i].x * rstd * g.x + b.x, o1 = v[i].y * rstd * g.y + b.y;
    const float o2 = v[i].z * rstd * g.z + b.z, o3 = v[i].w * rstd * g.w + b.w;
    if constexpr (sizeof(OutT) == 4) {
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + size_t(row) * DIM + c) = make_float4(o0, o1, o2, o3);
    } else {
      uint2 o;
      o.x = pack_bf16x2(o0, o1);
      o.y = pack_bf16x2(o2, o3);
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(y) + size_t(row) * DIM + c) = o;
    }
  }
}

// BatchNorm1d with running statistics (AU_BN1 in eval, models/heads.py:263,293) on strided rows.
template <typename OutT>
__global__ void bn_rows_kernel(const float* __restrict__ x, int ld_x, const float* __restrict__ g, const float* __restrict__ b,
                               const float* __restrict__ mean, const float* __restrict__ var, OutT* __restrict__ y,
                               int rows, int dim) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * dim) return;
  const int r = idx / dim, c = idx - r * dim;
  const float v = (x[size_t(r) * ld_x + c] - mean[c]) * rsqrtf(var[c] + 1e-5f) * g[c] + b[c];
  y[idx] = from_f32<OutT>(v);
}

// ---------------------------------------------------------------------------------------------
// SFormer token packing: fmap [F, dim, hw] -> x [F*hw, dim] + pos  (models/vformer.py:247-253) and back (:257-259).
// One frame per CTA iteration, staged in shared memory as fp32 in its NATURAL [dim][hw] order:
//   * the NCHW side is moved with 16-byte vectors over the flat frame (fully coalesced);
//   * the token side is moved one token row at a time, lane <-> channel: a warp instruction reads / writes 32 consecutive
//     fp32 of a token row (128 B, coalesced) and touches tile[(c0 + lane) * hw + t] in shared memory — conflict-free
//     whenever hw is odd (7x7 = 49: bank = (17 lane + t) mod 32), at most 2-way otherwise (pitch hw|1).
// ---------------------------------------------------------------------------------------------
template <typename T> struct Vec16;      // 16-byte global access of 8 bf16 / 4 fp32
template <> struct Vec16<__nv_bfloat16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&f)[8]) {
    const uint4 v = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) { f[2 * q] = __uint_as_float(w[q] << 16); f[2 * q + 1] = __uint_as_float(w[q] & 0xffff0000u); }
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&f)[8]) {
    uint4 v;
    v.x = pack_bf16x2(f[0], f[1]); v.y = pack_bf16x2(f[2], f[3]); v.z = pack_bf16x2(f[4], f[5]); v.w = pack_bf16x2(f[6], f[7]);
    *reinterpret_cast<uint4*>(p) = v;
  }
};
template <> struct Vec16<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ void load(const float* p, float (&f)[4]) {
    const float4 v = *reinterpret_cast<const float4*>(p);
    f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&f)[4]) { *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]); }
};

template <typename InT>
__global__ void __launch_bounds__(256) sformer_pack_kernel(const InT* __restrict__ fmap, const float* __restrict__ pos,
                                                           float* __restrict__ x, int n_frames, int dim, int hw) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  extern __shared__ float tile[];               // [dim][pitch], pitch = hw | 1
  constexpr int V = Vec16<InT>::N;
  const int pitch = hw | 1, n = dim * hw;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int f = blockIdx.x; f < n_frames; f += gridDim.x) {
    const InT* src = fmap + size_t(f) * n;
    for (int i = threadIdx.x * V; i < n; i += blockDim.x * V) {          // n % V == 0 is checked by the launcher
      float v[V];
      Vec16<InT>::load(src + i, v);
      if (pitch == hw) {                         // odd hw: the tile IS the flat frame -> 16-byte shared-memory stores
#pragma unroll
        for (int j = 0; j < V; j += 4) *reinterpret_cast<float4*>(&tile[i + j]) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      } else {
        int c = i / hw, t = i - c * hw;
#pragma unroll
        for (int j = 0; j < V; ++j) {
          tile[c * pitch + t] = v[j];
          if (++t == hw) { t = 0; ++c; }
        }
      }
    }
    __syncthreads();
    float* dst = x + size_t(f) * n;
    for (int t = warp; t < hw; t += 8) {
      for (int c = lane; c < dim; c += 32) {
        const float p = pos != nullptr ? __ldg(pos + t * dim + c) : 0.f;
        dst[t * dim + c] = tile[c * pitch + t] + p;
      }
    }
    __syncthreads();
  }
}

// x [F*hw, dim] -> fmap [F, dim, hw]   (models/vformer.py:257-259)
template <typename OutT>
__global__ void __launch_bounds__(256) sformer_unpack_kernel(const float* __restrict__ x, OutT* __restrict__ fmap, int n_frames, int dim, int hw) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  extern __shared__ float tile[];               // [dim][pitch]
  constexpr int V = Vec16<OutT>::N;
  const int pitch = hw | 1, n = dim * hw;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int f = blockIdx.x; f < n_frames; f += gridDim.x) {
    const float* src = x + size_t(f) * n;
    for (int t = warp; t < hw; t += 8)
      for (int c = lane; c < dim; c += 32) tile[c * pitch + t] = src[t * dim + c];
    __syncthreads();
    OutT* dst = fmap + size_t(f) * n;
    for (int i = threadIdx.x * V; i < n; i += blockDim.x * V) {
      float v[V];
      if (pitch == hw) {
#pragma unroll
        for (int j = 0; j < V; j += 4) {
          const float4 q = *reinterpret_cast<const float4*>(&tile[i + j]);
          v[j] = q.x; v[j + 1] = q.y; v[j + 2] = q.z; v[j + 3] = q.w;
        }
      } else {
        int c = i / hw, t = i - c * hw;
#pragma unroll
        for (int j = 0; j < V; ++j) {
          v[j] = tile[c * pitch + t];
          if (++t == hw) { t = 0; ++c; }
        }
      }
      Vec16<OutT>::store(dst + i, v);
    }
    __syncthreads();
  }
}

// TFormer embed: x[c, 0, :] = cls + pos[0]; x[c, t+1, :] = frames[c*T+t, :] + pos[t+1]   (models/vformer.py:283-286)
template <typename InT>
__global__ void tformer_embed_kernel(const InT* __restrict__ frames, const float* __restrict__ cls, const float* __restrict__ pos,
                                     float* __restrict__ x, int n_clips, int T, int dim) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const size_t idx = size_t(blockIdx.x) * blockDim.x + threadIdx.x;      // over float4 groups
  const int d4 = dim >> 2;
  const size_t total = size_t(n_clips) * (T + 1) * d4;
  if (idx >= total) return;
  const int c4 = int(idx % d4);
  const size_t r = idx / d4;
  const int tok = int(r % (T + 1));
  const size_t clip = r / (T + 1);
  float4 v;
  if (tok == 0) {
    v = __ldg(reinterpret_cast<const float4*>(cls) + c4);
  } else {
    const InT* fp = frames + (clip * T + (tok - 1)) * size_t(dim) + c4 * 4;
    v = make_float4(to_f32<InT>(fp[0]), to_f32<InT>(fp[1]), to_f32<InT>(fp[2]), to_f32<InT>(fp[3]));
  }
  const float4 p = __ldg(reinterpret_cast<const float4*>(pos + size_t(tok) * dim) + c4);
  reinterpret_cast<float4*>(x)[idx] = make_float4(v.x + p.x, v.y + p.y, v.z + p.z, v.w + p.w);
}

// The same embed with the frames gathered from a per-video frame bank (models/vformer.py:280-290 on clips described by frame indices):
// i = index[c*T + t]; x[c, t+1, :] = bank[i, :] + pos[t+1] when 0 <= i < n_bank, else pos[t+1] alone (a missing frame, value 0).
// keep[c, 0] = 1 and keep[c, t+1] = (0 <= i < n_bank): the attention mask of the layers that follow.  The bank is never read outside
// [0, n_bank), whatever the index holds.
template <typename InT>
__global__ void tformer_embed_indexed_kernel(const InT* __restrict__ bank, int n_bank, const int* __restrict__ index, const float* __restrict__ cls,
                                             const float* __restrict__ pos, float* __restrict__ x, uint8_t* __restrict__ keep, int n_clips, int T, int dim) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const size_t idx = size_t(blockIdx.x) * blockDim.x + threadIdx.x;      // over float4 groups
  const int d4 = dim >> 2;
  const size_t total = size_t(n_clips) * (T + 1) * d4;
  if (idx >= total) return;
  const int c4 = int(idx % d4);
  const size_t r = idx / d4;
  const int tok = int(r % (T + 1));
  const size_t clip = r / (T + 1);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  bool real = true;
  if (tok == 0) {
    v = __ldg(reinterpret_cast<const float4*>(cls) + c4);
  } else {
    const int i = __ldg(index + clip * T + (tok - 1));
    real = unsigned(i) < unsigned(n_bank);
    if (real) {
      const InT* fp = bank + size_t(i) * dim + c4 * 4;
      if constexpr (sizeof(InT) == 4) {
        v = __ldg(reinterpret_cast<const float4*>(fp));
      } else {
        const uint2 q = __ldg(reinterpret_cast<const uint2*>(fp));
        v = make_float4(__uint_as_float(q.x << 16), __uint_as_float(q.x & 0xffff0000u), __uint_as_float(q.y << 16), __uint_as_float(q.y & 0xffff0000u));
      }
    }
  }
  const float4 p = __ldg(reinterpret_cast<const float4*>(pos + size_t(tok) * dim) + c4);
  reinterpret_cast<float4*>(x)[idx] = make_float4(v.x + p.x, v.y + p.y, v.z + p.z, v.w + p.w);
  if (c4 == 0) keep[r] = real ? 1 : 0;
}

__global__ void rows_gather_kernel(const float* __restrict__ x, size_t src_row_stride, float* __restrict__ y, int rows, int dim) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * dim) return;
  const int r = idx / dim, c = idx - r * dim;
  y[idx] = x[size_t(r) * src_row_stride + c];
}

__global__ void add_row_periodic_kernel(float* __restrict__ x, int ld_x, const float* __restrict__ pos, int rows, int dim, int period) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * dim) return;
  const int r = idx / dim, c = idx - r * dim;
  x[size_t(r) * ld_x + c] += pos[size_t(r % period) * dim + c];
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ s, __nv_bfloat16* __restrict__ d, size_t n) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const size_t i = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(s + i);
    uint2 o;
    o.x = pack_bf16x2(v.x, v.y);
    o.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(d + i) = o;
  } else {
    for (size_t j = i; j < n; ++j) d[j] = __float2bfloat16_rn(s[j]);
  }
}
__global__ void cast_bf16_f32_kernel(const __nv_bfloat16* __restrict__ s, float* __restrict__ d, size_t n) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) d[i] = __bfloat162float(s[i]);
}

// ---------------------------------------------------------------------------------------------
// Fusion-head tail: 12 x Linear(dim,1,bias=False) on token i (models/tformer.py:389-401), zero-padded
// [B,21] output (models/avformer.py:102-105) and decisions round(sigmoid(x)) == x > 0 (train.py:155).
// One warp per (clip, AU).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) au_logits_kernel(const float* __restrict__ x, int ld_x, const float* __restrict__ w_last,
                                                        float* __restrict__ out21, int* __restrict__ decisions, int n_clips, int dim) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (gw >= n_clips * 12) return;
  const int au = gw % 12;
  const float* xp = x + size_t(gw) * ld_x;
  const float* wp = w_last + size_t(au) * dim;
  float s = 0.f;
  for (int c = lane * 4; c < dim; c += 128) {
    const float4 a = *reinterpret_cast<const float4*>(xp + c);
    const float4 b = __ldg(reinterpret_cast<const float4*>(wp + c));
    s += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
  }
  s = warp_sum(s);
  if (lane == 0) {
    const int clip = gw / 12;
    if (out21) out21[size_t(clip) * 21 + au] = s;
    if (decisions) decisions[gw] = s > 0.f ? 1 : 0;
  }
  if (out21 && au == 0 && lane < 9) out21[size_t(gw / 12) * 21 + 12 + lane] = 0.f;
}

// AULoss (models/loss.py:75-103) in one CTA: valid rows = labels[:,0] != -1; stable BCE-with-logits
//   l = (1-y) x + (1 + (w-1) y) softplus(-x);  loss = sum / (12 * n_valid)
// and its gradient (sigma(x)(1+(w-1)y) - w y) / (12 n_valid).
__global__ void __launch_bounds__(256) au_bce_kernel(const float* __restrict__ logits, int ld, const float* __restrict__ labels,
                                                     const float* __restrict__ pw, float* __restrict__ loss_out,
                                                     float* __restrict__ dlogits, int n_clips) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  __shared__ float red[2][8];
  __shared__ float tot[2];
  float lsum = 0.f, nvalid = 0.f;
  for (int i = threadIdx.x; i < n_clips * 12; i += blockDim.x) {
    const int r = i / 12, c = i - r * 12;
    if (labels[r * 12] == -1.0f) continue;
    const float xv = logits[size_t(r) * ld + c], y = labels[i], w = pw[c];
    const float sp = fmaxf(-xv, 0.f) + log1pf(expf(-fabsf(xv)));   // softplus(-x)
    lsum += (1.f - y) * xv + (1.f + (w - 1.f) * y) * sp;
    if (c == 0) nvalid += 1.f;
  }
  lsum = warp_sum(lsum);
  nvalid = warp_sum(nvalid);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = lsum; red[1][threadIdx.x >> 5] = nvalid; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int i = 0; i < 8; ++i) { a += red[0][i]; b += red[1][i]; }
    tot[0] = a; tot[1] = b;
    loss_out[0] = a / (12.f * b);      // 0/0 = NaN when every row is ignored, like .mean() of an empty tensor
    loss_out[1] = b;
  }
  if (dlogits == nullptr) return;
  __syncthreads();
  const float inv = 1.f / (12.f * fmaxf(tot[1], 1.f));
  for (int i = threadIdx.x; i < n_clips * 12; i += blockDim.x) {
    const int r = i / 12, c = i - r * 12;
    float g = 0.f;
    if (labels[r * 12] != -1.0f) {
      const float xv = logits[size_t(r) * ld + c], y = labels[i], w = pw[c];
      const float sg = 1.f / (1.f + expf(-xv));
      g = (sg * (1.f + (w - 1.f) * y) - w * y) * inv;
    }
    dlogits[i] = g;
  }
}

// Per-AU confusion counters for MultiLabelAccF1 (metrics/accf1.py:45-77): counts[au][0..3] += {TP, FP, FN, TN} over the entries
// whose label is not `ignore`.  pred > thresh is the positive decision (logits: thresh 0 == round(sigmoid(x)), train.py:155;
// already-rounded predictions: thresh 0.5).  Integer atomics: the result does not depend on the order of the additions.
__global__ void __launch_bounds__(256) au_confusion_kernel(const float* __restrict__ pred, int ld_pred, float thresh,
                                                           const float* __restrict__ labels, int ld_lab, float ignore,
                                                           unsigned long long* __restrict__ counts, int n_rows) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  __shared__ unsigned int sc[12][4];
  if (threadIdx.x < 48) sc[threadIdx.x / 4][threadIdx.x % 4] = 0;
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_rows * 12; i += gridDim.x * blockDim.x) {
    const int r = i / 12, c = i - r * 12;
    const float y = labels[size_t(r) * ld_lab + c];
    if (y == ignore) continue;
    const bool p = pred[size_t(r) * ld_pred + c] > thresh, t = y == 1.0f;
    atomicAdd(&sc[c][p ? (t ? 0 : 1) : (t ? 2 : 3)], 1u);
  }
  __syncthreads();
  if (threadIdx.x < 48 && sc[threadIdx.x / 4][threadIdx.x % 4] != 0)
    atomicAdd(&counts[threadIdx.x], (unsigned long long)sc[threadIdx.x / 4][threadIdx.x % 4]);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host launchers (internal C++ API used by avf_api.cu)
// ---------------------------------------------------------------------------------------------
int layernorm(int out_mode, const float* x, int ld_x, const float* g, const float* b, void* y, int rows, int dim, cudaStream_t st) {
  AVF_REQUIRE(rows > 0, AVF_EINVAL, "layernorm: rows=%d", rows);
  AVF_REQUIRE(dim % 128 == 0 && dim <= 1536 && ld_x % 4 == 0, AVF_EUNSUPPORTED, "layernorm: dim=%d must be a multiple of 128, <= 1536", dim);
  const int wpb = 8;
  dim3 grid(ceil_div(rows, wpb)), block(wpb * 32);
#define AVF_LN(V)                                                                                                   \
  case V:                                                                                                           \
    if (out_mode == AVF_BF16) launch_pdl(layernorm_kernel<__nv_bfloat16, V>, grid, block, 0, st, x, ld_x, g, b, static_cast<__nv_bfloat16*>(y), rows); \
    else launch_pdl(layernorm_kernel<float, V>, grid, block, 0, st, x, ld_x, g, b, static_cast<float*>(y), rows);             \
    break;
  switch (dim / 128) {
    AVF_LN(1) AVF_LN(2) AVF_LN(3) AVF_LN(4) AVF_LN(5) AVF_LN(6) AVF_LN(7) AVF_LN(8) AVF_LN(9) AVF_LN(10) AVF_LN(11) AVF_LN(12)
  }
#undef AVF_LN
  AVF_LAUNCH_CHECK("layernorm_kernel");
  return 0;
}

int bn_rows(int out_mode, const float* x, int ld_x, const float* g, const float* b, const float* mean, const float* var, void* y,
            int rows, int dim, cudaStream_t st) {
  const int n = rows * dim;
  if (out_mode == AVF_BF16) launch_pdl(bn_rows_kernel<__nv_bfloat16>, ceil_div(n, 256), 256, 0, st, x, ld_x, g, b, mean, var, static_cast<__nv_bfloat16*>(y), rows, dim);
  else launch_pdl(bn_rows_kernel<float>, ceil_div(n, 256), 256, 0, st, x, ld_x, g, b, mean, var, static_cast<float*>(y), rows, dim);
  AVF_LAUNCH_CHECK("bn_rows_kernel");
  return 0;
}

static int sformer_grid(int n_frames, size_t smem) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int per_sm = std::max(1, std::min(4, int((220 * 1024) / (smem + 1024))));
  return std::min(n_frames, sms * per_sm);
}

int sformer_pack(int io_mode, const void* fmap, const float* pos, float* x, int n_frames, int dim, int hw, cudaStream_t st) {
  AVF_REQUIRE(n_frames > 0 && dim > 0 && hw > 0, AVF_EINVAL, "sformer_tokens_pack: empty input");
  const size_t smem = size_t(dim) * (hw | 1) * 4;
  AVF_REQUIRE(smem <= 200 * 1024, AVF_EUNSUPPORTED, "sformer_tokens_pack: frame of %d x %d does not fit shared memory", dim, hw);
  AVF_REQUIRE((size_t(dim) * hw) % 8 == 0 && (reinterpret_cast<uintptr_t>(fmap) & 15) == 0, AVF_EUNSUPPORTED,
              "sformer_tokens_pack: frames must be 16-byte aligned multiples of 8 elements (dim=%d hw=%d)", dim, hw);
  static PerDeviceOnce once;
  if (once.first()) {
    AVF_CUDA(cudaFuncSetAttribute(sformer_pack_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    AVF_CUDA(cudaFuncSetAttribute(sformer_pack_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  const int grid = sformer_grid(n_frames, smem);
  if (io_mode == AVF_BF16) launch_pdl(sformer_pack_kernel<__nv_bfloat16>, grid, 256, smem, st, static_cast<const __nv_bfloat16*>(fmap), pos, x, n_frames, dim, hw);
  else launch_pdl(sformer_pack_kernel<float>, grid, 256, smem, st, static_cast<const float*>(fmap), pos, x, n_frames, dim, hw);
  AVF_LAUNCH_CHECK("sformer_pack_kernel");
  return 0;
}

int sformer_unpack(int io_mode, const float* x, void* fmap, int n_frames, int dim, int hw, cudaStream_t st) {
  AVF_REQUIRE(n_frames > 0 && dim > 0 && hw > 0, AVF_EINVAL, "sformer_tokens_unpack: empty input");
  const size_t smem = size_t(dim) * (hw | 1) * 4;
  AVF_REQUIRE(smem <= 200 * 1024, AVF_EUNSUPPORTED, "sformer_tokens_unpack: frame of %d x %d does not fit shared memory", dim, hw);
  AVF_REQUIRE((size_t(dim) * hw) % 8 == 0 && (reinterpret_cast<uintptr_t>(fmap) & 15) == 0, AVF_EUNSUPPORTED,
              "sformer_tokens_unpack: frames must be 16-byte aligned multiples of 8 elements (dim=%d hw=%d)", dim, hw);
  static PerDeviceOnce once;
  if (once.first()) {
    AVF_CUDA(cudaFuncSetAttribute(sformer_unpack_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    AVF_CUDA(cudaFuncSetAttribute(sformer_unpack_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  const int grid = sformer_grid(n_frames, smem);
  if (io_mode == AVF_BF16) launch_pdl(sformer_unpack_kernel<__nv_bfloat16>, grid, 256, smem, st, x, static_cast<__nv_bfloat16*>(fmap), n_frames, dim, hw);
  else launch_pdl(sformer_unpack_kernel<float>, grid, 256, smem, st, x, static_cast<float*>(fmap), n_frames, dim, hw);
  AVF_LAUNCH_CHECK("sformer_unpack_kernel");
  return 0;
}

int tformer_embed(int io_mode, const void* frames, const float* cls, const float* pos, float* x, int n_clips, int T, int dim, cudaStream_t st) {
  AVF_REQUIRE(n_clips > 0 && T > 0 && dim % 4 == 0, AVF_EINVAL, "tformer_embed: n_clips=%d T=%d dim=%d", n_clips, T, dim);
  const size_t total = size_t(n_clips) * (T + 1) * (dim / 4);
  const unsigned grid = unsigned((total + 255) / 256);
  if (io_mode == AVF_BF16) launch_pdl(tformer_embed_kernel<__nv_bfloat16>, grid, 256, 0, st, static_cast<const __nv_bfloat16*>(frames), cls, pos, x, n_clips, T, dim);
  else launch_pdl(tformer_embed_kernel<float>, grid, 256, 0, st, static_cast<const float*>(frames), cls, pos, x, n_clips, T, dim);
  AVF_LAUNCH_CHECK("tformer_embed_kernel");
  return 0;
}

int tformer_embed_indexed(int io_mode, const void* bank, int n_bank, const int* index, const float* cls, const float* pos, float* x, uint8_t* keep,
                          int n_clips, int T, int dim, cudaStream_t st) {
  AVF_REQUIRE(n_clips > 0 && T > 0 && dim % 4 == 0 && n_bank >= 0, AVF_EINVAL, "tformer_embed_indexed: n_clips=%d T=%d dim=%d n_bank=%d", n_clips, T,
              dim, n_bank);
  AVF_REQUIRE((reinterpret_cast<uintptr_t>(bank) & (io_mode == AVF_BF16 ? 7 : 15)) == 0, AVF_EINVAL,
              "tformer_embed_indexed: the bank must be %d-byte aligned", io_mode == AVF_BF16 ? 8 : 16);
  const size_t total = size_t(n_clips) * (T + 1) * (dim / 4);
  const unsigned grid = unsigned((total + 255) / 256);
  if (io_mode == AVF_BF16)
    launch_pdl(tformer_embed_indexed_kernel<__nv_bfloat16>, grid, 256, 0, st, static_cast<const __nv_bfloat16*>(bank), n_bank, index, cls, pos, x, keep,
               n_clips, T, dim);
  else
    launch_pdl(tformer_embed_indexed_kernel<float>, grid, 256, 0, st, static_cast<const float*>(bank), n_bank, index, cls, pos, x, keep, n_clips, T, dim);
  AVF_LAUNCH_CHECK("tformer_embed_indexed_kernel");
  return 0;
}

int rows_gather(const float* x, size_t src_row_stride, float* y, int rows, int dim, cudaStream_t st) {
  AVF_REQUIRE(rows > 0 && dim > 0, AVF_EINVAL, "cls_extract: empty input");
  launch_pdl(rows_gather_kernel, ceil_div(rows * dim, 256), 256, 0, st, x, src_row_stride, y, rows, dim);
  AVF_LAUNCH_CHECK("rows_gather_kernel");
  return 0;
}

int add_row_periodic(float* x, int ld_x, const float* pos, int rows, int dim, int period, cudaStream_t st) {
  AVF_REQUIRE(rows > 0 && dim > 0 && period > 0, AVF_EINVAL, "add_row_periodic: empty input");
  launch_pdl(add_row_periodic_kernel, ceil_div(rows * dim, 256), 256, 0, st, x, ld_x, pos, rows, dim, period);
  AVF_LAUNCH_CHECK("add_row_periodic_kernel");
  return 0;
}

int cast_f32_bf16(const float* s, void* d, size_t n, cudaStream_t st) {
  if (n == 0) return 0;
  AVF_REQUIRE((reinterpret_cast<uintptr_t>(s) & 15) == 0 && (reinterpret_cast<uintptr_t>(d) & 7) == 0, AVF_EINVAL, "cast: unaligned pointers");
  launch_pdl(cast_f32_bf16_kernel, unsigned((n / 4 + 256) / 256), 256, 0, st, s, static_cast<__nv_bfloat16*>(d), n);
  AVF_LAUNCH_CHECK("cast_f32_bf16_kernel");
  return 0;
}
int cast_bf16_f32(const void* s, float* d, size_t n, cudaStream_t st) {
  if (n == 0) return 0;
  launch_pdl(cast_bf16_f32_kernel, unsigned((n + 255) / 256), 256, 0, st, static_cast<const __nv_bfloat16*>(s), d, n);
  AVF_LAUNCH_CHECK("cast_bf16_f32_kernel");
  return 0;
}

int au_logits(const float* x, int ld_x, const float* w_last, float* out21, int* decisions, int n_clips, int dim, cudaStream_t st) {
  AVF_REQUIRE(n_clips > 0 && dim % 4 == 0 && ld_x % 4 == 0, AVF_EINVAL, "au_logits: n_clips=%d dim=%d", n_clips, dim);
  launch_pdl(au_logits_kernel, ceil_div(n_clips * 12, 8), 256, 0, st, x, ld_x, w_last, out21, decisions, n_clips, dim);
  AVF_LAUNCH_CHECK("au_logits_kernel");
  return 0;
}

int au_confusion(const float* pred, int ld_pred, float thresh, const float* labels, int ld_lab, float ignore, unsigned long long* counts, int n_rows,
                 cudaStream_t st) {
  AVF_REQUIRE(n_rows > 0 && pred && labels && counts, AVF_EINVAL, "au_confusion_update: n_rows=%d", n_rows);
  launch_pdl(au_confusion_kernel, std::min(ceil_div(n_rows * 12, 256), 296), 256, 0, st, pred, ld_pred, thresh, labels, ld_lab, ignore, counts, n_rows);
  AVF_LAUNCH_CHECK("au_confusion_kernel");
  return 0;
}

int au_bce(const float* logits, int ld, const float* labels, const float* pw, float* loss_out, float* dlogits, int n_clips, cudaStream_t st) {
  AVF_REQUIRE(n_clips > 0, AVF_EINVAL, "au_bce_loss: n_clips=%d", n_clips);
  launch_pdl(au_bce_kernel, 1, 256, 0, st, logits, ld, labels, pw, loss_out, dlogits, n_clips);
  AVF_LAUNCH_CHECK("au_bce_kernel");
  return 0;
}

}  // namespace avf
