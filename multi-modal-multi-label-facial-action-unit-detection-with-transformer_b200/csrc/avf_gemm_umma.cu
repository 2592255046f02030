// bf16 linear layer on the 5th-gen tensor cores:  C[M,N] = epi(A[M,K] * W[N,K]^T).
//
// Both operands are K-major (activations row-major, nn.Linear weights [out,in] row-major), so they go
// through TMA (128B swizzle, 64-column boxes) straight into the layout tcgen05.mma reads.  One CTA owns
// one 128 x BN output tile: warp 0 = TMA producer, warp 1 = TMEM allocator + single-thread MMA issuer,
// warps 2..5 = epilogue (TMEM -> registers -> bias / tanh-GELU / fp32 residual -> global).  The fp32
// accumulator never leaves TMEM until the epilogue.  Two CTAs fit per SM so one tile's epilogue
// overlaps the other's main loop.
//
// Replaces the cuBLAS calls behind nn.Linear at models/heads.py:192,195,212,215 of the reference.
//
// Training adds two operand orientations without any transposed copy in HBM (tools/umma_probe.cu T7-T9 pin the
// descriptors on hardware): an operand stored with the reduction index as its ROW index ([K, M] or [K, N] row-major) is
// fetched as 64x64 boxes and described to tcgen05.mma as MN-major SW128 (LBO = 8192 B between 64-wide panels,
// SBO = 1024 B between 8-row groups, +2048 B per UMMA_K).  That gives
//   dgrad  dX[R,Kin]  = dY[R,Nout] * W[Nout,Kin]        A K-major, B = W itself MN-major
//   wgrad  dW[Nout,Kin] = dY[R,Nout]^T * X[R,Kin]       A and B both MN-major, reduction over the token rows R,
// the latter split along R over CTAs (deterministic partial tiles + a reduction kernel).
#include <cuda.h>

#include <atomic>
#include <unordered_map>

#include <algorithm>
#include <mutex>

#include "avf_common.cuh"

namespace avf {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;        // one 128-byte swizzle span of bf16
constexpr int UMMA_K = 16;

template <int BN, int STAGES>
struct GemmCfg {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int W_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + W_BYTES;
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
  static constexpr int BIAS_OFF = BAR_OFF + 256;            // [2][BN] fp32: the tile's slice of the bias vector, staged per accumulator buffer
  static constexpr int SMEM_BYTES = BIAS_OFF + 2 * BN * 4 + 1024;   // barriers + bias slices + slack for 1024B alignment
  static constexpr int TMEM_COLS = 2 * BN;                  // double-buffered accumulator; power of two >= 32
};

// Epilogue math on one 32-column chunk held in registers, then the store of that chunk.
// 4 x 4 transpose of 16-byte pieces inside every quad of lanes: lane j of a quad enters with pieces 0..3 of ITS row and leaves
// with piece j of the rows of lanes 0..3 of the quad.  A store instruction then writes 64 contiguous bytes per row (8 rows =
// 8 lines per instruction) instead of 16 bytes in each of 32 rows: the tile write-back was bound by the number of memory
// transactions, not by bytes (CTA milestones: 4 us per 128 x 256 bf16 tile, the main loop of the next tile starved behind it).
__device__ __forceinline__ void quad_transpose(uint4 (&p)[4], int lane) {
  auto xchg = [&](uint4& keep_lo, uint4& keep_hi, bool upper, int mask) {     // lower lane sends keep_hi, upper lane sends keep_lo
    uint4 snd = upper ? keep_lo : keep_hi, rcv;
    rcv.x = __shfl_xor_sync(0xffffffffu, snd.x, mask);
    rcv.y = __shfl_xor_sync(0xffffffffu, snd.y, mask);
    rcv.z = __shfl_xor_sync(0xffffffffu, snd.z, mask);
    rcv.w = __shfl_xor_sync(0xffffffffu, snd.w, mask);
    if (upper) keep_lo = rcv; else keep_hi = rcv;
  };
  const bool b0 = lane & 1, b1 = lane & 2;
  xchg(p[0], p[1], b0, 1);
  xchg(p[2], p[3], b0, 1);
  xchg(p[0], p[2], b1, 2);
  xchg(p[1], p[3], b1, 2);
}

// The lane's own 16 fp32 columns [col, col + 16) of `src` (row pitch ld), fetched the same way: lane j of a quad reads piece j of
// the quad's four rows (64 contiguous bytes per row per instruction), then the quad transposes.  Rows beyond M read nothing.
__device__ __forceinline__ void quad_load16(const float* src, int ld, int row, int col, int M, int lane, float4 (&out)[4]) {
  const int row_q = row - (lane & 3);
  uint4 p[4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
    p[i] = row_q + i < M ? *reinterpret_cast<const uint4*>(src + size_t(row_q + i) * ld + col + (lane & 3) * 4) : make_uint4(0u, 0u, 0u, 0u);
  quad_transpose(p, lane);
#pragma unroll
  for (int j = 0; j < 4; ++j) out[j] = make_float4(__uint_as_float(p[j].x), __uint_as_float(p[j].y), __uint_as_float(p[j].z), __uint_as_float(p[j].w));
}

template <typename OutT>
__device__ __forceinline__ void epilogue_chunk(const uint32_t (&v)[32], int row, int col0, OutT* C, int ldc,
                                               const float* __restrict__ bias, const float* res, int ld_res, int flags,
                                               __nv_bfloat16* aux, int ld_aux, const DropSpec& drop, int n_total, int M,
                                               const float4* pre_res = nullptr) {
  // every lane of the warp runs this (the store below shuffles between lanes); rows beyond M only skip their memory accesses
  const bool valid = row < M;
  const int lane = threadIdx.x & 31;
  float f[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
  if ((flags & AVF_EPI_DGELU) && valid) {       // backward of the tanh-GELU: multiply by gelu'(pre-activation)
    const __nv_bfloat16* ap = aux + size_t(row) * ld_aux + col0;
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      const uint4 pk = *reinterpret_cast<const uint4*>(ap + j);
      const uint32_t w[4] = {pk.x, pk.y, pk.z, pk.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        f[j + 2 * q] *= gelu_tanh_grad(__uint_as_float(w[q] << 16));
        f[j + 2 * q + 1] *= gelu_tanh_grad(__uint_as_float(w[q] & 0xffff0000u));
      }
    }
  }
  if (flags & AVF_EPI_BIAS) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 b = *reinterpret_cast<const float4*>(bias + col0 + j);     // shared memory (staged per tile by the epilogue warps)
      f[j] += b.x; f[j + 1] += b.y; f[j + 2] += b.z; f[j + 3] += b.w;
    }
  }
  if ((flags & AVF_EPI_SAVE_PRE) && valid) {    // training forward: keep the pre-activation (bf16) for the GELU backward
    __nv_bfloat16* ap = aux + size_t(row) * ld_aux + col0;
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      uint4 o;
      o.x = pack_bf16x2(f[j], f[j + 1]);
      o.y = pack_bf16x2(f[j + 2], f[j + 3]);
      o.z = pack_bf16x2(f[j + 4], f[j + 5]);
      o.w = pack_bf16x2(f[j + 6], f[j + 7]);
      *reinterpret_cast<uint4*>(ap + j) = o;
    }
  }
  if (flags & AVF_EPI_GELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] = gelu_tanh<true>(f[j]);
  }
  if (flags & AVF_EPI_DROPOUT) {
    const uint32_t i0 = uint32_t(row) * uint32_t(n_total) + uint32_t(col0);
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] *= drop_factor(drop, i0 + j);
  }
  if (flags & AVF_EPI_RESIDUAL) {       // (warp-uniform: the un-prefetched form shuffles between lanes)
    float4 r8[8];
    if (pre_res == nullptr) {
      quad_load16(res, ld_res, row, col0, M, lane, reinterpret_cast<float4(&)[4]>(r8[0]));
      quad_load16(res, ld_res, row, col0 + 16, M, lane, reinterpret_cast<float4(&)[4]>(r8[4]));
    }
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 r = pre_res != nullptr ? pre_res[j >> 2] : r8[j >> 2];
      f[j] += r.x; f[j + 1] += r.y; f[j + 2] += r.z; f[j + 3] += r.w;
    }
  }
  const int row_q = row - (lane & 3);            // first row of this lane's quad
  if constexpr (sizeof(OutT) == 4) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {                // two halves of 16 columns = 4 pieces of 16 bytes
      uint4 p[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        p[j] = make_uint4(__float_as_uint(f[h * 16 + 4 * j]), __float_as_uint(f[h * 16 + 4 * j + 1]), __float_as_uint(f[h * 16 + 4 * j + 2]),
                          __float_as_uint(f[h * 16 + 4 * j + 3]));
      quad_transpose(p, lane);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (row_q + i < M) *reinterpret_cast<uint4*>(reinterpret_cast<float*>(C) + size_t(row_q + i) * ldc + col0 + h * 16 + (lane & 3) * 4) = p[i];
    }
  } else {
    uint4 p[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      p[j].x = pack_bf16x2(f[8 * j], f[8 * j + 1]);
      p[j].y = pack_bf16x2(f[8 * j + 2], f[8 * j + 3]);
      p[j].z = pack_bf16x2(f[8 * j + 4], f[8 * j + 5]);
      p[j].w = pack_bf16x2(f[8 * j + 6], f[8 * j + 7]);
    }
    quad_transpose(p, lane);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (row_q + i < M) *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(C) + size_t(row_q + i) * ldc + col0 + (lane & 3) * 8) = p[i];
  }
}

// Developer build -DAVF_GEMM_PROF: CTA 0 stamps %globaltimer (ns) at the milestones of its life into g_gemm_prof[16].
#ifdef AVF_GEMM_PROF
__device__ unsigned long long g_gemm_prof[16];
__device__ __forceinline__ void gprof(int i) {
  if (blockIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_gemm_prof[i] = t;
  }
}
#else
__device__ __forceinline__ void gprof(int) {}
#endif

// Persistent kernel: grid = min(#tiles, #SMs); every CTA walks tiles t = blockIdx.x, +gridDim.x, ...
// (n-block fastest, so CTAs that run concurrently share the A tile in L2).  The TMEM accumulator is double
// buffered (2 x BN columns): the MMA warp fills buffer (t+1)&1 while the 8 epilogue warps drain buffer t&1.
template <int BN, int STAGES, typename OutT, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(384, 1)
gemm_umma_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w,
                 OutT* C, int ldc, const float* __restrict__ bias,
                 const float* res, int ld_res, int M, int N, int K, int flags,
                 __nv_bfloat16* aux, int ld_aux, int splits, size_t split_stride, DropSpec drop) {
  using Cfg = GemmCfg<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::BAR_OFF);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* acc_full = empty_bar + STAGES;       // [2]
  uint64_t* acc_empty = acc_full + 2;            // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) gprof(0);                  // kernel entry
  const int kblocks_total = (K + BK - 1) / BK;     // a ragged last block is zero-filled by TMA
  const int kb_per_split = (kblocks_total + splits - 1) / splits;
  const int n_blocks = N / BN;
  const int mn_tiles = n_blocks * ((M + BM - 1) / BM);
  const int n_tiles = mn_tiles * splits;           // tile = split * mn_tiles + (m_blk * n_blocks + n_blk)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_w);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], 8);               // one arrive per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) gprof(1);                  // prologue done
  pdl_wait();        // the prologue above overlapped the previous kernel; its results are needed from here on
  pdl_trigger();
  if (threadIdx.x == 0) gprof(2);                  // predecessor complete

  // Warps 0 and 1 run their loops with all 32 lanes on warp-uniform values (addresses, descriptors and loop state then live in
  // uniform registers and the issue loops are a few instructions per TMA / MMA); only the elected lane issues.
  if (warp == 0) {
    const bool leader = elect_one();
    {
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int split = tile / mn_tiles, mn = tile - split * mn_tiles;
        const int m0 = (mn / n_blocks) * BM, n0 = (mn % n_blocks) * BN;
        const int kb0 = split * kb_per_split, kb1 = min(kblocks_total, kb0 + kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          uint8_t* st = smem + s * Cfg::STAGE_BYTES;
          if (leader) {
            mbar_expect_tx(&full_bar[s], Cfg::STAGE_BYTES);
            if constexpr (A_MN) {
#pragma unroll
              for (int p = 0; p < BM / 64; ++p) tma_load_2d(st + p * 8192, &tm_a, &full_bar[s], m0 + p * 64, kb * BK);
            } else {
              tma_load_2d(st, &tm_a, &full_bar[s], kb * BK, m0);
            }
            if constexpr (B_MN) {
#pragma unroll
              for (int p = 0; p < BN / 64; ++p) tma_load_2d(st + Cfg::A_BYTES + p * 8192, &tm_w, &full_bar[s], n0 + p * 64, kb * BK);
            } else {
              tma_load_2d(st + Cfg::A_BYTES, &tm_w, &full_bar[s], kb * BK, n0);
            }
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 1) {
    const bool leader = elect_one();
    {
      constexpr uint32_t idesc = make_idesc_bf16(BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      uint32_t it = 0, lt = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++lt) {
        const uint32_t buf = lt & 1, aph = (lt >> 1) & 1;
        mbar_wait(&acc_empty[buf], aph ^ 1);      // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + buf * BN;
        const int split = tile / mn_tiles;
        const int kb0 = split * kb_per_split, kb1 = min(kblocks_total, kb0 + kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          if (leader && it == 0) gprof(3);         // first operand stage has landed
          const uint32_t a_addr = smem_u32(smem + s * Cfg::STAGE_BYTES);
          // K-major: +32 bytes per UMMA_K inside the 128B swizzle span.  MN-major: 16 K-rows of 128 B = +2048 bytes,
          // panels of 64 MN elements 8192 B apart (LBO), 8-row groups 1024 B apart (SBO).
          const uint64_t da = A_MN ? make_desc(a_addr, 8192, 1024, 2) : make_desc_sw128_kmajor(a_addr);
          const uint64_t db = B_MN ? make_desc(a_addr + Cfg::A_BYTES, 8192, 1024, 2) : make_desc_sw128_kmajor(a_addr + Cfg::A_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            if (leader) umma_bf16(tmem_d, da + uint64_t(k * (A_MN ? 128 : 2)), db + uint64_t(k * (B_MN ? 128 : 2)), idesc, ((kb - kb0) | k) != 0 ? 1u : 0u);
          }
          if (leader) umma_commit(&empty_bar[s]); // frees the smem stage when these MMAs have read it
        }
        if (leader) umma_commit(&acc_full[buf]);  // accumulator complete
        if (leader) gprof(4 + min(int(lt), 3));    // all MMAs of tile lt issued
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    const int half = (warp - 4) >> 2;             // which half of the tile's columns
    constexpr int HALF_COLS = BN / 2;
    drop = drop_resolve(drop);
    uint32_t lt = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++lt) {
      const int split = tile / mn_tiles, mn = tile - split * mn_tiles;
      const int m0 = (mn / n_blocks) * BM, n0 = (mn % n_blocks) * BN;
      OutT* Cs = C + size_t(split) * split_stride;
      const uint32_t buf = lt & 1, aph = (lt >> 1) & 1;
      const int row = m0 + q * 32 + lane;
      const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + buf * BN + half * HALF_COLS;
      // The tile's bias slice goes to shared memory BEFORE the wait for the accumulator (one global load per thread, hidden
      // behind the main loop) instead of eight dependent L2 round trips per 32-column chunk inside the epilogue.  Two slices
      // (one per accumulator buffer) and the barrier below make the reuse safe: a warp reaches tile t+2 only after every
      // epilogue warp has passed the barrier of tile t+1, i.e. finished reading the slice of tile t.
      const float* bias_t = bias;
      if (flags & AVF_EPI_BIAS) {
        float* bs = reinterpret_cast<float*>(smem + Cfg::BIAS_OFF) + buf * BN;
        for (int i = threadIdx.x - 128; i < BN; i += 256) bs[i] = __ldg(bias + n0 + i);
        asm volatile("bar.sync 1, 256;" ::: "memory");
        bias_t = bs - n0;
      }
      if constexpr (HALF_COLS <= 64) {
        // Narrow tiles are epilogue-latency bound (K is short on this path): request the thread's residual fragment BEFORE
        // waiting for the accumulator, so that the HBM/L2 round trip overlaps the main loop of this tile.
        float4 pre[HALF_COLS / 4];
        const bool want_res = (flags & AVF_EPI_RESIDUAL) != 0;      // warp-uniform: the fetch shuffles inside lane quads
        if (want_res) {
#pragma unroll
          for (int j = 0; j < HALF_COLS / 16; ++j)
            quad_load16(res, ld_res, row, n0 + half * HALF_COLS + j * 16, M, lane, reinterpret_cast<float4(&)[4]>(pre[4 * j]));
        }
        mbar_wait(&acc_full[buf], aph);
        tc_fence_after();
        if (threadIdx.x == 128) gprof(8 + min(int(lt), 3));   // accumulator of tile lt complete
#pragma unroll
        for (int c0 = 0; c0 < HALF_COLS; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(taddr + uint32_t(c0), v);
          tmem_ld_wait();
          if (c0 + 32 >= HALF_COLS) {             // last chunk is in registers: hand the buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
          }
          epilogue_chunk<OutT>(v, row, n0 + half * HALF_COLS + c0, Cs, ldc, bias_t, res, ld_res, flags, aux, ld_aux, drop, N, M, want_res ? &pre[c0 / 4] : nullptr);
        }
      } else {
        mbar_wait(&acc_full[buf], aph);
        tc_fence_after();
        if (threadIdx.x == 128) gprof(8 + min(int(lt), 3));   // accumulator of tile lt complete
#pragma unroll 1
        for (int c0 = 0; c0 < HALF_COLS; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(taddr + uint32_t(c0), v);
          tmem_ld_wait();
          if (c0 + 32 >= HALF_COLS) {             // last chunk is in registers: hand the buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
          }
          epilogue_chunk<OutT>(v, row, n0 + half * HALF_COLS + c0, Cs, ldc, bias_t, res, ld_res, flags, aux, ld_aux, drop, N, M);
        }
      }
    }
  }

  if (threadIdx.x == 128) gprof(12);               // epilogue warp 0 done
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  if (threadIdx.x == 0) gprof(13);                 // kernel end
}

// ---------------------------------------------------------------------------------------------
// host: tensor maps
// ---------------------------------------------------------------------------------------------
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

}  // namespace

// 2-D bf16 row-major [rows, cols] (row stride ld elements), box = [box_rows x box_cols]: 64 cols with the 128B swizzle
// (default) or 32 cols with the 64B swizzle.
// A tensor map is a pure function of (pointer, shape, pitch, box): encoded maps are kept in a small per-thread cache keyed by exactly
// those values (SURVEY.md section 8b: "cached CUtensorMaps keyed by pointer/shape"), so the steady state of an eagerly launched
// step — the same activations and weights every iteration — costs a hash lookup per operand instead of a driver call
// (cuTensorMapEncodeTiled, ~1 us; two per GEMM launch, four per layer of a fused launch).  The map holds no reference to the memory:
// a freed and re-allocated buffer with the same address, shape and pitch yields the same, still correct, map.
namespace {
struct TmapKey {
  const void* ptr;
  uint64_t rows, cols, ld;
  uint32_t box_rows, box_cols;
  bool operator==(const TmapKey& o) const {
    return ptr == o.ptr && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows && box_cols == o.box_cols;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    uint64_t h = reinterpret_cast<uintptr_t>(k.ptr) * 0x9E3779B97F4A7C15ull;
    h ^= (k.rows * 0xBF58476D1CE4E5B9ull) ^ (k.cols << 21) ^ (k.ld << 42) ^ (uint64_t(k.box_rows) << 7) ^ k.box_cols;
    return size_t(h ^ (h >> 29));
  }
};
constexpr size_t TMAP_CACHE_MAX = 4096;      // ~600 KB at most; cleared wholesale when full (a training step touches a few hundred)
std::atomic<uint64_t> g_tmap_hits{0}, g_tmap_misses{0};
}  // namespace

void tmap_cache_stats(uint64_t* hits, uint64_t* misses) {
  *hits = g_tmap_hits.load();
  *misses = g_tmap_misses.load();
}

static int encode_tmap_bf16_2d(CUtensorMap* tm, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols);

int make_tmap_bf16_2d(CUtensorMap* tm, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols = 64) {
  static thread_local std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> cache;
  const TmapKey key{ptr, rows, cols, ld, box_rows, box_cols};
  auto it = cache.find(key);
  if (it != cache.end()) {
    *tm = it->second;
    g_tmap_hits.fetch_add(1, std::memory_order_relaxed);
    return 0;
  }
  const int e = encode_tmap_bf16_2d(tm, ptr, rows, cols, ld, box_rows, box_cols);
  if (e) return e;
  if (cache.size() >= TMAP_CACHE_MAX) cache.clear();
  cache.emplace(key, *tm);
  g_tmap_misses.fetch_add(1, std::memory_order_relaxed);
  return 0;
}

static int encode_tmap_bf16_2d(CUtensorMap* tm, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols) {
  EncodeTiledFn fn = get_encode_fn();
  AVF_REQUIRE(fn != nullptr, AVF_ENODEVICE, "cuTensorMapEncodeTiled is not available from the driver");
  AVF_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && (ld * 2) % 16 == 0, AVF_EINVAL,
              "TMA operand must be 16-byte aligned with a 16-byte multiple row pitch (ptr=%p ld=%llu)", ptr,
              (unsigned long long)ld);
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  AVF_REQUIRE(box_cols == 64 || box_cols == 32, AVF_EINVAL, "tensor map box must be 64 or 32 columns wide");
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  AVF_REQUIRE(r == CUDA_SUCCESS, AVF_EINVAL, "cuTensorMapEncodeTiled failed with CUresult %d", int(r));
  return 0;
}

static int sm_count() { return sm_count_of_current_device(); }

template <int BN, int STAGES, typename OutT, bool A_MN, bool B_MN>
static int launch_gemm(const void* a, int lda, const void* w, int ldw, OutT* c, int ldc, const float* bias,
                       const float* res, int ld_res, int m, int n, int k, int flags, const void* aux, int ld_aux,
                       int splits, size_t split_stride, cudaStream_t stream, DropSpec drop = DropSpec{}) {
  using Cfg = GemmCfg<BN, STAGES>;
  CUtensorMap ta, tw;
  // K-major operand: [rows = M|N, cols = K], box 64 x {128|BN}.  MN-major operand: [rows = K, cols = M|N], box 64 x 64.
  int e = A_MN ? make_tmap_bf16_2d(&ta, a, k, m, lda, 64) : make_tmap_bf16_2d(&ta, a, m, k, lda, BM);
  if (e) return e;
  e = B_MN ? make_tmap_bf16_2d(&tw, w, k, n, ldw, 64) : make_tmap_bf16_2d(&tw, w, n, k, ldw, BN);
  if (e) return e;
  auto kern = gemm_umma_kernel<BN, STAGES, OutT, A_MN, B_MN>;
  static PerDeviceOnce once;
  if (once.first()) AVF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  const int n_tiles = (n / BN) * ceil_div(m, BM) * splits;
  const int cap = sm_cap();
  launch_pdl(kern, min(n_tiles, cap > 0 ? min(cap, sm_count()) : sm_count()), 384, Cfg::SMEM_BYTES, stream, ta, tw, c, ldc, bias, res, ld_res, m, n, k, flags,
                                                                   static_cast<__nv_bfloat16*>(const_cast<void*>(aux)), ld_aux, splits, split_stride, drop);
  AVF_LAUNCH_CHECK("gemm_umma_kernel");
  return 0;
}

namespace {
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ part, int splits, size_t n, float* __restrict__ out,
                                                            int accumulate) {
  pdl_wait();      // programmatic dependent launch: everything above is launch overhead hidden behind the previous kernel
  pdl_trigger();
  const size_t i = (size_t(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  float4 acc = *reinterpret_cast<const float4*>(part + i);
  if (accumulate) {
    const float4 v = *reinterpret_cast<const float4*>(out + i);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  for (int s = 1; s < splits; ++s) {
    const float4 v = *reinterpret_cast<const float4*>(part + size_t(s) * n + i);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  *reinterpret_cast<float4*>(out + i) = acc;
}
}  // namespace

// General bf16 GEMM  C[M,N] = epi(op(A) op(B)), fp32 accumulation in TMEM.
//   trans_a = 0: A is [M,K] row-major (lda);  1: A is stored [K,M] row-major (reduction index = row).
//   trans_b = 0: B is [N,K] row-major (nn.Linear layout, C = A B^T);  1: B is stored [K,N] row-major.
// When both operands are MN-major (wgrad: K = token rows) the reduction is split over CTAs; `ws` then receives the
// partial tiles and a second kernel reduces them in a fixed order (bit-reproducible).
int gemm_umma(int trans_a, int trans_b, const void* a, int lda, const void* w, int ldw, const float* bias, const float* res,
              int ld_res, const void* aux, int ld_aux, void* c, int ldc, int c_mode, int m, int n, int k, int flags,
              void* ws, size_t ws_bytes, cudaStream_t stream, DropSpec drop) {
  AVF_REQUIRE(m > 0 && n > 0 && k > 0, AVF_EINVAL, "linear: empty problem m=%d n=%d k=%d", m, n, k);
  AVF_REQUIRE(n % 64 == 0, AVF_EUNSUPPORTED, "linear(bf16): N=%d must be a multiple of 64", n);
  AVF_REQUIRE(trans_a || trans_b || k % 8 == 0, AVF_EUNSUPPORTED, "linear(bf16): K=%d must be a multiple of 8", k);
  AVF_REQUIRE(!trans_a || m % 64 == 0, AVF_EUNSUPPORTED, "linear(bf16): M=%d of a transposed A must be a multiple of 64", m);
  AVF_REQUIRE(ldc % 8 == 0 && (!(flags & AVF_EPI_RESIDUAL) || ld_res % 4 == 0), AVF_EINVAL,
              "linear(bf16): ldc=%d / ld_res=%d break vector alignment", ldc, ld_res);
  AVF_REQUIRE(!(flags & (AVF_EPI_DGELU | AVF_EPI_SAVE_PRE)) || (aux != nullptr && ld_aux % 8 == 0), AVF_EINVAL,
              "linear(bf16): DGELU / SAVE_PRE epilogues need the pre-activation buffer");
  const int m_tiles = ceil_div(m, BM), sms = sm_count();
  if (trans_a && trans_b) {
    // wgrad: few output tiles, long reduction -> split K so that every SM has a tile
    const bool accumulate = (flags & AVF_EPI_ACCUMULATE) != 0;
    AVF_REQUIRE(c_mode == AVF_FP32 && (flags & ~AVF_EPI_ACCUMULATE) == 0, AVF_EUNSUPPORTED, "linear(bf16): the TN form writes (or accumulates into) plain fp32");
    const int bn = n % 128 == 0 ? 128 : 64;
    const int mn_tiles = m_tiles * (n / bn), kblocks = ceil_div(k, BK);
    int splits = std::max(1, std::min(kblocks, sms / std::max(1, mn_tiles)));
    const int per = ceil_div(kblocks, splits);
    splits = ceil_div(kblocks, per);
    const size_t elems = size_t(m) * n;
    float* out = static_cast<float*>(c);
    float* part = out;
    size_t stride = 0;
    if (splits > 1 || accumulate) {
      AVF_REQUIRE(ldc == n, AVF_EINVAL, "linear(bf16): split-K output must be dense (ldc=%d n=%d)", ldc, n);
      AVF_REQUIRE(ws != nullptr && ws_bytes >= elems * splits * sizeof(float), AVF_EWORKSPACE,
                  "linear(bf16): split-K workspace too small: %zu < %zu bytes", ws_bytes, elems * splits * sizeof(float));
      part = static_cast<float*>(ws);
      stride = elems;
    }
    int e = bn == 128 ? launch_gemm<128, 6, float, true, true>(a, lda, w, ldw, part, ldc, nullptr, nullptr, 0, m, n, k, 0, nullptr, 0, splits, stride, stream)
                      : launch_gemm<64, 8, float, true, true>(a, lda, w, ldw, part, ldc, nullptr, nullptr, 0, m, n, k, 0, nullptr, 0, splits, stride, stream);
    if (e) return e;
    if (splits > 1 || accumulate) {
      launch_pdl(splitk_reduce_kernel, unsigned((elems / 4 + 255) / 256), 256, 0, stream, part, splits, elems, out, accumulate ? 1 : 0);
      AVF_LAUNCH_CHECK("splitk_reduce_kernel");
    }
    return 0;
  }
  AVF_REQUIRE(!trans_a, AVF_EUNSUPPORTED, "linear(bf16): transposed A is only implemented together with transposed B");
  // widest tile that still gives every SM at least two tiles; small problems get narrower tiles for parallelism
  int bn = 64;
  // the wide tile halves the operand traffic per FLOP: bf16 outputs take it from 0.8 waves on, fp32 outputs (whose epilogue
  // then moves 128 KB per tile without the residual prefetch) only when there are at least two waves
  if (n % 256 == 0 && m_tiles * (n / 256) * 5 >= (c_mode == AVF_BF16 ? 4 : 10) * sms) bn = 256;
  else if (n % 128 == 0 && m_tiles * (n / 128) >= sms) bn = 128;
  else if (n % 128 == 0 && n / 128 * m_tiles >= sms / 2 && n >= 512) bn = 128;
#define AVF_GEMM(BN_, ST_, BMN_)                                                                                                   \
  if (bn == BN_ && bool(trans_b) == BMN_) {                                                                                        \
    if (c_mode == AVF_BF16)                                                                                                        \
      return launch_gemm<BN_, ST_, __nv_bfloat16, false, BMN_>(a, lda, w, ldw, static_cast<__nv_bfloat16*>(c), ldc, bias, res, ld_res, m, n, k, flags, aux, ld_aux, 1, 0, stream, drop); \
    return launch_gemm<BN_, ST_, float, false, BMN_>(a, lda, w, ldw, static_cast<float*>(c), ldc, bias, res, ld_res, m, n, k, flags, aux, ld_aux, 1, 0, stream, drop);          \
  }
  AVF_GEMM(256, 4, false)
  AVF_GEMM(128, 6, false)
  AVF_GEMM(64, 8, false)
  AVF_GEMM(256, 4, true)
  AVF_GEMM(128, 6, true)
  AVF_GEMM(64, 8, true)
#undef AVF_GEMM
  return AVF_EUNSUPPORTED;
}

int gemm_prof_read(unsigned long long* out16) {
#ifdef AVF_GEMM_PROF
  AVF_CUDA(cudaDeviceSynchronize());
  AVF_CUDA(cudaMemcpyFromSymbol(out16, g_gemm_prof, sizeof(unsigned long long) * 16));
  return 0;
#else
  (void)out16;
  return AVF_EUNSUPPORTED;
#endif
}

size_t gemm_umma_workspace_bytes(int m, int n, int k) {       // for the TN (wgrad) form
  const int sms = sm_count(), bn = n % 128 == 0 ? 128 : 64;
  const int mn_tiles = ceil_div(m, BM) * (n / bn), kblocks = ceil_div(k, BK);
  const int splits = std::max(1, std::min(kblocks, sms / std::max(1, mn_tiles)));
  return size_t(m) * n * splits * sizeof(float);      // splits == 1 still needs one tile set when the result is accumulated
}

// C = epi(A W^T) with bf16 operands; c_mode selects fp32 / bf16 output.
int linear_umma(const void* a, int lda, const void* w, const float* bias, const float* res, int ld_res, void* c,
                int ldc, int c_mode, int m, int n, int k, int flags, cudaStream_t stream) {
  AVF_REQUIRE(k % BK == 0, AVF_EUNSUPPORTED, "linear(bf16): K=%d must be a multiple of %d", k, BK);
  return gemm_umma(0, 0, a, lda, w, k, bias, res, ld_res, nullptr, 0, c, ldc, c_mode, m, n, k, flags, nullptr, 0, stream, DropSpec{});
}

}  // namespace avf
