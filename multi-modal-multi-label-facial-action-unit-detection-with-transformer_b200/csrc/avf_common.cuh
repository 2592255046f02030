// Shared device helpers for the AVFormer B200 kernels: PTX wrappers for mbarrier / TMA /
// tcgen05 (sm_100a), numeric helpers, and the host-side error plumbing of the C ABI.
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/avformer_b200.h"

namespace avf {

// ---------------------------------------------------------------------------------------------
// host-side error handling
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);
void count_launch();   // bumps the counter avf_launch_count() reports
int sm_cap();          // avf_set_sm_cap: upper bound on the grid of the persistent kernels (0 = all SMs)

#define AVF_REQUIRE(cond, code, ...)            \
  do {                                          \
    if (!(cond)) {                              \
      avf::set_error(__VA_ARGS__);              \
      return (code);                            \
    }                                           \
  } while (0)

#define AVF_CUDA(call)                                        \
  do {                                                        \
    int _e = avf::check_cuda((call), #call);                  \
    if (_e != 0) return _e;                                   \
  } while (0)

#define AVF_LAUNCH_CHECK(name)                                \
  do {                                                        \
    avf::count_launch();                                      \
    int _e = avf::check_cuda(cudaGetLastError(), name);       \
    if (_e != 0) return _e;                                   \
  } while (0)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// cudaFuncSetAttribute and the SM count are per DEVICE: one-time set-up is keyed by the current device ordinal, so a process that
// drives several GPUs configures every kernel on each of them.
constexpr int AVF_MAX_DEVICES = 64;
static inline int current_device_slot() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) dev = 0;
  return dev % AVF_MAX_DEVICES;
}
struct PerDeviceOnce {
  bool done[AVF_MAX_DEVICES] = {};
  bool first() {                       // true exactly once per device
    const int d = current_device_slot();
    if (done[d]) return false;
    done[d] = true;
    return true;
  }
};
static inline int sm_count_of_current_device() {
  static int n[AVF_MAX_DEVICES] = {};
  const int d = current_device_slot();
  if (n[d] == 0) {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    n[d] = v;
  }
  return n[d];
}

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch.  Every kernel of the library is launched with the programmatic-stream-serialization
// attribute and starts with pdl_wait() (griddepcontrol.wait: blocks until the preceding grid of the stream has completed and
// its writes are visible) followed by pdl_trigger() (lets the NEXT kernel of the stream be scheduled while this one runs; it
// blocks in its own pdl_wait()).  The launch latency and the prologue of a kernel (barrier set-up, TMEM allocation, tensor-map
// prefetch) thus overlap the tail of its predecessor — the hot path is a chain of 60 (forward) / 330 (training step) mostly
// short launches.  Captured CUDA graphs keep the programmatic edges.  avf_set_pdl_enabled(0) launches everything plainly.
// ---------------------------------------------------------------------------------------------
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

// ---------------------------------------------------------------------------------------------
// numeric helpers
// ---------------------------------------------------------------------------------------------
// models/heads.py:164-166.  kFast uses MUFU.TANH (rel. error 2^-11, below bf16 resolution).
template <bool kFast>
__device__ __forceinline__ float gelu_tanh(float x) {
  const float u = 0.7978845608028654f * (x + 0.044715f * x * x * x);
  float t;
  if (kFast) {
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  } else {
    t = tanhf(u);
  }
  return 0.5f * x * (1.0f + t);
}

// d/dx of the tanh-GELU above: 0.5 (1 + t) + 0.5 x (1 - t^2) c (1 + 3 * 0.044715 x^2),  t = tanh(c (x + 0.044715 x^3))
__device__ __forceinline__ float gelu_tanh_grad(float x) {
  const float c = 0.7978845608028654f;
  const float x2 = x * x;
  const float t = tanhf(c * x * fmaf(0.044715f, x2, 1.0f));
  return 0.5f * (1.0f + t) + 0.5f * x * (1.0f - t * t) * c * fmaf(3.0f * 0.044715f, x2, 1.0f);
}

// Dropout (nn.Dropout of models/heads.py:194,197,216) as a stateless counter-based mask: element `idx` of site `seed` is kept
// iff murmur3-finaliser(idx * golden ^ seed) >= thresh, kept values are scaled by 1/(1-p).  The same (seed, idx) regenerates the
// mask in the backward pass, so no mask is ever stored.
struct DropSpec {
  uint32_t seed = 0, thresh = 0;     // thresh = round(p * 2^32); 0 disables
  float scale = 1.f;                 // 1 / (1 - p)
  const uint32_t* salt = nullptr;    // optional DEVICE word xor-ed into the seed at kernel start: lets a captured CUDA graph
                                     // draw fresh masks on every replay (the host bumps / a graph node increments the word)
};
__host__ __device__ __forceinline__ uint32_t mix32(uint32_t h) {
  h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
  return h;
}
__device__ __forceinline__ DropSpec drop_resolve(DropSpec d) {      // once per thread, before the first drop_factor
  if (d.thresh != 0 && d.salt != nullptr) d.seed ^= mix32(__ldg(d.salt));
  return d;
}
__device__ __forceinline__ float drop_factor(const DropSpec& d, uint32_t idx) {
  return mix32(idx * 0x9E3779B1u ^ d.seed) >= d.thresh ? d.scale : 0.f;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// ---------------------------------------------------------------------------------------------
// PTX: shared-memory addresses, mbarrier, fences
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t.reg .b32 R;\n\t"
      "elect.sync R|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Non-blocking probe (mbarrier.try_wait may suspend the thread for a system-dependent time before it answers "not yet").
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// The same with a suspend-time hint (ns): the thread sleeps in hardware until the phase completes or the hint expires, so a
// waiting warp issues (almost) no instructions and leaves its scheduler's issue slots to the warps that have work.
constexpr uint32_t SPIN_HINT_NS = 20000;
__device__ __forceinline__ bool mbar_try_wait_sleep(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(SPIN_HINT_NS)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (-> a CUDA error the host reports) instead of hanging the GPU.  The spin loop
// lives out of line so that the many wait sites of the fused kernels stay small.
static __device__ __noinline__ void mbar_wait_slow(uint64_t* bar, uint32_t parity) {
  const long long t0 = clock64();
  while (!mbar_try_wait_sleep(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {   // ~2 s at 2 GHz
      printf("avf: mbarrier wait timed out (block %d,%d thread %d parity %u)\n", blockIdx.x, blockIdx.y, threadIdx.x, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (!mbar_try_wait(bar, parity)) mbar_wait_slow(bar, parity);
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// Make generic-proxy smem writes visible to the async proxy (TMA / tcgen05 operand reads).
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// PTX: TMA (cp.async.bulk.tensor) — SASS UTMALDG
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// 1-D bulk copy global -> shared (SASS UBLKCP); bytes must be a multiple of 16, addresses 16B aligned.
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---------------------------------------------------------------------------------------------
// PTX: tcgen05 / TMEM — SASS UTCHMMA, LDTM, STTM
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_in_smem, uint32_t ncols) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {         // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Instruction descriptor, kind::f16, bf16 x bf16 -> fp32 (cute/arch/mma_sm100_desc.hpp InstrDescriptor):
// c_format[4,6)=1 (F32), a_format[7,10)=1 (BF16), b_format[10,13)=1, a_major bit15, b_major bit16
// (0 = K-major, 1 = MN-major), n_dim[17,23)=N>>3, m_dim[24,29)=M>>4.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n, int a_mn_major = 0, int b_mn_major = 0) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(a_mn_major) << 15) | (uint32_t(b_mn_major) << 16) |
         (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}

// Shared-memory matrix descriptor (SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout type [61,64) (0 none, 2 = 128B, 4 = 64B, 6 = 32B swizzle).
// K-major, 128B swizzle: rows are 128 B (64 bf16), 8-row groups are 1024 B apart (SBO), LBO unused (1).
__device__ __forceinline__ uint64_t make_desc_sw128_kmajor(uint32_t smem_addr) {
  return uint64_t((smem_addr & 0x3FFFFu) >> 4) | (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
// Generic form for the other canonical layouts.
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
  return uint64_t((smem_addr & 0x3FFFFu) >> 4) | (uint64_t((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         (uint64_t((sbo_bytes >> 4) & 0x3FFFu) << 32) | (uint64_t(1) << 46) | (uint64_t(layout_type) << 61);
}

// Byte offset of element (row, col) of a K-major bf16 tile stored as 128B-swizzled [rows x 64] panels
// (what TMA SWIZZLE_128B writes and what make_desc_sw128_kmajor describes).  `panel_rows` = rows per panel.
__device__ __forceinline__ uint32_t sw128_offset(int row, int col, int panel_rows) {
  const int panel = col >> 6, c = col & 63;
  return uint32_t(panel) * uint32_t(panel_rows) * 128u + uint32_t(row) * 128u +
         (uint32_t(((c >> 3) ^ (row & 7))) << 4) + uint32_t(c & 7) * 2u;
}

// TMEM -> registers: 32 lanes x 32-bit, N consecutive columns; warp w may only touch lanes 32*(w%4)..+31.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

}  // namespace avf
