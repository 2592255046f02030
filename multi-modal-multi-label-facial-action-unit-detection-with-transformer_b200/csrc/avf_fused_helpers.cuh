// Device helpers of the fused encoder kernel (avf_layer_fused.cu): packed bf16x2 arithmetic,
// narrow TMEM load / store shapes, bulk stores, operand packing and the optional per-phase cycle counters.
#pragma once
#include "avf_common.cuh"

namespace avf {
namespace fused {

// Optional phase timing (-DAVF_FUSED_PROF): CTA 0's MMA thread and first worker thread accumulate clock64() deltas per phase.
#ifdef AVF_FUSED_PROF
static __device__ unsigned long long g_prof[64];   // one copy per translation unit (each fused kernel file has its own reader)
struct Prof {      // per-thread accumulators (local memory, L1-resident: a mark costs tens of cycles), flushed to g_prof once at the end
  long long t0;
  bool on;
  unsigned acc[64];
  __device__ __forceinline__ void start(bool enable) {
    on = enable;
    for (int i = 0; i < 64; ++i) acc[i] = 0;
    t0 = clock64();
  }
  __device__ __forceinline__ void mark(int idx) {
    if (on) {
      const long long t1 = clock64();
      acc[idx] += unsigned(t1 - t0);
      t0 = t1;
    }
  }
  __device__ __forceinline__ void count(int idx) { if (on) acc[idx] += 1; }
  __device__ __forceinline__ void flush(int lo, int hi) {
    if (on) for (int i = lo; i < hi; ++i) g_prof[i] += acc[i];
  }
};
#else
struct Prof {
  __device__ __forceinline__ void start(bool) {}
  __device__ __forceinline__ void mark(int) {}
  __device__ __forceinline__ void count(int) {}
  __device__ __forceinline__ void flush(int, int) {}
};
#endif

__device__ __forceinline__ void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
// Packed bf16x2 arithmetic for the two MUFU-heavy epilogues (softmax exponentials, tanh-GELU, models/heads.py:164-166).  Their
// results are rounded to bf16 anyway (P and gelu(h) are tensor-core operands), so evaluating the transcendental on a bf16 pair
// halves the MUFU work (16 results / clk / SM -> 32) and the surrounding multiply-adds.
__device__ __forceinline__ uint32_t cvt_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t ex2_bf16x2(uint32_t x) {
  uint32_t r;
  asm("ex2.approx.ftz.bf16x2 %0, %1;" : "=r"(r) : "r"(x));
  return r;
}
__device__ __forceinline__ uint32_t tanh_bf16x2(uint32_t x) {
  uint32_t r;
  asm("tanh.approx.bf16x2 %0, %1;" : "=r"(r) : "r"(x));
  return r;
}
__device__ __forceinline__ uint32_t mul_bf16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t fma_bf16x2(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm("fma.rn.bf16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
  return r;
}
// tanh-GELU of a bf16 pair: 0.5x(1 + tanh(x(c0 + c1 x^2))), 5 packed multiply-adds + 1 MUFU
__device__ __forceinline__ uint32_t gelu_bf16x2(uint32_t x) {
  constexpr uint32_t C0 = 0x3F4C3F4Cu;      // 0.796875  ~ sqrt(2/pi)
  constexpr uint32_t C1 = 0x3D123D12u;      // 0.035645  ~ sqrt(2/pi) * 0.044715
  constexpr uint32_t HALF = 0x3F003F00u;
  const uint32_t x2 = mul_bf16x2(x, x);
  const uint32_t u = mul_bf16x2(x, fma_bf16x2(x2, C1, C0));
  const uint32_t hx = mul_bf16x2(x, HALF);
  return fma_bf16x2(hx, tanh_bf16x2(u), hx);
}
// Packed fp32 pairs (Blackwell FADD2 / FMUL2 / FFMA2: one instruction, two fp32 results, bit-identical to the scalar forms).  The
// row workers are bound by the issue rate of their fp32 sweeps (LayerNorm statistics / normalisation, bias and positional adds,
// softmax scaling), so halving the instruction count of those loops is worth more than any reordering.  A pair lives in a 64-bit
// register; consecutive TMEM columns land in consecutive registers, so building a pair from two of them costs nothing.
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint32_t cvt_bf16x2_pair(uint64_t v) {      // (lo, hi) fp32 pair -> packed bf16 pair, round to nearest even
  float lo, hi;
  f2_unpack(v, lo, hi);
  return cvt_bf16x2(lo, hi);
}

__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
      "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]),
               "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st16_zero(uint32_t taddr) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(0u)
               : "memory");
}
// zero the TMEM columns [lo, hi) of this warp's lanes (lo, hi multiples of 4; warp-uniform; empty when hi <= lo)
__device__ __forceinline__ void zero_p_columns(uint32_t taddr, int lo, int hi) {
  int c = lo;
  for (; c + 16 <= hi; c += 16) tmem_st16_zero(taddr + c);
  for (; c + 4 <= hi; c += 4) tmem_st4(taddr + c, 0u, 0u, 0u, 0u);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void bulk_store_1d(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(reinterpret_cast<uint64_t>(gdst)), "r"(smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ uint64_t desc_sw64(uint32_t addr) { return make_desc(addr, 16, 512, 4); }

__device__ __forceinline__ uint4 pack8u(const uint32_t* r) {
  uint4 pk;
  pk.x = pack_bf16x2(__uint_as_float(r[0]), __uint_as_float(r[1]));
  pk.y = pack_bf16x2(__uint_as_float(r[2]), __uint_as_float(r[3]));
  pk.z = pack_bf16x2(__uint_as_float(r[4]), __uint_as_float(r[5]));
  pk.w = pack_bf16x2(__uint_as_float(r[6]), __uint_as_float(r[7]));
  return pk;
}

}  // namespace fused
}  // namespace avf
