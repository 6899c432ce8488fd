// Shared device helpers for the sm_100a kernels: mbarrier, TMA, tcgen05/TMEM inline PTX and the
// UMMA shared-memory / instruction descriptor encodings.  Hand-written; no CUTLASS dependency.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>

#ifndef SED_DEVICE_INLINE
#define SED_DEVICE_INLINE __device__ __forceinline__
#endif

namespace sed {

// ------------------------------------------------------------------ error codes (C-ABI)
enum : int {
  SED_OK = 0,
  SED_ERR_BAD_SHAPE = 1,
  SED_ERR_UNSUPPORTED = 2,
  SED_ERR_CUDA = 3,
  SED_ERR_NULL = 4,
  SED_ERR_DRIVER = 5,
};

// ------------------------------------------------------------------ generic helpers
SED_DEVICE_INLINE uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// 1024-byte aligned start of the dynamic shared memory window, computed as pointer + offset so that the compiler keeps
// the shared address space (an integer round trip turns every later access into a generic LD/ST)
SED_DEVICE_INLINE uint8_t* align_smem_1024(uint8_t* p) { return p + ((1024u - (smem_u32(p) & 1023u)) & 1023u); }

// x / d for a launch-invariant divisor: magic = ceil(2^32 / d) (0 encodes d == 1); exact while x * d < 2^32
SED_DEVICE_INLINE int fast_div(int x, uint32_t magic) {
  return magic ? static_cast<int>(__umulhi(static_cast<uint32_t>(x), magic)) : x;
}

SED_DEVICE_INLINE bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------ mbarrier
SED_DEVICE_INLINE void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
SED_DEVICE_INLINE void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
SED_DEVICE_INLINE void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
SED_DEVICE_INLINE void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
SED_DEVICE_INLINE bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
SED_DEVICE_INLINE void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// Register re-balancing between warpgroups (all four warps of a warpgroup execute the same one).
template <int R>
SED_DEVICE_INLINE void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(R)); }
template <int R>
SED_DEVICE_INLINE void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(R)); }

// ------------------------------------------------------------------ proxies / fences
SED_DEVICE_INLINE void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
SED_DEVICE_INLINE void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
SED_DEVICE_INLINE void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ------------------------------------------------------------------ TMA (cp.async.bulk.tensor)
SED_DEVICE_INLINE void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
SED_DEVICE_INLINE void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
SED_DEVICE_INLINE void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                   int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

SED_DEVICE_INLINE void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
          reinterpret_cast<uint64_t>(m)),
      "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
SED_DEVICE_INLINE void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until the bulk stores of this thread have finished READING shared memory (buffer reusable)
SED_DEVICE_INLINE void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
SED_DEVICE_INLINE void bulk_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
SED_DEVICE_INLINE void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ------------------------------------------------------------------ TMEM
SED_DEVICE_INLINE void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
SED_DEVICE_INLINE void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
SED_DEVICE_INLINE void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// 32 lanes x 16 consecutive 32-bit columns -> 16 registers per thread (lane = row, reg i = column i)
SED_DEVICE_INLINE void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
      "%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
SED_DEVICE_INLINE void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------ UMMA descriptors
// Shared-memory matrix descriptor, K-major operand, SWIZZLE_128B (one 128-byte row per matrix row,
// 8-row groups `sbo_bytes` apart).  Field layout: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), base_offset [49,52), layout_type [61,64) (2 = SWIZZLE_128B).
SED_DEVICE_INLINE uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;  // LBO: unused for swizzled K-major, canonical value 1
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;  // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;  // SWIZZLE_128B
  return d;
}

// Instruction descriptor for kind::f16, fp32 accumulate, both operands K-major.
// ab_fmt: 0 = f16, 1 = bf16.   c_format=1 (f32) at [4,6); a_format [7,10); b_format [10,13);
// n>>3 at [17,23); m>>4 at [24,29).
__host__ __device__ constexpr uint32_t umma_idesc_f16(uint32_t ab_fmt, uint32_t m, uint32_t n) {
  return (1u << 4) | (ab_fmt << 7) | (ab_fmt << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T, issued by one thread for the CTA.
SED_DEVICE_INLINE void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
SED_DEVICE_INLINE void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------ clusters / CTA pairs
SED_DEVICE_INLINE void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
SED_DEVICE_INLINE void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
SED_DEVICE_INLINE void mbar_arrive_remote(uint64_t* bar, uint32_t cta_rank) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(cta_rank)
      : "memory");
}
SED_DEVICE_INLINE void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// Remote arrive with the default (.release.cta) semantics: used where the barrier only orders tcgen05 / TMEM
// work (no generic-proxy global data is published), so no GPU-scope memory barrier is needed.
SED_DEVICE_INLINE void mbar_arrive_remote_light(uint64_t* bar, uint32_t cta_rank) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(cta_rank)
      : "memory");
}
// packed f32x2 arithmetic (sm_100): two float32 FMAs per instruction on a 64-bit register pair
SED_DEVICE_INLINE unsigned long long pack_f32x2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
SED_DEVICE_INLINE void unpack_f32x2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
SED_DEVICE_INLINE unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
SED_DEVICE_INLINE uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
SED_DEVICE_INLINE uint32_t map_to_cta(const void* smem_ptr, uint32_t cta_rank) {
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(smem_ptr)), "r"(cta_rank));
  return ra;
}
// cta_group::2 (CTA pair) variants: TMEM allocation, TMA load that signals the leader CTA's mbarrier,
// the paired MMA (M = 256 over both CTAs, B split N/2 + N/2) and the multicast commit.
SED_DEVICE_INLINE void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
SED_DEVICE_INLINE void tmem_relinquish2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
SED_DEVICE_INLINE void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
SED_DEVICE_INLINE void tma_load_4d_2sm(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1,
                                       int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
      "%5, %6}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
SED_DEVICE_INLINE void tma_load_2d_2sm(void* dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
SED_DEVICE_INLINE void umma_f16_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                    uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all prior MMAs of this thread completed) on the barrier at this shared-memory offset in
// every CTA of `cta_mask`
SED_DEVICE_INLINE void umma_commit_2sm(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}

// ------------------------------------------------------------------ input samples
// int16 PCM input follows the reference's HDF5 path: x = q / 32767 (utils/utilities.py:78-79).  The three-operation
// sequence below (multiply by the rounded reciprocal, exact residual, correction) returns the correctly rounded
// float32 quotient for every int16 q (checked exhaustively on the host) -- the value numpy's
// (q / 32767.).astype(float32) produces.  Used by the front-end and by the resampler's downmix.
SED_DEVICE_INLINE float load_sample(const float* p) { return *p; }
SED_DEVICE_INLINE float load_sample(const short* p) {
  const float q = static_cast<float>(*p);
  constexpr float kInv = 1.0f / 32767.0f;
  const float r = q * kInv;
  const float e = fmaf(-r, 32767.0f, q);
  return fmaf(e, kInv, r);
}

// ------------------------------------------------------------------ 16-bit element traits
template <typename T>
struct Elem16;
template <>
struct Elem16<__half> {
  static constexpr uint32_t kFmt = 0;
  SED_DEVICE_INLINE static uint32_t pack2(float a, float b) {
    uint32_t r;  // saturating: +-inf never enters the activation stream
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
  SED_DEVICE_INLINE static float to_float(uint16_t v) { return __half2float(__ushort_as_half(v)); }
  // {max(a,0), max(b,0)} rounded to 16 bits in ONE instruction (a in the low half)
  SED_DEVICE_INLINE static uint32_t pack2_relu(float a, float b) {
    uint32_t r;
    asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
};
template <>
struct Elem16<__nv_bfloat16> {
  static constexpr uint32_t kFmt = 1;
  SED_DEVICE_INLINE static uint32_t pack2(float a, float b) {
    uint32_t r;
    asm("cvt.rn.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
  SED_DEVICE_INLINE static float to_float(uint16_t v) { return __uint_as_float(static_cast<uint32_t>(v) << 16); }
  SED_DEVICE_INLINE static uint32_t pack2_relu(float a, float b) {
    uint32_t r;
    asm("cvt.rn.relu.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
  }
};

}  // namespace sed
