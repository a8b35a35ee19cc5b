// Shared device/host helpers for the biu_b200 engine (sm_100a only).
//
// PTX wrappers for the Blackwell async machinery used by the convolution kernels:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld) and TMEM.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <type_traits>

namespace biu {

// ----------------------------------------------------------------------------------------------
// Error plumbing: every C-ABI entry point returns 0 on success; the message is kept per thread.
// ----------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
const char* get_error();

#define BIU_CHECK_CUDA(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      biu::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,   \
                     __LINE__);                                                           \
      return -1;                                                                          \
    }                                                                                     \
  } while (0)

#define BIU_REQUIRE(cond, ...)                                                            \
  do {                                                                                    \
    if (!(cond)) {                                                                        \
      biu::set_error(__VA_ARGS__);                                                        \
      return -2;                                                                          \
    }                                                                                     \
  } while (0)

// Device-side fault word: kernels that time out on an mbarrier write a code here and trap.
// (one copy per translation unit; only conv_tc.cu's copy is ever written or read)
#ifdef __CUDACC__
static __device__ unsigned int g_device_fault = 0;
#endif

// ----------------------------------------------------------------------------------------------
// Small numeric helpers
// ----------------------------------------------------------------------------------------------
__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ inline long long ceil_div_ll(long long a, long long b) { return (a + b - 1) / b; }

// ----------------------------------------------------------------------------------------------
// Element formats of the activations and tcgen05 operands: the template argument of the kernels and the `fmt` of every
// launcher argument block. The values of bf16, fp16 and tf32 are the element codes of the layer C-ABI. FMT_TF32 is fp32
// storage rounded to tf32 (the tensor core's operand format); FMT_F32 is fp32 storage that is never rounded (the exact
// fp32 mode, CUDA-core kernels only).
// ----------------------------------------------------------------------------------------------
enum ElemFmt { FMT_BF16 = 2, FMT_F16 = 3, FMT_TF32 = 4, FMT_F32 = 5 };
__host__ __device__ constexpr int fmt_esz(int fmt) { return fmt == FMT_TF32 || fmt == FMT_F32 ? 4 : 2; }
// A / B format field of the tcgen05 instruction descriptor (make_idesc)
__host__ __device__ constexpr uint32_t fmt_idesc(int fmt) { return fmt == FMT_F16 ? 0u : (fmt == FMT_BF16 ? 1u : 2u); }

// Storage type of a format: with_elem_type(fmt, f) calls f(ElemTag<T>{}) with T = __nv_bfloat16, __half or float, and
// returns f's result (an error code). fmt_of<T> / ElemTag<T>::fmt is the tensor-core format of a storage type.
template <typename T>
constexpr int fmt_of = sizeof(T) == 4 ? FMT_TF32 : (std::is_same<T, __half>::value ? FMT_F16 : FMT_BF16);
template <typename T> struct ElemTag {
  using type = T;
  static constexpr int fmt = fmt_of<T>;
};
template <typename F>
int with_elem_type(int fmt, F&& f) {
  switch (fmt) {
    case FMT_BF16: return f(ElemTag<__nv_bfloat16>{});
    case FMT_F16: return f(ElemTag<__half>{});
    case FMT_TF32:
    case FMT_F32: return f(ElemTag<float>{});
  }
  BIU_REQUIRE(false, "unknown element format %d", fmt);
}

#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 rx;\n"
      ".reg .pred px;\n"
      "elect.sync rx|px, %1;\n"
      "@px mov.s32 %0, 1;\n"
      "}\n"
      : "+r"(pred)
      : "r"(0xFFFFFFFFu));
  return pred != 0;
}

// ---------------------------------------- mbarrier ------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)      // no suspend-time hint: it compiles to NANOSLEEP.SYNCS whose wake-up
      : "memory");                           // latency sits on every producer/consumer hand-off
  return ok != 0;
}
// Bounded wait: a pipeline bug must never hang the GPU box. ~4e9 cycles (≈2 s) then fault+trap.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, uint32_t fault_code) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      atomicExch(&g_device_fault, fault_code);
      __threadfence_system();
      asm volatile("trap;");
    }
  }
}

// ------------------------------------------ TMA ---------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0, int c1,
                                            int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, "
      "%7}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

// ---------------------------------------- tcgen05 -------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]; bf16/f16 inputs, fp32 accumulate.
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same, tf32 inputs (fp32 words in smem, low mantissa bits ignored by the tensor core).
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrive once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp receives row (lane base + i).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
      "%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
      "%15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor for a K-major operand tile whose rows are `row_bytes` (32/64/128) wide and
// stored with the matching TMA swizzle; groups of 8 rows are `sbo_bytes` apart.
//   bits [0,14)  start address >> 4      bits [16,30) leading byte offset >> 4 (unused for swizzled K-major)
//   bits [32,46) stride byte offset >> 4 bits [46,48) version = 1 (Blackwell)
//   bits [49,52) base offset             bits [61,64) layout: 2 = SW128, 4 = SW64, 6 = SW32
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout_type,
                                                   uint32_t base_offset = 0) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(base_offset & 7) << 49;
  d |= (uint64_t)(layout_type & 7) << 61;
  return d;
}

// Instruction descriptor, kind::f16 / kind::tf32, K-major A and B, fp32 accumulate, M = 128 (256 for a CTA pair).
//   fmt: 0 = f16, 1 = bf16, 2 = tf32 (fmt_idesc)
__device__ __forceinline__ uint32_t make_idesc(uint32_t fmt, uint32_t n, uint32_t m = 128u) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

// ------------------------------------ CTA pairs (cta_group::2) ------------------------------------
// Two CTAs of a cluster (the two SMs of a TPC) run ONE tcgen05.mma of M = 256: each CTA contributes the 128 rows of
// A in its own shared memory and HALF of the N rows of B, and receives its 128 accumulator rows in its own TMEM.
// The leader (cluster rank 0) issues the MMAs. A shared::cluster address of a CTA's own shared memory carries the
// CTA's rank within the pair in bit 24: clearing it addresses the same offset in the leader's shared memory.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same offset in the LEADER CTA's shared memory (from either CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask)
               : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// completion of all earlier MMAs of this thread -> arrive on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void tc_commit2(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}

// Two floats -> one 32-bit pair of a 2-byte format (a in the low half), each rounded to nearest even.
template <int FMT>
__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  if (FMT == FMT_F16) {
    __half2 h2 = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h2);
  }
  __nv_bfloat162 b2 = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&b2);
}
// Element-wise maximum of two 32-bit pairs of a 2-byte format.
template <int FMT>
__device__ __forceinline__ uint32_t max_half2(uint32_t a, uint32_t b) {
  if (FMT == FMT_F16) {
    __half2 m = __hmax2(*reinterpret_cast<__half2*>(&a), *reinterpret_cast<__half2*>(&b));
    return *reinterpret_cast<uint32_t*>(&m);
  }
  __nv_bfloat162 m = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
  return *reinterpret_cast<uint32_t*>(&m);
}

#endif  // __CUDACC__

// packed fp32 pairs (sm_100: fma.rn.f32x2 / mul.rn.f32x2 do two IEEE operations per issue slot, results bit-identical
// to the scalar forms)
__device__ __forceinline__ unsigned long long pack_f32x2(float a, float b) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(unsigned long long v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ unsigned long long fma_f32x2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ unsigned long long mul_f32x2(unsigned long long a, unsigned long long b) {
  unsigned long long d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}


}  // namespace biu
