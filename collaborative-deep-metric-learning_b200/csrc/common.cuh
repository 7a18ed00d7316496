// Shared device helpers for libcdml (sm_100a only): mbarrier, TMA, tcgen05/TMEM wrappers.
// Hand-written PTX; no CUTLASS/CuTe dependency.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

namespace cdml {

// ----------------------------------------------------------------------------------------------
// error plumbing (host)
// ----------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
#define CDML_CHECK_CUDA(expr)                                                              \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      cdml::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return -2;                                                                           \
    }                                                                                      \
  } while (0)
#define CDML_REQUIRE(cond, ...)                                                            \
  do {                                                                                     \
    if (!(cond)) {                                                                         \
      cdml::set_error(__VA_ARGS__);                                                        \
      return -1;                                                                           \
    }                                                                                      \
  } while (0)

// ----------------------------------------------------------------------------------------------
// small device utilities
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}
__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  // no suspend-time hint: measured on B200, a parked waiter wakes up too late for the 4-k-block tiles of the
  // KNN / mining scans (2x slower); the default try_wait window is short enough not to starve the epilogue warps
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// A wedged pipeline must not hang the GPU box: after ~4 s of waiting the kernel reports which
// barrier it was stuck on and traps (the launch then fails with an error the C ABI returns).
static __device__ __noinline__ void mbar_timeout(int tag, uint32_t parity) {
  printf("[cdml] mbarrier wait timeout: tag=%d parity=%u block=%d thread=%d\n", tag, parity,
         (int)blockIdx.x, (int)threadIdx.x);
  __trap();
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = global_timer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 255u) == 0u && global_timer_ns() - t0 > 4000000000ull) mbar_timeout(tag, parity);
  }
}

// ----------------------------------------------------------------------------------------------
// TMA (cp.async.bulk.tensor)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_hint(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1,
                                                 uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, "
      "%4}], [%2], %5;"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}
// TMA store of a shared-memory box (written by ordinary st.shared: fence_proxy_async first), bulk-group completion
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;
constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

// ----------------------------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers fp16 and bf16 operands, fp32 accumulate.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread t <-> TMEM lane base+t).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 16-byte shared-memory accesses by shared-space address (epilogue staging buffers)
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}

// Shared-memory matrix descriptor (sm_100 "version 1"), 128-byte swizzle.
//   K-major : rows of 128 B (64 x 16-bit along K); 8-row groups are SBO = 1024 B apart.
//   MN-major: 128 B (64 x 16-bit along M/N) per K row; 8-K-row groups SBO = 1024 B apart,
//             64-element MN atoms LBO bytes apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;  // descriptor version (Blackwell)
  d |= 2ull << 61;  // SWIZZLE_128B
  return d;
}
// Instruction descriptor for kind::f16: fp32 accumulate, A/B both fp16 (fmt 0) or bf16 (fmt 1).
__host__ __device__ constexpr uint32_t make_idesc_f16(int fmt, int a_mn_major, int b_mn_major, int m, int n) {
  return (1u << 4) | (static_cast<uint32_t>(fmt) << 7) | (static_cast<uint32_t>(fmt) << 10) |
         (static_cast<uint32_t>(a_mn_major) << 15) | (static_cast<uint32_t>(b_mn_major) << 16) |
         (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

// ----------------------------------------------------------------------------------------------
// Packed fp32x2 arithmetic and 3-input min/max (sm_100: FADD2 / FMNMX3 / VIMNMX3).  The selection epilogues of the
// KNN and mining scans are issue-bound (two epilogue warps per SM sub-partition against a 2048-cycle K=256 tile);
// these halve the instructions per accumulator element.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 sub2(float a0, float a1, float b0, float b1) {   // (a0-b0, a1-b1) in one FADD2
  float2 r;
  asm("{\n\t.reg .b64 a, b, c;\n\t"
      "mov.b64 a, {%2, %3};\n\t"
      "mov.b64 b, {%4, %5};\n\t"
      "sub.f32x2 c, a, b;\n\t"
      "mov.b64 {%0, %1}, c;\n\t}"
      : "=f"(r.x), "=f"(r.y)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
  return r;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ uint32_t umin3(uint32_t a, uint32_t b, uint32_t c) { return __vimin3_u32(a, b, c); }
__device__ __forceinline__ uint32_t umax3(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_u32(a, b, c); }

__device__ __forceinline__ uint32_t f2key(float f) {  // order-preserving float -> uint32
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

// Philox4x32-10 (Salmon et al., SC'11; pinned in tests to the Random123 known-answer vectors): the four output words of
// counter (c0, c1, c2, c3) under key (k0, k1).
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                               uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0, c1 = lo1, c2 = hi0 ^ c3 ^ k1, c3 = lo0;
    k0 += 0x9E3779B9u, k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

// ----------------------------------------------------------------------------------------------
// 16-bit element helpers (dtype 0 = fp16, 1 = bf16)
// ----------------------------------------------------------------------------------------------
template <int kBf16>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  if constexpr (kBf16) {
    __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&t);
  } else {
    __half2 t = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&t);
  }
}
template <int kBf16>
__device__ __forceinline__ float2 unpack2(uint32_t u) {
  if constexpr (kBf16) {
    return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u));
  } else {
    return __half22float2(*reinterpret_cast<__half2*>(&u));
  }
}

}  // namespace cdml
