// Shared helpers for libspotv2_gat.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/spotv2_gat.h"

namespace spotv2 {

// Thread-local error text behind spotv2_last_error().
void set_error(const char* fmt, ...);
int fail(spotv2_status st, const char* fmt, ...);

#define SPOTV2_CUDA_OK(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess)                                                                \
      return ::spotv2::fail(SPOTV2_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,              \
                            cudaGetErrorString(_e), __FILE__, __LINE__);                  \
  } while (0)

#define SPOTV2_REQUIRE(cond, ...)                                                         \
  do {                                                                                    \
    if (!(cond)) return ::spotv2::fail(SPOTV2_ERR_INVALID_ARG, __VA_ARGS__);              \
  } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }

int check_desc(const spotv2_gat_desc* d);
// p_format 1 pads every head's channel block to a multiple of 8 columns (16-byte aligned TMA tile starts for fp16 planes)
inline int head_pitch_of(const spotv2_gat_desc* d) { return d->p_format == 1 ? (d->C + 7) / 8 * 8 : d->C; }
inline int n_aug_of(const spotv2_gat_desc* d) { return d->H * head_pitch_of(d) + 2 * d->H; }
int sm_count();
size_t attn_bwd_ws_bytes(const spotv2_gat_desc* d);      // attn_bwd.cu

// ---- device helpers ---------------------------------------------------------------------
// Packed fp32 pair FMA (Blackwell FFMA2): d = a * b + c on both halves.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  unsigned long long ra, rb, rc, rd;
  ra = *reinterpret_cast<unsigned long long*>(&a);
  rb = *reinterpret_cast<unsigned long long*>(&b);
  rc = *reinterpret_cast<unsigned long long*>(&c);
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  return *reinterpret_cast<float2*>(&rd);
}

__device__ __forceinline__ uint32_t tf32_rna(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return u;
}

// Split an fp32 value into a tf32 "hi" and a tf32 "lo" with hi + lo == x to ~2^-22.
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = tf32_rna(x);
  lo = tf32_rna(x - __uint_as_float(hi));
}

// Cheap split for hot loops (cvt.rna.tf32 is emulated with ~5 ALU ops on sm_100): hi = x truncated to
// tf32, lo = (x - hi) truncated to tf32; x - hi is exact, so hi + lo == x to 2^-21 |x|.
__device__ __forceinline__ void split_tf32_trunc(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi)) & 0xffffe000u;
}

// tf32 split for mma.sync operands: the tensor core reads only the top 19 bits of a tf32 operand register
// (verified by the parity tests), so "hi" is the raw fp32 pattern and only lo = x - trunc(x) costs ALU work.
__device__ __forceinline__ void split_lean(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x);
  lo = __float_as_uint(x - __uint_as_float(hi & 0xffffe000u));
}

// D(16x8, f32) += A(16x8, tf32, row) * B(8x8, tf32, col)
__device__ __forceinline__ void mma_tf32_16x8x8(float (&c)[4], const uint32_t (&a)[4],
                                                const uint32_t (&b)[2]) {
  asm(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, "
      "{%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// D(16x8, f32) += A(16x16, f16, row) * B(16x8, f16, col)
__device__ __forceinline__ void mma_f16_k16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// ldmatrix: four 8x8 b16 matrices; lane l supplies the address of row (l & 7) of matrix (l >> 3)
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// Explicit shared-memory load: pointers that reach a helper through arrays or structs lose their
// address space and compile to generic LD, which is several times slower than LDS (measured: the edge
// logit loop ran at ~290 cycles per k-step with generic loads).
__device__ __forceinline__ float lds_f32(const float* p) {
  float v;
  asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(smem_u32(p)));      // not volatile: free to be hoisted
  return v;
}

// ---- shared memory by 32-bit shared-window address ----------------------------------------
// The hot loops' accesses (generic pointers make the compiler re-derive the window base before every access).  These
// are asm volatile: issued where written, in program order with each other; lds_f32 above is the hoistable form.
__device__ __forceinline__ float ldsa(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ int ldsa_s32(uint32_t a) {
  int v;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float2 lds64a(uint32_t a) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ uint2 lds64a_b32(uint32_t a) {
  uint2 v;
  asm volatile("ld.shared.v2.b32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ float4 lds128a(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void stsa(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void stsa_b32(uint32_t a, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts128a(uint32_t a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts128a_b32(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}

// named barrier kId over kCount threads (whole warps)
template <int kId, int kCount>
__device__ __forceinline__ void bar_sync() {
  asm volatile("bar.sync %0, %1;" ::"n"(kId), "n"(kCount) : "memory");
}

// ---- mbarrier + 1-D bulk async copy (TMA engine, no tensor map) ---------------------------
// Every mbarrier operation takes the barrier's 32-bit shared address; the uint64_t* forms forward to it.
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) { mbar_arrive(smem_u32(bar)); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) { mbar_expect_tx(smem_u32(bar), bytes); }
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) { return mbar_try_wait(smem_u32(bar), parity); }

// Bounded wait.  try_wait parks the thread for a short hardware-defined interval; after kSpins misses we back off with
// kSleepNs sleeps so parked warps do not eat issue slots (a suspend-time HINT compiles to a 200 us NANOSLEEP and
// serialises the pipeline - measured).  A lost transaction calls report() (e.g. a printf naming the barrier) and traps
// after kLimit cycles instead of hanging the GPU box.
struct NoReport {
  __device__ __forceinline__ void operator()() const {}
};
template <int kSpins, unsigned kSleepNs, long long kLimit, class Report = NoReport>
__device__ __forceinline__ void mbar_wait_bounded(uint32_t bar, uint32_t parity, Report report = Report()) {
  for (int spin = 0; spin < kSpins; ++spin)
    if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(kSleepNs);
    if (clock64() - t0 > kLimit) { report(); __trap(); }
  }
}
constexpr long long kWaitTrapCycles = 4000000000LL;     // ~2 s at the B200's SM clock (~1.9-2.0 GHz)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  constexpr int kSpins = 16;
  constexpr unsigned kSleepNs = 64;
  mbar_wait_bounded<kSpins, kSleepNs, kWaitTrapCycles>(smem_u32(bar), parity);
}
// Diagnostics: cycles spent parked on each class of barrier (one sampling thread per role adds its
// totals at kernel exit); read and reset through spotv2_diag_counters().
enum { kCntRingFull = 0, kCntTileEmpty, kCntTileFull, kCntPtileFull, kCntPtileEmpty, kCntRoleA, kCntRoleB, kCntRoleP,
       kCntAux0, kCntAux1, kCntAux2, kCntAux3, kNumCounters = 16 };
// Host side: adds the kNumCounters entries of the __device__ counter array `counters` into host_out[0, kNumCounters)
// and zeroes them on the device if reset.
inline int diag_add(unsigned long long* host_out, const void* counters, int reset) {
  unsigned long long tmp[kNumCounters];
  SPOTV2_CUDA_OK(cudaMemcpyFromSymbol(tmp, counters, sizeof(tmp)));
  for (int k = 0; k < kNumCounters; ++k) host_out[k] += tmp[k];
  if (reset) {
    unsigned long long zeros[kNumCounters] = {0};
    SPOTV2_CUDA_OK(cudaMemcpyToSymbol(counters, zeros, sizeof(zeros)));
  }
  return SPOTV2_OK;
}
// adds the cycles wait() took to acc; kOn = false only waits (reads no clock)
template <bool kOn = true, class Wait>
__device__ __forceinline__ void wait_timed(long long& acc, Wait&& wait) {
  if (!kOn) return wait();
  const long long t0 = clock64();
  wait();
  acc += clock64() - t0;
}
__device__ __forceinline__ void mbar_wait_timed(uint64_t* bar, uint32_t parity, long long& acc) {
  wait_timed(acc, [&] { mbar_wait(bar, parity); });
}

__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                         uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// L2 eviction-priority descriptors for the .L2::cache_hint forms of the bulk copies (the encodings CUTLASS
// ships as TMA::CacheHintSm90)
constexpr uint64_t kEvictNormal = 0x1000000000000000ull, kEvictFirst = 0x12F0000000000000ull, kEvictLast = 0x14F0000000000000ull;
__device__ __forceinline__ void bulk_g2s_hint(uint32_t smem_dst, const void* gmem_src, uint32_t bytes, uint32_t bar, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_dst),
      "l"(gmem_src), "r"(bytes), "r"(bar), "l"(hint)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s_hint(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar,
                                              uint64_t hint) {
  bulk_g2s_hint(smem_u32(smem_dst), gmem_src, bytes, smem_u32(bar), hint);
}

__device__ __forceinline__ float2 ldg_stream2(const float* p) {
  float2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ldg_stream4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

}  // namespace spotv2
