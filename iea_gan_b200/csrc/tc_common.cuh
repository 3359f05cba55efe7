// tc_common.cuh -- PTX wrappers shared by the tcgen05 kernels (mbarrier, TMA bulk copy, tcgen05
// alloc/mma/commit/ld, UMMA instruction and shared-memory descriptors) and the fused-prologue chunk loader.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace tc {
using namespace iea;
constexpr uint32_t SPIN_LIMIT = 1u << 20;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// makes the barrier initialisation visible to the async proxy (TMA, tcgen05.commit) before any use
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  // try_wait with a suspend-time hint: the hardware parks the thread until the phase completes (or the
  // hint expires), so a waiting role issues almost no instructions.  A plain poll loop costs thousands of
  // issue slots per tile here because every role spends most of its time waiting on another one.
  uint32_t ok = 0;
#pragma unroll 1
  for (uint32_t i = 0; i < SPIN_LIMIT; ++i) {
    asm volatile(
        "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3; selp.u32 %0, 1, 0, p; }"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(0x989680u)
        : "memory");
    if (ok) return;
  }
  __trap();  // a pipeline bug must never hang the GPU
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{ .reg .pred p; setp.ne.b32 p, %4, 0; tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p; }" ::"r"(tmem_c),
      "l"(da), "l"(db), "r"(idesc), "r"(acc)
      : "memory");
}
// UMMA instruction descriptor: bf16 A and B, fp32 accumulator, M = 128, N = n; a_mn / b_mn: the operand is
// MN-major (reduction along its rows) instead of K-major
__host__ __device__ constexpr uint32_t idesc(int n, bool a_mn, bool b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version for sm_100
  return d;                // layout_type = 0 (no swizzle), base_offset = 0
}
// tcgen05.ld of 16 accumulator columns of this warp's 32 lanes, split into issue and wait so that several loads
// can be in flight before one wait
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  tmem_ld16_issue(taddr, r);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// one warp allocates `cols` TMEM columns (address written to shared memory at `slot`) and gives up the permit;
// the same warp frees them at the end
__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_free(uint32_t base, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols));
}
// one lane of the (fully active) warp; warp-uniform code around it keeps the operands in uniform registers
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{ .reg .pred P; elect.sync _|P, 0xffffffff; selp.u32 %0, 1, 0, P; }" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void bar_sync_epi() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

// one 16-byte chunk (8 channels starting at ci) of T(x) at conv-resolution pixel (n, ih, iw)
__device__ __forceinline__ uint4 load_chunk(const iea_conv_desc& d, int hs, int ws, int64_t n, int ih, int iw, int ci) {
  if ((unsigned)ih >= (unsigned)d.h || (unsigned)iw >= (unsigned)d.w) return make_uint4(0, 0, 0, 0);
  const bf16* x = (const bf16*)d.x;
  const bool affine = d.in_scale != nullptr;
  if (d.in_mode == IEA_IN_DIRECT && !affine && !d.in_relu)
    return *reinterpret_cast<const uint4*>(x + ((n * hs + ih) * (int64_t)ws + iw) * d.x_ld + ci);
  float sc[8], sh[8];
  if (affine) {
    const int64_t si = (d.in_bcast ? 0 : n * d.cin) + ci;
    const float4 a0 = *reinterpret_cast<const float4*>(d.in_scale + si), a1 = *reinterpret_cast<const float4*>(d.in_scale + si + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(d.in_shift + si), b1 = *reinterpret_cast<const float4*>(d.in_shift + si + 4);
    sc[0] = a0.x; sc[1] = a0.y; sc[2] = a0.z; sc[3] = a0.w; sc[4] = a1.x; sc[5] = a1.y; sc[6] = a1.z; sc[7] = a1.w;
    sh[0] = b0.x; sh[1] = b0.y; sh[2] = b0.z; sh[3] = b0.w; sh[4] = b1.x; sh[5] = b1.y; sh[6] = b1.z; sh[7] = b1.w;
  }
  float acc[8];
  if (d.in_mode == IEA_IN_POOL2) {
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        float f[8];
        unpack8(*reinterpret_cast<const uint4*>(x + ((n * hs + 2 * ih + a) * (int64_t)ws + 2 * iw + b) * d.x_ld + ci), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float v = affine ? fmaf(f[j], sc[j], sh[j]) : f[j];
          if (d.in_relu) v = fmaxf(v, 0.f);
          acc[j] += v;
        }
      }
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] *= 0.25f;
  } else {
    const int s = d.in_mode == IEA_IN_UP2 ? 1 : 0;
    unpack8(*reinterpret_cast<const uint4*>(x + ((n * hs + (ih >> s)) * (int64_t)ws + (iw >> s)) * d.x_ld + ci), acc);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = affine ? fmaf(acc[j], sc[j], sh[j]) : acc[j];
      if (d.in_relu) v = fmaxf(v, 0.f);
      acc[j] = v;
    }
  }
  return pack8(acc);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda); null when the
// driver does not provide it
typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline encode_tiled_fn tma_encoder() {
  static encode_tiled_fn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (encode_tiled_fn)p;
  }
  return fn;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// division by a launch-time constant as multiply-high + shift (n < 2^31): pixel -> (image, row, column) in the
// tile loops of the persistent kernels
struct FastDiv { uint32_t mul, shr, d; };
inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f; f.d = d;
  if (d == 1) { f.mul = 0; f.shr = 0; return f; }
  uint32_t s = 0;
  while ((1u << s) < d) ++s;
  f.shr = s;
  f.mul = (uint32_t)(((1ull << (32 + s)) + d - 1) / d - (1ull << 32));
  return f;
}
__device__ __forceinline__ uint32_t fdiv(uint32_t n, const FastDiv& f) {
  if (f.d == 1) return n;
  const uint32_t t = __umulhi(n, f.mul);
  return (t + ((n - t) >> 1)) >> (f.shr - 1);
}

}  // namespace tc
