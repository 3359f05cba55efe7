// attn_tc.cu -- BigGAN self-attention core on tcgen05 / TMEM (layers.py:289-299):
//   beta = softmax(theta phi^T)  (no 1/sqrt(d)),   o = beta g
//   theta [n][hw][32], phi [n][hwk][32], g [n][hwk][128]  ->  o [n][hw][128]      (bf16, hw = 4 hwk)
// The (hw x hwk) attention map never leaves the SM: S = theta phi^T is a UMMA into TMEM, every thread
// owns one TMEM lane (= one query row, or one key row in the key-parallel backward pass), turns its
// row into bf16 probabilities in shared memory, and the second UMMA consumes them from there.
//
// Operand staging.  Every operand is copied with 16-byte cp.async into "planes":
//     plane c, row r  =  the 8 channels [8c, 8c+8) of row r            (plane pitch PL = 128*16+16 B)
// One such image serves BOTH operand orientations the backward pass needs:
//   * K-major  (reduction over channels): plane = K chunk  -> LBO = PL,  SBO = 128 B (8-row group)
//   * MN-major (reduction over rows):     plane = MN chunk -> SBO = PL,  LBO = 128 B (8-row group)
// (canonical no-swizzle UMMA layouts; the instruction descriptor's a_major / b_major bits select the
// orientation).  So g is staged once and read as the [keys x cv] B operand of o = P g (MN-major) and as
// the [keys x cv] operand of dP = dO g^T (K-major); the same holds for theta, phi, dO, P and dS.
//
// Kernels (128 threads = 128 TMEM lanes; 128-key blocks):
//   attn_fwd_tc    CTA = (image, 128 queries).  Pass 1: row max over all key blocks (S only).
//                  Pass 2: P = exp(S - max) -> smem, O += P g in TMEM; epilogue O / sum, lse.
//   attn_bwd_q_tc  CTA = (image, 128 queries): D = dO.O, then per key block S and dP = dO g^T,
//                  dS = P (dP - D) -> smem, dtheta += dS phi.
//   attn_bwd_kv_tc CTA = (image, 128 keys): per query tile S^T = phi theta^T and dP^T = g dO^T,
//                  P^T, dS^T -> smem, dphi += dS^T theta, dg += P^T dO.  Deterministic (no atomics).
// Other shapes / fp32 activations stay on the CUDA-core kernels of attn.cu.
#include "tc_common.cuh"
#include <stdlib.h>
using namespace iea;

namespace atc {
using namespace tc;

constexpr int CK = 32, CV = 128, BLK = 128, THREADS = 128;
constexpr int CKC = CK / 8, CVC = CV / 8;          // 16-byte chunks per row
constexpr uint32_t PL = BLK * 16 + 16;             // plane pitch (16-byte skew: conflict-free staging)
constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ uint64_t desc_k(uint32_t addr) { return make_desc(addr, PL, 128); }    // K-major
__device__ __forceinline__ uint64_t desc_mn(uint32_t addr) { return make_desc(addr, 128, PL); }   // MN-major

// 128 rows of CH 16-byte chunks (row pitch ld elements) -> planes
template <int CH>
__device__ __forceinline__ void stage(uint32_t dst, const bf16* src, int ld) {
#pragma unroll
  for (int e = threadIdx.x; e < BLK * CH; e += THREADS) {
    const int r = e / CH, c = e % CH;
    cp16(dst + c * PL + r * 16, src + (int64_t)r * ld + c * 8);
  }
}
__device__ __forceinline__ void staged_ready() {
  cp_async_commit();
  cp_async_wait<0>();
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
}
// K-major A x K-major B, KS 16-wide k-steps
template <int KS>
__device__ __forceinline__ void mma_kk(uint32_t tacc, uint32_t a, uint32_t b, int n, bool acc) {
#pragma unroll
  for (int j = 0; j < KS; ++j) tc_mma(tacc, desc_k(a + 2 * j * PL), desc_k(b + 2 * j * PL), idesc(n, false, false), (acc || j > 0) ? 1u : 0u);
}
// K-major A (rows = M, reduction over its 128 plane-chunked columns) x MN-major B (reduction over its 128 rows)
__device__ __forceinline__ void mma_kmn(uint32_t tacc, uint32_t a, uint32_t b, int n, bool acc) {
#pragma unroll
  for (int j = 0; j < BLK / 16; ++j) tc_mma(tacc, desc_k(a + 2 * j * PL), desc_mn(b + j * 256), idesc(n, false, true), (acc || j > 0) ? 1u : 0u);
}
__device__ __forceinline__ void st16(uint32_t addr, const uint4& q) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(q.x), "r"(q.y), "r"(q.z), "r"(q.w) : "memory");
}

struct Ctx {
  uint32_t bar, phase, tmem, lane_off;
  __device__ __forceinline__ void wait() {
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
  }
};
// barrier + TMEM set-up; returns with all threads synchronised
__device__ __forceinline__ Ctx setup(uint8_t* smem, uint32_t bar_off, uint32_t cols) {
  Ctx c;
  c.bar = smem_u32(smem) + bar_off;
  uint32_t* slot = reinterpret_cast<uint32_t*>(smem + bar_off + 8);
  if (threadIdx.x == 0) {
    mbar_init(c.bar, 1);
    fence_mbar_init();
  }
  if (threadIdx.x < 32) tmem_alloc(smem_u32(slot), cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  c.tmem = *slot;
  c.phase = 0;
  c.lane_off = (uint32_t)((threadIdx.x >> 5) * 32) << 16;  // warp w reads TMEM lanes 32w .. 32w+31
  return c;
}
__device__ __forceinline__ void teardown(const Ctx& c, uint32_t cols) {
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) {
    tc_fence_after();
    tmem_free(c.tmem, cols);
  }
}

// ------------------------------------------------------------------ forward
struct FwdP { const bf16 *th, *ph, *g; bf16* o; float* lse; int hw, hwk; };
constexpr uint32_t FWD_SMEM = (CKC + CKC + CVC + 16) * PL + 16;
constexpr uint32_t FWD_COLS = 256;

__global__ void __launch_bounds__(THREADS) attn_fwd_tc(const FwdP p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sTH = smem_u32(smem), sPH = sTH + CKC * PL, sG = sPH + CKC * PL, sP = sG + CVC * PL;
  Ctx c = setup(smem, (CKC + CKC + CVC + 16) * PL, FWD_COLS);
  const int tid = threadIdx.x;
  const int64_t n = blockIdx.y, q0 = (int64_t)blockIdx.x * BLK;
  const uint32_t tS = c.tmem, tO = c.tmem + 128;
  const int nkb = p.hwk / BLK;
  stage<CKC>(sTH, p.th + (n * p.hw + q0) * CK, CK);
  // ---- pass 1: row maximum over all keys
  float m = -3.0e38f;
  for (int kb = 0; kb < nkb; ++kb) {
    stage<CKC>(sPH, p.ph + (n * p.hwk + (int64_t)kb * BLK) * CK, CK);
    staged_ready();
    if (tid == 0) {
      tc_fence_after();
      mma_kk<CK / 16>(tS, sTH, sPH, BLK, false);
      tc_commit(c.bar);
    }
    c.wait();
#pragma unroll
    for (int j = 0; j < BLK / 16; ++j) {
      float s[16];
      tmem_ld16(tS + c.lane_off + j * 16, s);
#pragma unroll
      for (int i = 0; i < 16; ++i) m = fmaxf(m, s[i]);
    }
  }
  // ---- pass 2: P = exp(S - m) (bf16, shared memory), O += P g
  const float mb = m * LOG2E;
  float l = 0.f;
  for (int kb = 0; kb < nkb; ++kb) {
    tc_fence_before();
    __syncthreads();  // every thread has read S of the previous block
    if (nkb > 1) stage<CKC>(sPH, p.ph + (n * p.hwk + (int64_t)kb * BLK) * CK, CK);
    stage<CVC>(sG, p.g + (n * p.hwk + (int64_t)kb * BLK) * CV, CV);
    staged_ready();
    if (nkb > 1 || kb > 0) {  // (single key block: S of pass 1 is still in TMEM)
      if (tid == 0) {
        tc_fence_after();
        mma_kk<CK / 16>(tS, sTH, sPH, BLK, false);
        tc_commit(c.bar);
      }
      c.wait();
    }
#pragma unroll
    for (int j = 0; j < BLK / 16; ++j) {
      float s[16];
      tmem_ld16(tS + c.lane_off + j * 16, s);
#pragma unroll
      for (int i = 0; i < 16; ++i) { s[i] = exp2f(fmaf(s[i], LOG2E, -mb)); l += s[i]; }
      st16(sP + (2 * j) * PL + tid * 16, pack8(s));
      st16(sP + (2 * j + 1) * PL + tid * 16, pack8(s + 8));
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      mma_kmn(tO, sP, sG, CV, kb > 0);
      tc_commit(c.bar);
    }
    c.wait();  // P, g and phi may be overwritten
  }
  // ---- epilogue
  const float inv = 1.f / l;
  bf16* orow = p.o + (n * p.hw + q0 + tid) * CV;
#pragma unroll
  for (int j = 0; j < CV / 16; ++j) {
    float v[16];
    tmem_ld16(tO + c.lane_off + j * 16, v);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] *= inv;
    *reinterpret_cast<uint4*>(orow + j * 16) = pack8(v);
    *reinterpret_cast<uint4*>(orow + j * 16 + 8) = pack8(v + 8);
  }
  p.lse[n * p.hw + q0 + tid] = m + __logf(l);
  teardown(c, FWD_COLS);
}

// ------------------------------------------------------------------ backward, query-parallel: d theta, D = dO . O
struct BwdP {
  const bf16 *d_o, *th, *ph, *g, *o; const float* lse;
  bf16 *dth, *dph, *dg; float* dq; int hw, hwk;
};
constexpr uint32_t BQ_PLANES = CKC + CVC + CKC + CVC + 16;  // theta, dO, phi, g, dS
constexpr uint32_t BQ_SMEM = BQ_PLANES * PL + 16;
constexpr uint32_t BQ_COLS = 512;

__global__ void __launch_bounds__(THREADS) attn_bwd_q_tc(const BwdP p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sTH = smem_u32(smem), sDO = sTH + CKC * PL, sPH = sDO + CVC * PL, sG = sPH + CKC * PL, sDS = sG + CVC * PL;
  Ctx c = setup(smem, BQ_PLANES * PL, BQ_COLS);
  const int tid = threadIdx.x;
  const int64_t n = blockIdx.y, q0 = (int64_t)blockIdx.x * BLK;
  const int64_t row = n * p.hw + q0 + tid;
  const uint32_t tS = c.tmem, tDP = c.tmem + 128, tDT = c.tmem + 256;
  const int nkb = p.hwk / BLK;
  stage<CKC>(sTH, p.th + (n * p.hw + q0) * CK, CK);
  stage<CVC>(sDO, p.d_o + (n * p.hw + q0) * CV, CV);
  float D = 0.f;
  {
    const uint4* a = reinterpret_cast<const uint4*>(p.d_o + row * CV);
    const uint4* b = reinterpret_cast<const uint4*>(p.o + row * CV);
#pragma unroll 4
    for (int j = 0; j < CVC; ++j) {
      float x[8], y[8];
      unpack8(a[j], x);
      unpack8(b[j], y);
#pragma unroll
      for (int i = 0; i < 8; ++i) D = fmaf(x[i], y[i], D);
    }
    p.dq[row] = D;
  }
  const float lb = p.lse[row] * LOG2E;
  for (int kb = 0; kb < nkb; ++kb) {
    stage<CKC>(sPH, p.ph + (n * p.hwk + (int64_t)kb * BLK) * CK, CK);
    stage<CVC>(sG, p.g + (n * p.hwk + (int64_t)kb * BLK) * CV, CV);
    staged_ready();
    if (tid == 0) {
      tc_fence_after();
      mma_kk<CK / 16>(tS, sTH, sPH, BLK, false);   // S  = theta phi^T
      mma_kk<CV / 16>(tDP, sDO, sG, BLK, false);   // dP = dO g^T
      tc_commit(c.bar);
    }
    c.wait();
#pragma unroll
    for (int j = 0; j < BLK / 16; ++j) {
      float s[16], dp[16];
      tmem_ld16(tS + c.lane_off + j * 16, s);
      tmem_ld16(tDP + c.lane_off + j * 16, dp);
#pragma unroll
      for (int i = 0; i < 16; ++i) s[i] = exp2f(fmaf(s[i], LOG2E, -lb)) * (dp[i] - D);
      st16(sDS + (2 * j) * PL + tid * 16, pack8(s));
      st16(sDS + (2 * j + 1) * PL + tid * 16, pack8(s + 8));
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      mma_kmn(tDT, sDS, sPH, CK, kb > 0);          // d theta += dS phi
      tc_commit(c.bar);
    }
    c.wait();
  }
  bf16* drow = p.dth + row * CK;
#pragma unroll
  for (int j = 0; j < CK / 16; ++j) {
    float v[16];
    tmem_ld16(tDT + c.lane_off + j * 16, v);
    *reinterpret_cast<uint4*>(drow + j * 16) = pack8(v);
    *reinterpret_cast<uint4*>(drow + j * 16 + 8) = pack8(v + 8);
  }
  teardown(c, BQ_COLS);
}

// ------------------------------------------------------------------ backward, key-parallel: d phi, d g
constexpr uint32_t BK_PLANES = CKC + CVC + CKC + CVC + 16 + 16;  // phi, g, theta, dO, P^T, dS^T
constexpr uint32_t BK_STAT = BK_PLANES * PL;                    // lse[128], D[128] of the query tile
constexpr uint32_t BK_SMEM = BK_STAT + 2 * BLK * 4 + 16;
constexpr uint32_t BK_COLS = 512;

__global__ void __launch_bounds__(THREADS) attn_bwd_kv_tc(const BwdP p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sPH = smem_u32(smem), sG = sPH + CKC * PL, sTH = sG + CVC * PL, sDO = sTH + CKC * PL, sPT = sDO + CVC * PL,
                 sDST = sPT + 16 * PL;
  float* lq = reinterpret_cast<float*>(smem + BK_STAT);
  Ctx c = setup(smem, BK_STAT + 2 * BLK * 4, BK_COLS);
  const int tid = threadIdx.x;
  const int64_t n = blockIdx.y, k0 = (int64_t)blockIdx.x * BLK;
  const uint32_t tS = c.tmem, tDP = c.tmem + 128, tDG = c.tmem + 256, tDPH = c.tmem + 384;
  const int nqt = p.hw / BLK;
  stage<CKC>(sPH, p.ph + (n * p.hwk + k0) * CK, CK);
  stage<CVC>(sG, p.g + (n * p.hwk + k0) * CV, CV);
  for (int qt = 0; qt < nqt; ++qt) {
    const int64_t q0 = n * p.hw + (int64_t)qt * BLK;
    stage<CKC>(sTH, p.th + q0 * CK, CK);
    stage<CVC>(sDO, p.d_o + q0 * CV, CV);
    lq[tid] = p.lse[q0 + tid] * LOG2E;
    lq[BLK + tid] = p.dq[q0 + tid];
    staged_ready();
    if (tid == 0) {
      tc_fence_after();
      mma_kk<CK / 16>(tS, sPH, sTH, BLK, false);   // S^T  = phi theta^T
      mma_kk<CV / 16>(tDP, sG, sDO, BLK, false);   // dP^T = g dO^T
      tc_commit(c.bar);
    }
    c.wait();
#pragma unroll
    for (int j = 0; j < BLK / 16; ++j) {
      float s[16], dp[16];
      tmem_ld16(tS + c.lane_off + j * 16, s);
      tmem_ld16(tDP + c.lane_off + j * 16, dp);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        s[i] = exp2f(fmaf(s[i], LOG2E, -lq[j * 16 + i]));
        dp[i] = s[i] * (dp[i] - lq[BLK + j * 16 + i]);
      }
      st16(sPT + (2 * j) * PL + tid * 16, pack8(s));
      st16(sPT + (2 * j + 1) * PL + tid * 16, pack8(s + 8));
      st16(sDST + (2 * j) * PL + tid * 16, pack8(dp));
      st16(sDST + (2 * j + 1) * PL + tid * 16, pack8(dp + 8));
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      mma_kmn(tDPH, sDST, sTH, CK, qt > 0);        // d phi += dS^T theta
      mma_kmn(tDG, sPT, sDO, CV, qt > 0);          // d g   += P^T dO
      tc_commit(c.bar);
    }
    c.wait();
  }
  const int64_t krow = n * p.hwk + k0 + tid;
#pragma unroll
  for (int j = 0; j < CK / 16; ++j) {
    float v[16];
    tmem_ld16(tDPH + c.lane_off + j * 16, v);
    *reinterpret_cast<uint4*>(p.dph + krow * CK + j * 16) = pack8(v);
    *reinterpret_cast<uint4*>(p.dph + krow * CK + j * 16 + 8) = pack8(v + 8);
  }
#pragma unroll
  for (int j = 0; j < CV / 16; ++j) {
    float v[16];
    tmem_ld16(tDG + c.lane_off + j * 16, v);
    *reinterpret_cast<uint4*>(p.dg + krow * CV + j * 16) = pack8(v);
    *reinterpret_cast<uint4*>(p.dg + krow * CV + j * 16 + 8) = pack8(v + 8);
  }
  teardown(c, BK_COLS);
}

}  // namespace atc

// 1: this shape runs on the tcgen05 kernels (IEA_ATTN_IMPL=generic forces the CUDA-core kernels)
int iea_attn_tc_ok(int dtype, int64_t n, int hw, int hwk, int ck, int cv, const void* a, const void* b, const void* c,
                   const void* d) {
  const char* e = getenv("IEA_ATTN_IMPL");
  if (e && e[0] == 'g') return 0;
  return dtype == IEA_BF16 && ck == atc::CK && cv == atc::CV && hw > 0 && hwk > 0 && hw % atc::BLK == 0 &&
         hwk % atc::BLK == 0 && n > 0 && n < 65536 && tc::aligned16(a) && tc::aligned16(b) && tc::aligned16(c) &&
         tc::aligned16(d);
}

int iea_attn_fwd_tc(const void* theta, const void* phi, const void* g, int64_t n, int hw, int hwk, void* o, float* lse,
                    cudaStream_t s) {
  atc::FwdP p{(const bf16*)theta, (const bf16*)phi, (const bf16*)g, (bf16*)o, lse, hw, hwk};
  IEA_CUDA(cudaFuncSetAttribute(atc::attn_fwd_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)atc::FWD_SMEM));
  atc::attn_fwd_tc<<<dim3(hw / atc::BLK, (unsigned)n), atc::THREADS, atc::FWD_SMEM, s>>>(p);
  return check_launch("iea_attn_fwd(tcgen05)");
}

int iea_attn_bwd_tc(const void* d_o, const void* theta, const void* phi, const void* g, const void* o, const float* lse,
                    int64_t n, int hw, int hwk, void* dtheta, void* dphi, void* dg, float* dq, cudaStream_t s) {
  atc::BwdP p{(const bf16*)d_o, (const bf16*)theta, (const bf16*)phi, (const bf16*)g, (const bf16*)o, lse,
              (bf16*)dtheta, (bf16*)dphi, (bf16*)dg, dq, hw, hwk};
  IEA_CUDA(cudaFuncSetAttribute(atc::attn_bwd_q_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)atc::BQ_SMEM));
  atc::attn_bwd_q_tc<<<dim3(hw / atc::BLK, (unsigned)n), atc::THREADS, atc::BQ_SMEM, s>>>(p);
  IEA_CUDA(cudaFuncSetAttribute(atc::attn_bwd_kv_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)atc::BK_SMEM));
  atc::attn_bwd_kv_tc<<<dim3(hwk / atc::BLK, (unsigned)n), atc::THREADS, atc::BK_SMEM, s>>>(p);
  return check_launch("iea_attn_bwd(tcgen05)");
}
