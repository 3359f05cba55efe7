// linear_skinny.cu -- the head linears of G and D (layers.py:223-224 SNLinear; the grouped ccbn gain/bias
// GEMM, G.linear, the RRM / D-head projections) and their data gradients: fp32 feature matrices with only
// M = 40*E rows (one per image) but K or N up to 24576.  As a convolution (h = w = 1) they give the generic
// kernel 3 x 8 CTAs that each walk K = 12096 serially (2.9 ms for 1 GMAC).
//
// Here: 64 x 64 output tile per CTA, fp32 FFMA with 4 x 4 register tiles, 16-byte loads of both K-contiguous
// operands -- and split-K over a THREAD-BLOCK CLUSTER: the up-to-8 CTAs of a cluster take consecutive K
// slices of the same tile, park their partial tile in shared memory and every CTA then sums its 1/8 of the
// tile over all ranks through distributed shared memory in rank order (deterministic, no global scratch,
// no atomics) before the fused epilogue (1/sigma, bias, residual, accumulate, activation).
#include "common.cuh"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;
using namespace iea;

namespace lsk {
constexpr int BM = 64, BN = 64, BK = 16;

// 4 consecutive K elements of row r (fp32 or bf16 storage), zero beyond k_end
__device__ __forceinline__ float4 load4(const void* base, int dtype, int64_t row_off, int k, int k_end) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (k + 3 < k_end) {
    if (dtype == IEA_F32) {
      v = *reinterpret_cast<const float4*>((const float*)base + row_off + k);
    } else {
      const uint2 q = *reinterpret_cast<const uint2*>((const bf16*)base + row_off + k);
      v = make_float4(__uint_as_float(q.x << 16), __uint_as_float(q.x & 0xFFFF0000u), __uint_as_float(q.y << 16),
                      __uint_as_float(q.y & 0xFFFF0000u));
    }
  } else {
    float t[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j = 0; j < 4; ++j)
      if (k + j < k_end) t[j] = ld_act(base, dtype, row_off + k + j);
    v = make_float4(t[0], t[1], t[2], t[3]);
  }
  return v;
}

__global__ void __launch_bounds__(256) linear_skinny_kernel(const iea_conv_desc d, int M, int k_per_cta) {
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank(), nrank = (int)cluster.num_blocks();
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];
  __shared__ __align__(16) float part[BM * BN];  // this CTA's partial tile (row-major)
  const int tid = threadIdx.x;
  const int m0 = blockIdx.x * BM, c0 = blockIdx.y * BN;
  const int kb = rank * k_per_cta;
  const int ke = kb + k_per_cta < d.cin ? kb + k_per_cta : d.cin;
  const int tx = tid & 15, ty = tid >> 4;   // 16 x 16 threads, 4 x 4 outputs each
  const int lr = tid >> 2, lk = (tid & 3) * 4;  // loader: 64 rows x 4 k-quads
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const bool a_ok = m0 + lr < M, b_ok = c0 + lr < d.cout;
  const int64_t a_off = (int64_t)(m0 + lr) * d.x_ld, b_off = (int64_t)(c0 + lr) * d.cin;
  const int64_t s_off = d.in_scale ? (d.in_bcast ? 0 : (int64_t)(m0 + lr) * d.cin) : 0;
  for (int k0 = kb; k0 < ke; k0 += BK) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    const int k = k0 + lk;
    if (a_ok && k < ke) {
      a = load4(d.x, d.x_dtype, a_off, k, ke);
      if (d.in_scale) {  // fused prologue T(x) = relu?(x * scale + shift)
        const float4 s = load4(d.in_scale, IEA_F32, s_off, k, ke), h = load4(d.in_shift, IEA_F32, s_off, k, ke);
        a.x = fmaf(a.x, s.x, h.x); a.y = fmaf(a.y, s.y, h.y); a.z = fmaf(a.z, s.z, h.z); a.w = fmaf(a.w, s.w, h.w);
        if (k + 3 >= ke) {  // (the zero fill beyond k_end must stay zero)
          if (k + 1 >= ke) a.y = 0.f;
          if (k + 2 >= ke) a.z = 0.f;
          if (k + 3 >= ke) a.w = 0.f;
        }
      }
      if (d.in_relu) { a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f); }
    }
    if (b_ok && k < ke) b = load4(d.wpack, d.w_dtype, b_off, k, ke);
    __syncthreads();  // previous tile fully consumed
    As[lk][lr] = a.x; As[lk + 1][lr] = a.y; As[lk + 2][lr] = a.z; As[lk + 3][lr] = a.w;
    Bs[lk][lr] = b.x; Bs[lk + 1][lr] = b.y; Bs[lk + 2][lr] = b.z; Bs[lk + 3][lr] = b.w;
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float a4[4] = {av.x, av.y, av.z, av.w}, b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], b4[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
    *reinterpret_cast<float4*>(&part[(ty * 4 + i) * BN + tx * 4]) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
  cluster.sync();
  // every CTA reduces its slice of the tile over all ranks (rank order: deterministic) and runs the epilogue
  const int per = BM * BN / nrank;
  for (int e = rank * per + tid; e < (rank + 1) * per; e += 256) {
    float v = 0.f;
    for (int r = 0; r < nrank; ++r) v += cluster.map_shared_rank(part, r)[e];
    const int row = e / BN, col = e - row * BN;
    const int64_t m = m0 + row;
    const int c = c0 + col;
    if (m >= M || c >= d.cout) continue;
    if (d.out_scale) v *= d.out_scale[d.out_scale_stride ? c : 0];
    if (d.bias) v += d.bias[c];
    if (d.res && c < d.res_c) v += ld_act(d.res, d.res_dtype, m * d.res_ld + c);
    if (d.acc_c0 >= 0 && c >= d.acc_c0) v += ld_act(d.y, d.y_dtype, m * d.y_ld + c);
    if (d.act == IEA_ACT_RELU) v = fmaxf(v, 0.f);
    else if (d.act == IEA_ACT_TANH) v = tanhf(v);
    st_act(d.y, d.y_dtype, m * d.y_ld + c, v);
  }
  cluster.sync();  // nobody leaves while its shared memory may still be read
}
}  // namespace lsk

int iea_linear_skinny_ok(const iea_conv_desc* d) {
  if (d->h != 1 || d->w != 1 || d->ksize != 1 || d->in_mode != IEA_IN_DIRECT || d->stats) return 0;
  if (d->n > 4096 || d->n < 1) return 0;
  if (d->res && d->res_mode != IEA_IN_DIRECT) return 0;
  if ((int64_t)d->cin * d->cout < 64 * 1024) return 0;  // small layers: the generic kernel is fine
  // 16-byte loads: K-contiguous rows must stay aligned
  const int xa = d->x_dtype == IEA_F32 ? 4 : 8, wa = d->w_dtype == IEA_F32 ? 4 : 8;
  if (d->x_ld % xa || d->cin % wa || d->cin % 4) return 0;
  if ((reinterpret_cast<uintptr_t>(d->x) & 15) || (reinterpret_cast<uintptr_t>(d->wpack) & 15)) return 0;
  if (d->in_scale && ((reinterpret_cast<uintptr_t>(d->in_scale) & 15) || (reinterpret_cast<uintptr_t>(d->in_shift) & 15))) return 0;
  return 1;
}

int iea_linear_skinny(const iea_conv_desc* d, cudaStream_t s) {
  const int M = (int)d->n;
  const int tiles = cdiv(M, lsk::BM) * cdiv(d->cout, lsk::BN);
  const int sms = sm_count();
  int split = 1;  // cluster size: enough CTAs to fill the chip, at least 128 K elements per CTA
  while (split < 8 && tiles * split < 2 * sms && d->cin / (split * 2) >= 128) split *= 2;
  int kper = cdiv(d->cin, split);
  kper = (kper + lsk::BK - 1) / lsk::BK * lsk::BK;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(cdiv(M, lsk::BM), cdiv(d->cout, lsk::BN), split);
  cfg.blockDim = dim3(256);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = split;
  cfg.attrs = attr; cfg.numAttrs = 1;
  IEA_CUDA(cudaLaunchKernelEx(&cfg, lsk::linear_skinny_kernel, *d, M, kper));
  return check_launch("iea_conv_fprop(skinny linear)");
}
