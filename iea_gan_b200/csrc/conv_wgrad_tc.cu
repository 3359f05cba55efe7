// conv_wgrad_tc.cu -- tcgen05 / TMEM weight gradient for the wide (>= 64-channel), low-resolution convolutions.
//
//   dW[co][tap][ci] = sum over pixels  g[px][co] * T(x)[px + tap][ci]            (backward of layers.py:198-206)
//
// As a UMMA the pixels are the K dimension: D[M = 128 output channels][N = 64 / 128 input channels] accumulates
// in TMEM over ALL pixel tiles a CTA owns (fp32, never leaves the SM until the end), A = g^T and B = T(x) shifted
// by the tap.  Both operands live in shared memory exactly as the forward kernels stage them -- 16-byte chunks of
// 8 channels per pixel, planes of [128 pixels][16 B] -- and are read through MN-major descriptors (pixels = K along
// the rows), so no transpose is ever materialised.  One CTA owns a (pixel split, group of up to 3 (tap, ci-block)
// accumulators, 128-wide co block); partials of the pixel splits are summed in a fixed order afterwards.
//
// Why only these layers: the mma.sync kernel of conv_wgrad_mma.cu is HBM-bound and fine on the 16..32-channel
// layers at 128^2..256^2 (UMMA's M >= 64 would waste 4-8x the shared-memory reads there), but on 128 -> 128 3x3 at
// 4^2..16^2 it took 200-270 us per call whatever the size (6 GFLOP: 7-30 TFLOP/s), 9 ms of the 164 ms train step.
#include "tc_common.cuh"
using namespace iea;

namespace wg {
__global__ void wgrad_reduce_kernel(const float* gpart, int nsplit, int64_t total, float* out);
}

namespace wtc {
using namespace tc;

constexpr int BK = 128;             // pixels per tile (the UMMA K extent per staged tile)
constexpr int THREADS = 256;
constexpr int MAXSLOT = 3;          // (tap, ci-block) accumulators per CTA: 3 x 128 fp32 columns of TMEM
constexpr uint32_t PL = BK * 16 + 16;  // plane pitch (16-byte skew, as attn_tc.cu)

struct Params {
  iea_conv_desc d;
  const bf16* g;
  int g_ld;
  float* parts;       // [S][cout][taps][cin]
  int64_t M;
  int hs, ws, nb, cprx, units, cin_blocks, n_tiles, S, slots, nbuf;
  uint32_t g_bytes, x_bytes, buf_bytes, bar_off, tmem_cols;
};

__device__ __forceinline__ uint64_t desc_mn(uint32_t addr) { return make_desc(addr, 128, PL); }

__global__ void __launch_bounds__(THREADS, 1) wgrad_tc_kernel(const Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const iea_conv_desc& d = p.d;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + p.bar_off;  // mma_done[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + p.bar_off + 16);
  if (tid == 0) {
    mbar_init(bar0, 1);
    mbar_init(bar0 + 8, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int split = blockIdx.x, group = blockIdx.y, cob = blockIdx.z;
  const int u0 = group * p.slots;
  const int nslot = p.units - u0 < p.slots ? p.units - u0 : p.slots;
  const int co0 = cob * 128;
  const int taps = d.ksize * d.ksize;
  // zero the g planes of output channels beyond cout once (both buffers): they are never written again
  const int g_planes = (d.cout - co0 >= 128) ? 16 : (d.cout - co0) / 8;
  for (int b = 0; b < p.nbuf; ++b)
    for (int e = tid; e < (16 - g_planes) * BK; e += THREADS) {
      const int c = g_planes + e / BK, r = e % BK;
      *reinterpret_cast<uint4*>(smem + b * p.buf_bytes + c * PL + r * 16) = make_uint4(0, 0, 0, 0);
    }

  int it = 0;
  const int nbuf = p.nbuf;
  for (int t = split; t < p.n_tiles; t += p.S, ++it) {
    const int b = it % nbuf;
    if (it >= nbuf) {  // the MMAs that read buffer b `nbuf` tiles ago must have completed
      mbar_wait(bar0 + 8 * b, (it / nbuf - 1) & 1);
      tc_fence_after();
    }
    uint8_t* buf = smem + b * p.buf_bytes;
    const int m0 = t * BK;
    // ---- g tile: [g_planes][128 px][8 co]
    for (int e = tid; e < g_planes * BK; e += THREADS) {
      const int c = e % g_planes, r = e / g_planes;
      const int m = m0 + r;
      uint4 v = make_uint4(0, 0, 0, 0);
      if (m < (int)p.M) v = __ldg(reinterpret_cast<const uint4*>(p.g + (int64_t)m * p.g_ld + co0 + c * 8));
      *reinterpret_cast<uint4*>(buf + c * PL + r * 16) = v;
    }
    // ---- x tiles, one per accumulator slot: T(x) at the tap-shifted pixel, [cprx][128 px][8 ci].
    // A thread owns the same rows in every slot: their (image, row, column) are computed once per tile.
    constexpr int MAXR = BK * 16 / THREADS;  // rows per thread at 16 planes
    int rn[MAXR], roh[MAXR], row_[MAXR];
    const int nrow = BK * p.cprx / THREADS;
#pragma unroll
    for (int i = 0; i < MAXR; ++i) {
      rn[i] = -1; roh[i] = 0; row_[i] = 0;
      if (i < nrow) {
        const int r = (i * THREADS + tid) / p.cprx;
        const unsigned m = (unsigned)(m0 + r);
        if (m < (unsigned)p.M) {
          const unsigned q = m / (unsigned)d.w;
          row_[i] = (int)(m - q * (unsigned)d.w);
          rn[i] = (int)(q / (unsigned)d.h);
          roh[i] = (int)(q - (unsigned)rn[i] * (unsigned)d.h);
        }
      }
    }
    for (int s = 0; s < nslot; ++s) {
      const int u = u0 + s, tap = u / p.cin_blocks, cb = u - tap * p.cin_blocks;
      int dh = 0, dw = 0;
      if (d.ksize == 3) { dh = tap / 3 - 1; dw = tap % 3 - 1; }
      uint8_t* xb = buf + p.g_bytes + s * p.x_bytes;
#pragma unroll
      for (int i = 0; i < MAXR; ++i) {
        if (i < nrow) {
          const int e = i * THREADS + tid;
          const int c = e % p.cprx, r = e / p.cprx;
          uint4 v = make_uint4(0, 0, 0, 0);
          if (rn[i] >= 0) v = load_chunk(d, p.hs, p.ws, rn[i], roh[i] + dh, row_[i] + dw, cb * p.nb + c * 8);
          *reinterpret_cast<uint4*>(xb + c * PL + r * 16) = v;
        }
      }
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      const uint32_t a0 = sbase + b * p.buf_bytes;
      const uint32_t id = idesc(p.nb, true, true);
      for (int s = 0; s < nslot; ++s) {
        const uint32_t x0 = a0 + p.g_bytes + s * p.x_bytes;
#pragma unroll
        for (int j = 0; j < BK / 16; ++j)
          tc_mma(tmem + s * 128, desc_mn(a0 + j * 256), desc_mn(x0 + j * 256), id, (it > 0 || j > 0) ? 1u : 0u);
      }
      tc_commit(bar0 + 8 * b);
    }
  }
  // ---- all MMAs done: wait for the last commit of every buffer that was used
  const int n_it = it;
  for (int j = n_it - 1; j >= 0 && j >= n_it - nbuf; --j) mbar_wait(bar0 + 8 * (j % nbuf), (j / nbuf) & 1);
  tc_fence_after();
  // ---- epilogue: TMEM lane = output channel; warps 0-3 cover the 128 lanes
  if (warp < 4) {
    const int co = co0 + tid;  // tid = lane index 0..127
    float* out = p.parts + (int64_t)split * d.cout * taps * d.cin;
    for (int s = 0; s < nslot; ++s) {
      const int u = u0 + s, tap = u / p.cin_blocks, cb = u - tap * p.cin_blocks;
      for (int c16 = 0; c16 < p.nb / 16; ++c16) {
        float v[16];
        if (n_it > 0) {
          tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + s * 128 + c16 * 16, v);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = 0.f;
        }
        if (co < d.cout) {
          float* o = out + ((int64_t)co * taps + tap) * d.cin + cb * p.nb + c16 * 16;
#pragma unroll
          for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_free(tmem, p.tmem_cols);
}

static bool plan(const iea_conv_desc* d, int g_dtype, int g_ld, Params* p) {
  const int64_t M = d->n * (int64_t)d->h * d->w;
  if (d->x_dtype != IEA_BF16 || g_dtype != IEA_BF16) return false;
  if (!(d->cin == 64 || d->cin % 128 == 0) || d->cout < 64 || d->cout % 8) return false;
  if (d->ksize != 1 && d->ksize != 3) return false;
  if (M < 512 || M > 131072) return false;  // the low-resolution, tensor / latency-bound regime
  if (d->x_ld % 8 || g_ld % 8 || !aligned16(d->x)) return false;
  if (d->in_scale && (!aligned16(d->in_scale) || !aligned16(d->in_shift) || d->cin % 4)) return false;
  p->d = *d;
  p->M = M;
  p->hs = stored_res(*d, d->h);
  p->ws = stored_res(*d, d->w);
  p->nb = d->cin < 128 ? d->cin : 128;
  p->cprx = p->nb / 8;
  p->cin_blocks = d->cin / p->nb;
  p->units = d->ksize * d->ksize * p->cin_blocks;
  p->slots = p->units < MAXSLOT ? p->units : MAXSLOT;
  p->n_tiles = (int)((M + BK - 1) / BK);
  const int groups = (p->units + p->slots - 1) / p->slots, cobs = (d->cout + 127) / 128;
  int S = 148 / (groups * cobs);
  if (S < 1) S = 1;
  if (S > p->n_tiles) S = p->n_tiles;
  if (S > 64) S = 64;
  p->S = S;
  p->g_bytes = 16 * PL;
  p->x_bytes = p->cprx * PL;
  p->buf_bytes = p->g_bytes + p->slots * p->x_bytes;
  p->nbuf = 2 * p->buf_bytes + 64 <= 220 * 1024 ? 2 : 1;  // (128 input channels: 3 x 33 KB of x tiles -> one buffer)
  p->bar_off = p->nbuf * p->buf_bytes;
  p->tmem_cols = 512;
  return true;
}

}  // namespace wtc

// number of pixel splits (partial slices) the tcgen05 weight-gradient kernel writes; 0: shape not handled
int iea_conv_wgrad_tc_splits(const iea_conv_desc* d, int g_dtype, int g_ld) {
  wtc::Params p;
  return wtc::plan(d, g_dtype, g_ld, &p) ? p.S : 0;
}

// gpart: slice 0 receives the sum, slices 1..S the per-split partials
int iea_conv_wgrad_tc(const iea_conv_desc* d, const void* g, int g_dtype, int g_ld, float* gpart, cudaStream_t s) {
  wtc::Params p;
  IEA_CHECK_ARG(wtc::plan(d, g_dtype, g_ld, &p) && tc::aligned16(g), "iea_conv_wgrad_tc: shape not handled");
  p.g = (const bf16*)g;
  p.g_ld = g_ld;
  const int64_t total = (int64_t)d->cout * d->ksize * d->ksize * d->cin;
  p.parts = gpart + total;
  const uint32_t smem = p.bar_off + 64;
  IEA_CUDA(cudaFuncSetAttribute(wtc::wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int groups = (p.units + p.slots - 1) / p.slots, cobs = (d->cout + 127) / 128;
  wtc::wgrad_tc_kernel<<<dim3(p.S, groups, cobs), wtc::THREADS, smem, s>>>(p);
  int rb = (int)((total + 255) / 256);
  if (rb > 592) rb = 592;
  wg::wgrad_reduce_kernel<<<rb, 256, 0, s>>>(p.parts, p.S, total, gpart);
  return check_launch("iea_conv_wgrad_tc");
}
