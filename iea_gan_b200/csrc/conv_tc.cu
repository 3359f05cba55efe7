// conv_tc.cu -- tcgen05 / TMEM implicit-GEMM convolutions for sm_100a whose weights do not fit shared memory
// next to a staged patch (>= 128-channel 3x3 and 512-channel 1x1 layers at 4x4..16x16).  Two persistent,
// warp-specialised kernels share one epilogue (epilogue_role):
//
// conv_tc_kernel -- streaming im2col, any shape the tcgen05 path takes (416 threads):
//   warp 0      : TMEM allocation + the single MMA-issuing thread (tcgen05.mma, M=128, N=Cout tile,
//                 K=16 per instruction, fp32 accumulators double-buffered in TMEM)
//   warps 1-8   : A-operand producers.  They read the NHWC bf16 activation, apply the fused prologue
//                 T(x) = [avgpool2|up2](relu(x*scale[n,c]+shift[n,c])) in registers (this is what removes
//                 the separate BN-apply / ReLU / upsample / pool passes over HBM) and write the UMMA
//                 K-major core-matrix layout into the smem ring, once per (tap, k block).  One of them also
//                 streams the matching weight slice with TMA bulk copies (cp.async.bulk, mbarrier complete_tx).
//   warps 9-12  : epilogue.
//   smem ring: `stages` x {A: cpr planes of [128 rows][16 B], B: cpr planes of [BN rows][16 B]} in the
//   no-swizzle ("interleave") canonical layout: 8x16-byte core matrices, SBO = 128 B between 8-row
//   groups, LBO = plane stride between the two 16-byte K chunks of one MMA.
//
// conv_lr_kernel -- staged patch + streamed weights, for 3x3 layers on same-resolution or nearest-up2 inputs
// whose 128-pixel tiles are whole image rows (8x8, 16x16, ...; 448 threads):
//   warp 0      : MMA issuer.  The nine taps are shifted UMMA descriptors on one staged halo patch.
//   warp 1      : weight loader: the (tap, k block) B slices through an mbarrier ring with cp.async.bulk.
//   warps 2-9   : patch producers: each input chunk of the tile's halo patch is loaded, transformed and
//                 stored ONCE (the streaming kernel does it nine times); patches are double-buffered so
//                 tile t+1 loads while tile t multiplies.
//   warps 10-13 : epilogue.
//   Patch layout (per 16-byte channel chunk, one plane each): the tile's 16 groups of 8 output pixels
//   (an image row's 8-column block) are ordered row-major over (tile row, segment), segment = (image of the
//   tile, 8-column block); patch row r holds for every segment the 8 pixels plus a 1-pixel halo on each side
//   (10 pixels).  Group g then starts at g*160 B for every tap, so each tap is the same descriptor (SBO =
//   160 B) with start address + ((dh+1)*segments*10 + dw+1)*16 B.  The MMAs accumulate in the streaming
//   kernel's order (tap, k block, 16-channel step), so both kernels produce bit-identical outputs.
#include "tc_common.cuh"
using namespace iea;

namespace tc {

constexpr int BM = 128;
constexpr int THREADS = 416;   // warp 0: MMA issuer, warps 1-8: A producers, warps 9-12: epilogue
constexpr int NPT = 256;       // producer threads (8 warps: a lone producer warp per scheduler walked ~550 dependent
                               // instructions per K step; twice the warps, half the chunks per thread)

struct Params {
  iea_conv_desc d;
  const bf16* wtc;
  int64_t M;
  int hs, ws, KB, nkb, BN, n_tiles_m, n_tiles_n, stages, taps;
  uint32_t a_bytes, b_bytes, lbo_a, lbo_b, stage_bytes, staging_off, staging_ld, bar_off, stat_off, tmem_cols;
  uint32_t tab_off;  // bf16 scale / shift table of the images of the current tile: [TAB_IMGS][cin] x 2
  uint32_t tfull_off;  // byte offset of the accumulator barriers (tfull[2], tempty[2]) from bar_off
  // conv_lr_kernel only: segments per patch row, 8-column blocks per image row, patch pixels, bytes per patch
  // plane (one 16-byte channel chunk of every patch pixel), bytes per patch, offset of the weight ring
  int nseg, ncb, ppx, hw;
  uint32_t plane, patch_bytes, ring_off;
};
constexpr int TAB_IMGS = 8;


// Epilogue role (warps whose TMEM lane quadrant is q): tcgen05.ld the accumulator, *1/sigma, +bias, +residual
// (direct / up2 / pool2), activation, bf16 pack into the smem staging tile, coalesced 16-byte stores, and the
// per-tile (sum, sum^2) batch-norm partials for the next layer.  `row` is the tile pixel (0..127, offset from the
// tile's first flattened output pixel) that this thread's TMEM lane holds: the staging tile is in pixel order, so
// stores and statistics do not depend on how a kernel orders the MMA rows.
__device__ __forceinline__ void epilogue_role(const Params& p, uint32_t tmem_base, int q, int lane, int row) {
  extern __shared__ __align__(128) uint8_t smem[];
  const iea_conv_desc& d = p.d;
  const int et = q * 32 + lane;
  const uint32_t bar0 = smem_u32(smem) + p.bar_off;
  auto tfull_bar = [&](int b) { return bar0 + p.tfull_off + 8u * b; };
  auto tempty_bar = [&](int b) { return bar0 + p.tfull_off + 8u * (2 + b); };
  const int num_tiles = p.n_tiles_m * p.n_tiles_n;
  uint8_t* stg = smem + p.staging_off;
  float* stat = reinterpret_cast<float*>(smem + p.stat_off);
  uint32_t tcount = 0;
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++tcount) {
    const int tn = tile / p.n_tiles_m, tm = tile - tn * p.n_tiles_m;
    const int64_t m0 = (int64_t)tm * BM;
    const int n0 = tn * p.BN;
    const uint32_t ab = tcount & 1, aph = (tcount >> 1) & 1;
    const int64_t m = m0 + row;
    const bool valid = m < p.M;
    int ow = 0, oh = 0;
    int64_t n = 0;
    if (valid) { ow = (int)(m % d.w); const int64_t t = m / d.w; oh = (int)(t % d.h); n = t / d.h; }
    mbar_wait(tfull_bar(ab), aph);
    tc_fence_after();
    const float osc0 = (d.out_scale && !d.out_scale_stride) ? d.out_scale[0] : 1.f;
    for (int cb = 0; cb < p.BN / 16; ++cb) {
      float v[16];
      tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + ab * p.BN + cb * 16, v);
      const int c0 = n0 + cb * 16;
      if (valid) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float sc = d.out_scale_stride ? d.out_scale[c0 + j] : osc0;
          v[j] = d.bias ? fmaf(v[j], sc, d.bias[c0 + j]) : v[j] * sc;
        }
        if (d.res && c0 < d.res_c) {
          const bf16* rp = (const bf16*)d.res;
          float f[16];
          if (d.res_mode == IEA_IN_POOL2) {
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = 0.f;
            for (int a = 0; a < 2; ++a)
              for (int b = 0; b < 2; ++b) {
                const bf16* sp = rp + ((n * (2 * d.h) + 2 * oh + a) * (int64_t)(2 * d.w) + 2 * ow + b) * d.res_ld + c0;
                float t8[16];
                unpack8(*reinterpret_cast<const uint4*>(sp), t8);
                unpack8(*reinterpret_cast<const uint4*>(sp + 8), t8 + 8);
#pragma unroll
                for (int j = 0; j < 16; ++j) f[j] += 0.25f * t8[j];
              }
          } else {
            const int s = d.res_mode == IEA_IN_UP2 ? 1 : 0;
            const bf16* sp = rp + ((n * (d.h >> s) + (oh >> s)) * (int64_t)(d.w >> s) + (ow >> s)) * d.res_ld + c0;
            unpack8(*reinterpret_cast<const uint4*>(sp), f);
            unpack8(*reinterpret_cast<const uint4*>(sp + 8), f + 8);
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] += f[j];
        }
        if (d.acc_c0 >= 0 && c0 >= d.acc_c0) {
          const bf16* yp = (const bf16*)d.y + m * d.y_ld + c0;
          float f[16];
          unpack8(*reinterpret_cast<const uint4*>(yp), f);
          unpack8(*reinterpret_cast<const uint4*>(yp + 8), f + 8);
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] += f[j];
        }
        if (d.act == IEA_ACT_RELU) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
        } else if (d.act == IEA_ACT_TANH) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = tanhf(v[j]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0.f;
      }
      uint4* dst = reinterpret_cast<uint4*>(stg + (size_t)row * p.staging_ld + cb * 32);
      dst[0] = pack8(v);
      dst[1] = pack8(v + 8);
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(tempty_bar(ab));  // accumulator drained: the MMA warp may start the next tile
    bar_sync_epi();
    // coalesced 16-byte stores of the bf16 tile
    const int cg = p.BN / 8;
    int64_t rows_valid = p.M - m0;
    if (rows_valid > BM) rows_valid = BM;
    bf16* yb = (bf16*)d.y;
    for (int i = et; i < (int)rows_valid * cg; i += 128) {
      const int row = i / cg, g8 = i - row * cg;
      *reinterpret_cast<uint4*>(yb + (m0 + row) * d.y_ld + n0 + g8 * 8) =
          *reinterpret_cast<const uint4*>(stg + (size_t)row * p.staging_ld + g8 * 16);
    }
    if (d.stats) {  // per-tile column (sum, sum^2) of the rounded outputs; fixed order -> deterministic
      int parts = 1;                                            // row parts handled in parallel (power of two)
      while (parts * 2 * cg <= 128) parts *= 2;
      const int rows_per = BM / parts;
      for (int w0 = et; w0 < cg * parts; w0 += 128) {
        const int g8 = w0 % cg, part = w0 / cg;
        float s1[8], s2[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { s1[j] = 0.f; s2[j] = 0.f; }
        for (int r = part * rows_per; r < (part + 1) * rows_per; ++r) {
          float f[8];
          unpack8(*reinterpret_cast<const uint4*>(stg + (size_t)r * p.staging_ld + g8 * 16), f);
#pragma unroll
          for (int j = 0; j < 8; ++j) { s1[j] += f[j]; s2[j] = fmaf(f[j], f[j], s2[j]); }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          stat[(part * p.BN + g8 * 8 + j) * 2] = s1[j];
          stat[(part * p.BN + g8 * 8 + j) * 2 + 1] = s2[j];
        }
      }
      bar_sync_epi();
      for (int c = et; c < p.BN * 2; c += 128) {
        float a = 0.f;
        for (int part = 0; part < parts; ++part) a += stat[part * p.BN * 2 + c];
        d.stats[((int64_t)tm * d.cout + n0) * 2 + c] = a;
      }
    }
    bar_sync_epi();  // staging / stat scratch are reused by the next tile
  }
}

template <int CPR>
__global__ void __launch_bounds__(THREADS, 1) conv_tc_kernel(const Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const iea_conv_desc& d = p.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + p.bar_off;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (p.stages + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * p.stages + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * p.stages + 2 + b); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + p.bar_off + 8 * (2 * p.stages + 4));

  if (tid == 0) {
    // one arrival per producer WARP (+1: the expect_tx of the weight copy) -- 128 per-thread arrivals on one
    // mbarrier serialise and wake the parked MMA thread 128 times per step
    for (int s = 0; s < p.stages; ++s) { mbar_init(full_bar(s), NPT / 32 + 1); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 4); }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int num_tiles = p.n_tiles_m * p.n_tiles_n;
  const int k_iters = p.taps * p.nkb;

  if (warp == 0) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t id = idesc(p.BN, false, false);
      uint32_t g = 0, tcount = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++tcount) {
        const uint32_t ab = tcount & 1, aph = (tcount >> 1) & 1;
        mbar_wait(tempty_bar(ab), aph ^ 1);
        tc_fence_after();
        const uint32_t tacc = tmem_base + ab * p.BN;
        for (int it = 0; it < k_iters; ++it, ++g) {
          const uint32_t s = g % p.stages, ph = (g / p.stages) & 1;
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t a0 = sbase + s * p.stage_bytes, b0 = a0 + p.a_bytes;
#pragma unroll
          for (int j = 0; j < CPR / 2; ++j) {
            const uint64_t da = make_desc(a0 + 2 * j * p.lbo_a, p.lbo_a, 128);
            const uint64_t db = make_desc(b0 + 2 * j * p.lbo_b, p.lbo_b, 128);
            tc_mma(tacc, da, db, id, (it > 0 || j > 0) ? 1u : 0u);
          }
          tc_commit(empty_bar(s));
        }
        tc_commit(tfull_bar(ab));
      }
    }
  } else if (warp <= NPT / 32) {
    // ===================== A producers (+ weight TMA) =====================
    constexpr int NCH = CPR * 128 / NPT;  // 16-byte chunks per thread and K step
    const int pt = tid - 32;
    uint32_t g = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int tn = tile / p.n_tiles_m, tm = tile - tn * p.n_tiles_m;
      const int64_t m0 = (int64_t)tm * BM;
      const int n0 = tn * p.BN;
      int r_[NCH], oh_[NCH], ow_[NCH];
      int64_t n_[NCH], base_[NCH];  // base_: element offset of (n, oh, ow) in a same-resolution input
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int e = i * NPT + pt;
        r_[i] = e / CPR;
        const int64_t m = m0 + r_[i];
        if (m < p.M) {
          ow_[i] = (int)(m % d.w);
          const int64_t t = m / d.w;
          oh_[i] = (int)(t % d.h);
          n_[i] = t / d.h;
        } else {
          ow_[i] = -100000; oh_[i] = -100000; n_[i] = 0;  // out of range -> zero rows
        }
        base_[i] = ((n_[i] * p.hs + oh_[i]) * (int64_t)p.ws + ow_[i]) * d.x_ld;
      }
      const int cc = pt % CPR;  // chunk handled by this thread (e % CPR is the same for every i)
      // ---- software-pipelined path (same-resolution / nearest-up2 inputs): the raw 16-byte chunks of step
      // it+1 are requested BEFORE step it is transformed and stored, so a step no longer pays a full global
      // load round trip (these 4x4..16x16 layers are pure latency: 18 steps per tile, 2 tiles per CTA)
      if (d.in_mode != IEA_IN_POOL2) {
        const bool affine = d.in_scale != nullptr, relu = d.in_relu != 0;
        const int sh_ = d.in_mode == IEA_IN_UP2 ? 1 : 0;
        const bf16* xb = (const bf16*)d.x;
        // fused-prologue constants of the (<= TAB_IMGS) images this tile touches, as bf16 pairs in shared memory:
        // the per-chunk transform is then 2 LDS + 4 packed fma.relu (the same rounding as conv_thin / conv_tc2)
        // instead of four dependent global loads and ~40 fp32 instructions per 16-byte chunk
        const int hw_ = d.h * d.w;
        const int64_t img0 = m0 / hw_;
        int64_t img1 = (m0 + BM - 1 < p.M ? m0 + BM - 1 : p.M - 1) / hw_;
        const int nimg = d.in_bcast ? 1 : (int)(img1 - img0 + 1);
        const bool tab = affine && nimg <= TAB_IMGS;
        bf16* const tsc = reinterpret_cast<bf16*>(smem + p.tab_off);
        bf16* const tsh = tsc + TAB_IMGS * d.cin;
        if (affine) {
          asm volatile("bar.sync 2, 256;" ::: "memory");  // every producer is done with the previous tile's table
          if (tab) {
            const int c8n = d.cin >> 3;
            for (int e = pt; e < nimg * c8n; e += NPT) {
              const int li = e / c8n, c8 = e - li * c8n;
              const int64_t si = (d.in_bcast ? 0 : (img0 + li) * d.cin) + c8 * 8;
              float a[8], b[8];
              *reinterpret_cast<float4*>(a) = *reinterpret_cast<const float4*>(d.in_scale + si);
              *reinterpret_cast<float4*>(a + 4) = *reinterpret_cast<const float4*>(d.in_scale + si + 4);
              *reinterpret_cast<float4*>(b) = *reinterpret_cast<const float4*>(d.in_shift + si);
              *reinterpret_cast<float4*>(b + 4) = *reinterpret_cast<const float4*>(d.in_shift + si + 4);
              *reinterpret_cast<uint4*>(tsc + li * d.cin + c8 * 8) = pack8(a);
              *reinterpret_cast<uint4*>(tsh + li * d.cin + c8 * 8) = pack8(b);
            }
          }
          asm volatile("bar.sync 2, 256;" ::: "memory");
        }
        uint4 nxt[NCH];
        uint32_t nxt_ok = 0;
        auto raw_load = [&](int it) {
          const int tap = it / p.nkb, kb = it - tap * p.nkb;
          int dh = 0, dw = 0;
          if (d.ksize == 3) { dh = tap / 3 - 1; dw = tap % 3 - 1; }
          const int ci = kb * p.KB + cc * 8;
          const int toff = (dh * p.ws + dw) * d.x_ld + ci;  // same-resolution input: one add per chunk
          nxt_ok = 0;
#pragma unroll
          for (int i = 0; i < NCH; ++i) {
            const int ih = oh_[i] + dh, iw = ow_[i] + dw;
            if ((unsigned)ih < (unsigned)d.h && (unsigned)iw < (unsigned)d.w) {
              const bf16* src = sh_ ? xb + ((n_[i] * p.hs + (ih >> 1)) * (int64_t)p.ws + (iw >> 1)) * d.x_ld + ci
                                    : xb + base_[i] + toff;
              nxt[i] = __ldg(reinterpret_cast<const uint4*>(src));
              nxt_ok |= 1u << i;
            }
          }
        };
        raw_load(0);
        for (int it = 0; it < k_iters; ++it, ++g) {
          const uint32_t s = g % p.stages, ph = (g / p.stages) & 1;
          const int tap = it / p.nkb, kb = it - tap * p.nkb;
          uint4 cur[NCH];
          const uint32_t cur_ok = nxt_ok;
#pragma unroll
          for (int i = 0; i < NCH; ++i) cur[i] = nxt[i];
          if (it + 1 < k_iters) raw_load(it + 1);
          mbar_wait(empty_bar(s), ph ^ 1);
          const uint32_t a0 = sbase + s * p.stage_bytes;
          if (pt == 0) {
            mbar_expect_tx(full_bar(s), p.b_bytes);
#pragma unroll
            for (int c = 0; c < CPR; ++c)
              bulk_g2s(a0 + p.a_bytes + c * p.lbo_b,
                       p.wtc + ((((int64_t)tap * p.nkb + kb) * CPR + c) * d.cout + n0) * 8, p.BN * 16, full_bar(s));
          }
          const int ci = kb * p.KB + cc * 8;
#pragma unroll
          for (int i = 0; i < NCH; ++i) {
            uint4 v = make_uint4(0, 0, 0, 0);
            if (cur_ok >> i & 1) {
              v = cur[i];
              if (tab) {
                const int li = d.in_bcast ? 0 : (int)(n_[i] - img0);
                const uint4 s4 = *reinterpret_cast<const uint4*>(tsc + li * d.cin + ci), h4 = *reinterpret_cast<const uint4*>(tsh + li * d.cin + ci);
                __nv_bfloat162* x2 = reinterpret_cast<__nv_bfloat162*>(&v);
                const __nv_bfloat162* s2 = reinterpret_cast<const __nv_bfloat162*>(&s4);
                const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&h4);
                if (relu) {
#pragma unroll
                  for (int j = 0; j < 4; ++j) x2[j] = __hfma2_relu(x2[j], s2[j], h2[j]);
                } else {
#pragma unroll
                  for (int j = 0; j < 4; ++j) x2[j] = __hfma2(x2[j], s2[j], h2[j]);
                }
              } else if (affine || relu) {
                float f[8];
                unpack8(v, f);
                if (affine) {
                  const int64_t si = (d.in_bcast ? 0 : n_[i] * d.cin) + ci;
                  const float4 s0 = *reinterpret_cast<const float4*>(d.in_scale + si), s1 = *reinterpret_cast<const float4*>(d.in_scale + si + 4);
                  const float4 h0 = *reinterpret_cast<const float4*>(d.in_shift + si), h1 = *reinterpret_cast<const float4*>(d.in_shift + si + 4);
                  f[0] = fmaf(f[0], s0.x, h0.x); f[1] = fmaf(f[1], s0.y, h0.y); f[2] = fmaf(f[2], s0.z, h0.z); f[3] = fmaf(f[3], s0.w, h0.w);
                  f[4] = fmaf(f[4], s1.x, h1.x); f[5] = fmaf(f[5], s1.y, h1.y); f[6] = fmaf(f[6], s1.z, h1.z); f[7] = fmaf(f[7], s1.w, h1.w);
                }
                if (relu) {
#pragma unroll
                  for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], 0.f);
                }
                v = pack8(f);
              }
            }
            *reinterpret_cast<uint4*>(smem + s * p.stage_bytes + cc * p.lbo_a + (r_[i] >> 3) * 128 + (r_[i] & 7) * 16) = v;
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(full_bar(s));
        }
        continue;
      }
      for (int it = 0; it < k_iters; ++it, ++g) {
        const uint32_t s = g % p.stages, ph = (g / p.stages) & 1;
        const int tap = it / p.nkb, kb = it - tap * p.nkb;
        mbar_wait(empty_bar(s), ph ^ 1);
        const uint32_t a0 = sbase + s * p.stage_bytes;
        if (pt == 0) {
          mbar_expect_tx(full_bar(s), p.b_bytes);
#pragma unroll
          for (int c = 0; c < CPR; ++c)
            bulk_g2s(a0 + p.a_bytes + c * p.lbo_b,
                     p.wtc + ((((int64_t)tap * p.nkb + kb) * CPR + c) * d.cout + n0) * 8, p.BN * 16, full_bar(s));
        }
        int dh = 0, dw = 0;
        if (d.ksize == 3) { dh = tap / 3 - 1; dw = tap % 3 - 1; }
        const int ci = kb * p.KB + cc * 8;
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          const uint4 v = load_chunk(d, p.hs, p.ws, n_[i], oh_[i] + dh, ow_[i] + dw, ci);
          *reinterpret_cast<uint4*>(smem + s * p.stage_bytes + cc * p.lbo_a + (r_[i] >> 3) * 128 + (r_[i] & 7) * 16) = v;
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(full_bar(s));
      }
    }
  } else {
    // ===================== epilogue =====================
    const int et = (warp & 3) * 32 + lane;  // TMEM lane == tile row
    epilogue_role(p, tmem_base, warp & 3, lane, et);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_free(tmem_base, p.tmem_cols);
  }
}


// ---------------------------------------------------------------------------------------------------------------
// conv_lr_kernel: staged halo patch (A) + streamed weights (B); see the header.
constexpr int LR_THREADS = 448;  // warp 0: MMA, warp 1: weight loader, warps 2-9: patch producers, 10-13: epilogue
constexpr int LR_NPT = 256;      // patch producer threads
constexpr int LR_NCH = 16;       // patch chunks per producer thread: (ppx x cin/8) <= LR_NCH * LR_NPT
constexpr int LR_CPR = 8;        // 16-byte chunks per 64-channel k block

// tile pixel (offset from the tile's first flattened output pixel) held by MMA row `r`
__device__ __forceinline__ int lr_row_pixel(const Params& p, int r) {
  const int g = r >> 3, tr = g / p.nseg, seg = g - tr * p.nseg, img = seg / p.ncb, cb = seg - img * p.ncb;
  return img * p.hw + tr * p.d.w + cb * 8 + (r & 7);
}

__global__ void __launch_bounds__(LR_THREADS, 1) conv_lr_kernel(const Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const iea_conv_desc& d = p.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + p.bar_off;
  auto wfull_bar = [&](int s) { return bar0 + 8u * s; };
  auto wempty_bar = [&](int s) { return bar0 + 8u * (p.stages + s); };
  auto pfull_bar = [&](int b) { return bar0 + 8u * (2 * p.stages + b); };
  auto pempty_bar = [&](int b) { return bar0 + 8u * (2 * p.stages + 2 + b); };
  auto tfull_bar = [&](int b) { return bar0 + p.tfull_off + 8u * b; };
  auto tempty_bar = [&](int b) { return bar0 + p.tfull_off + 8u * (2 + b); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + p.bar_off + p.tfull_off + 32);

  if (tid == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(wfull_bar(s), 1); mbar_init(wempty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) {
      mbar_init(pfull_bar(b), LR_NPT / 32); mbar_init(pempty_bar(b), 1);  // one arrival per producer warp
      mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 4);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int num_tiles = p.n_tiles_m * p.n_tiles_n;

  if (warp == 0) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t id = idesc(p.BN, false, false);
      const uint64_t da0 = make_desc(sbase, p.plane, 160);
      const uint64_t db0 = make_desc(sbase + p.ring_off, p.lbo_b, 128);
      const uint32_t plane16 = p.plane >> 4, lbo16 = p.lbo_b >> 4, stage16 = p.b_bytes >> 4, patch16 = p.patch_bytes >> 4;
      uint32_t s = 0, ph = 0, tcount = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++tcount) {
        const uint32_t ab = tcount & 1, aph = (tcount >> 1) & 1;
        mbar_wait(tempty_bar(ab), aph ^ 1);
        mbar_wait(pfull_bar(ab), aph);
        tc_fence_after();
        const uint32_t tacc = tmem_base + ab * p.BN;
        for (int tap = 0; tap < 9; ++tap) {
          const uint32_t a_tap = ab * patch16 + (uint32_t)((tap / 3) * p.nseg * 10 + tap % 3);
          for (int kb = 0; kb < p.nkb; ++kb) {
            mbar_wait(wfull_bar(s), ph);
            tc_fence_after();
            const uint32_t a16 = a_tap + kb * LR_CPR * plane16, b16 = s * stage16;
#pragma unroll
            for (int j = 0; j < LR_CPR / 2; ++j)
              tc_mma(tacc, da0 + (a16 + 2 * j * plane16), db0 + (b16 + 2 * j * lbo16), id,
                     (tap > 0 || kb > 0 || j > 0) ? 1u : 0u);
            tc_commit(wempty_bar(s));
            if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1; }
          }
        }
        tc_commit(pempty_bar(ab));
        tc_commit(tfull_bar(ab));
      }
    }
  } else if (warp == 1) {
    // ===================== weight loader =====================
    if (lane == 0) {
      uint32_t s = 0, ph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int n0 = (tile / p.n_tiles_m) * p.BN;
        for (int it = 0; it < 9 * p.nkb; ++it) {  // (tap, k block) in the MMA order
          mbar_wait(wempty_bar(s), ph ^ 1);
          const uint32_t dst = sbase + p.ring_off + s * p.b_bytes;
          mbar_expect_tx(wfull_bar(s), p.b_bytes);
#pragma unroll
          for (int c = 0; c < LR_CPR; ++c)
            bulk_g2s(dst + c * p.lbo_b, p.wtc + (((int64_t)it * LR_CPR + c) * d.cout + n0) * 8, p.BN * 16, wfull_bar(s));
          if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp < 2 + LR_NPT / 32) {
    // ===================== patch producers =====================
    const int pt = tid - 64;
    const int cpt = d.cin >> 3;                    // patch planes (divides LR_NPT: cin is 64 or 128)
    const int pl = pt % cpt, pstep = LR_NPT / cpt;  // this thread's plane and its pixel stride
    const int ci = pl * 8;
    const int sh_ = d.in_mode == IEA_IN_UP2 ? 1 : 0;
    const bool affine = d.in_scale != nullptr, relu = d.in_relu != 0;
    const bf16* xb = (const bf16*)d.x;
    const int imgs = p.nseg / p.ncb;              // images per tile (1, or 2 when an image is 64 pixels)
    // tile-independent coordinates of this thread's chunks: patch row, input column + 1, image of the tile
    int meta[LR_NCH];
#pragma unroll
    for (int i = 0; i < LR_NCH; ++i) {
      const int px = pt / cpt + i * pstep;
      if (px < p.ppx) {
        const int pr = px / (p.nseg * 10), rem = px - pr * p.nseg * 10, seg = rem / 10, x = rem - seg * 10;
        const int img = seg / p.ncb, cb = seg - img * p.ncb;
        meta[i] = pr | ((cb * 8 + x) << 8) | (img << 20);
      } else {
        meta[i] = -1;
      }
    }
    const uint32_t a_thr = pl * p.plane + (pt / cpt) * 16;  // + patch buffer + i*pstep*16
    uint32_t tcount = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++tcount) {
      const uint32_t pb = tcount & 1, pph = (tcount >> 1) & 1;
      const int tm = tile % p.n_tiles_m;
      const int64_t m0 = (int64_t)tm * BM;
      const int64_t img0 = m0 / p.hw;
      const int h0 = (int)(m0 - img0 * p.hw) / d.w;
      // fused-prologue constants of this thread's 8 channels as bf16 pairs (the rounding of conv_tc_kernel's table)
      __nv_bfloat162 sc0[4], sh0[4], sc1[4], sh1[4];
      auto load_ss2 = [&](int li, __nv_bfloat162* sc2, __nv_bfloat162* sh2) {
        if (!affine || li >= imgs || img0 + li >= d.n) return;
        const int64_t si = (d.in_bcast ? 0 : (img0 + li) * d.cin) + ci;
        const float4 a0 = *reinterpret_cast<const float4*>(d.in_scale + si), a1 = *reinterpret_cast<const float4*>(d.in_scale + si + 4);
        const float4 b0 = *reinterpret_cast<const float4*>(d.in_shift + si), b1 = *reinterpret_cast<const float4*>(d.in_shift + si + 4);
        sc2[0] = __floats2bfloat162_rn(a0.x, a0.y); sc2[1] = __floats2bfloat162_rn(a0.z, a0.w);
        sc2[2] = __floats2bfloat162_rn(a1.x, a1.y); sc2[3] = __floats2bfloat162_rn(a1.z, a1.w);
        sh2[0] = __floats2bfloat162_rn(b0.x, b0.y); sh2[1] = __floats2bfloat162_rn(b0.z, b0.w);
        sh2[2] = __floats2bfloat162_rn(b1.x, b1.y); sh2[3] = __floats2bfloat162_rn(b1.z, b1.w);
      };
      load_ss2(0, sc0, sh0);
      load_ss2(1, sc1, sh1);
      uint4 v[LR_NCH];
      uint32_t ok = 0;
#pragma unroll
      for (int i = 0; i < LR_NCH; ++i) {
        v[i] = make_uint4(0, 0, 0, 0);
        if (meta[i] < 0) continue;
        const int ih = h0 + (meta[i] & 0xFF) - 1, iw = ((meta[i] >> 8) & 0xFFF) - 1, li = meta[i] >> 20;
        const int64_t n = img0 + li;
        if ((unsigned)ih < (unsigned)d.h && (unsigned)iw < (unsigned)d.w && n < d.n) {
          v[i] = __ldg(reinterpret_cast<const uint4*>(xb + ((n * p.hs + (ih >> sh_)) * (int64_t)p.ws + (iw >> sh_)) * d.x_ld + ci));
          ok |= 1u << i;
        }
      }
      mbar_wait(pempty_bar(pb), pph ^ 1);
      uint8_t* a1 = smem + pb * p.patch_bytes + a_thr;
#pragma unroll
      for (int i = 0; i < LR_NCH; ++i) {
        if (meta[i] < 0) continue;
        uint4 x = v[i];
        if ((ok >> i & 1) && (affine || relu)) {  // zero padding stays zero
          if (affine) {
            auto fma8 = [&](const __nv_bfloat162* sc2, const __nv_bfloat162* sh2) {
              __nv_bfloat162* x2 = reinterpret_cast<__nv_bfloat162*>(&x);
              if (relu) {
#pragma unroll
                for (int j = 0; j < 4; ++j) x2[j] = __hfma2_relu(x2[j], sc2[j], sh2[j]);
              } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) x2[j] = __hfma2(x2[j], sc2[j], sh2[j]);
              }
            };
            if (!d.in_bcast && (meta[i] >> 20)) fma8(sc1, sh1);
            else fma8(sc0, sh0);
          } else {
            float f[8];
            unpack8(x, f);
#pragma unroll
            for (int j = 0; j < 8; ++j) f[j] = fmaxf(f[j], 0.f);
            x = pack8(f);
          }
        }
        *reinterpret_cast<uint4*>(a1 + i * pstep * 16) = x;
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(pfull_bar(pb));
    }
  } else {
    // ===================== epilogue =====================
    const int q = warp & 3;
    epilogue_role(p, tmem_base, q, lane, lr_row_pixel(p, q * 32 + lane));
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_free(tmem_base, p.tmem_cols);
  }
}


}  // namespace tc

// shared eligibility of the tcgen05 kernels; `padded` admits cout < 16 (weights padded to 16 rows,
// direct fp32/bf16 store of the real channels) which only the resident-weights kernel implements
int iea_conv_tc_base_ok(const iea_conv_desc* d, int padded) {
  if (!d->wpack_tc) return 0;
  // 1-channel input (the discriminator stem, fp32 or bf16 image): the resident kernel zero-extends it
  const bool thin_a = padded && d->cin == 1 && !d->in_scale && !d->in_relu && d->in_mode == IEA_IN_DIRECT;
  if (thin_a) {
    if (d->cout % 16 || d->y_dtype != IEA_BF16 || d->y_ld % 8 || !tc::aligned16(d->y) || !tc::aligned16(d->wpack_tc)) return 0;
    if (d->res && (d->res_dtype != IEA_BF16 || d->res_ld % 8 || !tc::aligned16(d->res) || d->res_c % 16)) return 0;
    if (d->acc_c0 >= 0 && d->acc_c0 % 16) return 0;
    return 1;
  }
  if (d->cin % 16) return 0;
  if (padded && d->cout < 16) {
    if (d->cout_tc != 16 || d->res || d->acc_c0 >= 0 || d->stats) return 0;
  } else {
    if (d->cout % 16 || d->y_dtype != IEA_BF16) return 0;
  }
  if (!(d->cin == 16 || d->cin == 32 || d->cin % 64 == 0)) return 0;
  if (d->x_dtype != IEA_BF16) return 0;
  if (d->res && d->res_dtype != IEA_BF16) return 0;
  const bool direct_store = padded && d->cout < 16;  // real channels stored straight from registers
  if (d->x_ld % 8 || (!direct_store && d->y_ld % 8) || (d->res && d->res_ld % 8)) return 0;
  if (!tc::aligned16(d->x) || (!direct_store && !tc::aligned16(d->y)) || !tc::aligned16(d->wpack_tc) || (d->res && !tc::aligned16(d->res)))
    return 0;
  if (d->res && (d->res_c % 16)) return 0;
  if (d->acc_c0 >= 0 && d->acc_c0 % 16) return 0;
  if (d->in_scale && (!tc::aligned16(d->in_scale) || !tc::aligned16(d->in_shift))) return 0;
  return 1;
}
int iea_conv_tc_ok(const iea_conv_desc* d) { return iea_conv_tc_base_ok(d, 0); }

int iea_conv_fprop_tc(const iea_conv_desc* d, cudaStream_t s) {
  tc::Params p;
  p.d = *d;
  p.wtc = (const bf16*)d->wpack_tc;
  p.M = d->n * (int64_t)d->h * d->w;
  p.hs = stored_res(*d, d->h);
  p.ws = stored_res(*d, d->w);
  p.KB = d->cin < 64 ? d->cin : 64;
  p.nkb = d->cin / p.KB;
  p.taps = d->ksize * d->ksize;
  p.BN = d->cout <= 256 ? d->cout : 256;
  IEA_CHECK_ARG(d->cout % p.BN == 0, "iea_conv_fprop(tcgen05): cout=%d is not a multiple of the N tile %d", d->cout, p.BN);
  p.n_tiles_n = d->cout / p.BN;
  p.n_tiles_m = (int)((p.M + tc::BM - 1) / tc::BM);
  const int cpr = p.KB / 8;
  p.lbo_a = 128 * 16 + (cpr == 8 ? 64 : 0);
  p.lbo_b = p.BN * 16;
  p.a_bytes = cpr * p.lbo_a;
  p.b_bytes = cpr * p.lbo_b;
  p.stage_bytes = (p.a_bytes + p.b_bytes + 127) / 128 * 128;
  p.staging_ld = p.BN * 2 + 16;
  const uint32_t staging_bytes = (tc::BM * p.staging_ld + 127) / 128 * 128;
  const uint32_t stat_bytes = 1024 * 2 * 4 > p.BN * 2 * 4 ? 1024 * 2 * 4 : p.BN * 2 * 4;
  const uint32_t tab_bytes = d->in_scale ? (uint32_t)(tc::TAB_IMGS * d->cin * 2 * 2) : 0;
  const uint32_t fixed = staging_bytes + stat_bytes + tab_bytes + 256;
  int stages = (int)((200 * 1024 - fixed) / p.stage_bytes);
  if (stages > 6) stages = 6;
  IEA_CHECK_ARG(stages >= 2, "iea_conv_fprop(tcgen05): tile does not fit shared memory (cin=%d cout=%d)", d->cin, d->cout);
  p.stages = stages;
  p.staging_off = stages * p.stage_bytes;
  p.stat_off = p.staging_off + staging_bytes;
  p.tab_off = p.stat_off + stat_bytes;
  p.bar_off = p.tab_off + tab_bytes;
  p.tfull_off = 8u * 2 * stages;
  const uint32_t smem = p.bar_off + 256;
  const uint32_t cols = tmem_cols_for(2 * p.BN);
  p.tmem_cols = cols;
  const int sms = sm_count();
  const int tiles = p.n_tiles_m * p.n_tiles_n;
  const int occ = (smem <= 100 * 1024 && cols <= 256) ? 2 : 1;
  int grid = tiles < sms * occ ? tiles : sms * occ;
  auto launch = [&](auto kern) -> int {
    IEA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, tc::THREADS, smem, s>>>(p);
    return 0;
  };
  int rc = cpr == 2 ? launch(tc::conv_tc_kernel<2>) : (cpr == 4 ? launch(tc::conv_tc_kernel<4>) : launch(tc::conv_tc_kernel<8>));
  if (rc) return rc;
  return check_launch("iea_conv_fprop(tcgen05)");
}

// Geometry of conv_lr_kernel for a descriptor, or false when the kernel does not take it: 3x3 on a same-resolution
// or nearest-up2 input with 64 or 128 input channels, and 128-pixel tiles that are whole rows of one image or two
// whole 64-pixel images (w a multiple of 8 that divides 128).  Everything else stays on conv_tc_kernel.
static bool lr_geometry(const iea_conv_desc* d, int& nseg, int& ncb, int& ppx) {
  if (!iea_conv_tc_ok(d) || d->ksize != 3 || (d->in_mode != IEA_IN_DIRECT && d->in_mode != IEA_IN_UP2)) return false;
  if ((d->cin != 64 && d->cin != 128) || d->cout > 256 || d->cout % 16) return false;
  if (d->w % 8 || 128 % d->w) return false;
  const int hw = d->h * d->w;
  int imgs;
  if (hw % tc::BM == 0) imgs = 1;
  else if (hw == tc::BM / 2) imgs = 2;
  else return false;
  ncb = d->w / 8;
  nseg = imgs * ncb;
  const int rows = 16 / nseg;  // tile rows
  ppx = (rows + 2) * nseg * 10;
  return ppx * (d->cin / 8) <= tc::LR_NCH * tc::LR_NPT;
}

// shared-memory plan of conv_lr_kernel: two patches, the weight ring, staging, statistics scratch, barriers
static bool lr_plan(const iea_conv_desc* d, tc::Params& p) {
  int nseg, ncb, ppx;
  if (!lr_geometry(d, nseg, ncb, ppx)) return false;
  p.nseg = nseg; p.ncb = ncb; p.ppx = ppx; p.hw = d->h * d->w;
  p.BN = d->cout;
  p.lbo_b = p.BN * 16;
  p.b_bytes = tc::LR_CPR * p.lbo_b;
  p.plane = (ppx * 16 + 127) / 128 * 128 + 16;  // odd multiple of 16 B: the producers' chunk stores spread over banks
  p.patch_bytes = (d->cin / 8) * p.plane;
  p.ring_off = 2 * p.patch_bytes;
  p.staging_ld = p.BN * 2 + 16;
  const uint32_t staging_bytes = (tc::BM * p.staging_ld + 127) / 128 * 128;
  const uint32_t stat_bytes = 1024 * 2 * 4 > p.BN * 2 * 4 ? 1024 * 2 * 4 : p.BN * 2 * 4;
  const uint32_t fixed = p.ring_off + staging_bytes + stat_bytes + 256;
  const uint32_t limit = 225 * 1024;
  if (fixed + 2 * p.b_bytes > limit) return false;
  int stages = (int)((limit - fixed) / p.b_bytes);
  if (stages > 6) stages = 6;
  p.stages = stages;
  p.staging_off = p.ring_off + stages * p.b_bytes;
  p.stat_off = p.staging_off + staging_bytes;
  p.bar_off = p.stat_off + stat_bytes;
  p.tfull_off = 8u * (2 * stages + 4);
  return true;
}

int iea_conv_lowres_ok(const iea_conv_desc* d) {
  tc::Params p;
  return lr_plan(d, p) ? 1 : 0;
}

int iea_conv_fprop_lowres(const iea_conv_desc* d, cudaStream_t s) {
  tc::Params p;
  IEA_CHECK_ARG(lr_plan(d, p), "iea_conv_fprop(tcgen05 low-res): unsupported shape (cin=%d cout=%d %dx%d)", d->cin,
                d->cout, d->h, d->w);
  p.d = *d;
  p.wtc = (const bf16*)d->wpack_tc;
  p.M = d->n * (int64_t)d->h * d->w;
  p.hs = stored_res(*d, d->h);
  p.ws = stored_res(*d, d->w);
  p.KB = 64;
  p.nkb = d->cin / 64;
  p.taps = 9;
  p.n_tiles_n = 1;
  p.n_tiles_m = (int)((p.M + tc::BM - 1) / tc::BM);
  const uint32_t smem = p.bar_off + 256;
  p.tmem_cols = tmem_cols_for(2 * p.BN);
  const int sms = sm_count();
  const int grid = p.n_tiles_m < sms ? p.n_tiles_m : sms;
  IEA_CUDA(cudaFuncSetAttribute(tc::conv_lr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  tc::conv_lr_kernel<<<grid, tc::LR_THREADS, smem, s>>>(p);
  return check_launch("iea_conv_fprop(tcgen05 low-res)");
}
