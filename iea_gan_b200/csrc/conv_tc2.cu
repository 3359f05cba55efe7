// conv_tc2.cu -- tcgen05 / TMEM convolution, "resident weights + staged patch" variant.
//
// The heavy IEA-GAN layers are thin (16..64 channels) at high resolution and therefore HBM bound.
// For them this kernel
//   * TMA-bulk-loads the whole (1/sigma-free) bf16 weight once per persistent CTA and keeps it in smem;
//   * stages every input pixel ONCE per tile: a 1x1 conv stages its 128 pixels, a 3x3 conv stages the
//     18x10 halo patch of a 16x8 output tile and addresses the 9 taps as shifted UMMA descriptors on
//     that single patch (start address + (dh*10+dw)*16 B, SBO = 160 B), so shared-memory write traffic
//     is 1.4x the input instead of 9x and each tile costs one global-load round trip instead of nine;
//   * keeps `depth` patches in flight per CTA with cp.async straight into their final UMMA slots
//     (Little's law: ~44 KB per SM must be in flight to saturate HBM3e) and applies the fused prologue
//     (BN affine + ReLU, nearest-up2 by address mapping) IN PLACE on the landed chunks;
//   * runs the same fused epilogue as conv_tc.cu out of double-buffered TMEM accumulators.
// Index arithmetic is 32-bit with one division set per tile (not per chunk): at 16 channels the kernel
// has ~1400 issue slots per tile at the HBM rate, so 64-bit div/mod per chunk would dominate.
// Layers whose weights do not fit (>= 128-channel 3x3, 512-channel 1x1) use the streaming kernel.
#include "tc_common.cuh"
#include <type_traits>
using namespace iea;

namespace tc2 {
using namespace tc;

constexpr int BM = 128;
constexpr int THREADS = 288;
constexpr int PW = 10, PH = 18;  // 3x3 halo patch of a 16x8 tile

struct Params {
  FastDiv fd_tw, fd_th, fd_w, fd_h, fd_hw, fd_tpe;  // fd_tpe: tiles per event (lean-epilogue statistics slots)
  iea_conv_desc d;
  const bf16* wtc;
  int64_t M;
  int n_tiles, hw, hs, ws, KB, nkb, BN, taps, tiles_w, tiles_h, npix, stages, uniform_n, depth;
  uint32_t plane, stage_bytes, w_bytes, stage_off, staging_off, staging_ld, stat_off, bar_off, tmem_cols;
};

// tile -> (image, top-left output pixel) for 3x3 tiles, first flattened row for 1x1 tiles
struct Origin { int n, h0, w0; int64_t m0; };
template <bool IS3>
__device__ __forceinline__ Origin tile_origin(const Params& p, int tile) {
  Origin o;
  if (IS3) {
    const unsigned t = fdiv((unsigned)tile, p.fd_tw);
    o.w0 = (int)((unsigned)tile - t * (unsigned)p.tiles_w) * 8;
    o.n = (int)fdiv(t, p.fd_th);
    o.h0 = (int)(t - (unsigned)o.n * (unsigned)p.tiles_h) * 16;
    o.m0 = 0;
  } else {
    o.m0 = (int64_t)tile * BM; o.n = 0; o.h0 = 0; o.w0 = 0;
  }
  return o;
}

// (image, tile row, tile column) of a tile, advanced without divisions.  1x1 layers use tiles_h = 1 and
// tiles_w = tiles per image (or "never wraps" when an image is not a whole number of tiles).
struct TilePos { int n, th, tw; };
__device__ __forceinline__ TilePos tile_pos(const Params& p, int tile) {
  TilePos c;
  const unsigned t = fdiv((unsigned)tile, p.fd_tw);
  c.tw = (int)((unsigned)tile - t * (unsigned)p.tiles_w);
  c.n = (int)fdiv(t, p.fd_th);
  c.th = (int)(t - (unsigned)c.n * (unsigned)p.tiles_h);
  return c;
}
__device__ __forceinline__ void tile_next(const Params& p, TilePos& c) {
  if (++c.tw == p.tiles_w) { c.tw = 0; if (++c.th == p.tiles_h) { c.th = 0; ++c.n; } }
}
template <bool IS3>
__device__ __forceinline__ Origin origin_of(const TilePos& c, int tile) {
  Origin o;
  if (IS3) { o.n = c.n; o.h0 = c.th * 16; o.w0 = c.tw * 8; o.m0 = 0; }
  else { o.m0 = (int64_t)tile * BM; o.n = 0; o.h0 = 0; o.w0 = 0; }
  return o;
}

__device__ __forceinline__ uint4 transform(const uint4& raw, const float* sc, const float* sh, bool affine, bool relu) {
  float f[8];
  unpack8(raw, f);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float v = affine ? fmaf(f[j], sc[j], sh[j]) : f[j];
    f[j] = relu ? fmaxf(v, 0.f) : v;
  }
  return pack8(f);
}

__device__ __forceinline__ void load_ss(const iea_conv_desc& d, int64_t n, int ci, float* sc, float* sh) {
  const int64_t si = (d.in_bcast ? 0 : n * d.cin) + ci;
  const float4 a0 = *reinterpret_cast<const float4*>(d.in_scale + si), a1 = *reinterpret_cast<const float4*>(d.in_scale + si + 4);
  const float4 b0 = *reinterpret_cast<const float4*>(d.in_shift + si), b1 = *reinterpret_cast<const float4*>(d.in_shift + si + 4);
  sc[0] = a0.x; sc[1] = a0.y; sc[2] = a0.z; sc[3] = a0.w; sc[4] = a1.x; sc[5] = a1.y; sc[6] = a1.z; sc[7] = a1.w;
  sh[0] = b0.x; sh[1] = b0.y; sh[2] = b0.z; sh[3] = b0.w; sh[4] = b1.x; sh[5] = b1.y; sh[6] = b1.z; sh[7] = b1.w;
}

template <int CPR, bool IS3, int LEANB, int OCC>
__global__ void __launch_bounds__(THREADS, OCC) conv_tc2_kernel(const Params p) {
  constexpr int NPIX = IS3 ? PH * PW : BM;
  constexpr int NL = (NPIX * CPR + 127) / 128;  // chunks per producer thread per patch
  constexpr int TAPS = IS3 ? 9 : 1;
  constexpr int GP = 128 / CPR;                 // patch pixels covered by one pass of the 128 producer threads
  extern __shared__ __align__(128) uint8_t smem[];
  const iea_conv_desc& d = p.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + p.bar_off;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (p.stages + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * p.stages + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * p.stages + 2 + b); };
  const uint32_t w_bar = bar0 + 8u * (2 * p.stages + 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + p.bar_off + 8 * (2 * p.stages + 5));

  if (tid == 0) {
    // one arrival per WARP on full / tempty (128 per-thread arrivals on one mbarrier serialise)
    for (int s = 0; s < p.stages; ++s) { mbar_init(full_bar(s), 4); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 4); }
    mbar_init(w_bar, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // blocked tile partition: each CTA owns a contiguous run of tiles, so consecutive tiles share the image
  // (per-image scale/shift stay in registers), halos hit L1/L2 and the event-boundary flushes are rare
  const int t_base = p.n_tiles / (int)gridDim.x, t_rem = p.n_tiles % (int)gridDim.x;
  const int my_tiles = t_base + ((int)blockIdx.x < t_rem ? 1 : 0);
  const int tile0 = (int)blockIdx.x * t_base + ((int)blockIdx.x < t_rem ? (int)blockIdx.x : t_rem);

  if (warp == 0) {
    // ===================== weight TMA + MMA issuer =====================
    if (lane == 0) {
      mbar_expect_tx(w_bar, p.w_bytes);
      for (uint32_t off = 0; off < p.w_bytes; off += 32768) {
        const uint32_t nb = p.w_bytes - off < 32768 ? p.w_bytes - off : 32768;
        bulk_g2s(sbase + off, (const uint8_t*)p.wtc + off, nb, w_bar);
      }
      mbar_wait(w_bar, 0);
      const uint32_t id = idesc(p.BN, false, false);
      const uint32_t lbo_b = p.BN * 16;
      const uint32_t sbo_a = IS3 ? PW * 16 : 128;
      // descriptors differ only in their 16-byte-unit start address: build the two bases once and add offsets
      const uint64_t da_base = make_desc(sbase + p.stage_off, p.plane, sbo_a);
      const uint64_t db_base = make_desc(sbase, lbo_b, 128);
      const uint32_t stage16 = p.stage_bytes >> 4, plane16 = p.plane >> 4, lbo16 = lbo_b >> 4;
      uint32_t s = 0, ph = 0;
      for (int tcount = 0; tcount < my_tiles; ++tcount) {
        const uint32_t ab = tcount & 1, aph = (tcount >> 1) & 1;
        mbar_wait(tempty_bar(ab), aph ^ 1);
        tc_fence_after();
        const uint32_t tacc = tmem_base + ab * p.BN;
        for (int kb = 0; kb < p.nkb; ++kb) {
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t a16 = s * stage16;
#pragma unroll
          for (int tap = 0; tap < TAPS; ++tap) {
            const uint32_t a_tap = a16 + (IS3 ? (tap / 3) * PW + (tap % 3) : 0);
            const uint32_t b_tap = (uint32_t)(tap * p.nkb + kb) * CPR * lbo16;
#pragma unroll
            for (int j = 0; j < CPR / 2; ++j) {
              const uint64_t da = da_base + (a_tap + 2 * j * plane16);
              const uint64_t db = db_base + (b_tap + 2 * j * lbo16);
              tc_mma(tacc, da, db, id, (kb > 0 || tap > 0 || j > 0) ? 1u : 0u);
            }
          }
          tc_commit(empty_bar(s));
          if (++s == (uint32_t)p.stages) { s = 0; ph ^= 1; }
        }
        tc_commit(tfull_bar(ab));
      }
    }
  } else if (warp <= 4) {
    // ===================== patch producers =====================
    const int pt = tid - 32;
    const int cc = pt % CPR, pp0 = pt / CPR;
    const bool affine = d.in_scale != nullptr;
    const bool relu = d.in_relu != 0;
    const bool pool = d.in_mode == IEA_IN_POOL2;
    const bool thin_a = d.cin < 16;                             // 1-channel image (D stem): zero-extended chunks
    const bool flat = !IS3 && d.in_mode == IEA_IN_DIRECT;      // 1x1 on a same-resolution input: pixel index == row
    const bool slow = pool || (affine && !p.uniform_n) || (!IS3 && !flat);  // rare shapes: per-chunk generic path
    const bool fast = !slow && !thin_a;                         // interior tiles: precomputed chunk offsets
    const int D = p.depth;                                       // patches kept in flight by cp.async
    const int n_items = my_tiles * p.nkb;
    const int sh_ = d.in_mode == IEA_IN_UP2 ? 1 : 0;
    const bf16* xb = (const bf16*)d.x;

    // Tile-independent part of this thread's chunk addresses.  Slot i of a patch is pixel pp = i*GP + pp0,
    // chunk cc; its global element offset from the tile's base pixel and its smem offset never change, so an
    // interior tile costs one 64-bit add + one cp.async per chunk (nearest-up2 is folded into the offsets:
    // tile origins are even, hence (h0 - 1 + pi) >> 1 == h0/2 + ((pi - 1) >> 1)).
    // 2x2-average-pooled input of a 1x1 layer (every DBlock's conv4 / shortcut): a tile of 128 output pixels is whole
    // rows (or a piece of one row) of one image, so the four source pixels of slot i sit at fixed offsets from the
    // tile's first source pixel as well -- all loads of an item are issued before the first use, no index arithmetic.
    const bool pool_fast = pool && !IS3 && !affine && p.uniform_n && (d.w % BM == 0 || BM % d.w == 0);
    int dlt[NL];
#pragma unroll
    for (int i = 0; i < NL; ++i) {
      const int pp = i * GP + pp0;
      if (IS3) {
        const int pi = pp / PW, pj = pp - pi * PW;
        dlt[i] = (((pi - 1) >> sh_) * p.ws + ((pj - 1) >> sh_)) * d.x_ld;
      } else if (pool_fast) {
        const int pr = pp / d.w, pc = pp - pr * d.w;
        dlt[i] = (pr * 2 * p.ws + pc * 2) * d.x_ld;
      } else {
        dlt[i] = pp * d.x_ld;
      }
    }
    const bool last_ok = (NL - 1) * GP + pp0 < NPIX;
    const uint32_t a_thr = sbase + p.stage_off + cc * p.plane + pp0 * 16;  // + stage offset + i*GP*16

    // position of a pipeline item (tile, k block) and of its ring slot
    struct Cur { int tl, kb; uint32_t s, ph; TilePos t; };
    auto cur_next = [&](Cur& c) {
      if (++c.s == (uint32_t)p.stages) { c.s = 0; c.ph ^= 1; }
      if (++c.kb == p.nkb) { c.kb = 0; ++c.tl; tile_next(p, c.t); }
    };
    auto interior_of = [&](const Cur& c) -> bool {
      if (IS3) return c.t.th > 0 && c.t.th < p.tiles_h - 1 && c.t.tw > 0 && c.t.tw < p.tiles_w - 1;
      return (int64_t)(tile0 + c.tl + 1) * BM <= p.M;
    };

    // generic (slow-path) coordinates of patch pixel pp
    auto coords_slow = [&](const Origin& o, int pp, int64_t& nn, int& ih, int& iw) -> bool {
      if (IS3) { nn = o.n; ih = o.h0 - 1 + pp / PW; iw = o.w0 - 1 + pp % PW; }
      else {
        const int64_t m = o.m0 + pp;
        if (m >= p.M) return false;
        iw = (int)(m % d.w); const int64_t t = m / d.w; ih = (int)(t % d.h); nn = t / d.h;
      }
      return (unsigned)ih < (unsigned)d.h && (unsigned)iw < (unsigned)d.w;
    };
    // asynchronous copy of this thread's raw chunks of item `c` straight into their final smem slots
    auto issue = [&](const Cur& c) {
      mbar_wait(empty_bar(c.s), c.ph ^ 1);
      if (slow) return;
      const int ci = c.kb * p.KB + cc * 8;
      const uint32_t a1 = a_thr + c.s * p.stage_bytes;
      if (fast && interior_of(c)) {
        int64_t base;
        if (IS3) base = ((int64_t)(c.t.n * p.hs + ((c.t.th * 16) >> sh_)) * p.ws + ((c.t.tw * 8) >> sh_)) * d.x_ld + ci;
        else base = (int64_t)(tile0 + c.tl) * BM * d.x_ld + ci;
        const bf16* bp = xb + base;
#pragma unroll
        for (int i = 0; i < NL; ++i)
          if (i < NL - 1 || last_ok) cp16(a1 + i * GP * 16, bp + dlt[i]);
        return;
      }
      const Origin o = origin_of<IS3>(c.t, tile0 + c.tl);
#pragma unroll
      for (int i = 0; i < NL; ++i) {
        const int pp = i * GP + pp0;
        if (pp >= NPIX) continue;
        int64_t pix;
        bool in;
        if (IS3) {
          const int pi = pp / PW, ih = o.h0 - 1 + pi, iw = o.w0 - 1 + (pp - pi * PW);
          in = (unsigned)ih < (unsigned)d.h && (unsigned)iw < (unsigned)d.w;
          pix = ((int64_t)o.n * p.hs + (ih >> sh_)) * p.ws + (iw >> sh_);
        } else {
          in = o.m0 + pp < p.M;
          pix = o.m0 + pp;
        }
        if (in && thin_a) {
          const float v = cc == 0 ? ld_act(d.x, d.x_dtype, pix * d.x_ld) : 0.f;
          const uint32_t lo = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v));
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%2,%2};" ::"r"(a1 + i * GP * 16), "r"(lo), "r"(0) : "memory");
        } else if (in) {
          cp16(a1 + i * GP * 16, xb + pix * d.x_ld + ci);
        } else {
          asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(a1 + i * GP * 16), "r"(0) : "memory");
        }
      }
    };

    Cur ci_, ct_;  // issue cursor (runs D-1 items ahead) and transform cursor
    ci_.tl = 0; ci_.kb = 0; ci_.s = 0; ci_.ph = 0; ci_.t = tile_pos(p, tile0);
    ct_ = ci_;
    int issued = 0;
    for (int k = 0; k < D - 1; ++k) {
      if (issued < n_items) { issue(ci_); cur_next(ci_); ++issued; }
      cp_async_commit();
    }
    // fused prologue constants as packed bf16x2: relu(x*scale+shift) is ONE fma.rn.relu.bf16x2 per channel
    // pair (single rounding of the fused result; scale/shift carry bf16 precision like the weights do)
    __nv_bfloat162 sc2[4], sh2[4];
    const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
    int ss_n = -1, ss_ci = -1;
    for (int it = 0; it < n_items; ++it) {
      if (issued < n_items) { issue(ci_); cur_next(ci_); ++issued; }
      cp_async_commit();
      switch (D) {  // wait until item `it` (this thread's part) has landed
        case 2: cp_async_wait<1>(); break;
        case 3: cp_async_wait<2>(); break;
        case 4: cp_async_wait<3>(); break;
        case 6: cp_async_wait<5>(); break;
        default: cp_async_wait<0>(); break;
      }
      const Cur& c = ct_;
      const int ci = c.kb * p.KB + cc * 8;
      uint8_t* a1 = smem + (a_thr - sbase) + c.s * p.stage_bytes;
      if (pool_fast) {
        const unsigned m0u = (unsigned)(tile0 + c.tl) * BM, r0 = m0u / (unsigned)d.w, ow0 = m0u - r0 * (unsigned)d.w;
        const bf16* bp = xb + ((int64_t)r0 * 2 * p.ws + 2 * ow0) * d.x_ld + ci;
        const int64_t o1 = d.x_ld, o2 = (int64_t)p.ws * d.x_ld;
#pragma unroll
        for (int i0 = 0; i0 < NL; i0 += 2) {  // two slots (eight 16-byte loads) in flight per thread
          uint4 r[2][4];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int i = i0 + u;
            if (i < NL && (i < NL - 1 || last_ok)) {
              const bf16* q = bp + dlt[i];
              r[u][0] = __ldg(reinterpret_cast<const uint4*>(q));
              r[u][1] = __ldg(reinterpret_cast<const uint4*>(q + o1));
              r[u][2] = __ldg(reinterpret_cast<const uint4*>(q + o2));
              r[u][3] = __ldg(reinterpret_cast<const uint4*>(q + o2 + o1));
            }
          }
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int i = i0 + u;
            if (i < NL && (i < NL - 1 || last_ok)) {
              float acc[8], f[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                unpack8(r[u][q], f);
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[j] += relu ? fmaxf(f[j], 0.f) : f[j];
              }
#pragma unroll
              for (int j = 0; j < 8; ++j) acc[j] *= 0.25f;
              *reinterpret_cast<uint4*>(a1 + i * GP * 16) = pack8(acc);
            }
          }
        }
      } else if (slow) {
        const Origin o = origin_of<IS3>(c.t, tile0 + c.tl);
#pragma unroll
        for (int i = 0; i < NL; ++i) {
          const int pp = i * GP + pp0;
          if (pp >= NPIX) continue;
          int64_t nn; int ih, iw;
          const bool in = coords_slow(o, pp, nn, ih, iw);
          *reinterpret_cast<uint4*>(a1 + i * GP * 16) = in ? load_chunk(d, p.hs, p.ws, nn, ih, iw, ci) : make_uint4(0, 0, 0, 0);
        }
      } else if (affine || relu) {  // in-place fused prologue on the chunks this thread copied
        const int nn = c.t.n;  // (affine on a 1x1 layer implies uniform_n, so the cursor's image index is exact)
        if (affine && (nn != ss_n || ci != ss_ci)) {
          float sc[8], sh[8];
          load_ss(d, nn, ci, sc, sh);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            sc2[j] = __floats2bfloat162_rn(sc[2 * j], sc[2 * j + 1]);
            sh2[j] = __floats2bfloat162_rn(sh[2 * j], sh[2 * j + 1]);
          }
          ss_n = nn; ss_ci = ci;
        }
        const bool inter = fast && interior_of(c);
        const Origin o = origin_of<IS3>(c.t, tile0 + c.tl);
#pragma unroll
        for (int i = 0; i < NL; ++i) {
          if (i == NL - 1 && !last_ok) continue;
          if (!inter) {  // border tile: padding pixels stay zero
            const int pp = i * GP + pp0;
            bool in;
            if (IS3) {
              const int pi = pp / PW, ih = o.h0 - 1 + pi, iw = o.w0 - 1 + (pp - pi * PW);
              in = (unsigned)ih < (unsigned)d.h && (unsigned)iw < (unsigned)d.w;
            } else {
              in = o.m0 + pp < p.M;
            }
            if (!in) continue;
          }
          uint4* q = reinterpret_cast<uint4*>(a1 + i * GP * 16);
          uint4 v = *q;
          __nv_bfloat162* x2 = reinterpret_cast<__nv_bfloat162*>(&v);
          if (affine && relu) {
#pragma unroll
            for (int j = 0; j < 4; ++j) x2[j] = __hfma2_relu(x2[j], sc2[j], sh2[j]);
          } else if (affine) {
#pragma unroll
            for (int j = 0; j < 4; ++j) x2[j] = __hfma2(x2[j], sc2[j], sh2[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) x2[j] = __hmax2(x2[j], zero2);
          }
          *q = v;
        }
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(full_bar(c.s));
      cur_next(ct_);
    }
    cp_async_wait<0>();
  } else {
    // ===================== epilogue =====================
    const int q = warp & 3, et = q * 32 + lane;  // TMEM lane == tile row
    uint8_t* stg = smem + p.staging_off;
    float* stat = reinterpret_cast<float*>(smem + p.stat_off);
    // per-channel epilogue constants (1/sigma or the grouped-GEMM column scale, bias) staged once per CTA
    float* ep_sc = reinterpret_cast<float*>(smem + p.bar_off + 256);
    float* ep_bs = ep_sc + p.BN;
    for (int c = et; c < p.BN; c += 128) {
      float s_ = 1.f, b_ = 0.f;
      if (c < d.cout) {
        if (d.out_scale) s_ = d.out_scale[d.out_scale_stride ? c : 0];
        if (d.bias) b_ = d.bias[c];
      }
      ep_sc[c] = s_; ep_bs[c] = b_;
    }
    bar_sync_epi();
    const bool need_px = IS3 || (d.res && d.res_mode != IEA_IN_DIRECT);  // (n, oh, ow) only where it is used
    if constexpr (LEANB > 0) {
      // ---- lean epilogue for Cout = 16 / 32 (the HBM-bound thin layers): no smem staging, no CTA
      // barriers.  Each thread owns one output pixel: scale/bias/residual in registers, two or four
      // 16-byte stores straight to its NHWC row, and batch-norm partial sums kept in registers ACROSS
      // tiles; they are folded (warp shuffles + 4-warp smem) only when the CTA moves to the next event,
      // into the slot [event][blockIdx.x][C][2] (bn_finalize then reduces gridDim.x slots per event).
      constexpr int BN_ = 16 * LEANB;
      // (the sums are taken on the fp32 values before the bf16 rounding of the store: the rounding error is
      // zero-mean and 2^-9 relative, far below the batch statistics' own noise; it saves the unpack)
      float2 s1[BN_ / 2], s2[BN_ / 2];
#pragma unroll
      for (int j = 0; j < BN_ / 2; ++j) { s1[j] = make_float2(0.f, 0.f); s2[j] = s1[j]; }
      float* fold = reinterpret_cast<float*>(smem + p.stat_off);  // [4 warps][2*BN_]
      auto flush = [&](int ev) {
#pragma unroll
        for (int j = 0; j < BN_ / 2; ++j) {
          s1[j].x = warp_sum(s1[j].x); s1[j].y = warp_sum(s1[j].y);
          s2[j].x = warp_sum(s2[j].x); s2[j].y = warp_sum(s2[j].y);
        }
        if (lane == 0)
#pragma unroll
          for (int j = 0; j < BN_ / 2; ++j) {
            fold[(q * BN_ + 2 * j) * 2] = s1[j].x; fold[(q * BN_ + 2 * j) * 2 + 1] = s2[j].x;
            fold[(q * BN_ + 2 * j + 1) * 2] = s1[j].y; fold[(q * BN_ + 2 * j + 1) * 2 + 1] = s2[j].y;
          }
        bar_sync_epi();
        for (int c = et; c < BN_ * 2; c += 128) {
          const float a = fold[c] + fold[BN_ * 2 + c] + fold[2 * BN_ * 2 + c] + fold[3 * BN_ * 2 + c];
          d.stats[((int64_t)ev * gridDim.x + blockIdx.x) * d.cout * 2 + c] = a;
        }
        bar_sync_epi();
#pragma unroll
        for (int j = 0; j < BN_ / 2; ++j) { s1[j] = make_float2(0.f, 0.f); s2[j] = s1[j]; }
      };
      const bool has_sb = d.out_scale != nullptr || d.bias != nullptr;
      const bool has_stats = d.stats != nullptr;
      const int tpe = (int)p.fd_tpe.d;                     // tiles per event (statistics are per event)
      int ev = (int)fdiv((unsigned)tile0, p.fd_tpe), ev_pos = tile0 - ev * tpe;
      TilePos tp = tile_pos(p, tile0);
      const int er = et >> 3, ec = et & 7;
      bf16* const yb = (bf16*)d.y;
      for (int tcount = 0; tcount < my_tiles; ++tcount) {
        const uint32_t ab = tcount & 1, aph = (tcount >> 1) & 1;
        int m; int nn = 0, oh = 0, ow = 0; bool valid = true;  // (M < 2^31 is checked on the host)
        if (IS3) {
          nn = tp.n; oh = tp.th * 16 + er; ow = tp.tw * 8 + ec;
          m = (nn * d.h + oh) * d.w + ow;
        } else {
          m = (tile0 + tcount) * BM + et;
          valid = m < p.M;
          if (valid && need_px) {
            const unsigned mm = (unsigned)m, t = fdiv(mm, p.fd_w);
            ow = (int)(mm - t * (unsigned)d.w); nn = (int)fdiv(t, p.fd_h); oh = (int)(t - (unsigned)nn * (unsigned)d.h);
          }
        }
        tile_next(p, tp);
        if (has_stats) {
          if (ev_pos == tpe) { flush(ev); ++ev; ev_pos = 0; }
          ++ev_pos;
        }
        mbar_wait(tfull_bar(ab), aph);
        tc_fence_after();
#pragma unroll
        for (int cb = 0; cb < LEANB; ++cb) {
          float2 v[8];
          {
            float t16[16];
            tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + ab * p.BN + cb * 16, t16);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = make_float2(t16[2 * j], t16[2 * j + 1]);
          }
          const int c0 = cb * 16;
          if (valid) {  // (no early `continue`: all lanes must reconverge before the next aligned tcgen05.ld)
          if (has_sb) {
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const float4 s4 = *reinterpret_cast<const float4*>(ep_sc + c0 + 4 * j4);
              const float4 b4 = *reinterpret_cast<const float4*>(ep_bs + c0 + 4 * j4);
              v[2 * j4] = ffma2(v[2 * j4], make_float2(s4.x, s4.y), make_float2(b4.x, b4.y));
              v[2 * j4 + 1] = ffma2(v[2 * j4 + 1], make_float2(s4.z, s4.w), make_float2(b4.z, b4.w));
            }
          }
          if (d.res && c0 < d.res_c) {
            const bf16* rp = (const bf16*)d.res;
            if (d.res_mode == IEA_IN_POOL2) {
              const float2 quarter = make_float2(0.25f, 0.25f);
              for (int a = 0; a < 2; ++a)
                for (int b = 0; b < 2; ++b) {
                  const bf16* sp = rp + (((int64_t)nn * (2 * d.h) + 2 * oh + a) * (2 * d.w) + 2 * ow + b) * d.res_ld + c0;
                  const uint4 r0 = *reinterpret_cast<const uint4*>(sp), r1 = *reinterpret_cast<const uint4*>(sp + 8);
                  const uint32_t w[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
                  for (int j = 0; j < 8; ++j) v[j] = ffma2(bf2_to_f2(w[j]), quarter, v[j]);
                }
            } else {
              const bf16* sp = d.res_mode == IEA_IN_UP2
                                   ? rp + (((int64_t)nn * (d.h >> 1) + (oh >> 1)) * (d.w >> 1) + (ow >> 1)) * d.res_ld + c0
                                   : rp + (int64_t)m * d.res_ld + c0;
              const uint4 r0 = *reinterpret_cast<const uint4*>(sp), r1 = *reinterpret_cast<const uint4*>(sp + 8);
              const uint32_t w[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] = fadd2(v[j], bf2_to_f2(w[j]));
            }
          }
          uint4* yp = reinterpret_cast<uint4*>(yb + (int64_t)m * d.y_ld + c0);
          if (d.acc_c0 >= 0 && c0 >= d.acc_c0) {
            const uint4 r0 = yp[0], r1 = yp[1];
            const uint32_t w[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fadd2(v[j], bf2_to_f2(w[j]));
          }
          if (d.act == IEA_ACT_RELU) {
#pragma unroll
            for (int j = 0; j < 8; ++j) { v[j].x = fmaxf(v[j].x, 0.f); v[j].y = fmaxf(v[j].y, 0.f); }
          } else if (d.act == IEA_ACT_TANH) {
#pragma unroll
            for (int j = 0; j < 8; ++j) { v[j].x = tanhf(v[j].x); v[j].y = tanhf(v[j].y); }
          }
          uint32_t o[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = pack2(v[j].x, v[j].y);
          yp[0] = make_uint4(o[0], o[1], o[2], o[3]); yp[1] = make_uint4(o[4], o[5], o[6], o[7]);
          if (has_stats) {
#pragma unroll
            for (int j = 0; j < 8; ++j) { s1[cb * 8 + j] = fadd2(s1[cb * 8 + j], v[j]); s2[cb * 8 + j] = ffma2(v[j], v[j], s2[cb * 8 + j]); }
          }
          }  // valid
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(ab));
      }
      if (has_stats && my_tiles > 0) flush(ev);
    } else {
    const int cg = p.BN / 8;
    const bool cg_pow2 = (cg & (cg - 1)) == 0;
    const int cg_sh = 31 - __clz(cg);
    int parts = 1;
    while (parts * 2 * cg <= 128) parts *= 2;
    const int rows_per = BM / parts;
    // ---- fast staged epilogue: the shapes of the generator / discriminator main path (no accumulate, no
    // activation, residual absent / same-resolution / nearest-up2).  Straight-line per flavour (compile-time
    // residual and statistics switches), packed fp32x2 math, copy-out with per-thread constant strides, and
    // the batch-norm partial sums taken from the 16-byte chunks while they are copied out (no second pass).
    const bool fast = d.acc_c0 < 0 && d.act == IEA_ACT_NONE && d.cout >= 16 && cg_pow2 && cg <= 32 &&
                      (!d.res || d.res_mode != IEA_IN_POOL2);
    auto fast_loop = [&](auto res_c_, auto stats_c_) {
      constexpr bool RES = decltype(res_c_)::value, STATS = decltype(stats_c_)::value;
      const int g8 = et & (cg - 1), r0 = et >> cg_sh, step = 128 >> cg_sh;  // copy-out: rows r0, r0+step, ... of chunk g8
      const bf16* const rp_ = (const bf16*)d.res;
      bf16* const yb = (bf16*)d.y;
      const int ncb = p.BN / 16;
      for (int tcount = 0; tcount < my_tiles; ++tcount) {
        const int tile = tile0 + tcount;
        const Origin o = tile_origin<IS3>(p, tile);
        const uint32_t ab = tcount & 1, aph = (tcount >> 1) & 1;
        int64_t m; int nn = 0, oh = 0, ow = 0; bool valid = true;
        if (IS3) {
          nn = o.n; oh = o.h0 + (et >> 3); ow = o.w0 + (et & 7);
          m = ((int64_t)nn * d.h + oh) * d.w + ow;
        } else {
          m = o.m0 + et;
          valid = m < p.M;
          if (RES && valid && need_px) {
            const unsigned mm = (unsigned)m, t = fdiv(mm, p.fd_w);
            ow = (int)(mm - t * (unsigned)d.w); nn = (int)fdiv(t, p.fd_h); oh = (int)(t - (unsigned)nn * (unsigned)d.h);
          }
        }
        const bf16* rrow = nullptr;
        uint4 pr0, pr1;
        if (RES && valid) {
          rrow = d.res_mode == IEA_IN_UP2 ? rp_ + (((int64_t)nn * (d.h >> 1) + (oh >> 1)) * (d.w >> 1) + (ow >> 1)) * d.res_ld
                                          : rp_ + m * d.res_ld;
          if (0 < d.res_c) { pr0 = __ldg(reinterpret_cast<const uint4*>(rrow)); pr1 = __ldg(reinterpret_cast<const uint4*>(rrow + 8)); }
        }
        mbar_wait(tfull_bar(ab), aph);
        tc_fence_after();
        uint8_t* const srow = stg + (size_t)et * p.staging_ld;
        for (int cb = 0; cb < ncb; ++cb) {
          const int c0 = cb * 16;
          uint32_t raw[16];
          tmem_ld16_issue(tmem_base + ((uint32_t)(q * 32) << 16) + ab * p.BN + c0, raw);
          tmem_ld_wait();
          float2 v[8];
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 s4 = *reinterpret_cast<const float4*>(ep_sc + c0 + 4 * j4);
            const float4 b4 = *reinterpret_cast<const float4*>(ep_bs + c0 + 4 * j4);
            v[2 * j4] = ffma2(make_float2(__uint_as_float(raw[4 * j4]), __uint_as_float(raw[4 * j4 + 1])), make_float2(s4.x, s4.y),
                              make_float2(b4.x, b4.y));
            v[2 * j4 + 1] = ffma2(make_float2(__uint_as_float(raw[4 * j4 + 2]), __uint_as_float(raw[4 * j4 + 3])),
                                  make_float2(s4.z, s4.w), make_float2(b4.z, b4.w));
          }
          if (RES) {
            if (valid && c0 < d.res_c) {
              const uint32_t w[8] = {pr0.x, pr0.y, pr0.z, pr0.w, pr1.x, pr1.y, pr1.z, pr1.w};
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] = fadd2(v[j], bf2_to_f2(w[j]));
            }
            if (valid && cb + 1 < ncb && c0 + 16 < d.res_c) {  // next block's residual: in flight during pack + staging store
              pr0 = __ldg(reinterpret_cast<const uint4*>(rrow + c0 + 16));
              pr1 = __ldg(reinterpret_cast<const uint4*>(rrow + c0 + 24));
            }
          }
          uint4 o0, o1;
          if (valid) {
            o0 = make_uint4(pack2(v[0].x, v[0].y), pack2(v[1].x, v[1].y), pack2(v[2].x, v[2].y), pack2(v[3].x, v[3].y));
            o1 = make_uint4(pack2(v[4].x, v[4].y), pack2(v[5].x, v[5].y), pack2(v[6].x, v[6].y), pack2(v[7].x, v[7].y));
          } else {
            o0 = make_uint4(0, 0, 0, 0); o1 = o0;  // rows beyond the last pixel: zeros (they enter the statistics)
          }
          *reinterpret_cast<uint4*>(srow + cb * 32) = o0;
          *reinterpret_cast<uint4*>(srow + cb * 32 + 16) = o1;
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(ab));  // accumulator drained: the MMA warp may start the next tile
        bar_sync_epi();
        // coalesced copy-out: this thread moves chunk g8 of rows r0, r0 + step, ... (cg rows) -- rows of the tile
        // are contiguous pixel runs in NHWC -- and sums its chunks for the batch-norm statistics on the way
        float2 s1[4], s2[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { s1[j] = make_float2(0.f, 0.f); s2[j] = s1[j]; }
        {
          const uint8_t* sp = stg + (size_t)r0 * p.staging_ld + g8 * 16;
          const size_t sstep = (size_t)step * p.staging_ld;
          bf16* yp; int64_t ystep; int rows_left = cg;
          if (IS3) {  // row r -> pixel (r >> 3, r & 7) of the 16x8 tile; step is 4, 8 or 16 rows
            yp = yb + (((int64_t)o.n * d.h + o.h0 + (r0 >> 3)) * d.w + o.w0 + (r0 & 7)) * d.y_ld + g8 * 8;
            ystep = (int64_t)(step >> 3) * d.w * d.y_ld;  // (step >= 8 on this path: Cout <= 128 for 3x3)
          } else {
            yp = yb + (o.m0 + r0) * d.y_ld + g8 * 8;
            ystep = (int64_t)step * d.y_ld;
            const int64_t left = p.M - o.m0 - r0;  // rows of this tile that exist, from r0 on
            if (left < (int64_t)(cg - 1) * step + 1) rows_left = left <= 0 ? 0 : (int)((left - 1) / step) + 1;
          }
          int it = 0;
          for (; it + 4 <= rows_left; it += 4) {  // four rows per pass: the shared-memory reads are issued back to back
            uint4 v4[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v4[u] = *reinterpret_cast<const uint4*>(sp + u * sstep);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              *reinterpret_cast<uint4*>(yp + u * ystep) = v4[u];
              if (STATS) {
                const uint32_t w[4] = {v4[u].x, v4[u].y, v4[u].z, v4[u].w};
#pragma unroll
                for (int j = 0; j < 4; ++j) { const float2 f = bf2_to_f2(w[j]); s1[j] = fadd2(s1[j], f); s2[j] = ffma2(f, f, s2[j]); }
              }
            }
            sp += 4 * sstep; yp += 4 * ystep;
          }
          for (; it < rows_left; ++it) {
            const uint4 v4 = *reinterpret_cast<const uint4*>(sp);
            *reinterpret_cast<uint4*>(yp) = v4;
            if (STATS) {
              const uint32_t w[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) { const float2 f = bf2_to_f2(w[j]); s1[j] = fadd2(s1[j], f); s2[j] = ffma2(f, f, s2[j]); }
            }
            sp += sstep; yp += ystep;
          }
        }
        if (STATS) {  // [part = r0][BN][2] partials, then a fixed-order fold over the parts
          // (16-byte stores: the scalar version was a 16-way bank conflict -- the r0 rows of partials are 2 BN floats apart)
          float4* st4 = reinterpret_cast<float4*>(stat + (r0 * p.BN + g8 * 8) * 2);
#pragma unroll
          for (int j = 0; j < 4; ++j) st4[j] = make_float4(s1[j].x, s2[j].x, s1[j].y, s2[j].y);
          bar_sync_epi();
          for (int c = et; c < p.BN * 2; c += 128) {
            float a = 0.f;
            for (int part = 0; part < step; ++part) a += stat[part * p.BN * 2 + c];
            d.stats[(int64_t)tile * d.cout * 2 + c] = a;
          }
        }
        bar_sync_epi();  // staging / stat scratch are reused by the next tile
      }
    };
    if (fast) {
      if (d.res && d.stats) fast_loop(std::true_type{}, std::true_type{});
      else if (d.res) fast_loop(std::true_type{}, std::false_type{});
      else if (d.stats) fast_loop(std::false_type{}, std::true_type{});
      else fast_loop(std::false_type{}, std::false_type{});
    } else
    for (int tcount = 0; tcount < my_tiles; ++tcount) {
      const int tile = tile0 + tcount;
      const Origin o = tile_origin<IS3>(p, tile);
      const uint32_t ab = tcount & 1, aph = (tcount >> 1) & 1;
      // this thread's output pixel
      int64_t m; int nn = 0, oh = 0, ow = 0; bool valid = true;
      if (IS3) {
        nn = o.n; oh = o.h0 + (et >> 3); ow = o.w0 + (et & 7);
        m = ((int64_t)nn * d.h + oh) * d.w + ow;
      } else {
        m = o.m0 + et;
        valid = m < p.M;
        if (valid && need_px) {
          const unsigned mm = (unsigned)m, t = fdiv(mm, p.fd_w);
          ow = (int)(mm - t * (unsigned)d.w); nn = (int)fdiv(t, p.fd_h); oh = (int)(t - (unsigned)nn * (unsigned)d.h);
        }
      }
      // residual / accumulate operands of a 16-channel block are fetched one block AHEAD of their use (the
      // first block before the wait for the accumulator): their global-load latency is hidden behind the
      // TMEM load, the packing and the staging store of the previous block instead of being paid per block
      const bf16* const rp_ = (const bf16*)d.res;
      const bool pf_res = valid && d.res != nullptr;
      const bool pf_acc = valid && d.acc_c0 >= 0;
      const int res_q = d.res_mode == IEA_IN_POOL2 ? 4 : 1;  // source pixels per output pixel
      int64_t res_px[4];
      if (pf_res) {
        if (d.res_mode == IEA_IN_POOL2) {
#pragma unroll
          for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) res_px[a * 2 + b] = (((int64_t)nn * (2 * d.h) + 2 * oh + a) * (2 * d.w) + 2 * ow + b) * d.res_ld;
        } else {
          res_px[0] = d.res_mode == IEA_IN_UP2 ? (((int64_t)nn * (d.h >> 1) + (oh >> 1)) * (d.w >> 1) + (ow >> 1)) * d.res_ld
                                               : m * d.res_ld;
        }
      }
      uint4 pr[4][2], pa[2];
      auto prefetch = [&](int cb) {
        const int c0 = cb * 16;
        if (pf_res && c0 < d.res_c) {
#pragma unroll
          for (int s4 = 0; s4 < 4; ++s4)
            if (s4 < res_q) {
              pr[s4][0] = __ldg(reinterpret_cast<const uint4*>(rp_ + res_px[s4] + c0));
              pr[s4][1] = __ldg(reinterpret_cast<const uint4*>(rp_ + res_px[s4] + c0 + 8));
            }
        }
        if (pf_acc && c0 >= d.acc_c0) {
          const uint4* yp = reinterpret_cast<const uint4*>((const bf16*)d.y + m * d.y_ld + c0);
          pa[0] = yp[0]; pa[1] = yp[1];
        }
      };
      prefetch(0);
      mbar_wait(tfull_bar(ab), aph);
      tc_fence_after();
      const int ncb = p.BN / 16;
      for (int cb = 0; cb < ncb; ++cb) {
        float v[16];
        tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + ab * p.BN + cb * 16, v);
        const int c0 = cb * 16;
        if (valid) {
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 s4 = *reinterpret_cast<const float4*>(ep_sc + c0 + 4 * j4);
            const float4 b4 = *reinterpret_cast<const float4*>(ep_bs + c0 + 4 * j4);
            v[4 * j4] = fmaf(v[4 * j4], s4.x, b4.x); v[4 * j4 + 1] = fmaf(v[4 * j4 + 1], s4.y, b4.y);
            v[4 * j4 + 2] = fmaf(v[4 * j4 + 2], s4.z, b4.z); v[4 * j4 + 3] = fmaf(v[4 * j4 + 3], s4.w, b4.w);
          }
          if (d.res && c0 < d.res_c) {
            float f[16];
            if (d.res_mode == IEA_IN_POOL2) {
#pragma unroll
              for (int j = 0; j < 16; ++j) f[j] = 0.f;
#pragma unroll
              for (int s4 = 0; s4 < 4; ++s4) {
                float t8[16];
                unpack8(pr[s4][0], t8);
                unpack8(pr[s4][1], t8 + 8);
#pragma unroll
                for (int j = 0; j < 16; ++j) f[j] += 0.25f * t8[j];
              }
            } else {
              unpack8(pr[0][0], f);
              unpack8(pr[0][1], f + 8);
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] += f[j];
          }
          if (d.acc_c0 >= 0 && c0 >= d.acc_c0) {
            float f[16];
            unpack8(pa[0], f);
            unpack8(pa[1], f + 8);
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] += f[j];
          }
          if (cb + 1 < ncb) prefetch(cb + 1);  // (the operands of this block are consumed: refill for the next one)
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
        if (d.cout < 16) {  // padded output channels (32->1 convs): store the real ones straight from registers
          if (valid)
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (j < d.cout) st_act(d.y, d.y_dtype, m * d.y_ld + j, v[j]);
          continue;
        }
        uint4* dst = reinterpret_cast<uint4*>(stg + (size_t)et * p.staging_ld + cb * 32);
        dst[0] = pack8(v);
        dst[1] = pack8(v + 8);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(ab));  // accumulator drained: the MMA warp may start the next tile
      if (d.cout < 16) continue;
      bar_sync_epi();
      // coalesced 16-byte stores: rows of the tile are contiguous runs of pixels in NHWC
      bf16* yb = (bf16*)d.y;
      for (int i = et; i < BM * cg; i += 128) {
        const int row = cg_pow2 ? (i >> cg_sh) : i / cg, g8 = i - row * cg;
        int64_t m2;
        if (IS3) m2 = ((int64_t)o.n * d.h + o.h0 + (row >> 3)) * d.w + o.w0 + (row & 7);
        else { m2 = o.m0 + row; if (m2 >= p.M) continue; }
        *reinterpret_cast<uint4*>(yb + m2 * d.y_ld + g8 * 8) =
            *reinterpret_cast<const uint4*>(stg + (size_t)row * p.staging_ld + g8 * 16);
      }
      if (d.stats) {  // per-tile column (sum, sum^2) of the rounded outputs; fixed order -> deterministic
        for (int w0_ = et; w0_ < cg * parts; w0_ += 128) {
          const int part = cg_pow2 ? (w0_ >> cg_sh) : w0_ / cg, g8 = w0_ - part * cg;
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
          d.stats[(int64_t)tile * d.cout * 2 + c] = a;
        }
      }
      bar_sync_epi();  // staging / stat scratch are reused by the next tile
    }
    }  // staged epilogue
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_free(tmem_base, p.tmem_cols);
  }
}

}  // namespace tc2

int iea_conv_tc_base_ok(const iea_conv_desc* d, int padded);

int iea_conv_tc2_ok(const iea_conv_desc* d) {
  if (!iea_conv_tc_base_ok(d, 1)) return 0;
  if (d->cout > 256) return 0;
  const int64_t wbytes = (int64_t)(d->cout < 16 ? 16 : d->cout) * (d->cin < 16 ? 16 : d->cin) * d->ksize * d->ksize * 2;
  if (wbytes > 96 * 1024) return 0;
  if (d->ksize == 3 && (d->h % 16 || d->w % 8 || d->cin > 64)) return 0;
  if (d->n * (int64_t)d->h * d->w >= (1ll << 31)) return 0;  // 32-bit pixel arithmetic inside the kernel
  return 1;
}

// tiles of one event (40 images) in this kernel's tiling; 0 when a tile could straddle two events
static int tc2_tiles_per_event(const iea_conv_desc* d) {
  const int64_t px = 40ll * d->h * d->w;
  if (d->n % 40 || px % 128) return 0;
  return (int)(px / 128);
}
// 0: staged epilogue; 1 / 2: lean register epilogue for Cout = 16 / 32
int iea_conv_tc2_lean(const iea_conv_desc* d) {
  if (d->cout != 16 && d->cout != 32) return 0;
  if (d->y_dtype != IEA_BF16) return 0;
  if (d->stats && !tc2_tiles_per_event(d)) return 0;
  return d->cout / 16;
}
static int tc2_grid(const iea_conv_desc* d);
// number of statistics slots per event the chosen kernel writes (engine sizes / zero-fills the buffer)
int iea_conv_tc2_stats_slots(const iea_conv_desc* d) {
  if (iea_conv_tc2_lean(d)) return tc2_grid(d);
  return tc2_tiles_per_event(d);
}

// launch geometry shared by the launcher and the statistics-slot query; occ_out: CTAs per SM it is sized for
static int tc2_prepare(const iea_conv_desc* d, tc2::Params& p, int& grid, uint32_t& smem_out, int& cpr_out, bool& is3_out,
                       int& occ_out) {
  p.d = *d;
  p.wtc = (const bf16*)d->wpack_tc;
  p.M = d->n * (int64_t)d->h * d->w;
  p.hw = d->h * d->w;
  p.fd_w = tc::make_fastdiv(d->w); p.fd_h = tc::make_fastdiv(d->h); p.fd_hw = tc::make_fastdiv(p.hw);
  p.hs = stored_res(*d, d->h);
  p.ws = stored_res(*d, d->w);
  const int cin_eff = d->cin < 16 ? 16 : d->cin;  // 1-channel stem: K padded to one 16-wide MMA step
  p.KB = cin_eff < 64 ? cin_eff : 64;
  p.nkb = cin_eff / p.KB;
  p.taps = d->ksize * d->ksize;
  p.BN = d->cout < 16 ? 16 : d->cout;
  const bool is3 = d->ksize == 3;
  p.uniform_n = is3 ? 1 : (((int64_t)d->h * d->w) % 128 == 0 ? 1 : 0);
  p.n_tiles = (int)(is3 ? d->n * (int64_t)(d->w / 8) * (d->h / 16) : (p.M + 127) / 128);
  // 1x1: a "tile row" is one image when images are whole tiles; otherwise the column counter never wraps
  p.tiles_w = is3 ? d->w / 8 : (p.uniform_n ? p.hw / 128 : p.n_tiles + 1);
  p.tiles_h = is3 ? d->h / 16 : 1;
  p.fd_tw = tc::make_fastdiv(p.tiles_w); p.fd_th = tc::make_fastdiv(p.tiles_h);
  p.npix = is3 ? tc2::PH * tc2::PW : 128;
  const int cpr = p.KB / 8;
  // planes (8 channels each) are skewed by 128 / CPR bytes: the CPR chunks of a pixel are copied / transformed by
  // consecutive threads and must fall into different banks (ncu, 32 -> 64 1x1 @128^2 with unskewed planes: 122 M
  // shared-memory bank conflicts, L1 data pipe 76 % busy)
  p.plane = (p.npix * 16 + 127) / 128 * 128 + 128 / cpr;
  p.stage_bytes = (cpr * p.plane + 127) / 128 * 128;
  p.w_bytes = (uint32_t)((int64_t)p.BN * cin_eff * p.taps * 2);
  p.stage_off = (p.w_bytes + 127) / 128 * 128;
  p.staging_ld = p.BN * 2 + 16;
  const uint32_t staging_bytes = (128 * p.staging_ld + 127) / 128 * 128;
  const uint32_t stat_bytes = 8192;
  const uint32_t fixed = p.stage_off + staging_bytes + stat_bytes + 256 + 2 * p.BN * 4;
  // ring depth: enough patches in flight to cover HBM latency (~44 KB per SM), bounded by shared memory
  int stages = 8;
  while (stages > 3 && fixed + stages * p.stage_bytes > 110 * 1024) --stages;  // prefer 2 CTAs / SM
  if (stages < 5) {
    stages = 8;
    while (stages > 3 && fixed + stages * p.stage_bytes > 200 * 1024) --stages;
  }
  IEA_CHECK_ARG(fixed + stages * p.stage_bytes <= 220 * 1024, "iea_conv_fprop(tcgen05 resident): tile does not fit "
                "shared memory (cin=%d cout=%d k=%d)", d->cin, d->cout, d->ksize);
  p.depth = stages >= 8 ? 6 : (stages >= 6 ? 4 : (stages >= 5 ? 3 : 2));
  p.stages = stages;
  p.staging_off = p.stage_off + stages * p.stage_bytes;
  p.stat_off = p.staging_off + staging_bytes;
  p.bar_off = p.stat_off + stat_bytes;
  const uint32_t smem = p.bar_off + 256 + 2 * p.BN * 4;
  const uint32_t cols = tmem_cols_for(2 * p.BN);
  p.tmem_cols = cols;
  const int occ = (cpr == 2 && smem <= 72 * 1024 && cols <= 128) ? 3 : ((cpr <= 4 && smem <= 110 * 1024 && cols <= 256) ? 2 : 1);
  const int cap = sm_count() * occ;
  grid = p.n_tiles < cap ? p.n_tiles : cap;
  smem_out = smem; cpr_out = cpr; is3_out = is3; occ_out = occ;
  return 0;
}
static int tc2_grid(const iea_conv_desc* d) {
  tc2::Params p; int grid = 0, cpr, occ; uint32_t smem; bool is3;
  if (tc2_prepare(d, p, grid, smem, cpr, is3, occ)) return 0;
  return grid;
}

int iea_conv_fprop_tc2(const iea_conv_desc* d, cudaStream_t s) {
  tc2::Params p; int grid = 0, cpr, occ; uint32_t smem; bool is3;
  int rc0 = tc2_prepare(d, p, grid, smem, cpr, is3, occ);
  if (rc0) return rc0;
  auto launch = [&](auto kern) -> int {
    IEA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, tc2::THREADS, smem, s>>>(p);
    return 0;
  };
  const int leanb = iea_conv_tc2_lean(d);
  const int tpe_ = tc2_tiles_per_event(d);
  p.fd_tpe = tc::make_fastdiv(tpe_ > 0 ? tpe_ : 1);
  int rc = -2;
  const int ko = cpr == 2 ? (occ == 3 ? 3 : 2) : (cpr == 4 ? 2 : 1);  // launch-bound variant of the kernel
#define TC2_LAUNCH(C_, I_, L_, O_) \
  if (cpr == C_ && is3 == I_ && leanb == L_ && ko == O_) rc = launch(tc2::conv_tc2_kernel<C_, I_, L_, O_>);
  TC2_LAUNCH(2, true, 0, 3) TC2_LAUNCH(2, true, 1, 3) TC2_LAUNCH(2, true, 2, 3)
  TC2_LAUNCH(2, true, 0, 2) TC2_LAUNCH(2, true, 1, 2) TC2_LAUNCH(2, true, 2, 2)
  TC2_LAUNCH(4, true, 0, 2) TC2_LAUNCH(4, true, 1, 2) TC2_LAUNCH(4, true, 2, 2)
  TC2_LAUNCH(8, true, 0, 1) TC2_LAUNCH(8, true, 1, 1) TC2_LAUNCH(8, true, 2, 1)
  TC2_LAUNCH(2, false, 0, 3) TC2_LAUNCH(2, false, 1, 3) TC2_LAUNCH(2, false, 2, 3)
  TC2_LAUNCH(2, false, 0, 2) TC2_LAUNCH(2, false, 1, 2) TC2_LAUNCH(2, false, 2, 2)
  TC2_LAUNCH(4, false, 0, 2) TC2_LAUNCH(4, false, 1, 2) TC2_LAUNCH(4, false, 2, 2)
  TC2_LAUNCH(8, false, 0, 1) TC2_LAUNCH(8, false, 1, 1) TC2_LAUNCH(8, false, 2, 1)
#undef TC2_LAUNCH
  if (rc) return rc;
  return check_launch("iea_conv_fprop(tcgen05 resident)");
}
