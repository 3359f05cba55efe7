// conv_thin.cu -- tcgen05 / TMEM convolution for the thin, high-resolution IEA-GAN layers
// (Cin 16..64, Cout 16/32; 3x3 and 1x1), the layers that carry most of the HBM traffic of G and D
// (SURVEY.md Appendix A: 16->16 / 32->32 3x3 at 128^2..256^2, 64->16 / 16->32 1x1, layers.py:169-206).
//
// These layers move 64..192 bytes per output pixel, so at the HBM rate an SM has only a few hundred
// issue slots per 128-pixel UMMA tile.  conv_tc2.cu spends ~2000; this kernel is built to spend ~400:
//   * MACRO TILES: one pipeline item is MT side-by-side 16x8 tiles (3x3: one 18 x (8*MT+2) halo patch,
//     1x1: MT*128 consecutive pixels).  Barrier hand-offs, tile bookkeeping and halo re-reads are paid
//     once per macro tile; the MT accumulators live side by side in TMEM.
//   * every producer thread owns the same chunk slots of every patch, so the global / shared offsets of
//     its 16-byte cp.async copies are computed once per kernel (nearest-up2 folded into the offsets);
//     a macro tile costs one 64-bit add + one cp.async per chunk, and one LDS / 4 HFMA2 / STS for the
//     fused BN-affine + ReLU prologue in place.  Border patches use per-slot side masks (no coordinates).
//   * the MMA issuer is warp-uniform code around elect.sync, so descriptors stay in uniform registers;
//   * the epilogue keeps one pixel per thread: packed fp32x2 math (FFMA2 / FADD2), 16-byte stores to
//     its own NHWC row, batch-norm partial sums in registers across the whole run of tiles.
// Shapes outside this envelope (pooled inputs, Cout > 32, Cin > 64, the 1-channel stem) stay on
// conv_tc2.cu / conv_tc.cu.
#include "tc_common.cuh"
#include <stdlib.h>
#include <string.h>
using namespace iea;

namespace thin {
using namespace tc;

constexpr int BM = 128;
constexpr int RES_RING = 4;    // residual sub-tiles in flight per epilogue group (TMA-store flavour)
constexpr int THREADS = 512;  // warps 0-7: two producer groups (they also issue their tiles' MMAs), warps 8-15: two epilogue groups
                              // (one CTA per SM; the groups take alternate macro tiles so every hand-off latency is
                              // covered by the other group's tile)


// compile-time geometry shared by the kernel and the launcher
template <int CPR, bool IS3, int MT, bool TMA = false>
struct Geo {
  static constexpr int PW = 8 * MT + 2;                       // patch pitch in pixels (3x3)
  static constexpr int NPIX = IS3 ? 18 * PW : BM * MT;        // staged pixels per macro tile
  static constexpr int NCH = NPIX * CPR;                      // 16-byte chunks per macro tile
  static constexpr int NS = (NCH + 127) / 128;                // chunk slots per producer thread
  // planes (8 channels each) are skewed by 128/CPR bytes so that the CPR chunks of a pixel, written by
  // consecutive threads, fall into different shared-memory banks
  // (TMA box loads write whole planes: no skew there, the transform threads walk a plane pixel by pixel instead)
  static constexpr uint32_t PLANE = (NPIX * 16 + 127) / 128 * 128 + (TMA ? 0 : 128 / CPR);
  static constexpr uint32_t BOX_BYTES = NPIX * 16;            // bytes one plane receives per macro tile
  static constexpr uint32_t STAGE = (CPR * PLANE + 127) / 128 * 128;
};

struct Params {
  iea_conv_desc d;
  const bf16* wtc;
  FastDiv fd_mtw, fd_mth, fd_tpe, fd_w, fd_h;
  int M;                  // output pixels (< 2^31)
  int n_macro;            // macro tiles
  int mtw, mth;           // macro tiles per image row / per image column (1x1: per image / 1)
  int hs, ws;             // stored input resolution
  int stages;
  uint32_t w_bytes, stage_off, misc_off, bar_off, tmem_cols, tst_off, res_off, res_slot;  // tst_off: output staging of the TMA-store epilogue; res_off / res_slot: its residual ring
  int depth;              // (behind the uint32_t block, which stays 8-byte aligned: pairs of it load as one 64-bit constant)
};

struct Pos { int n, th, tw; };
__device__ __forceinline__ Pos pos_of(const Params& p, int g) {
  Pos c;
  const unsigned t = fdiv((unsigned)g, p.fd_mtw);
  c.tw = (int)((unsigned)g - t * (unsigned)p.mtw);
  c.n = (int)fdiv(t, p.fd_mth);
  c.th = (int)(t - (unsigned)c.n * (unsigned)p.mth);
  return c;
}
__device__ __forceinline__ void pos_next(const Params& p, Pos& c) {
  if (++c.tw == p.mtw) { c.tw = 0; if (++c.th == p.mth) { c.th = 0; ++c.n; } }
}

// EPI: epilogue flavour, fixed at compile time so that each is straight-line code (run-time flags made the
// compiler shuffle the 16 accumulator registers at every merge point: ~200 instructions per 128x16 block
// where ~70 do the work).  1: scale/bias + residual read, same-resolution or nearest-up2 [+ statistics]
// (the GBlock conv4 layers);  2: everything (pooled residual, accumulate, activation, padded 1-channel store);
// 3: flavour 1 with the output leaving through TMA: one pixel per thread means a warp's 16-byte stores hit 16 different
// 128-byte lines per instruction, and those wavefronts (not HBM, not the math) kept the L1 data pipe of the dominant
// launch 55 % busy.  The group writes its 128 x 64 B (or 32 B) sub-tile into a swizzled shared-memory image
// (conflict-free) and one thread hands it to the TMA unit, which writes whole lines.
// TMA: same-resolution inputs are fetched by TMA box loads, one per 8-channel plane ({8 ch, patch width, 18 rows}
// for 3x3 with out-of-image pixels zero-filled by the unit; {8 ch, 128 pixels} for 1x1): one elected thread per
// producer group issues them, the other producer threads only run the fused prologue (nothing at all for the
// prologue-free data-gradient convolutions).  Nearest-up2 inputs keep the cp.async slot tables.
template <int CPR, bool IS3, int NB, int MT, int EPI, bool TMA>
__global__ void __launch_bounds__(THREADS, 1) conv_thin_kernel(const __grid_constant__ Params p,
                                                               const __grid_constant__ CUtensorMap tmap,
                                                               const __grid_constant__ CUtensorMap tmap_y,
                                                               const __grid_constant__ CUtensorMap tmap_r) {
  using G = Geo<CPR, IS3, MT, TMA>;
  constexpr int PW = G::PW, NCH = G::NCH, NS = G::NS;
  constexpr uint32_t PLANE = G::PLANE, STAGE = G::STAGE;
  constexpr int TAPS = IS3 ? 9 : 1;
  constexpr int BN = 16 * NB;
  constexpr int NI = IS3 ? MT : 1;  // MMA-issuing warps per group: 3x3 -> producer warp w issues the 9*CPR/2 MMAs of sub-tile w
  extern __shared__ __align__(128) uint8_t smem[];
  const iea_conv_desc& d = p.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + p.bar_off;
  const int S = p.stages;  // even: ring slot s belongs to group s & 1
  // barriers: full[S] | empty[S] | tfull[4] | tempty[4] | w
  const uint32_t full0 = bar0, empty0 = bar0 + 8u * S, tfull0 = bar0 + 16u * S, tempty0 = tfull0 + 32, w_bar = tfull0 + 64;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + p.bar_off + 16 * S + 72);
  const uint32_t land0 = bar0 + 16u * S + 80;  // land[S]: TMA completion (transaction bytes) per ring slot

  if (tid == 0) {
    // one arrival per WARP on full / tempty (per-thread arrivals would wake every parked waiter 128 times)
    for (int s = 0; s < S; ++s) { mbar_init(full0 + 8 * s, 4); mbar_init(empty0 + 8 * s, NI); }
    for (int b = 0; b < 4; ++b) { mbar_init(tfull0 + 8 * b, NI); mbar_init(tempty0 + 8 * b, 4); }
    mbar_init(w_bar, 1);
    if (TMA) for (int s = 0; s < S; ++s) mbar_init(land0 + 8 * s, 1);
    if (EPI == 3) for (int i = 0; i < 2 * RES_RING; ++i) mbar_init(bar0 + 24u * S + 80 + 8 * i, 1);  // residual ring: TMA landing
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // blocked partition: each CTA owns a contiguous run of macro tiles; inside the CTA the two producer
  // groups and the two epilogue groups take alternate macro tiles (group = item & 1)
  const int g_base = p.n_macro / (int)gridDim.x, g_rem = p.n_macro % (int)gridDim.x;
  const int my_n = g_base + ((int)blockIdx.x < g_rem ? 1 : 0);
  const int g0 = (int)blockIdx.x * g_base + ((int)blockIdx.x < g_rem ? (int)blockIdx.x : g_rem);

  if (warp < 8) {
    // ===================== patch producers: two groups of 4 warps, alternate macro tiles =====================
    const int grp = warp >> 2, pw = warp & 3;
    const int pt = tid & 127;
    // this thread's 8-channel plane (fixed: 128 % CPR == 0).  cp.async: the CPR chunks of a pixel go to consecutive
    // threads (coalesced global reads); TMA: a thread walks one plane, consecutive threads = consecutive pixels
    constexpr int TPP = 128 / CPR;                             // threads per plane (TMA mapping)
    const int cc = TMA ? pt / TPP : pt % CPR;
    const bool affine = d.in_scale != nullptr;
    const bool relu = d.in_relu != 0;
    const int sh_ = d.in_mode == IEA_IN_UP2 ? 1 : 0;
    const int D = p.depth;
    // slot table: chunk q = pt + 128*i of the macro patch -> (global element offset, smem byte offset) and,
    // for 3x3, which patch sides it lies on (bit i of top/bot/left/right).  Tile independent.
    int goff[NS];
    uint32_t soff[NS];
    uint32_t m_top = 0, m_bot = 0, m_left = 0, m_right = 0, m_valid = 0;
#pragma unroll
    for (int i = 0; i < NS; ++i) {
      const int q = pt + 128 * i;
      const int pp = TMA ? (pt % TPP) + TPP * i : q / CPR;  // patch pixel
      if (TMA ? pp < G::NPIX : q < NCH) m_valid |= 1u << i;
      if (IS3) {
        const int pi = pp / PW, pj = pp - pi * PW;
        goff[i] = (((pi - 1) >> sh_) * p.ws + ((pj - 1) >> sh_)) * d.x_ld + cc * 8;
        if (pi == 0) m_top |= 1u << i;
        if (pi == 17) m_bot |= 1u << i;
        if (pj == 0) m_left |= 1u << i;
        if (pj == PW - 1) m_right |= 1u << i;
      } else {
        goff[i] = pp * d.x_ld + cc * 8;
      }
      soff[i] = cc * PLANE + pp * 16;
    }
    const bf16* xb = (const bf16*)d.x;
    const uint32_t st0 = sbase + p.stage_off;

    struct Cur { uint32_t s, ph; int t; Pos c; };
    auto cur_next = [&](Cur& c) {  // two macro tiles on: the other group owns the one in between
      c.s += 2;
      if (c.s >= (uint32_t)S) { c.s -= S; c.ph ^= 1; }
      c.t += 2;
      pos_next(p, c.c);
      pos_next(p, c.c);
    };
    // slots of this macro tile that are conv padding (3x3) or beyond the last pixel (1x1 tail)
    auto pad_mask = [&](const Cur& c) -> uint32_t {
      if (IS3) {
        return (c.c.th == 0 ? m_top : 0u) | (c.c.th == p.mth - 1 ? m_bot : 0u) | (c.c.tw == 0 ? m_left : 0u) |
               (c.c.tw == p.mtw - 1 ? m_right : 0u);
      }
      const int left = p.M - (g0 + c.t) * (BM * MT);  // pixels left from the macro tile's first one
      if (left >= BM * MT) return 0u;
      uint32_t m = 0;
#pragma unroll
      for (int i = 0; i < NS; ++i)
        if ((TMA ? (pt % TPP) + TPP * i : (pt + 128 * i) / CPR) >= left) m |= 1u << i;
      return m;
    };
    auto issue = [&](const Cur& c) {
      mbar_wait(empty0 + 8 * c.s, c.ph ^ 1);
      int64_t base;
      if (IS3) base = ((int64_t)(c.c.n * p.hs + ((c.c.th * 16) >> sh_)) * p.ws + ((c.c.tw * (8 * MT)) >> sh_)) * d.x_ld;
      else base = (int64_t)(g0 + c.t) * (BM * MT) * d.x_ld;
      const bf16* bp = xb + base;
      const uint32_t a = st0 + c.s * STAGE;
      const uint32_t pad = pad_mask(c);
      if (pad == 0) {
#pragma unroll
        for (int i = 0; i < NS; ++i)
          if (i < NS - 1 || (m_valid >> i & 1)) cp16(a + soff[i], bp + goff[i]);
      } else {
#pragma unroll
        for (int i = 0; i < NS; ++i) {
          if (!(m_valid >> i & 1)) continue;
          if (pad >> i & 1) asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(a + soff[i]), "r"(0) : "memory");
          else cp16(a + soff[i], bp + goff[i]);
        }
      }
    };

    auto issue_tma = [&](const Cur& c) {  // one thread per group
      mbar_wait(empty0 + 8 * c.s, c.ph ^ 1);
      const uint32_t a = st0 + c.s * STAGE, bar = land0 + 8 * c.s;
      mbar_expect_tx(bar, CPR * G::BOX_BYTES);
      const uint64_t tm = reinterpret_cast<uint64_t>(&tmap);
      if (IS3) {
        const int w0 = c.c.tw * (8 * MT) - 1, h0 = c.c.th * 16 - 1;
#pragma unroll
        for (int k = 0; k < CPR; ++k)
          asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
                       ::"r"(a + k * PLANE), "l"(tm), "r"(k * 8), "r"(w0), "r"(h0), "r"(c.c.n), "r"(bar) : "memory");
      } else {
        const int m0 = (g0 + c.t) * (BM * MT);
#pragma unroll
        for (int k = 0; k < CPR; ++k)
#pragma unroll
          for (int j = 0; j < MT; ++j)
            asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                         ::"r"(a + k * PLANE + j * (BM * 16)), "l"(tm), "r"(k * 8), "r"(m0 + j * BM), "r"(bar) : "memory");
      }
    };

    // ---- MMA issue: warp pw < NI of the group issues sub-tile pw (3x3) / the whole item (1x1) of the group's
    // items; warp-uniform code around elect.sync keeps the descriptors in uniform registers
    if (tid == 0) {
      mbar_expect_tx(w_bar, p.w_bytes);
      for (uint32_t off = 0; off < p.w_bytes; off += 32768) {
        const uint32_t nb = p.w_bytes - off < 32768 ? p.w_bytes - off : 32768;
        bulk_g2s(sbase + off, (const uint8_t*)p.wtc + off, nb, w_bar);
      }
    }
    constexpr uint32_t ID = idesc(BN, false, false);
    constexpr uint32_t LBO_B = BN * 16;
    const uint64_t da_base = make_desc(sbase + p.stage_off, PLANE, IS3 ? PW * 16 : 128);
    const uint64_t db_base = make_desc(sbase, LBO_B, 128);
    auto mma_item = [&](int t, uint32_t s, uint32_t ph) {  // macro tile t of this CTA sits in ring slot s
      const uint32_t ab = t & 3, aph = (t >> 2) & 1;
      if (t < 2) mbar_wait(w_bar, 0);  // weights landed
      mbar_wait(tempty0 + 8 * ab, aph ^ 1);
      mbar_wait(full0 + 8 * s, ph);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a16 = s * (STAGE >> 4);
        const uint32_t tacc = tmem_base + ab * (MT * BN);
        for (int sb = IS3 ? pw : 0; sb < MT; sb += NI) {
#pragma unroll
          for (int tap = 0; tap < TAPS; ++tap) {
#pragma unroll
            for (int j = 0; j < CPR / 2; ++j) {
              const uint32_t a_off = a16 + (IS3 ? sb * 8 + (tap / 3) * PW + (tap % 3) : sb * BM) + 2 * j * (PLANE >> 4);
              const uint32_t b_off = (uint32_t)((tap * CPR + 2 * j) * (LBO_B >> 4));
              tc_mma(tacc + sb * BN, da_base + a_off, db_base + b_off, ID, (tap > 0 || j > 0) ? 1u : 0u);
            }
          }
        }
        tc_commit(empty0 + 8 * s);
        tc_commit(tfull0 + 8 * ab);
      }
      __syncwarp();
    };

    Cur ci, ct;
    ci.s = grp; ci.ph = 0; ci.t = grp; ci.c = pos_of(p, g0 + grp);
    ct = ci;
    for (int k = 0; k < D - 1; ++k) {
      if (ci.t < my_n) {
        if (!TMA) issue(ci);
        else if (pt == 0) issue_tma(ci);
        cur_next(ci);
      }
      if (!TMA) cp_async_commit();
    }
    __nv_bfloat162 sc2[4], sh2[4];
    const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
    int ss_n = -1;
    for (; ct.t < my_n;) {
      if (ci.t < my_n) {
        if (!TMA) issue(ci);
        else if (pt == 0) issue_tma(ci);
        cur_next(ci);
      }
      if (!TMA) {
        cp_async_commit();
        if (D == 2) cp_async_wait<1>();
        else if (D == 3) cp_async_wait<2>();
        else cp_async_wait<3>();
      } else {
        mbar_wait(land0 + 8 * ct.s, ct.ph);  // the boxes of this macro tile have landed
      }
      if (affine || relu) {  // fused prologue, in place on the chunks this thread copied
        if (affine && ct.c.n != ss_n) {
          ss_n = ct.c.n;
          const int64_t si = (d.in_bcast ? 0 : (int64_t)ss_n * d.cin) + cc * 8;
          const float4 a0 = *reinterpret_cast<const float4*>(d.in_scale + si), a1 = *reinterpret_cast<const float4*>(d.in_scale + si + 4);
          const float4 b0 = *reinterpret_cast<const float4*>(d.in_shift + si), b1 = *reinterpret_cast<const float4*>(d.in_shift + si + 4);
          sc2[0] = __floats2bfloat162_rn(a0.x, a0.y); sc2[1] = __floats2bfloat162_rn(a0.z, a0.w);
          sc2[2] = __floats2bfloat162_rn(a1.x, a1.y); sc2[3] = __floats2bfloat162_rn(a1.z, a1.w);
          sh2[0] = __floats2bfloat162_rn(b0.x, b0.y); sh2[1] = __floats2bfloat162_rn(b0.z, b0.w);
          sh2[2] = __floats2bfloat162_rn(b1.x, b1.y); sh2[3] = __floats2bfloat162_rn(b1.z, b1.w);
        }
        const uint32_t live = m_valid & ~pad_mask(ct);  // padding stays zero: relu(shift) != 0
        uint8_t* a = smem + p.stage_off + ct.s * STAGE;
        // loads first, then the math, then the stores (predicated, no branches), at most 6 chunks at a time
        constexpr int XB = 6;
#pragma unroll
        for (int i0 = 0; i0 < NS; i0 += XB) {
          uint4 v[XB];
#pragma unroll
          for (int i = 0; i < XB; ++i)
            if (i0 + i < NS && (live >> (i0 + i) & 1)) v[i] = *reinterpret_cast<const uint4*>(a + soff[i0 + i]);
#pragma unroll
          for (int i = 0; i < XB; ++i) {
            if (i0 + i >= NS) continue;
            __nv_bfloat162* x2 = reinterpret_cast<__nv_bfloat162*>(&v[i]);
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
          }
#pragma unroll
          for (int i = 0; i < XB; ++i)
            if (i0 + i < NS && (live >> (i0 + i) & 1)) *reinterpret_cast<uint4*>(a + soff[i0 + i]) = v[i];
        }
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(full0 + 8 * ct.s);
      if (pw < NI) mma_item(ct.t, ct.s, ct.ph);
      cur_next(ct);
    }
    if (!TMA) cp_async_wait<0>();
  } else {
    // ===================== epilogue: two groups of 4 warps, alternate macro tiles; one pixel per thread =====================
    const int grp = (warp - 8) >> 2;
    const int q = warp & 3, et = q * 32 + lane;  // TMEM lane == tile row (a warp may only touch lanes 32*(warp%4)..+31)
    float* ep_sc = reinterpret_cast<float*>(smem + p.misc_off);
    float* ep_bs = ep_sc + BN;
    float* fold = ep_bs + BN + grp * (4 * 2 * BN);  // [4 warps][2*BN] per group
    if (grp == 0)
      for (int c = et; c < BN; c += 128) {
        ep_sc[c] = d.out_scale ? d.out_scale[d.out_scale_stride && c < d.cout ? c : 0] : 1.f;
        ep_bs[c] = d.bias && c < d.cout ? d.bias[c] : 0.f;
      }
    asm volatile("bar.sync 3, 256;" ::: "memory");  // both epilogue groups: constants staged
    auto bar_grp = [&]() {
      if (grp == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
      else asm volatile("bar.sync 2, 128;" ::: "memory");
    };
    const bool has_stats = d.stats != nullptr;
    constexpr bool TST = EPI == 3;  // TMA store of the output sub-tiles
    const bool has_res = (EPI == 1 || EPI == 3) ? true : (EPI == 2 ? d.res != nullptr : false);
    const bool res_pool = EPI == 2 && d.res_mode == IEA_IN_POOL2;
    const bool res_up2 = EPI >= 1 && d.res_mode == IEA_IN_UP2;
    const bool need_px = IS3 || (has_res && d.res_mode != IEA_IN_DIRECT);
    // per-channel scale / bias in registers (smem loads in the tile loop would queue behind the MMA operand reads)
    constexpr int NREG = NB == 1 ? BN / 2 : 1;  // (32 output channels: the registers go to the statistics instead)
    float2 esc[NREG], ebs[NREG];
    if (NB == 1) {
#pragma unroll
      for (int j = 0; j < NREG; ++j) { esc[j] = make_float2(ep_sc[2 * j], ep_sc[2 * j + 1]); ebs[j] = make_float2(ep_bs[2 * j], ep_bs[2 * j + 1]); }
    }
    // (sums are taken on the fp32 values before the bf16 rounding of the store: the rounding error is
    // zero-mean and 2^-9 relative, far below the noise of the batch statistics themselves)
    float2 s1[BN / 2], s2[BN / 2];
#pragma unroll
    for (int j = 0; j < BN / 2; ++j) { s1[j] = make_float2(0.f, 0.f); s2[j] = s1[j]; }
    auto flush = [&](int ev) {
#pragma unroll
      for (int j = 0; j < BN / 2; ++j) {
        s1[j].x = warp_sum(s1[j].x); s1[j].y = warp_sum(s1[j].y);
        s2[j].x = warp_sum(s2[j].x); s2[j].y = warp_sum(s2[j].y);
      }
      if (lane == 0)
#pragma unroll
        for (int j = 0; j < BN / 2; ++j) {
          fold[(q * BN + 2 * j) * 2] = s1[j].x; fold[(q * BN + 2 * j) * 2 + 1] = s2[j].x;
          fold[(q * BN + 2 * j + 1) * 2] = s1[j].y; fold[(q * BN + 2 * j + 1) * 2 + 1] = s2[j].y;
        }
      bar_grp();
      for (int c = et; c < BN * 2; c += 128) {
        const float a = fold[c] + fold[BN * 2 + c] + fold[2 * BN * 2 + c] + fold[3 * BN * 2 + c];
        d.stats[((int64_t)ev * (2 * gridDim.x) + 2 * blockIdx.x + grp) * BN * 2 + c] = a;
      }
      bar_grp();
#pragma unroll
      for (int j = 0; j < BN / 2; ++j) { s1[j] = make_float2(0.f, 0.f); s2[j] = s1[j]; }
    };
    const int tpe = (int)p.fd_tpe.d;  // macro tiles per event (batch statistics are per event)
    int ev = (int)fdiv((unsigned)(g0 + grp), p.fd_tpe), ev_pos = g0 + grp - ev * tpe;
    Pos c = pos_of(p, g0 + grp);
    const int er = et >> 3, ec = et & 7;
    bf16* const yb = (bf16*)d.y;
    const bf16* const rp = (const bf16*)d.res;
    bool any = false;
    const int64_t ystep = (int64_t)(IS3 ? 8 : BM) * d.y_ld;
    // TMA-store staging: two sub-tile images per group, rows of RB bytes, 16-byte chunks XOR-swizzled like the
    // tensor map (64B / 32B swizzle) so that the row-per-thread writes are conflict-free
    constexpr uint32_t RB = BN * 2, ST_IMG = BM * RB;
    const uint32_t st_al = ((sbase + p.tst_off + 1023u) & ~1023u) - sbase;  // (the swizzle works on absolute addresses)
    const uint32_t st_u32 = sbase + st_al + grp * (2 * ST_IMG);
    uint8_t* const st_ptr = smem + st_al + grp * (2 * ST_IMG);
    const int st_sw = NB == 2 ? ((et >> 1) & 3) : ((et >> 2) & 1);
    int st_cnt = 0;
    // ... and the residual ENTERS through TMA as well: the rows of a sub-tile (64 source pixels for a nearest-up2
    // residual, 128 otherwise; <= 64 bytes each, swizzled) land in a ring slot RES_RING sub-tiles ahead of their use.
    // The per-pixel 16-byte loads they replace were an exposed L2 round trip per 16-channel block: 45 % of the
    // epilogue's time on the dominant launch.
    const uint32_t rr_al = ((sbase + p.res_off + 1023u) & ~1023u) - sbase;
    const uint32_t rr_u32 = sbase + rr_al + grp * (RES_RING * p.res_slot), rr_bar = bar0 + 24u * S + 80 + grp * (RES_RING * 8);
    const uint8_t* const rr_ptr = smem + rr_al + grp * (RES_RING * p.res_slot);
    const int rr_sub = my_n > grp ? ((my_n - grp + 1) >> 1) * MT : 0;  // sub-tiles of this group
    const uint32_t rr_rb = (uint32_t)d.res_c * 2;                       // bytes per residual row (64 or 32)
    const int rr_row = res_up2 ? (et >> 1) : et;
    const uint8_t* const rr_mine = rr_ptr + rr_row * rr_rb;
    const int rr_sw = rr_rb == 64 ? ((rr_row >> 1) & 3) : ((rr_row >> 2) & 1);
    auto rr_issue = [&](int sidx) {  // one thread: TMA load of the residual rows of this group's sub-tile `sidx`
      if (sidx >= rr_sub) return;
      const int msub = (g0 + grp + 2 * (sidx / MT)) * (BM * MT) + (sidx % MT) * BM;
      int src0 = msub;
      if (res_up2) {
        const unsigned r1 = fdiv((unsigned)msub, p.fd_w);
        src0 = (int)(r1 >> 1) * (d.w >> 1) + (int)(((unsigned)msub - r1 * (unsigned)d.w) >> 1);
      }
      const uint32_t bar = rr_bar + 8 * (sidx % RES_RING);
      mbar_expect_tx(bar, (res_up2 ? 64u : 128u) * rr_rb);
      asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                   ::"r"(rr_u32 + (sidx % RES_RING) * p.res_slot), "l"(reinterpret_cast<uint64_t>(&tmap_r)), "r"(0), "r"(src0), "r"(bar) : "memory");
    };
    if (TST && et == 0)
      for (int i = 0; i < RES_RING; ++i) rr_issue(i);
    for (int t = grp; t < my_n; t += 2) {
      const uint32_t ab = t & 3, aph = (t >> 2) & 1;
      int m0, oh = 0, ow0 = 0;
      const int nn = c.n;
      if (IS3) {
        oh = c.th * 16 + er; ow0 = c.tw * (8 * MT) + ec;
        m0 = (nn * d.h + oh) * d.w + ow0;
      } else {
        m0 = (g0 + t) * (BM * MT) + et;
      }
      bf16* const ytile = yb + (int64_t)m0 * d.y_ld;  // sub-tile sb of this thread's pixel: + sb * ystep
      pos_next(p, c);
      pos_next(p, c);
      if (has_stats) {
        if (ev_pos >= tpe) { if (any) flush(ev); ++ev; ev_pos -= tpe; }
        ev_pos += 2;
        any = true;
      }
      // residual rows are pulled into L1 one batch of sub-tiles ahead of their use (prefetch: no registers),
      // so the loads below do not stall every sub-tile on an L2 / HBM round trip
      const bool res_l1 = !TST && !IS3 && has_res && !res_pool;
      auto res_prefetch = [&](int m) {
        if (m >= p.M) return;
        const bf16* sp;
        if (res_up2) {
          const unsigned t1 = fdiv((unsigned)m, p.fd_w);
          const int row = (int)((unsigned)m - t1 * (unsigned)d.w), rn = (int)fdiv(t1, p.fd_h), roh = (int)(t1 - (unsigned)rn * (unsigned)d.h);
          sp = rp + (((int64_t)rn * (d.h >> 1) + (roh >> 1)) * (d.w >> 1) + (row >> 1)) * d.res_ld;
        } else {
          sp = rp + (int64_t)m * d.res_ld;
        }
        asm volatile("prefetch.global.L1 [%0];" ::"l"(sp));
      };
      if (res_l1 && t == grp) {
#pragma unroll
        for (int u = 0; u < (NB == 1 ? (MT < 2 ? MT : 2) : 1); ++u) res_prefetch(m0 + u * BM);
      }
      mbar_wait(tfull0 + 8 * ab, aph);
      tc_fence_after();
      // TMEM -> registers in batches of GRP sub-tiles: the loads are issued back to back and waited for
      // once, and the sub-tiles of a batch are independent instruction streams
      constexpr int GRP = NB == 1 ? (MT < 2 ? MT : 2) : 1;
#pragma unroll
      for (int sg = 0; sg < MT; sg += GRP) {
        uint32_t raw[GRP][NB][16];
#pragma unroll
        for (int u = 0; u < GRP; ++u)
#pragma unroll
          for (int cb = 0; cb < NB; ++cb)
            tmem_ld16_issue(tmem_base + ((uint32_t)(q * 32) << 16) + ab * (MT * BN) + (sg + u) * BN + cb * 16, raw[u][cb]);
        if (res_l1) {  // next batch of this macro tile, or the first batch of this group's next macro tile
#pragma unroll
          for (int u = 0; u < GRP; ++u) {
            if (sg + GRP < MT) res_prefetch(m0 + (sg + GRP + u) * BM);
            else if (t + 2 < my_n) res_prefetch(m0 + 2 * (BM * MT) + u * BM);
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int u = 0; u < GRP; ++u) {
          const int sb = sg + u;
          const int m = m0 + (IS3 ? sb * 8 : sb * BM);
          const bool valid = IS3 || m < p.M;
          if (!valid) continue;  // (the aligned tcgen05.ld of this batch are already done)
          int rn = nn, roh = oh, row = ow0 + sb * 8;
          if (!TST && !IS3 && need_px) {
            const unsigned t1 = fdiv((unsigned)m, p.fd_w);
            row = (int)((unsigned)m - t1 * (unsigned)d.w); rn = (int)fdiv(t1, p.fd_h); roh = (int)(t1 - (unsigned)rn * (unsigned)d.h);
          }
          const bf16* rsp = nullptr;  // this pixel's residual row (same resolution / nearest-up2 source pixel)
          if (!TST && has_res && !res_pool)
            rsp = res_up2 ? rp + (((int64_t)rn * (d.h >> 1) + (roh >> 1)) * (d.w >> 1) + (row >> 1)) * d.res_ld
                          : rp + (int64_t)m * d.res_ld;
          const uint8_t* rr_slot = rr_mine + (st_cnt % RES_RING) * p.res_slot;
          if (TST) mbar_wait(rr_bar + 8 * (st_cnt % RES_RING), (st_cnt / RES_RING) & 1);  // this sub-tile's residual rows
#pragma unroll
          for (int cb = 0; cb < NB; ++cb) {
            const int c0 = cb * 16;
            // scale / bias applied unconditionally (identity constants when the layer has none): no branch, and
            // the accumulator words feed the FFMA2 directly
            float2 v[8];
            if (NB == 1) {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                v[j] = ffma2(make_float2(__uint_as_float(raw[u][cb][2 * j]), __uint_as_float(raw[u][cb][2 * j + 1])), esc[j % NREG], ebs[j % NREG]);
            } else {
#pragma unroll
              for (int j4 = 0; j4 < 4; ++j4) {
                const float4 s4 = *reinterpret_cast<const float4*>(ep_sc + c0 + 4 * j4);
                const float4 b4 = *reinterpret_cast<const float4*>(ep_bs + c0 + 4 * j4);
                v[2 * j4] = ffma2(make_float2(__uint_as_float(raw[u][cb][4 * j4]), __uint_as_float(raw[u][cb][4 * j4 + 1])),
                                  make_float2(s4.x, s4.y), make_float2(b4.x, b4.y));
                v[2 * j4 + 1] = ffma2(make_float2(__uint_as_float(raw[u][cb][4 * j4 + 2]), __uint_as_float(raw[u][cb][4 * j4 + 3])),
                                      make_float2(s4.z, s4.w), make_float2(b4.z, b4.w));
              }
            }
            if (has_res && c0 < d.res_c) {
              if (res_pool) {
                const float2 quarter = make_float2(0.25f, 0.25f);
                for (int a = 0; a < 2; ++a)
                  for (int b = 0; b < 2; ++b) {
                    const bf16* sp = rp + (((int64_t)rn * (2 * d.h) + 2 * roh + a) * (2 * d.w) + 2 * row + b) * d.res_ld + c0;
                    const uint4 r0 = *reinterpret_cast<const uint4*>(sp), r1 = *reinterpret_cast<const uint4*>(sp + 8);
                    const uint32_t w[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = ffma2(bf2_to_f2(w[j]), quarter, v[j]);
                  }
              } else {
                uint4 r0, r1;
                if (TST) {
                  r0 = *reinterpret_cast<const uint4*>(rr_slot + (((2 * cb) ^ rr_sw) << 4));
                  r1 = *reinterpret_cast<const uint4*>(rr_slot + (((2 * cb + 1) ^ rr_sw) << 4));
                } else {
                  r0 = *reinterpret_cast<const uint4*>(rsp + c0);
                  r1 = *reinterpret_cast<const uint4*>(rsp + c0 + 8);
                }
                const uint32_t w[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = fadd2(v[j], bf2_to_f2(w[j]));
              }
            }
            if (EPI == 2 && NB == 1 && d.cout == 1) {  // padded output conv: one real channel
              float v0 = v[0].x;
              if (d.act == IEA_ACT_RELU) v0 = fmaxf(v0, 0.f);
              else if (d.act == IEA_ACT_TANH) v0 = tanhf(v0);
              st_act(d.y, d.y_dtype, (int64_t)m * d.y_ld, v0);
              continue;
            }
            uint4* yp = reinterpret_cast<uint4*>(ytile + sb * ystep + c0);
            if (EPI == 2 && d.acc_c0 >= 0 && c0 >= d.acc_c0) {
              const uint4 r0 = yp[0], r1 = yp[1];
              const uint32_t w[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] = fadd2(v[j], bf2_to_f2(w[j]));
            }
            if (EPI == 2 && d.act == IEA_ACT_RELU) {
#pragma unroll
              for (int j = 0; j < 8; ++j) { v[j].x = fmaxf(v[j].x, 0.f); v[j].y = fmaxf(v[j].y, 0.f); }
            } else if (EPI == 2 && d.act == IEA_ACT_TANH) {
#pragma unroll
              for (int j = 0; j < 8; ++j) { v[j].x = tanhf(v[j].x); v[j].y = tanhf(v[j].y); }
            }
            uint32_t o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = pack2(v[j].x, v[j].y);
            if (TST) {
              uint8_t* row_ = st_ptr + (st_cnt & 1) * ST_IMG + et * RB;
              *reinterpret_cast<uint4*>(row_ + (((2 * cb) ^ st_sw) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
              *reinterpret_cast<uint4*>(row_ + (((2 * cb + 1) ^ st_sw) << 4)) = make_uint4(o[4], o[5], o[6], o[7]);
            } else {
              yp[0] = make_uint4(o[0], o[1], o[2], o[3]);
              yp[1] = make_uint4(o[4], o[5], o[6], o[7]);
            }
            if (has_stats) {
#pragma unroll
              for (int j = 0; j < 8; ++j) { s1[cb * 8 + j] = fadd2(s1[cb * 8 + j], v[j]); s2[cb * 8 + j] = ffma2(v[j], v[j], s2[cb * 8 + j]); }
            }
          }
          if (TST) {  // the sub-tile image is complete: hand it to the TMA unit (host guarantees whole sub-tiles)
            fence_async_smem();
            // the OTHER image, which the group writes next, must have been read by its store (issued a sub-tile ago)
            if (et == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            bar_grp();
            if (et == 0) {
              asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                           ::"l"(reinterpret_cast<uint64_t>(&tmap_y)), "r"(0), "r"(m - et), "r"(st_u32 + (st_cnt & 1) * ST_IMG) : "memory");
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
              rr_issue(st_cnt + RES_RING);  // (every thread of the group is past its reads of this slot: bar_grp above)
            }
            ++st_cnt;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty0 + 8 * ab);
    }
    if (has_stats && any) flush(ev);
    if (TST && et == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_free(tmem_base, p.tmem_cols);
  }
}

}  // namespace thin

int iea_conv_tc_base_ok(const iea_conv_desc* d, int padded);

// macro-tile width (in 16x8 / 128-pixel tiles) the kernel uses for this layer; 0: layer not eligible
static int thin_mt(const iea_conv_desc* d) {
  if (!iea_conv_tc_base_ok(d, d->cout == 1 ? 1 : 0)) return 0;
  // (cout 1 with a 16-row weight pack: the generator's 32->1 output conv; its real channel is stored
  //  straight from the accumulator registers in the storage type of y)
  const bool pad1 = d->cout == 1 && d->cout_tc == 16;
  if (d->cout != 16 && d->cout != 32 && !pad1) return 0;
  if (d->cin != 16 && d->cin != 32 && d->cin != 64) return 0;
  if ((!pad1 && d->y_dtype != IEA_BF16) || d->cin < 16) return 0;
  if (pad1 && (d->stats || d->res || d->acc_c0 >= 0)) return 0;
  if (d->in_mode == IEA_IN_POOL2) return 0;
  const int64_t M = d->n * (int64_t)d->h * d->w;
  if (M >= (1ll << 31) || M * (int64_t)(d->x_ld > d->y_ld ? d->x_ld : d->y_ld) >= (1ll << 40)) return 0;
  // (the 32 -> 1 output conv takes 4-wide macro tiles as well: 6 % less halo, half the hand-offs per pixel)
  const int want = d->cin == 16 ? 4 : (d->cin == 32 ? (d->cout == 1 && d->ksize == 3 ? 4 : 2) : 1);
  if (d->ksize == 3) {
    if (d->h % 16 || d->w % 8) return 0;
    int mt = want;
    while (mt > 1 && d->w % (8 * mt)) mt >>= 1;
    return mt;
  }
  if (d->in_mode != IEA_IN_DIRECT) return 0;
  int mt = want;
  const int64_t hw = (int64_t)d->h * d->w;
  // images must be whole macro tiles when a per-image prologue or per-event statistics are fused
  while (mt > 1 && hw % (128 * mt)) mt >>= 1;
  if ((d->in_scale || d->stats) && hw % (128 * mt)) return 0;
  return mt;
}
int iea_conv_thin_ok(const iea_conv_desc* d) {
  if (!thin_mt(d)) return 0;
  if (d->stats && (d->n % 40)) return 0;
  return 1;
}

// ---- TMA tensor maps of the input, output and residual
// output of a 1x1 layer as {cout channels, pixels}: boxes {cout, 128}, chunks swizzled inside the 64 / 32-byte rows
static bool thin_tensor_map_y(const iea_conv_desc* d, CUtensorMap* tm) {
  tc::encode_tiled_fn enc = tc::tma_encoder();
  if (!enc || d->y_dtype != IEA_BF16 || d->y_ld % 8 || ((uintptr_t)d->y & 15) || (d->cout != 16 && d->cout != 32)) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)d->cout, (cuuint64_t)(d->n * (int64_t)d->h * d->w)};
  const cuuint64_t strides[1] = {(cuuint64_t)d->y_ld * 2};
  const cuuint32_t box[2] = {(cuuint32_t)d->cout, 128}, es[2] = {1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, d->y, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
             d->cout == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// residual of a 1x1 layer as {res_c channels, source pixels}: boxes {res_c, 64} (nearest-up2: the 64 source pixels under
// 128 consecutive output pixels of one row) or {res_c, 128} (same resolution)
static bool thin_tensor_map_r(const iea_conv_desc* d, CUtensorMap* tm) {
  tc::encode_tiled_fn enc = tc::tma_encoder();
  const bool up2 = d->res_mode == IEA_IN_UP2;
  if (!enc || !d->res || d->res_dtype != IEA_BF16 || d->res_ld % 8 || ((uintptr_t)d->res & 15)) return false;
  if ((d->res_c != 16 && d->res_c != 32) || d->res_c > d->cout) return false;
  if (up2 && (d->w % 128 || d->h % 2)) return false;
  if (!up2 && d->res_mode != IEA_IN_DIRECT) return false;
  const int64_t px = up2 ? d->n * (int64_t)(d->h / 2) * (d->w / 2) : d->n * (int64_t)d->h * d->w;
  const cuuint64_t dims[2] = {(cuuint64_t)d->res_c, (cuuint64_t)px};
  const cuuint64_t strides[1] = {(cuuint64_t)d->res_ld * 2};
  const cuuint32_t box[2] = {(cuuint32_t)d->res_c, up2 ? 64u : 128u}, es[2] = {1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(d->res), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
             d->res_c == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// {8 channels, patch width, 18 rows, 1 image} boxes of the NHWC input for 3x3; {8 channels, 128 pixels} for 1x1
static bool thin_tensor_map(const iea_conv_desc* d, bool is3, int mt, CUtensorMap* tm) {
  tc::encode_tiled_fn enc = tc::tma_encoder();
  if (!enc) return false;
  const cuuint64_t ld = (cuuint64_t)d->x_ld * 2;
  if (is3) {
    const cuuint64_t dims[4] = {(cuuint64_t)d->cin, (cuuint64_t)d->w, (cuuint64_t)d->h, (cuuint64_t)d->n};
    const cuuint64_t strides[3] = {ld, ld * d->w, ld * d->w * d->h};
    const cuuint32_t box[4] = {8, (cuuint32_t)(8 * mt + 2), 18, 1}, es[4] = {1, 1, 1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(d->x), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  }
  const cuuint64_t dims[2] = {(cuuint64_t)d->cin, (cuuint64_t)(d->n * (int64_t)d->h * d->w)};
  const cuuint64_t strides[1] = {ld};
  const cuuint32_t box[2] = {8, 128}, es[2] = {1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(d->x), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int CPR, bool IS3, int MT, bool TMA>
static int thin_prepare(const iea_conv_desc* d, thin::Params& p, int& grid, uint32_t& smem, bool tst = false) {
  using G = thin::Geo<CPR, IS3, MT, TMA>;
  p.d = *d;
  p.wtc = (const bf16*)d->wpack_tc;
  p.M = (int)(d->n * (int64_t)d->h * d->w);
  p.hs = stored_res(*d, d->h);
  p.ws = stored_res(*d, d->w);
  const int hw = d->h * d->w;
  if (IS3) {
    p.mtw = d->w / (8 * MT); p.mth = d->h / 16;
    p.n_macro = (int)(d->n * (int64_t)p.mtw * p.mth);
  } else {
    p.n_macro = (p.M + 128 * MT - 1) / (128 * MT);
    p.mtw = hw % (128 * MT) == 0 ? hw / (128 * MT) : p.n_macro + 1;  // (never wraps when images are not whole tiles)
    p.mth = 1;
  }
  p.fd_mtw = thin::make_fastdiv(p.mtw); p.fd_mth = thin::make_fastdiv(p.mth);
  p.fd_w = thin::make_fastdiv(d->w); p.fd_h = thin::make_fastdiv(d->h);
  const int64_t per_event = IS3 ? 40ll * p.mtw * p.mth : (40ll * hw) / (128 * MT);
  p.fd_tpe = thin::make_fastdiv(per_event > 0 ? (uint32_t)per_event : 1u);
  const int taps = IS3 ? 9 : 1;
  const int cout_e = d->cout == 1 ? 16 : d->cout;  // rows of the weight pack / accumulator columns
  p.w_bytes = (uint32_t)(cout_e * d->cin * taps * 2);
  p.stage_off = (p.w_bytes + 127) / 128 * 128;
  const uint32_t misc = (2 * cout_e + 2 * 4 * 2 * cout_e) * 4;  // scale, bias, statistics fold of both groups
  const uint32_t tail = misc + 512;
  p.res_slot = tst ? (d->res_mode == IEA_IN_UP2 ? 64u : 128u) * (uint32_t)d->res_c * 2 : 0;
  const uint32_t ring_bytes = tst ? 2 * thin::RES_RING * p.res_slot + 1024 : 0;
  const uint32_t tst_bytes = tst ? 2 * 2 * 128 * 64 + 2048 + ring_bytes : 0;  // two groups x two sub-tile images (+ alignment)
  int stages = 8;  // even: the two producer groups own alternate ring slots
  while (stages > 4 && p.stage_off + stages * G::STAGE + tail + tst_bytes > 208 * 1024) stages -= 2;
  p.stages = stages;
  p.depth = stages >= 8 ? 3 : 2;  // items each group keeps in flight (it owns stages/2 slots)
  p.tst_off = (p.stage_off + stages * G::STAGE + 1023) / 1024 * 1024;
  p.res_off = p.tst_off + 2 * 2 * 128 * 64 + 1024;
  p.misc_off = tst ? p.res_off + ring_bytes : p.stage_off + stages * G::STAGE;
  p.bar_off = (p.misc_off + misc + 15) / 16 * 16;
  smem = p.bar_off + 512;  // barriers: full, empty, landing (8 B x stages each), 2 x 4 accumulator, weights; TMEM slot
  const uint32_t cols = tmem_cols_for(4 * MT * cout_e);
  p.tmem_cols = cols;
  IEA_CHECK_ARG(smem <= 220 * 1024 && cols <= 512, "iea_conv_fprop(tcgen05 thin): tile does not fit (cin=%d cout=%d k=%d)",
                d->cin, d->cout, d->ksize);
  const int sms = sm_count();
  grid = p.n_macro < sms ? p.n_macro : sms;
  return 0;
}

template <int CPR, bool IS3, int NB, int MT>
static int thin_launch(const iea_conv_desc* d, cudaStream_t s, int* grid_only) {
  thin::Params p; int grid = 0; uint32_t smem = 0;
  alignas(64) CUtensorMap tm;
  memset(&tm, 0, sizeof(tm));
  // TMA producer: same-resolution bf16 input; IEA_THIN_TMA=0 keeps the cp.async producer (tests cover both)
  constexpr bool TMA_OK = true;  // (also worth it where the epilogue paces the kernel: 16 -> 32 1x1 + residual 2.05 -> 1.79 ms)
  bool tma = TMA_OK && !grid_only && d->in_mode == IEA_IN_DIRECT && d->x_ld % 8 == 0;
  if (tma) { const char* e_ = getenv("IEA_THIN_TMA"); if (e_ && e_[0] == '0') tma = false; }
  if (tma) tma = thin_tensor_map(d, IS3, MT, &tm);
  // TMA store of the output: the residual flavour of the 1x1 layers, whole sub-tiles only
  alignas(64) CUtensorMap tmy;
  memset(&tmy, 0, sizeof(tmy));
  const bool simple = d->acc_c0 < 0 && d->act == IEA_ACT_NONE && d->cout != 1;
  bool tst = !IS3 && tma && simple && d->res && d->res_mode != IEA_IN_POOL2 && (d->n * (int64_t)d->h * d->w) % (128 * MT) == 0;
  alignas(64) CUtensorMap tmr;
  memset(&tmr, 0, sizeof(tmr));
  if (tst) tst = thin_tensor_map_y(d, &tmy) && thin_tensor_map_r(d, &tmr);
  int rc = tma ? thin_prepare<CPR, IS3, MT, TMA_OK>(d, p, grid, smem, tst) : thin_prepare<CPR, IS3, MT, false>(d, p, grid, smem);
  if (rc) return rc;
  if (grid_only) { *grid_only = grid; return 0; }
  auto run = [&](auto kern) -> int {
    IEA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, thin::THREADS, smem, s>>>(p, tm, tmy, tmr);
    return check_launch("iea_conv_fprop(tcgen05 thin)");
  };
  // (a compile-time "plain" flavour measured no faster than the generic one -- without a residual the
  //  producers, not the epilogue, pace these kernels -- so only the residual flavour is specialised)
  if constexpr (TMA_OK) {
    if (tma) {
      if constexpr (!IS3) {
        if (tst) return run(thin::conv_thin_kernel<CPR, IS3, NB, MT, 3, true>);
        if (simple && d->res && d->res_mode != IEA_IN_POOL2) return run(thin::conv_thin_kernel<CPR, IS3, NB, MT, 1, true>);
      }
      return run(thin::conv_thin_kernel<CPR, IS3, NB, MT, 2, true>);
    }
  }
  if constexpr (!IS3) {
    if (simple && d->res && d->res_mode != IEA_IN_POOL2) return run(thin::conv_thin_kernel<CPR, IS3, NB, MT, 1, false>);
  }
  return run(thin::conv_thin_kernel<CPR, IS3, NB, MT, 2, false>);
}

static int thin_dispatch(const iea_conv_desc* d, cudaStream_t s, int* grid_only) {
  const int mt = thin_mt(d), cpr = d->cin / 8, nb = d->cout == 1 ? 1 : d->cout / 16;
  const bool is3 = d->ksize == 3;
#define IEA_THIN_CASE(C_, I_, N_, M_) \
  if (cpr == C_ && is3 == I_ && nb == N_ && mt == M_) return thin_launch<C_, I_, N_, M_>(d, s, grid_only);
#define IEA_THIN_MTS(C_, I_, N_) IEA_THIN_CASE(C_, I_, N_, 1) IEA_THIN_CASE(C_, I_, N_, 2)
  IEA_THIN_MTS(2, true, 1) IEA_THIN_MTS(2, true, 2) IEA_THIN_CASE(2, true, 1, 4) IEA_THIN_CASE(2, true, 2, 4)
  IEA_THIN_MTS(4, true, 1) IEA_THIN_MTS(4, true, 2) IEA_THIN_CASE(4, true, 1, 4)
  IEA_THIN_CASE(8, true, 1, 1) IEA_THIN_CASE(8, true, 2, 1)
  IEA_THIN_MTS(2, false, 1) IEA_THIN_MTS(2, false, 2) IEA_THIN_CASE(2, false, 1, 4) IEA_THIN_CASE(2, false, 2, 4)
  IEA_THIN_MTS(4, false, 1) IEA_THIN_MTS(4, false, 2)
  IEA_THIN_CASE(8, false, 1, 1) IEA_THIN_CASE(8, false, 2, 1)
#undef IEA_THIN_MTS
#undef IEA_THIN_CASE
  set_error("iea_conv_fprop(tcgen05 thin): no kernel for cin=%d cout=%d k=%d mt=%d", d->cin, d->cout, d->ksize, mt);
  return -2;
}

int iea_conv_fprop_thin(const iea_conv_desc* d, cudaStream_t s) { return thin_dispatch(d, s, nullptr); }
// statistics slots per event = 2 x CTAs of the launch (each epilogue group folds its tiles per event)
int iea_conv_thin_stats_slots(const iea_conv_desc* d) {
  int grid = 0;
  if (thin_dispatch(d, nullptr, &grid)) return 0;
  return 2 * grid;
}
