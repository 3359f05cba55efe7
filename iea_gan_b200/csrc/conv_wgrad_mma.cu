// conv_wgrad_mma.cu -- weight gradient of the thin, high-resolution convolutions.
//
//   dW[co][tap][ci] = sum over pixels  g[px][co] * T(x)[px + tap][ci]
//
// The outputs are tiny (16x144 ... 64x576 values) while the reduction runs over 10^6..10^8 pixels, so
// the kernel is a persistent split-K: every CTA streams pixel tiles (the same 18x10 halo patch /
// 128-pixel staging, cp.async ring and in-place fused prologue as the forward kernel), keeps the whole
// dW in registers across all its tiles and writes one fp32 partial per warp group at the end;
// iea_sn_weight_bwd reduces the partials in a fixed order (deterministic).
//
// Why warp-level mma.sync here and not tcgen05: the UMMA M dimension is >= 64 but Cout (and Cin) of the
// heavy layers is 16..64, and the 9 taps are non-uniformly strided views of the patch, so they cannot
// be stacked into one UMMA operand.  Padding M to 128 makes the MMA read 8x the useful shared-memory
// bytes (331 KB per 128-pixel tile at 16 channels = 2.6k cycles, vs ~350 cycles of HBM time).  The
// m16n8k16 shape matches the 16-channel blocks exactly, ldmatrix takes per-lane row addresses (so the
// shifted tap views are free) and each g fragment is reused by all 9 taps: ~40 KB of smem reads/tile.
#include "tc_common.cuh"
using namespace iea;

namespace wg {
using namespace tc;

constexpr int PW = 10, PH = 18;


struct Params {
  FastDiv fd_tw, fd_th, fd_hw, fd_w, fd_h;
  iea_conv_desc d;
  const void* g; int g_dtype, g_ld;
  float* gpart;
  float* cs_parts;  // [gridDim.x][cout] column sums of g (bias gradient) or NULL
  int64_t M;
  int n_tiles, tiles_w, tiles_h, hs, ws, cpa, cpg, cpa_sh, cpg_sh, cin_eff, cout_eff, stages, depth, P, WP;
  int per_px_affine;     // 1x1 layers whose images are not whole 128-pixel tiles: fused-prologue constants per pixel
  int nib_l, ncb_l, gi;  // output split over blockIdx.y: ci blocks / co blocks per CTA, groups along ci
  uint32_t plane_a, plane_g, stage_bytes, g_off;
};

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
    o.m0 = (int64_t)tile * 128; o.n = (int)fdiv((unsigned)o.m0, p.fd_hw); o.h0 = 0; o.w0 = 0;
  }
  return o;
}

__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int TAPS, int NPAIR>
__global__ void __launch_bounds__(256) wgrad_mma_kernel(const Params p) {
  constexpr bool IS3 = TAPS == 9;
  constexpr int NPIX = IS3 ? PH * PW : 128;
  extern __shared__ __align__(128) uint8_t smem[];
  const iea_conv_desc& d = p.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const int my_tiles = (int)blockIdx.x < p.n_tiles ? (p.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const bool affine = d.in_scale != nullptr, relu = d.in_relu != 0;
  const bool thin_a = d.cin < 16, thin_g = d.cout < 16;  // 1-channel stem input / 1-channel output conv
  const bool pool = d.in_mode == IEA_IN_POOL2;
  const int sh_ = d.in_mode == IEA_IN_UP2 ? 1 : 0;
  const int D = p.depth;
  const int total_a = NPIX * p.cpa, total_g = 128 * p.cpg;            // cpa / cpg: planes staged by THIS CTA
  const int ib0 = ((int)blockIdx.y % p.gi) * p.nib_l, cb0 = ((int)blockIdx.y / p.gi) * p.ncb_l;
  const int ca0 = ib0 * 16, cg0 = cb0 * 16;                           // first input / output channel of this CTA

  float acc[NPAIR][TAPS][2][4];
#pragma unroll
  for (int q = 0; q < NPAIR; ++q)
#pragma unroll
    for (int t = 0; t < TAPS; ++t)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[q][t][j][r] = 0.f;

  // bias gradient for free: the g fragments are already in registers, one extra MMA against an all-ones B
  // fragment per k-step gives sum_px g[px][co] (warps that own the first input-channel block only)
  const bool cs_cta = p.cs_parts != nullptr && ib0 == 0;
  float acc_cs[NPAIR][4];
#pragma unroll
  for (int q = 0; q < NPAIR; ++q)
#pragma unroll
    for (int r = 0; r < 4; ++r) acc_cs[q][r] = 0.f;

  // conv-resolution coordinates of patch pixel pp; false = padding / beyond the last row
  auto pix_a = [&](const Origin& o, int pp, int& ih, int& iw, int64_t& m) -> bool {
    if (IS3) {
      const int pi = pp / PW;
      ih = o.h0 - 1 + pi; iw = o.w0 - 1 + (pp - pi * PW);
      return (unsigned)ih < (unsigned)d.h && (unsigned)iw < (unsigned)d.w;
    }
    m = o.m0 + pp;
    return m < p.M;
  };
  auto issue = [&](int it) {
    const Origin o = tile_origin<IS3>(p, (int)blockIdx.x + it * (int)gridDim.x);
    const uint32_t s0 = sbase + (uint32_t)(it % p.stages) * p.stage_bytes;
    // ---- input patch (raw; transformed in place after it landed)
    for (int e = tid; e < total_a; e += 256) {
      const int pp = e >> p.cpa_sh, c = e & (p.cpa - 1);  // (cpa, cpg are powers of two)
      int ih = 0, iw = 0; int64_t m = 0;
      const bool in = pix_a(o, pp, ih, iw, m);
      const uint32_t dst = s0 + c * p.plane_a + pp * 16;
      if (!in) { asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(dst), "r"(0) : "memory"); continue; }
      const int64_t pix = IS3 ? (((int64_t)o.n * p.hs + (ih >> sh_)) * p.ws + (iw >> sh_)) : m;
      if (pool) {  // 1x1 conv behind AvgPool2d (DBlock conv4 / conv_sc): average of 4 transformed chunks
        const unsigned mm = (unsigned)m, t = fdiv(mm, p.fd_w);
        const int ow = (int)(mm - t * (unsigned)d.w), nn = (int)fdiv(t, p.fd_h), oh = (int)(t - (unsigned)nn * (unsigned)d.h);
        float a8[8], s8[8], h8[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { a8[j] = 0.f; s8[j] = 1.f; h8[j] = 0.f; }
        if (affine) {
          const int64_t si = (d.in_bcast ? 0 : (int64_t)nn * d.cin) + ca0 + c * 8;
#pragma unroll
          for (int j = 0; j < 8; ++j) { s8[j] = d.in_scale[si + j]; h8[j] = d.in_shift[si + j]; }
        }
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int b = 0; b < 2; ++b) {
            float f[8];
            unpack8(*reinterpret_cast<const uint4*>((const bf16*)d.x + (((int64_t)nn * p.hs + 2 * oh + a) * p.ws + 2 * ow + b) * d.x_ld + ca0 + c * 8), f);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float v = affine ? fmaf(f[j], s8[j], h8[j]) : f[j];
              a8[j] += relu ? fmaxf(v, 0.f) : v;
            }
          }
#pragma unroll
        for (int j = 0; j < 8; ++j) a8[j] *= 0.25f;
        const uint4 q4 = pack8(a8);
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(dst), "r"(q4.x), "r"(q4.y), "r"(q4.z), "r"(q4.w) : "memory");
      } else if (thin_a) {  // 1 input channel (fp32 or bf16): zero-extend to a 16-byte chunk
        const float v = c == 0 ? ld_act(d.x, d.x_dtype, pix * d.x_ld) : 0.f;
        const uint32_t lo = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v));
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%2,%2};" ::"r"(dst), "r"(lo), "r"(0) : "memory");
      } else {
        cp16(dst, (const bf16*)d.x + pix * d.x_ld + ca0 + c * 8);
      }
    }
    // ---- output-gradient tile: 128 pixels x cout, pixel r = (r>>3, r&7) inside a 16x8 tile
    for (int e = tid; e < total_g; e += 256) {
      const int r = e >> p.cpg_sh, c = e & (p.cpg - 1);
      int64_t m;
      bool in = true;
      if (IS3) {  // (images smaller than / not a multiple of the 16x8 tile: rows and columns beyond the edge are zero)
        m = ((int64_t)o.n * d.h + o.h0 + (r >> 3)) * d.w + o.w0 + (r & 7);
        in = o.h0 + (r >> 3) < d.h && o.w0 + (r & 7) < d.w;
      } else { m = o.m0 + r; in = m < p.M; }
      const uint32_t dst = s0 + p.g_off + c * p.plane_g + r * 16;
      if (!in) { asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(dst), "r"(0) : "memory"); continue; }
      if (thin_g) {
        uint32_t w4[4] = {0, 0, 0, 0};
        if (c == 0)
          for (int j = 0; j < d.cout; ++j) {
            const uint32_t h = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(ld_act(p.g, p.g_dtype, m * p.g_ld + j)));
            w4[j >> 1] |= h << ((j & 1) * 16);
          }
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(dst), "r"(w4[0]), "r"(w4[1]), "r"(w4[2]), "r"(w4[3]) : "memory");
      } else {
        cp16(dst, (const bf16*)p.g + m * p.g_ld + cg0 + c * 8);
      }
    }
  };

  for (int k = 0; k < D - 1; ++k) {
    if (k < my_tiles) issue(k);
    cp_async_commit();
  }
  // warp -> (output block pairs, k-step group)
  const int nib = p.nib_l;  // 16-wide ci blocks of this CTA
  int kg = 0, pair0 = 0;
  if (p.P <= 8) { pair0 = warp % p.P; kg = warp / p.P; } else { pair0 = warp * NPAIR; }
  float sc[8], sh[8];
  int ss_n = -1;
  const int my_c = tid & (p.cpa - 1);  // 256 % cpa == 0: the chunk column of this thread is fixed

  for (int it = 0; it < my_tiles; ++it) {
    if (it + D - 1 < my_tiles) issue(it + D - 1);
    cp_async_commit();
    switch (D) {
      case 2: cp_async_wait<1>(); break;
      case 3: cp_async_wait<2>(); break;
      case 4: cp_async_wait<3>(); break;
      default: cp_async_wait<0>(); break;
    }
    const Origin o = tile_origin<IS3>(p, (int)blockIdx.x + it * (int)gridDim.x);
    const uint32_t s0 = sbase + (uint32_t)(it % p.stages) * p.stage_bytes;
    uint8_t* sp = smem + (size_t)(it % p.stages) * p.stage_bytes;
    if ((affine || relu) && !pool) {  // fused prologue, in place, on the chunks this thread copied
      if (affine && !p.per_px_affine && o.n != ss_n) {
        const int64_t si = (d.in_bcast ? 0 : (int64_t)o.n * d.cin) + ca0 + my_c * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) { sc[j] = d.in_scale[si + j]; sh[j] = d.in_shift[si + j]; }
        ss_n = o.n;
      }
      for (int e = tid; e < total_a; e += 256) {
        const int pp = e >> p.cpa_sh;
        int ih = 0, iw = 0; int64_t m = 0;
        if (!pix_a(o, pp, ih, iw, m)) continue;
        if (p.per_px_affine) {  // images smaller than a tile (8x8, 4x4 layers): the constants change inside the tile
          const int nn = (int)fdiv((unsigned)m, p.fd_hw);
          if (nn != ss_n) {
            const int64_t si = (d.in_bcast ? 0 : (int64_t)nn * d.cin) + ca0 + my_c * 8;
#pragma unroll
            for (int j = 0; j < 8; ++j) { sc[j] = d.in_scale[si + j]; sh[j] = d.in_shift[si + j]; }
            ss_n = nn;
          }
        }
        uint4* q = reinterpret_cast<uint4*>(sp + my_c * p.plane_a + pp * 16);
        float f[8];
        unpack8(*q, f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float v = affine ? fmaf(f[j], sc[j], sh[j]) : f[j];
          f[j] = relu ? fmaxf(v, 0.f) : v;
        }
        *q = pack8(f);
      }
    }
    __syncthreads();
    // ---- tensor-core accumulation
    const int mat = lane >> 3, rr = lane & 7;
#pragma unroll
    for (int q = 0; q < NPAIR; ++q) {
      const int pair = pair0 + q;
      const int cb = pair / nib, ib = pair - cb * nib;
      for (int ks = kg; ks < 8; ks += p.WP) {
        uint32_t a[4];
        ldsm_x4_t(s0 + p.g_off + (cb * 2 + (mat & 1)) * p.plane_g + (ks * 16 + (mat >> 1) * 8 + rr) * 16, a[0], a[1], a[2], a[3]);
        if (cs_cta && ib == 0) mma16816(acc_cs[q], a, 0x3F803F80u, 0x3F803F80u);
        const uint32_t brow = s0 + (ib * 2 + (mat >> 1)) * p.plane_a;
#pragma unroll
        for (int t = 0; t < TAPS; ++t) {
          int pp;
          if (IS3) pp = (2 * ks + (mat & 1) + t / 3) * PW + rr + t % 3;   // (i + 1 + dh) * PW + (j + 1 + dw)
          else pp = ks * 16 + (mat & 1) * 8 + rr;
          uint32_t b0, b1, b2, b3;
          ldsm_x4_t(brow + pp * 16, b0, b1, b2, b3);
          mma16816(acc[q][t][0], a, b0, b1);
          mma16816(acc[q][t][1], a, b2, b3);
        }
      }
    }
    __syncthreads();  // the stage is overwritten by the cp.async of the next iteration
  }
  cp_async_wait<0>();
  // ---- fold the k-step groups of the CTA (fixed order), then one partial per CTA:
  //      gpart[blockIdx.x][cout][taps][cin]
  if (p.WP > 1) {  // NPAIR == 1 here; scratch [P][TAPS*8][32] floats re-uses the pipeline smem
    float* scr = reinterpret_cast<float*>(smem);
    __syncthreads();
    for (int kgi = 1; kgi < p.WP; ++kgi) {
      if (kg == kgi) {
#pragma unroll
        for (int t = 0; t < TAPS; ++t)
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int r = 0; r < 4; ++r) scr[(pair0 * TAPS * 8 + t * 8 + j * 4 + r) * 32 + lane] = acc[0][t][j][r];
#pragma unroll
        for (int r = 0; r < 4; ++r) scr[(p.P * TAPS * 8 + pair0 * 4 + r) * 32 + lane] = acc_cs[0][r];
      }
      __syncthreads();
      if (kg == 0) {
#pragma unroll
        for (int t = 0; t < TAPS; ++t)
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[0][t][j][r] += scr[(pair0 * TAPS * 8 + t * 8 + j * 4 + r) * 32 + lane];
#pragma unroll
        for (int r = 0; r < 4; ++r) acc_cs[0][r] += scr[(p.P * TAPS * 8 + pair0 * 4 + r) * 32 + lane];
      }
      __syncthreads();
    }
  }
  if (kg != 0) return;
  float* out = p.gpart + (int64_t)blockIdx.x * d.cout * TAPS * d.cin;
#pragma unroll
  for (int q = 0; q < NPAIR; ++q) {
    const int pair = pair0 + q;
    const int cb = pair / nib, ib = pair - cb * nib;
#pragma unroll
    for (int t = 0; t < TAPS; ++t)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int co = cg0 + cb * 16 + (lane >> 2) + (r >= 2 ? 8 : 0);
          const int ci = ca0 + ib * 16 + j * 8 + 2 * (lane & 3) + (r & 1);
          if (co < d.cout && ci < d.cin) out[((int64_t)co * TAPS + t) * d.cin + ci] = acc[q][t][j][r];
        }
    if (cs_cta && ib == 0 && (lane & 3) == 0) {  // every column of the ones-MMA holds the same sum
      const int co = cg0 + cb * 16 + (lane >> 2);
      if (co < d.cout) p.cs_parts[(int64_t)blockIdx.x * d.cout + co] = acc_cs[q][0];
      if (co + 8 < d.cout) p.cs_parts[(int64_t)blockIdx.x * d.cout + co + 8] = acc_cs[q][2];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Macro-tile variant for the thin 3x3 layers at high resolution (Cin, Cout in {16, 32}; same-resolution or
// nearest-up2 input): one pipeline item is MT side-by-side 16x8 tiles -- an 18 x (8*MT+2) halo patch of x and
// 128*MT rows of g -- so the two block barriers, the tile bookkeeping and the halo re-reads are paid once per
// 128*MT pixels, and every thread owns the same chunk slots of every patch: global / shared offsets of its
// cp.async copies are computed once per kernel (no divisions or coordinate tests in the tile loop), the fused
// BN-affine + ReLU prologue is one LDS / 4 packed-bf16 FMA / STS per chunk (the same rounding as the forward
// kernel, conv_thin.cu), border patches use per-slot side masks.
struct P3 {
  iea_conv_desc d;
  const bf16* g; int g_ld;
  float* gpart; float* cs_parts;
  int n_macro, mtw, mth, hs, ws, stages, depth;
  FastDiv fd_mtw, fd_mth;
};

template <int CPA, int CPG, int MT, bool IS3 = true>
struct G3 {
  static constexpr int PWM = 8 * MT + 2;
  static constexpr int NPA = IS3 ? PH * PWM : 128 * MT;  // staged input pixels (3x3: halo patch; 1x1: the pixel run)
  static constexpr int NPG = 128 * MT;                 // g rows
  static constexpr int NSA = (NPA * CPA + 255) / 256;  // chunk slots per thread
  static constexpr int NSG = NPG * CPG / 256;
  static constexpr uint32_t PLA = (NPA * 16 + 127) / 128 * 128 + 128 / CPA;
  static constexpr uint32_t PLG = NPG * 16 + 128 / CPG;
  static constexpr uint32_t GOFF = CPA * PLA;
  static constexpr uint32_t STAGE = (GOFF + CPG * PLG + 127) / 128 * 128;
};

template <int CPA, int CPG, int MT, bool IS3>
__global__ void __launch_bounds__(256) wgrad3_kernel(const P3 p) {
  using G = G3<CPA, CPG, MT, IS3>;
  constexpr int PWM = G::PWM, NSA = G::NSA, NSG = G::NSG, TAPS = IS3 ? 9 : 1;
  constexpr int NIB = CPA / 2, NCB = CPG / 2, P = NIB * NCB, WP = 8 / P, KS = 8 * MT;
  extern __shared__ __align__(128) uint8_t smem[];
  const iea_conv_desc& d = p.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const int my_n = (int)blockIdx.x < p.n_macro ? (p.n_macro - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const bool affine = d.in_scale != nullptr, relu = d.in_relu != 0;
  const int sh_ = d.in_mode == IEA_IN_UP2 ? 1 : 0;
  const int D = p.depth;

  // ---- slot tables (tile independent)
  const int ca = tid % CPA, cg = tid % CPG;
  int goa[NSA], gog[NSG];
  uint32_t soa[NSA], sog[NSG];
  uint32_t m_top = 0, m_bot = 0, m_left = 0, m_right = 0, m_valid = 0;
#pragma unroll
  for (int i = 0; i < NSA; ++i) {
    const int q = tid + 256 * i, pp = q / CPA;
    if (q < G::NPA * CPA) m_valid |= 1u << i;
    soa[i] = ca * G::PLA + pp * 16;
    if (IS3) {
      const int pi = pp / PWM, pj = pp - pi * PWM;
      goa[i] = (((pi - 1) >> sh_) * p.ws + ((pj - 1) >> sh_)) * d.x_ld + ca * 8;
      if (pi == 0) m_top |= 1u << i;
      if (pi == PH - 1) m_bot |= 1u << i;
      if (pj == 0) m_left |= 1u << i;
      if (pj == PWM - 1) m_right |= 1u << i;
    } else {
      goa[i] = pp * d.x_ld + ca * 8;
    }
  }
#pragma unroll
  for (int i = 0; i < NSG; ++i) {
    const int q = tid + 256 * i, r = q / CPG;            // r = sb*128 + (row*8 + col) inside the sub-tile
    const int sb = r >> 7, lr = r & 127;
    gog[i] = IS3 ? ((lr >> 3) * d.w + sb * 8 + (lr & 7)) * p.g_ld + cg * 8 : r * p.g_ld + cg * 8;
    sog[i] = G::GOFF + cg * G::PLG + r * 16;
  }
  struct Pos { int n, th, tw; };
  auto pos_of = [&](int item) {
    Pos c;
    if (!IS3) {  // mtw = macro tiles per image: n = item / mtw
      c.n = (int)fdiv((unsigned)item, p.fd_mtw); c.th = 0; c.tw = item;
      return c;
    }
    const unsigned t = fdiv((unsigned)item, p.fd_mtw);
    c.tw = (int)((unsigned)item - t * (unsigned)p.mtw);
    c.n = (int)fdiv(t, p.fd_mth);
    c.th = (int)(t - (unsigned)c.n * (unsigned)p.mth);
    return c;
  };
  auto pad_of = [&](const Pos& c) -> uint32_t {
    if (!IS3) return 0u;
    return (c.th == 0 ? m_top : 0u) | (c.th == p.mth - 1 ? m_bot : 0u) | (c.tw == 0 ? m_left : 0u) |
           (c.tw == p.mtw - 1 ? m_right : 0u);
  };
  const bf16* xb = (const bf16*)d.x;
  auto issue = [&](int it) {
    const Pos c = pos_of((int)blockIdx.x + it * (int)gridDim.x);
    const uint32_t s0 = sbase + (uint32_t)(it % p.stages) * G::STAGE;
    const bf16* ap = IS3 ? xb + ((int64_t)(c.n * p.hs + ((c.th * 16) >> sh_)) * p.ws + ((c.tw * (8 * MT)) >> sh_)) * d.x_ld
                         : xb + (int64_t)c.tw * (128 * MT) * d.x_ld;
    const bf16* gp = IS3 ? p.g + ((int64_t)(c.n * d.h + c.th * 16) * d.w + c.tw * (8 * MT)) * p.g_ld
                         : p.g + (int64_t)c.tw * (128 * MT) * p.g_ld;
    const uint32_t pad = pad_of(c);
#pragma unroll
    for (int i = 0; i < NSA; ++i) {
      if (!(m_valid >> i & 1)) continue;
      if (pad >> i & 1) asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(s0 + soa[i]), "r"(0) : "memory");
      else cp16(s0 + soa[i], ap + goa[i]);
    }
#pragma unroll
    for (int i = 0; i < NSG; ++i)
      cp16(s0 + sog[i], gp + gog[i]);
  };

  const int pair = warp % P, kg = warp / P;
  const int cb = pair / NIB, ib = pair - cb * NIB;
  const bool cs_on = p.cs_parts != nullptr && ib == 0;
  float acc[TAPS][2][4], acc_cs[4];
#pragma unroll
  for (int t = 0; t < TAPS; ++t)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int r = 0; r < 4; ++r) acc[t][j][r] = 0.f;
#pragma unroll
  for (int r = 0; r < 4; ++r) acc_cs[r] = 0.f;

  for (int k = 0; k < D - 1; ++k) {
    if (k < my_n) issue(k);
    cp_async_commit();
  }
  __nv_bfloat162 sc2[4], sh2[4];
  const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
  int ss_n = -1;
  const int mat = lane >> 3, rr = lane & 7;
  for (int it = 0; it < my_n; ++it) {
    if (it + D - 1 < my_n) issue(it + D - 1);
    cp_async_commit();
    if (D == 2) cp_async_wait<1>();
    else cp_async_wait<2>();
    const uint32_t s0 = sbase + (uint32_t)(it % p.stages) * G::STAGE;
    if (affine || relu) {  // fused prologue, in place on the chunks this thread copied; padding stays zero
      const Pos c = pos_of((int)blockIdx.x + it * (int)gridDim.x);
      if (affine && c.n != ss_n) {
        ss_n = c.n;
        const int64_t si = (d.in_bcast ? 0 : (int64_t)ss_n * d.cin) + ca * 8;
        const float4 a0 = *reinterpret_cast<const float4*>(d.in_scale + si), a1 = *reinterpret_cast<const float4*>(d.in_scale + si + 4);
        const float4 b0 = *reinterpret_cast<const float4*>(d.in_shift + si), b1 = *reinterpret_cast<const float4*>(d.in_shift + si + 4);
        sc2[0] = __floats2bfloat162_rn(a0.x, a0.y); sc2[1] = __floats2bfloat162_rn(a0.z, a0.w);
        sc2[2] = __floats2bfloat162_rn(a1.x, a1.y); sc2[3] = __floats2bfloat162_rn(a1.z, a1.w);
        sh2[0] = __floats2bfloat162_rn(b0.x, b0.y); sh2[1] = __floats2bfloat162_rn(b0.z, b0.w);
        sh2[2] = __floats2bfloat162_rn(b1.x, b1.y); sh2[3] = __floats2bfloat162_rn(b1.z, b1.w);
      }
      const uint32_t live = m_valid & ~pad_of(c);
      uint8_t* a = smem + (size_t)(it % p.stages) * G::STAGE;
#pragma unroll
      for (int i = 0; i < NSA; ++i) {
        if (!(live >> i & 1)) continue;
        uint4* q = reinterpret_cast<uint4*>(a + soa[i]);
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
    __syncthreads();
    // ---- tensor-core accumulation: this warp's (co block, ci block) pair over its share of the k-steps
    for (int ks = kg; ks < KS; ks += WP) {
      const int sb = ks >> 3, kl = ks & 7;
      uint32_t a[4];
      ldsm_x4_t(s0 + G::GOFF + (cb * 2 + (mat & 1)) * G::PLG + (sb * 128 + kl * 16 + (mat >> 1) * 8 + rr) * 16, a[0], a[1], a[2], a[3]);
      if (cs_on) mma16816(acc_cs, a, 0x3F803F80u, 0x3F803F80u);
      const uint32_t brow = s0 + (ib * 2 + (mat >> 1)) * G::PLA +
                            (uint32_t)(IS3 ? (2 * kl + (mat & 1)) * PWM + sb * 8 + rr : ks * 16 + (mat & 1) * 8 + rr) * 16;
#pragma unroll
      for (int t = 0; t < TAPS; ++t) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4_t(brow + (uint32_t)(IS3 ? (t / 3) * PWM + t % 3 : 0) * 16, b0, b1, b2, b3);
        mma16816(acc[t][0], a, b0, b1);
        mma16816(acc[t][1], a, b2, b3);
      }
    }
    __syncthreads();  // the stage is overwritten by the cp.async of the next iteration
  }
  cp_async_wait<0>();
  // ---- fold the k-step groups (fixed order), then one partial per CTA: gpart[blockIdx.x][cout][9][cin]
  if (WP > 1) {
    float* scr = reinterpret_cast<float*>(smem);  // [P][TAPS*8 + 4][32]
    constexpr int FS = TAPS * 8 + 4;
    __syncthreads();
    for (int kgi = 1; kgi < WP; ++kgi) {
      if (kg == kgi) {
#pragma unroll
        for (int t = 0; t < TAPS; ++t)
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int r = 0; r < 4; ++r) scr[(pair * FS + t * 8 + j * 4 + r) * 32 + lane] = acc[t][j][r];
#pragma unroll
        for (int r = 0; r < 4; ++r) scr[(pair * FS + TAPS * 8 + r) * 32 + lane] = acc_cs[r];
      }
      __syncthreads();
      if (kg == 0) {
#pragma unroll
        for (int t = 0; t < TAPS; ++t)
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[t][j][r] += scr[(pair * FS + t * 8 + j * 4 + r) * 32 + lane];
#pragma unroll
        for (int r = 0; r < 4; ++r) acc_cs[r] += scr[(pair * FS + TAPS * 8 + r) * 32 + lane];
      }
      __syncthreads();
    }
  }
  if (kg != 0) return;
  float* out = p.gpart + (int64_t)blockIdx.x * d.cout * TAPS * d.cin;
#pragma unroll
  for (int t = 0; t < TAPS; ++t)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int co = cb * 16 + (lane >> 2) + (r >= 2 ? 8 : 0);
        const int ci = ib * 16 + j * 8 + 2 * (lane & 3) + (r & 1);
        out[((int64_t)co * TAPS + t) * d.cin + ci] = acc[t][j][r];
      }
  if (cs_on && (lane & 3) == 0) {
    const int co = cb * 16 + (lane >> 2);
    p.cs_parts[(int64_t)blockIdx.x * d.cout + co] = acc_cs[0];
    p.cs_parts[(int64_t)blockIdx.x * d.cout + co + 8] = acc_cs[2];
  }
}

// sum of the per-CTA partials in a fixed order: out[i] = sum_s gpart[s][i]
__global__ void wgrad_reduce_kernel(const float* gpart, int nsplit, int64_t total, float* out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    float a = 0.f;
    for (int s = 0; s < nsplit; ++s) a += gpart[(int64_t)s * total + i];
    out[i] = a;
  }
}

}  // namespace wg

// The weight-gradient kernel a shape runs on, with its launch geometry.  wgrad_plan() is the one place that
// chooses it: iea_conv_wgrad_mma_slices sizes gpart from the plan and iea_conv_wgrad_mma launches it.
struct WgradPlan {
  enum Kernel { none, c1, tc, macro, mma } kernel = none;
  int grid = 0;      // per-CTA (tc: per-split) partials, in slices 1..grid of gpart
  int slices = 0;    // slices of gpart the launch uses; 0: shape not handled (use iea_conv_wgrad)
  uint32_t smem = 0;
  wg::P3 p3;                        // macro-tile kernel
  void (*k3)(wg::P3) = nullptr;
  wg::Params pm;                    // generic mma.sync kernel
  void (*km)(wg::Params) = nullptr;
  int grid_y = 1;
};

// generic mma.sync kernel: parameters, instance and grid (0: shape not handled by this kernel)
static int wgrad_mma_plan(const iea_conv_desc* d, int g_dtype, int g_ld, WgradPlan& pl) {
  wg::Params* p = &pl.pm;
  const bool thin_a = d->cin < 16, thin_g = d->cout < 16;
  if (!thin_a && (d->cin % 16 || d->x_dtype != IEA_BF16 || d->x_ld % 8 || (reinterpret_cast<uintptr_t>(d->x) & 15))) return 0;
  if (thin_a && (d->cin != 1 || d->in_scale || d->in_relu || d->in_mode != IEA_IN_DIRECT)) return 0;
  if (!thin_g && (d->cout % 16 || g_dtype != IEA_BF16 || g_ld % 8)) return 0;
  if (thin_g && d->cout > 8) return 0;
  if (d->in_mode == IEA_IN_POOL2 && (d->ksize != 1 || thin_a)) return 0;
  const int cin_eff = thin_a ? 16 : d->cin, cout_eff = thin_g ? 16 : d->cout;
  const bool is3 = d->ksize == 3;
  if (is3 && d->in_mode == IEA_IN_UP2 && (d->h % 2 || d->w % 2)) return 0;
  p->per_px_affine = (!is3 && (((int64_t)d->h * d->w) % 128) && d->in_scale) ? 1 : 0;  // a tile straddles images
  if (!is3 && d->in_mode == IEA_IN_UP2) return 0;
  const int64_t M = d->n * (int64_t)d->h * d->w;
  if (M >= (1ll << 31) || M < 512) return 0;  // tiny problems stay on the generic kernel
  const int taps = d->ksize * d->ksize;
  const int npix = is3 ? wg::PH * wg::PW : 128;
  const uint32_t plane_a = (npix * 16 + 127) / 128 * 128, plane_g = 128 * 16;
  // split the output blocks over blockIdx.y until the accumulators fit the registers and a stage fits smem
  const int nib = cin_eff / 16, ncb = cout_eff / 16;
  if ((nib & (nib - 1)) || (ncb & (ncb - 1))) return 0;
  int nib_l = nib, ncb_l = ncb;
  const int maxpairs = taps == 9 ? 16 : 128;
  while (nib_l * ncb_l > maxpairs || (uint32_t)(nib_l * 2) * plane_a + (uint32_t)(ncb_l * 2) * plane_g > 80 * 1024) {
    if (nib_l >= ncb_l && nib_l > 1) nib_l >>= 1;
    else if (ncb_l > 1) ncb_l >>= 1;
    else return 0;
  }
  const int P = nib_l * ncb_l;
  int npair = 1, WP = 1;
  if (P <= 8) WP = 8 / P; else npair = P / 8;
  p->d = *d;
  p->M = M;
  p->hs = stored_res(*d, d->h);
  p->ws = stored_res(*d, d->w);
  p->fd_w = wg::make_fastdiv(d->w); p->fd_h = wg::make_fastdiv(d->h);
  p->tiles_w = is3 ? (d->w + 7) / 8 : 1;    // edge tiles are masked (8x8 / 4x4 layers: one partly filled tile per image)
  p->tiles_h = is3 ? (d->h + 15) / 16 : 1;
  p->n_tiles = (int)(is3 ? d->n * (int64_t)p->tiles_w * p->tiles_h : (M + 127) / 128);
  p->fd_tw = wg::make_fastdiv(p->tiles_w); p->fd_th = wg::make_fastdiv(p->tiles_h);
  p->fd_hw = wg::make_fastdiv(d->h * d->w);
  p->cpa = nib_l * 2; p->cpg = ncb_l * 2; p->cin_eff = cin_eff; p->cout_eff = cout_eff;
  p->cpa_sh = 0; while ((1 << p->cpa_sh) < p->cpa) ++p->cpa_sh;
  p->cpg_sh = 0; while ((1 << p->cpg_sh) < p->cpg) ++p->cpg_sh;
  p->nib_l = nib_l; p->ncb_l = ncb_l; p->gi = nib / nib_l;
  p->plane_a = plane_a;
  p->plane_g = plane_g;
  p->g_off = p->cpa * p->plane_a;
  p->stage_bytes = p->g_off + p->cpg * p->plane_g;
  int stages = 4;
  while (stages > 2 && stages * p->stage_bytes > 100 * 1024) --stages;
  if (stages * p->stage_bytes > 200 * 1024) return 0;
  p->stages = stages;
  p->depth = stages >= 4 ? 3 : 2;
  p->P = P; p->WP = WP;
  const int sms = sm_count();
  pl.smem = p->stages * p->stage_bytes;
  const int occ = pl.smem <= 100 * 1024 ? 2 : 1;
  if (WP > 1 && pl.smem < (uint32_t)(P * (taps * 8 + 4) * 32 * 4)) pl.smem = P * (taps * 8 + 4) * 32 * 4;  // fold scratch
  pl.grid = p->n_tiles < sms * occ ? p->n_tiles : sms * occ;
  pl.grid_y = p->gi * (ncb / ncb_l);
  if (is3) pl.km = npair == 1 ? wg::wgrad_mma_kernel<9, 1> : npair == 2 ? wg::wgrad_mma_kernel<9, 2> : nullptr;
  else pl.km = npair == 1 ? wg::wgrad_mma_kernel<1, 1> : npair == 2 ? wg::wgrad_mma_kernel<1, 2>
             : npair == 4 ? wg::wgrad_mma_kernel<1, 4> : npair == 8 ? wg::wgrad_mma_kernel<1, 8>
             : npair == 16 ? wg::wgrad_mma_kernel<1, 16> : nullptr;
  return 1;
}

int iea_conv_c1_wgrad_grid(const iea_conv_desc* d, int g_dtype, int g_ld);
int iea_conv_c1_wgrad(const iea_conv_desc* d, const void* g, int g_dtype, int g_ld, float* parts, cudaStream_t s);

// macro-tile kernel: 0 = shape not handled, else MT (sub-tiles per macro tile)
static int wgrad3_mt(const iea_conv_desc* d, int g_dtype, int g_ld) {
  const bool is3 = d->ksize == 3;
  if (is3) {
    if ((d->cin != 16 && d->cin != 32) || (d->cout != 16 && d->cout != 32)) return 0;
  } else {
    if ((d->cin != 16 && d->cin != 32 && d->cin != 64) || (d->cout != 16 && d->cout != 32 && d->cout != 64)) return 0;
    if (d->cin * d->cout > 64 * 32 || d->in_mode != IEA_IN_DIRECT) return 0;  // <= 8 (16x16) block pairs: one per warp
  }
  if (d->in_mode == IEA_IN_POOL2 || d->x_dtype != IEA_BF16 || g_dtype != IEA_BF16) return 0;
  if (d->x_ld % 8 || g_ld % 8 || (reinterpret_cast<uintptr_t>(d->x) & 15)) return 0;
  if (is3 && (d->h % 16 || d->w % 16)) return 0;
  if (d->in_scale && ((reinterpret_cast<uintptr_t>(d->in_scale) & 15) || (reinterpret_cast<uintptr_t>(d->in_shift) & 15))) return 0;
  const int64_t M = d->n * (int64_t)d->h * d->w;
  if (M >= (1ll << 31) || M * (int64_t)(d->x_ld > g_ld ? d->x_ld : g_ld) >= (1ll << 31) || M < 8192) return 0;
  if (!is3) {  // 1x1: runs of 128*mt pixels inside one image; three stages must fit next to a second CTA
    const int planes = (d->cin + d->cout) / 8;
    int mt = planes <= 4 ? 4 : (planes <= 8 ? 2 : 1);
    const int64_t hw = (int64_t)d->h * d->w;
    while (mt > 1 && hw % (128 * mt)) mt >>= 1;
    return hw % (128 * mt) == 0 ? mt : 0;
  }
  int mt = (d->cin == 16 && d->cout == 16) ? 4 : 2;
  while (mt > 1 && d->w % (8 * mt)) mt >>= 1;
  return mt >= 2 ? mt : 0;
}
template <int CPA, int CPG, int MT, bool IS3>
static int wgrad3_setup(const iea_conv_desc* d, wg::P3& p, int& grid, uint32_t& smem) {
  using G = wg::G3<CPA, CPG, MT, IS3>;
  p.d = *d;
  p.hs = stored_res(*d, d->h);
  p.ws = stored_res(*d, d->w);
  if (IS3) { p.mtw = d->w / (8 * MT); p.mth = d->h / 16; }
  else { p.mtw = (int)(((int64_t)d->h * d->w) / (128 * MT)); p.mth = 1; }  // macro tiles per image
  p.n_macro = (int)(d->n * (int64_t)p.mtw * p.mth);
  p.fd_mtw = wg::make_fastdiv(p.mtw); p.fd_mth = wg::make_fastdiv(p.mth);
  p.stages = 3; p.depth = 3;
  if (p.stages * G::STAGE > 110 * 1024) { p.stages = 2; p.depth = 2; }
  smem = p.stages * G::STAGE;
  constexpr uint32_t fold = (uint32_t)((CPA / 2) * (CPG / 2)) * ((IS3 ? 72 : 8) + 4) * 32 * 4;
  if (smem < fold) smem = fold;
  const int sms = sm_count();
  const int occ = smem <= 110 * 1024 ? 2 : 1;
  grid = p.n_macro < sms * occ ? p.n_macro : sms * occ;
  return 0;
}
// macro-tile kernel: instance, parameters and grid (false: shape not handled by this kernel)
static bool wgrad3_plan(const iea_conv_desc* d, int g_dtype, int g_ld, WgradPlan& pl) {
  const int mt = wgrad3_mt(d, g_dtype, g_ld);
  if (!mt) return false;
  const int cpa = d->cin / 8, cpg = d->cout / 8;
  const bool is3 = d->ksize == 3;
#define IEA_W3(A_, G_, M_, I_)                                  \
  if (cpa == A_ && cpg == G_ && mt == M_ && is3 == I_) {        \
    wgrad3_setup<A_, G_, M_, I_>(d, pl.p3, pl.grid, pl.smem);   \
    pl.k3 = wg::wgrad3_kernel<A_, G_, M_, I_>;                  \
    return true;                                                \
  }
  IEA_W3(2, 2, 4, true) IEA_W3(2, 2, 2, true) IEA_W3(2, 4, 2, true) IEA_W3(4, 2, 2, true) IEA_W3(4, 4, 2, true)
  IEA_W3(2, 2, 4, false) IEA_W3(2, 2, 2, false) IEA_W3(2, 2, 1, false) IEA_W3(2, 4, 2, false) IEA_W3(2, 4, 1, false)
  IEA_W3(4, 2, 2, false) IEA_W3(4, 2, 1, false) IEA_W3(4, 4, 2, false) IEA_W3(4, 4, 1, false) IEA_W3(2, 8, 1, false)
  IEA_W3(8, 2, 1, false) IEA_W3(4, 8, 1, false) IEA_W3(8, 4, 1, false)
#undef IEA_W3
  return false;
}

int iea_conv_wgrad_tc_splits(const iea_conv_desc* d, int g_dtype, int g_ld);
int iea_conv_wgrad_tc(const iea_conv_desc* d, const void* g, int g_dtype, int g_ld, float* gpart, cudaStream_t s);

// first kernel that takes the shape: the 1-channel side (conv_c1.cu), the TMEM-accumulating tcgen05 kernel of the
// wide low-resolution layers (conv_wgrad_tc.cu), the macro-tile kernel, the generic mma.sync kernel
static WgradPlan wgrad_plan(const iea_conv_desc* d, int g_dtype, int g_ld) {
  WgradPlan pl;
  if ((pl.grid = iea_conv_c1_wgrad_grid(d, g_dtype, g_ld))) pl.kernel = WgradPlan::c1;
  else if ((pl.grid = iea_conv_wgrad_tc_splits(d, g_dtype, g_ld))) pl.kernel = WgradPlan::tc;
  else if (wgrad3_plan(d, g_dtype, g_ld, pl)) pl.kernel = WgradPlan::macro;
  else if (wgrad_mma_plan(d, g_dtype, g_ld, pl)) pl.kernel = WgradPlan::mma;
  else return pl;
  // the per-CTA partials + one slot for their sum (slice 0 after the call); the mma.sync kernels also need room
  // for their per-CTA column sums of g (grid * cout floats) behind them
  pl.slices = pl.grid + 1;
  if (pl.kernel == WgradPlan::macro || pl.kernel == WgradPlan::mma) {
    const int64_t total = (int64_t)d->cout * d->ksize * d->ksize * d->cin;
    pl.slices += (int)(((int64_t)pl.grid * d->cout + total - 1) / total);
  }
  return pl;
}

extern "C" int iea_conv_wgrad_mma_slices(const iea_conv_desc* d, int g_dtype, int g_ld) {
  return wgrad_plan(d, g_dtype, g_ld).slices;
}

extern "C" int iea_conv_wgrad_mma(const iea_conv_desc* d, const void* g, int g_dtype, int g_ld, float* gpart,
                                  float* dbias, iea_stream_t stream) {
  WgradPlan pl = wgrad_plan(d, g_dtype, g_ld);
  IEA_CHECK_ARG(pl.kernel != WgradPlan::none, "iea_conv_wgrad_mma: shape not handled (cin=%d cout=%d k=%d)", d->cin,
                d->cout, d->ksize);
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t total = (int64_t)d->cout * d->ksize * d->ksize * d->cin;
  float* parts = gpart + total;  // slices 1..grid hold the per-CTA partials, slice 0 receives their sum
  float* cs_parts = dbias ? gpart + (int64_t)(pl.grid + 1) * total : nullptr;
  int rb = (int)((total + 255) / 256);
  const char* what = "iea_conv_wgrad_mma";
  switch (pl.kernel) {
    case WgradPlan::none: break;
    case WgradPlan::tc:  // (0: the bias gradient is not produced by this path)
      return iea_conv_wgrad_tc(d, g, g_dtype, g_ld, gpart, s);
    case WgradPlan::c1: {
      const int rc = iea_conv_c1_wgrad(d, g, g_dtype, g_ld, parts, s);
      if (rc) return rc;
      cs_parts = nullptr;  // (the bias gradient is not produced by this path)
      what = "iea_conv_wgrad_mma(1-channel)";
      break;
    }
    case WgradPlan::macro:
      pl.p3.g = (const bf16*)g; pl.p3.g_ld = g_ld; pl.p3.gpart = parts; pl.p3.cs_parts = cs_parts;
      IEA_CHECK_ARG(cudaFuncSetAttribute(pl.k3, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem) == cudaSuccess,
                    "iea_conv_wgrad_mma(macro tile): launch set-up failed");
      pl.k3<<<pl.grid, 256, pl.smem, s>>>(pl.p3);
      what = "iea_conv_wgrad_mma(macro tile)";
      break;
    case WgradPlan::mma:
      IEA_CHECK_ARG(pl.km, "iea_conv_wgrad_mma: no kernel instance for %d block pairs", pl.pm.P);
      pl.pm.g = g; pl.pm.g_dtype = g_dtype; pl.pm.g_ld = g_ld; pl.pm.gpart = parts; pl.pm.cs_parts = cs_parts;
      IEA_CUDA(cudaFuncSetAttribute(pl.km, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
      pl.km<<<dim3(pl.grid, pl.grid_y), 256, pl.smem, s>>>(pl.pm);
      if (rb > 592) rb = 592;
      break;
  }
  wg::wgrad_reduce_kernel<<<rb, 256, 0, s>>>(parts, pl.grid, total, gpart);
  if (cs_parts) wg::wgrad_reduce_kernel<<<(d->cout + 255) / 256, 256, 0, s>>>(cs_parts, pl.grid, d->cout, dbias);
  const int rc = check_launch(what);
  return rc ? rc : (cs_parts ? 1 : 0);  // 1: dbias holds the column sums of g
}
