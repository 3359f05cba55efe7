// conv_wide.cu -- tcgen05 / TMEM kernel for the 1x1 convolutions with 64..256 output channels (every GBlock conv4:
// expansion + shortcut residual + batch-norm statistics, and the 256 -> 64 conv1 layers at 16^2 / 32^2).
//
// conv_tc2.cu runs these shapes with one 288-thread CTA per SM at Cin >= 64: one epilogue warp per SM sub-partition
// for a 128 x 64..256-channel tile, per-pixel residual loads and a second copy-out pass through shared memory, so
// the kernel waits on its epilogue at 30 % of the HBM rate.  This kernel moves every byte of the epilogue through
// TMA and gives it two groups of four warps on alternate tiles, following conv_thin.cu:
//   * one persistent 512-thread CTA per SM over a blocked run of 128-pixel tiles; the weight pack (<= 64 KB) is
//     bulk-loaded once and stays resident;
//   * inputs arrive by TMA box loads {8 channels, 128 pixels} into the K-major planes of a ring of 64-channel
//     k blocks; four warps apply the fused BN-affine + ReLU prologue in place;
//   * one thread issues the MMAs (M = 128, N = Cout, K = 16 in ascending channel order), into one of 2..4
//     accumulators in TMEM;
//   * epilogue warps 8..15: each group owns alternate tiles and works in {64 channels, 128 pixels} sub-tiles held
//     as 128B-swizzled images in a ring of NB buffers per group.  A same-resolution residual is TMA-loaded into
//     the image buffer itself (each thread reads its residual chunks and writes its output chunks at the same
//     place); a nearest-up2 residual lands as the contiguous run of source pixels under the tile in a ring of its
//     own.  The finished image leaves with one cp.async.bulk.tensor store.
// Results are bitwise those of conv_tc2: the same MMA instruction shape and order, the same fp32 epilogue
// arithmetic and bf16 rounding, and batch-norm partial sums taken from the rounded values in conv_tc2's order and
// stored in its per-tile slots.  Shapes outside iea_conv_wide_ok stay on conv_tc2.
#include "tc_common.cuh"
#include <string.h>
using namespace iea;

namespace wide {
using namespace tc;

constexpr int BM = 128;
constexpr int THREADS = 512;  // warp 0: TMA loads, warp 1: MMA, warps 4-7: prologue, warps 8-15: two epilogue groups
constexpr uint32_t PLANE = BM * 16;   // one 8-channel K-major plane of a tile
constexpr uint32_t IMG = BM * 128;    // one {64 channels, 128 pixels} output sub-tile

struct Params {
  iea_conv_desc d;
  const bf16* wtc;
  int n_tiles, hw, cpr, nkb, stages, nb, nacc, run;  // cpr: 8-channel planes per k block; run: up2 residual rows per sub-tile
  uint32_t w_bytes, stage_bytes, img_off, rr_off, stage_off, stat_off, ep_off, bar_off, tmem_cols, smem;
};

// RES: 0 none, 1 same resolution, 2 nearest-up2
template <int BN, int RES>
__global__ void __launch_bounds__(THREADS, 1) conv_wide_kernel(const __grid_constant__ Params p,
                                                               const __grid_constant__ CUtensorMap tmap_x,
                                                               const __grid_constant__ CUtensorMap tmap_y,
                                                               const __grid_constant__ CUtensorMap tmap_r) {
  constexpr int NSB = BN / 64;  // sub-tiles per tile
  extern __shared__ uint8_t smem_raw[];
  const iea_conv_desc& d = p.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // the 128B swizzle of the images works on absolute shared addresses: align the layout to 1 KB
  const uint32_t sraw = smem_u32(smem_raw);
  const uint32_t sbase = (sraw + 1023u) & ~1023u;
  uint8_t* const smem = smem_raw + (sbase - sraw);
  const int S = p.stages, NB = p.nb, NACC = p.nacc;
  // barriers: full[S] | land[S] | empty[S] | tfull[NACC] | tempty[NACC] | w | res[2][NB] | TMEM slot
  const uint32_t full0 = sbase + p.bar_off, land0 = full0 + 8u * S, empty0 = land0 + 8u * S;
  const uint32_t tfull0 = empty0 + 8u * S, tempty0 = tfull0 + 8u * NACC, w_bar = tempty0 + 8u * NACC;
  const uint32_t res0 = w_bar + 8u;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + p.bar_off + 8 * (3 * S + 2 * NACC + 1 + 2 * NB));
  const bool affine = d.in_scale != nullptr, relu = d.in_relu != 0, pro = affine || relu;

  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(full0 + 8 * s, 4); mbar_init(land0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
    for (int a = 0; a < NACC; ++a) { mbar_init(tfull0 + 8 * a, 1); mbar_init(tempty0 + 8 * a, 4); }
    mbar_init(w_bar, 1);
    for (int i = 0; i < 2 * NB; ++i) mbar_init(res0 + 8 * i, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // blocked partition: each CTA owns a contiguous run of tiles (the per-image prologue constants rarely change)
  const int t_base = p.n_tiles / (int)gridDim.x, t_rem = p.n_tiles % (int)gridDim.x;
  const int my_n = t_base + ((int)blockIdx.x < t_rem ? 1 : 0);
  const int tile0 = (int)blockIdx.x * t_base + ((int)blockIdx.x < t_rem ? (int)blockIdx.x : t_rem);
  const int KB = p.cpr * 8, n_items = my_n * p.nkb;

  if (warp == 0) {
    // ===================== TMA producer: weights once, then one k block of one tile per ring slot =====================
    if (lane == 0) {
      mbar_expect_tx(w_bar, p.w_bytes);
      for (uint32_t off = 0; off < p.w_bytes; off += 32768) {
        const uint32_t nb = p.w_bytes - off < 32768 ? p.w_bytes - off : 32768;
        bulk_g2s(sbase + off, (const uint8_t*)p.wtc + off, nb, w_bar);
      }
      const uint64_t tm = reinterpret_cast<uint64_t>(&tmap_x);
      uint32_t s = 0, ph = 0;
      for (int it = 0; it < n_items; ++it) {
        const int t = it / p.nkb, kb = it - t * p.nkb;
        mbar_wait(empty0 + 8 * s, ph ^ 1);
        const uint32_t a = sbase + p.stage_off + s * p.stage_bytes, bar = land0 + 8 * s;
        mbar_expect_tx(bar, p.stage_bytes);
        const int m0 = (tile0 + t) * BM;
        for (int k = 0; k < p.cpr; ++k)
          asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                       ::"r"(a + k * PLANE), "l"(tm), "r"(kb * KB + k * 8), "r"(m0), "r"(bar) : "memory");
        if (++s == (uint32_t)S) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: the order of conv_tc2 (k block, then 16-channel step) =====================
    constexpr uint32_t ID = idesc(BN, false, false);
    constexpr uint32_t LBO_B = BN * 16;
    const uint64_t da_base = make_desc(sbase + p.stage_off, PLANE, 128);
    const uint64_t db_base = make_desc(sbase, LBO_B, 128);
    const uint32_t stage16 = p.stage_bytes >> 4;
    mbar_wait(w_bar, 0);
    uint32_t s = 0, ph = 0;
    for (int t = 0; t < my_n; ++t) {
      const int a = t % NACC;
      mbar_wait(tempty0 + 8 * a, ((t / NACC) & 1) ^ 1);
      tc_fence_after();
      const uint32_t tacc = tmem_base + a * BN;
      for (int kb = 0; kb < p.nkb; ++kb) {
        mbar_wait((pro ? full0 : land0) + 8 * s, ph);
        tc_fence_after();
        if (elect_one()) {
          for (int j = 0; j < p.cpr / 2; ++j)
            tc_mma(tacc, da_base + (s * stage16 + 2 * j * (PLANE >> 4)), db_base + (uint32_t)(kb * p.cpr + 2 * j) * (LBO_B >> 4), ID,
                   (kb > 0 || j > 0) ? 1u : 0u);
          tc_commit(empty0 + 8 * s);
        }
        __syncwarp();
        if (++s == (uint32_t)S) { s = 0; ph ^= 1; }
      }
      if (elect_one()) tc_commit(tfull0 + 8 * a);
      __syncwarp();
    }
  } else if (warp >= 4 && warp < 8) {
    // ===================== fused prologue, in place on the landed planes =====================
    if (pro) {
      // a thread walks one plane: consecutive threads take consecutive pixels (conflict-free 16-byte accesses)
      const int pt = tid - 128;
      const int tpp = BM / p.cpr;
      const int k = pt / tpp, px0 = pt - k * tpp;
      __nv_bfloat162 sc2[4], sh2[4];
      const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
      int ss_n = -1, ss_ci = -1;
      uint32_t s = 0, ph = 0;
      for (int it = 0; it < n_items; ++it) {
        const int t = it / p.nkb, kb = it - t * p.nkb;
        const int ci = kb * KB + k * 8;
        if (affine) {
          const int nn = (tile0 + t) * BM / p.hw;  // (images are whole tiles)
          if (nn != ss_n || ci != ss_ci) {
            const int64_t si = (d.in_bcast ? 0 : (int64_t)nn * d.cin) + ci;
            const float4 a0 = *reinterpret_cast<const float4*>(d.in_scale + si), a1 = *reinterpret_cast<const float4*>(d.in_scale + si + 4);
            const float4 b0 = *reinterpret_cast<const float4*>(d.in_shift + si), b1 = *reinterpret_cast<const float4*>(d.in_shift + si + 4);
            sc2[0] = __floats2bfloat162_rn(a0.x, a0.y); sc2[1] = __floats2bfloat162_rn(a0.z, a0.w);
            sc2[2] = __floats2bfloat162_rn(a1.x, a1.y); sc2[3] = __floats2bfloat162_rn(a1.z, a1.w);
            sh2[0] = __floats2bfloat162_rn(b0.x, b0.y); sh2[1] = __floats2bfloat162_rn(b0.z, b0.w);
            sh2[2] = __floats2bfloat162_rn(b1.x, b1.y); sh2[3] = __floats2bfloat162_rn(b1.z, b1.w);
            ss_n = nn; ss_ci = ci;
          }
        }
        mbar_wait(land0 + 8 * s, ph);
        uint8_t* a = smem + p.stage_off + s * p.stage_bytes + k * PLANE + px0 * 16;
        uint4 v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (i < p.cpr) v[i] = *reinterpret_cast<const uint4*>(a + i * tpp * 16);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
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
        for (int i = 0; i < 8; ++i)
          if (i < p.cpr) *reinterpret_cast<uint4*>(a + i * tpp * 16) = v[i];
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(full0 + 8 * s);
        if (++s == (uint32_t)S) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp >= 8) {
    // ===================== epilogue: two groups of 4 warps on alternate tiles; TMEM lane = pixel =====================
    const int grp = (warp - 8) >> 2;
    const int q = warp & 3, et = q * 32 + lane;
    float* ep_sc = reinterpret_cast<float*>(smem + p.ep_off);
    float* ep_bs = ep_sc + BN;
    if (grp == 0)  // the per-channel constants exactly as conv_tc2 stages them
      for (int c = et; c < BN; c += 128) {
        float s_ = 1.f, b_ = 0.f;
        if (c < d.cout) {
          if (d.out_scale) s_ = d.out_scale[d.out_scale_stride ? c : 0];
          if (d.bias) b_ = d.bias[c];
        }
        ep_sc[c] = s_; ep_bs[c] = b_;
      }
    asm volatile("bar.sync 3, 256;" ::: "memory");
    auto bar_grp = [&]() {
      if (grp == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
      else asm volatile("bar.sync 2, 128;" ::: "memory");
    };
    const bool has_stats = d.stats != nullptr;
    float* const fold = reinterpret_cast<float*>(smem + p.stat_off) + grp * (BM / 8 * 8 * 2 * 8);  // [step][BN][2] = 8 KB
    const uint32_t img0 = sbase + p.img_off + grp * NB * IMG;
    uint8_t* const img0_ptr = smem + p.img_off + grp * NB * IMG;
    const uint32_t rslot = RES == 2 ? (uint32_t)p.run * 128 : IMG;
    const uint32_t rr0 = RES == 2 ? sbase + p.rr_off + grp * NB * rslot : img0;
    const uint8_t* const rr0_ptr = RES == 2 ? smem + p.rr_off + grp * NB * rslot : img0_ptr;
    const uint32_t rbar0 = res0 + 8u * grp * NB;
    const int sw = et & 7;  // 128B swizzle: chunk c of row r sits at r * 128 + ((c ^ (r & 7)) << 4)
    // row of this pixel's nearest-up2 source in the run of source pixels under the tile
    int rr_row = et;
    if (RES == 2) rr_row = d.w >= BM ? et >> 1 : ((et / d.w) >> 1) * (d.w >> 1) + ((et % d.w) >> 1);
    const int n_sub = my_n > grp ? ((my_n - grp + 1) >> 1) * NSB : 0;  // sub-tiles of this group
    auto res_issue = [&](int j) {  // one thread: residual of this group's sub-tile j into ring slot j % NB
      if (RES == 0 || j >= n_sub) return;
      const int m0 = (tile0 + grp + 2 * (j / NSB)) * BM, c0 = (j % NSB) * 64;
      int src0 = m0;
      if (RES == 2) {
        const int nn = m0 / p.hw, pix = m0 - nn * p.hw, oh = pix / d.w, ow = pix - oh * d.w;
        src0 = nn * (p.hw >> 2) + (oh >> 1) * (d.w >> 1) + (ow >> 1);
      }
      const uint32_t bar = rbar0 + 8 * (j % NB);
      mbar_expect_tx(bar, rslot);
      asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                   ::"r"(rr0 + (j % NB) * rslot), "l"(reinterpret_cast<uint64_t>(&tmap_r)), "r"(c0), "r"(src0), "r"(bar) : "memory");
    };
    if (RES && et == 0)
      for (int j = 0; j < NB - 1; ++j) res_issue(j);
    // statistics of a sub-tile, in conv_tc2's order: with cg = BN / 8 chunks per row and step = 128 / cg, part r0 of
    // chunk g sums rows r0, r0 + step, ... (cg rows); the 8 x step (chunk, part) pairs of a sub-tile rotate over the
    // group's threads from one sub-tile to the next
    constexpr int CG = BN / 8, STEP = BM / CG, PAIRS = 8 * STEP;
    int i = 0;  // sub-tile counter of this group
    for (int t = grp; t < my_n; t += 2) {
      const int a = t % NACC;
      const int tile = tile0 + t, m0 = tile * BM;
      mbar_wait(tfull0 + 8 * a, (t / NACC) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int sb = 0; sb < NSB; ++sb, ++i) {
        const int slot = i % NB;
        uint8_t* const img = img0_ptr + slot * IMG;
        if (RES) mbar_wait(rbar0 + 8 * slot, (i / NB) & 1);
        uint32_t raw[4][16];
#pragma unroll
        for (int cb = 0; cb < 4; ++cb)
          tmem_ld16_issue(tmem_base + ((uint32_t)(q * 32) << 16) + a * BN + sb * 64 + cb * 16, raw[cb]);
        tmem_ld_wait();
        if (sb == NSB - 1) {  // accumulator drained: the MMA warp may start the tile after next
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tempty0 + 8 * a);
        }
        const uint8_t* const rrow = RES == 2 ? rr0_ptr + slot * rslot + rr_row * 128 : img + et * 128;
        const int rsw = RES == 2 ? (rr_row & 7) : sw;
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
          const int c0 = sb * 64 + cb * 16;
          float2 v[8];
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 s4 = *reinterpret_cast<const float4*>(ep_sc + c0 + 4 * j4);
            const float4 b4 = *reinterpret_cast<const float4*>(ep_bs + c0 + 4 * j4);
            v[2 * j4] = ffma2(make_float2(__uint_as_float(raw[cb][4 * j4]), __uint_as_float(raw[cb][4 * j4 + 1])),
                              make_float2(s4.x, s4.y), make_float2(b4.x, b4.y));
            v[2 * j4 + 1] = ffma2(make_float2(__uint_as_float(raw[cb][4 * j4 + 2]), __uint_as_float(raw[cb][4 * j4 + 3])),
                                  make_float2(s4.z, s4.w), make_float2(b4.z, b4.w));
          }
          if (RES) {
            const uint4 r0 = *reinterpret_cast<const uint4*>(rrow + (((2 * cb) ^ rsw) << 4));
            const uint4 r1 = *reinterpret_cast<const uint4*>(rrow + (((2 * cb + 1) ^ rsw) << 4));
            const uint32_t w[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fadd2(v[j], bf2_to_f2(w[j]));
          }
          uint8_t* const row = img + et * 128;
          *reinterpret_cast<uint4*>(row + (((2 * cb) ^ sw) << 4)) =
              make_uint4(pack2(v[0].x, v[0].y), pack2(v[1].x, v[1].y), pack2(v[2].x, v[2].y), pack2(v[3].x, v[3].y));
          *reinterpret_cast<uint4*>(row + (((2 * cb + 1) ^ sw) << 4)) =
              make_uint4(pack2(v[4].x, v[4].y), pack2(v[5].x, v[5].y), pack2(v[6].x, v[6].y), pack2(v[7].x, v[7].y));
        }
        fence_async_smem();
        // the buffer the group writes next must have been read by its store (issued NB - 1 sub-tiles ago)
        if (et == 0) {
          if (NB == 2) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          else asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        }
        bar_grp();
        if (et == 0) {
          asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                       ::"l"(reinterpret_cast<uint64_t>(&tmap_y)), "r"(sb * 64), "r"(m0), "r"(img0 + slot * IMG) : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          if (RES) {
            // the slot of sub-tile i + NB - 1 is the one of sub-tile i - 1: its store must have read it (same-resolution
            // residuals land in the image buffer), and every thread is past its residual reads (bar_grp above)
            if (RES == 1 && NB > 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            res_issue(i + NB - 1);
          }
        }
        if (has_stats) {
          const int e = (et - sb * PAIRS) & (BM - 1);
          if (e < PAIRS) {
            const int g = e & 7, r0 = e >> 3;
            float2 s1[4], s2[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) { s1[j] = make_float2(0.f, 0.f); s2[j] = s1[j]; }
#pragma unroll 4
            for (int k = 0; k < CG; ++k) {
              const int r = r0 + k * STEP;
              const uint4 c = *reinterpret_cast<const uint4*>(img + r * 128 + ((g ^ (r & 7)) << 4));
              const uint32_t w[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) { const float2 f = bf2_to_f2(w[j]); s1[j] = fadd2(s1[j], f); s2[j] = ffma2(f, f, s2[j]); }
            }
            float4* st4 = reinterpret_cast<float4*>(fold + (r0 * BN + sb * 64 + g * 8) * 2);
#pragma unroll
            for (int j = 0; j < 4; ++j) st4[j] = make_float4(s1[j].x, s2[j].x, s1[j].y, s2[j].y);
          }
        }
      }
      if (has_stats) {  // fixed-order fold over the parts into this tile's slot
        bar_grp();
        for (int c = et; c < BN * 2; c += 128) {
          float s_ = 0.f;
          for (int part = 0; part < STEP; ++part) s_ += fold[part * BN * 2 + c];
          d.stats[(int64_t)tile * d.cout * 2 + c] = s_;
        }
      }
    }
    if (et == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_free(tmem_base, p.tmem_cols);
  }
}

}  // namespace wide

int iea_conv_tc_base_ok(const iea_conv_desc* d, int padded);
int iea_conv_tc2_ok(const iea_conv_desc* d);

// {cols channels, pixels} view of an NHWC bf16 tensor with `ld` elements per pixel, boxes {box_c, box_px}
static bool wide_tensor_map(CUtensorMap* tm, const void* base, int cols, int64_t px, int ld, int box_c, int box_px,
                            CUtensorMapSwizzle sw) {
  tc::encode_tiled_fn enc = tc::tma_encoder();
  if (!enc) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)px};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  const cuuint32_t box[2] = {(cuuint32_t)box_c, (cuuint32_t)box_px}, es[2] = {1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
             sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct WidePlan {
  wide::Params p;
  int grid;
  alignas(64) CUtensorMap tx, ty, tr;
};

// Envelope, shared-memory plan and tensor maps of one layer; false: the layer stays on conv_tc2.  Both the router
// and the launcher call it, so a shape that cannot be planned never reaches the launch.
static bool wide_plan(const iea_conv_desc* d, WidePlan& w) {
  if (!iea_conv_tc_base_ok(d, 0) || !iea_conv_tc2_ok(d)) return false;
  if (d->ksize != 1 || d->in_mode != IEA_IN_DIRECT || d->y_dtype != IEA_BF16) return false;
  if (d->cout != 64 && d->cout != 128 && d->cout != 256) return false;
  if (d->cin != 16 && d->cin != 32 && d->cin != 64 && d->cin != 128 && d->cin != 256) return false;
  const int64_t hw = (int64_t)d->h * d->w, M = d->n * hw;
  if (hw % wide::BM || M >= (1ll << 31)) return false;  // a tile never straddles two images
  if (d->stats && d->n % 40) return false;
  if (d->acc_c0 >= 0 || d->act != IEA_ACT_NONE) return false;
  int res = 0, run = 0;
  if (d->res) {
    if (d->res_dtype != IEA_BF16 || d->res_c != d->cout || d->res_ld < d->res_c) return false;
    if (d->res_mode == IEA_IN_DIRECT) {
      res = 1;
    } else if (d->res_mode == IEA_IN_UP2) {
      // the source pixels under a tile are one contiguous run: 64 at w >= 128, 32 at w = 16, 32, 64
      if (d->h % 2 || !(d->w % 128 == 0 || (d->w <= 64 && 128 % d->w == 0 && d->w >= 2))) return false;
      res = 2;
      run = d->w >= 128 ? 64 : 32;
    } else {
      return false;
    }
  }
  memset(&w, 0, sizeof(w));
  wide::Params& p = w.p;
  p.d = *d;
  p.wtc = (const bf16*)d->wpack_tc;
  p.n_tiles = (int)(M / wide::BM);
  p.hw = (int)hw;
  const int kb = d->cin < 64 ? d->cin : 64;
  p.cpr = kb / 8;
  p.nkb = d->cin / kb;
  p.run = run;
  p.w_bytes = (uint32_t)(d->cout * d->cin * 2);
  p.stage_bytes = p.cpr * wide::PLANE;
  p.nacc = d->cout == 256 ? 2 : 4;
  p.tmem_cols = tmem_cols_for(p.nacc * d->cout);
  // shared memory: weights | images [2][NB] | up2 residual ring [2][NB] | input ring [S] | statistics fold [2] |
  // epilogue constants | barriers.  Three images per group when the input ring still keeps >= 48 KB in flight,
  // else two with >= 32 KB (and never fewer than three k blocks).
  const uint32_t limit = 227 * 1024;
  bool ok = false;
  for (int nb = 3; nb >= 2 && !ok; --nb) {
    p.nb = nb;
    p.img_off = (p.w_bytes + 1023) / 1024 * 1024;
    p.rr_off = p.img_off + 2 * nb * wide::IMG;
    p.stage_off = p.rr_off + (res == 2 ? 2 * nb * run * 128 : 0);
    const uint32_t fixed = p.stage_off + (d->stats ? 2 * 8192 : 0) + 2 * d->cout * 4 + 512 + 1024;  // (+ 1 KB alignment)
    if (fixed >= limit) continue;
    int s = (int)((limit - fixed) / p.stage_bytes);
    if (s > 12) s = 12;
    if (s < 3 || s * p.stage_bytes < (nb == 3 ? 48u : 32u) * 1024) continue;
    p.stages = s;
    p.stat_off = p.stage_off + s * p.stage_bytes;
    p.ep_off = p.stat_off + (d->stats ? 2 * 8192 : 0);
    p.bar_off = p.ep_off + 2 * d->cout * 4;
    p.smem = p.bar_off + 512 + 1024;
    ok = true;
  }
  if (!ok) return false;
  const int64_t M_res = res == 2 ? d->n * (hw / 4) : M;
  if (!wide_tensor_map(&w.tx, d->x, d->cin, M, d->x_ld, 8, wide::BM, CU_TENSOR_MAP_SWIZZLE_NONE)) return false;
  if (!wide_tensor_map(&w.ty, d->y, d->cout, M, d->y_ld, 64, wide::BM, CU_TENSOR_MAP_SWIZZLE_128B)) return false;
  if (res && !wide_tensor_map(&w.tr, d->res, d->res_c, M_res, d->res_ld, 64, res == 2 ? run : wide::BM, CU_TENSOR_MAP_SWIZZLE_128B))
    return false;
  const int sms = sm_count();
  w.grid = p.n_tiles < sms ? p.n_tiles : sms;
  return true;
}

int iea_conv_wide_ok(const iea_conv_desc* d) {
  WidePlan w;
  return wide_plan(d, w) ? 1 : 0;
}

int iea_conv_fprop_wide(const iea_conv_desc* d, cudaStream_t s) {
  WidePlan w;
  IEA_CHECK_ARG(wide_plan(d, w), "iea_conv_fprop(tcgen05 wide): layer outside the kernel's envelope (cin=%d cout=%d)", d->cin,
                d->cout);
  const int res = !d->res ? 0 : (d->res_mode == IEA_IN_UP2 ? 2 : 1);
  auto run = [&](auto kern) -> int {
    IEA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)w.p.smem));
    kern<<<w.grid, wide::THREADS, w.p.smem, s>>>(w.p, w.tx, w.ty, w.tr);
    return check_launch("iea_conv_fprop(tcgen05 wide)");
  };
#define IEA_WIDE_CASE(B_, R_) \
  if (d->cout == B_ && res == R_) return run(wide::conv_wide_kernel<B_, R_>);
  IEA_WIDE_CASE(64, 0) IEA_WIDE_CASE(64, 1) IEA_WIDE_CASE(64, 2)
  IEA_WIDE_CASE(128, 0) IEA_WIDE_CASE(128, 1) IEA_WIDE_CASE(128, 2)
  IEA_WIDE_CASE(256, 0) IEA_WIDE_CASE(256, 1) IEA_WIDE_CASE(256, 2)
#undef IEA_WIDE_CASE
  set_error("iea_conv_fprop(tcgen05 wide): no kernel for cout=%d", d->cout);
  return -2;
}
