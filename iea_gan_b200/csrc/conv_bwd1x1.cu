// conv_bwd1x1.cu -- the WHOLE backward of a 1x1 SNConv2d layer as one tcgen05 / TMEM kernel.
//
// Forward (layers.py:198-206 with the fused prologue / epilogue of this build):
//     xt = relu(x * scale[n,c] + shift[n,c])          (ccbn / bn apply + ReLU, or a plain ReLU, or nothing)
//     y  = xt . W^T / sigma + b                       (+ batch-norm statistics of y taken by the epilogue)
// Backward, per pixel row and with NO spatial halo (that is what makes a 1x1 layer fusable end to end):
//     geff = g + ds1[e,co] + 2 y ds2[e,co]            adjoint of the statistics epilogue   (was iea_conv_out_bwd)
//     dW  += geff^T . xt ,  db += colsum(geff)        weight / bias gradient                (was iea_conv_wgrad_mma)
//     da   = geff . W / sigma                         data gradient                         (was iea_conv_fprop on the dgrad pack)
//     gm   = da * 1[x*scale+shift > 0]
//     dx   = beta*dx + gm * scale ; dscale[n,c] = sum_px gm*x ; dshift[n,c] = sum_px gm     (was iea_conv_input_bwd)
// Unfused these are four passes that move 5 (Cout + Cin) channel-rows per pixel through HBM (write geff, read it
// twice, write da, read it, read x twice, ...); here g, y and x are read once and dx is written once:
// 2 (Cout + Cin).  The 1x1 layers are half of all convolutions of G and D and their backward was ~52 ms of the
// 157 ms train step (8 events).
//
// One persistent CTA per SM, 544 threads.  Warps 0-3 and 4-7 are two producer groups that stage alternate tiles
// (cp.async into UMMA planes, then the elementwise transforms IN PLACE in shared memory: a 128-pixel tile of a thin
// layer is only 12-40 KB, so the per-tile chain wait -> barrier -> transform -> fence -> hand-over of ONE group cannot
// keep up with HBM; two groups overlap it), warps 8-11 and 12-15 are two epilogue groups that take alternate tiles
// (each owns one of the two D1 accumulators), warp 16 issues the MMAs.  Per 128-pixel tile:
//     MMA1  D1[128 px][Cin]        = geff (K-major A, K = Cout)  x  Wd (K-major B, resident)          -> da
//     MMA2  D2[128 (co)][Cin + 16] += geff^T (MN-major A, K = 128 px)  x  [xt | 1] (MN-major B)       -> dW, db
// D2 stays in TMEM for ALL tiles of the CTA (fp32) and is written once at the end; D1 is double buffered against the
// epilogue.  The same staged images serve both products (pixels are the rows of every plane: K-major for MMA1,
// MN-major for MMA2), so nothing is transposed.  Deterministic: per-CTA partials, fixed-order reduces.
#include "tc_common.cuh"
using namespace iea;

namespace wg {
__global__ void wgrad_reduce_kernel(const float* gpart, int nsplit, int64_t total, float* out);
}

namespace b1 {
using namespace tc;

constexpr int BM = 128;
constexpr int THREADS = 544;   // warps 0-3 / 4-7: producer groups; 8-11 / 12-15: epilogue groups; warp 16: MMA issuer
constexpr uint32_t PL = BM * 16 + 16;  // plane pitch: 128 rows x 16 B + 16 B skew

struct Params {
  iea_conv_desc d;          // forward geometry: x, x_ld, cin, cout, in_scale / in_shift / in_relu / in_bcast
  iea_bwd1x1_args a;
  int64_t M;
  int hw, tpi, tiles, tpc, nbuf, want_w, want_x, want_ss, has_ds, g_planes, x_planes, sl_img, inplace;
  uint32_t off_y, off_x, off_xt, off_tab, buf_bytes, off_w, off_stage, off_bar, stage_ld, tmem_cols;
};

__device__ __forceinline__ uint64_t desc_mn(uint32_t addr) { return make_desc(addr, 128, PL); }

__global__ void __launch_bounds__(THREADS, 1) bwd1x1_kernel(const Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const iea_conv_desc& d = p.d;
  const iea_bwd1x1_args& a = p.a;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + p.off_bar;
  // barriers: full[8], empty[8], d1_full[2], d1_empty[2], d2_full
  auto full = [&](int b) { return bar0 + 8u * b; };
  auto empty = [&](int b) { return bar0 + 64u + 8u * b; };
  auto d1_full = [&](int b) { return bar0 + 128u + 8u * b; };
  auto d1_empty = [&](int b) { return bar0 + 144u + 8u * b; };
  const uint32_t d2_full = bar0 + 160u;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + p.off_bar + 176);
  const int cin = d.cin, cout = d.cout;
  if (tid == 0) {
    for (int b = 0; b < 8; ++b) {
      mbar_init(full(b), 4);
      mbar_init(empty(b), 1 + 4);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(d1_full(b), 1);
      mbar_init(d1_empty(b), 4);
    }
    mbar_init(d2_full, 1);
    fence_mbar_init();
  }
  if (warp == 16) tmem_alloc(smem_u32(tmem_slot), p.tmem_cols);
  // one-time shared-memory images: the resident dgrad weights and the ones plane behind xt (bias-gradient column of
  // MMA2).  Neither geff^T (A of MMA2, 128 rows) nor [xt | 1] (B, Cin + 16 columns) is padded: the descriptors simply
  // run on into whatever follows the real planes -- those operand rows / columns only produce accumulator rows >= Cout
  // and columns > Cin, which nobody reads.
  {
    const uint4* wsrc = reinterpret_cast<const uint4*>(a.wd_tc);
    uint4* wdst = reinterpret_cast<uint4*>(smem + p.off_w);
    for (int e = tid; e < cout * cin / 8; e += THREADS) wdst[e] = __ldg(wsrc + e);
    for (int e = tid; e < p.nbuf * BM; e += THREADS)  // plane x_planes of xt: channel `cin` = 1.0 (bf16 0x3F80)
      *reinterpret_cast<uint4*>(smem + (e / BM) * p.buf_bytes + p.off_xt + p.x_planes * PL + (e % BM) * 16) =
          make_uint4(0x3F80u, 0, 0, 0);
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int t0 = blockIdx.x * p.tpc;
  int t1 = t0 + p.tpc;
  if (t1 > p.tiles) t1 = p.tiles;
  const int ntile = t1 > t0 ? t1 - t0 : 0;
  const int nbuf = p.nbuf;

  if (warp == 16) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int b = 0;
      uint32_t ph = 0;  // ring slot of tile i and the parity of its fill
      for (int i = 0; i < ntile; ++i) {
        const int db = i & 1;
        mbar_wait(full(b), ph);
        if (p.want_x && i >= 2) mbar_wait(d1_empty(db), ((i >> 1) - 1) & 1);  // group db released its accumulator
        tc_fence_after();
        const uint32_t g0 = sbase + b * p.buf_bytes;
        if (p.want_x) {
          const uint32_t w0 = sbase + p.off_w, id1 = idesc(cin, false, false);
          for (int j = 0; j < cout / 16; ++j)
            tc_mma(tmem + db * cin, make_desc(g0 + 2 * j * PL, PL, 128), make_desc(w0 + 2 * j * (cin * 16), cin * 16, 128), id1,
                   j > 0 ? 1u : 0u);
          tc_commit(d1_full(db));
        }
        if (p.want_w) {
          const uint32_t x0 = g0 + p.off_xt, id2 = idesc(cin + 16, true, true);
#pragma unroll
          for (int j = 0; j < BM / 16; ++j)
            tc_mma(tmem + 2 * cin, desc_mn(g0 + j * 256), desc_mn(x0 + j * 256), id2, (i > 0 || j > 0) ? 1u : 0u);
        }
        tc_commit(empty(b));  // every MMA that read buffer b has completed when this arrives
        if (++b == nbuf) { b = 0; ph ^= 1u; }
      }
      tc_commit(d2_full);
    }
  } else if (warp < 8) {
    // ===================== producers: two groups on alternate tiles; stage g, y, x and transform in place ===========
    const int pg = warp >> 2, pt = tid & 127;
    const bf16* gp = (const bf16*)a.g;
    const bf16* yp = (const bf16*)a.y;
    const bf16* xp = (const bf16*)d.x;
    // 128 % planes == 0, so a thread always handles the SAME 8-channel chunk (plane) of g / y and of x, at rows
    // r0, r0 + 128 / planes, ...: no index arithmetic inside the loops and the per-channel constants of the chunk
    // (scale / shift, ds1 / 2 ds2) live in registers, reloaded when the image changes (one image per tile).
    const int gc = pt % p.g_planes, gr0 = pt / p.g_planes, grs = BM / p.g_planes;
    const int xc = pt % p.x_planes, xr0 = pt / p.x_planes, xrs = BM / p.x_planes;
    const uint32_t g_so = gc * PL + gr0 * 16, x_so = xc * PL + xr0 * 16;  // shared-memory offsets inside a plane set
    const int64_t g_go = (int64_t)gr0 * a.g_ld + gc * 8, y_go = (int64_t)gr0 * a.y_ld + gc * 8, x_go = (int64_t)xr0 * d.x_ld + xc * 8;
    const int64_t g_gs = (int64_t)grs * a.g_ld, y_gs = (int64_t)grs * a.y_ld, x_gs = (int64_t)xrs * d.x_ld;
    const int kmax = ntile > pg ? (ntile - pg + 1) >> 1 : 0;  // this group's tiles: i = pg + 2 k
    // ring state of the NEXT tile to request: slot, how often the slot has been filled before, first pixel row
    int is_b = pg % nbuf, is_u = pg / nbuf;
    int64_t is_m0 = (int64_t)(t0 + pg) * BM;
    auto issue = [&]() {  // cp.async of the group's next tile into its slot (waits until the slot is free)
      // (one slot shared by both groups: this group skips the other group's phase, and a parity wait cannot tell
      //  release u - 2 from release u -- pass release u - 1 first)
      if (nbuf == 1 && is_u > 1) mbar_wait(empty(0), is_u & 1);
      if (is_u > 0) mbar_wait(empty(is_b), (is_u - 1) & 1);
      const uint32_t bu = sbase + is_b * p.buf_bytes;
      {
        const bf16* src = gp + is_m0 * a.g_ld + g_go;
        uint32_t dst = bu + g_so;
#pragma unroll 1
        for (int k = 0; k < p.g_planes; ++k, src += g_gs, dst += grs * 16) cp16(dst, src);
      }
      if (p.has_ds) {
        const bf16* src = yp + is_m0 * a.y_ld + y_go;
        uint32_t dst = bu + p.off_y + g_so;
#pragma unroll 1
        for (int k = 0; k < p.g_planes; ++k, src += y_gs, dst += grs * 16) cp16(dst, src);
      }
      {
        const bf16* src = xp + is_m0 * d.x_ld + x_go;
        uint32_t dst = bu + p.off_x + x_so;
#pragma unroll 2
        for (int k = 0; k < p.x_planes; ++k, src += x_gs, dst += xrs * 16) cp16(dst, src);
      }
      cp_async_commit();
      is_m0 += 2 * BM;
      is_b += 2;
      while (is_b >= nbuf) { is_b -= nbuf; ++is_u; }
    };
    // A group owns nbuf / 2 slots (even nbuf) and requests PDg of its own tiles ahead, always AFTER a hand-over.  The
    // request after the hand-over of own tile k (tile k + PDg) recycles the slot of own tile k + PDg - nbuf / 2 <= k - 1,
    // which has had a whole iteration to be consumed; PDg - 1 requests are in flight while a tile is transformed and the
    // other group covers the rest.  With two slots a group works strictly load -> transform -> hand over.
    const int PDg = nbuf >= 8 ? 3 : (nbuf >= 6 ? 2 : (nbuf >= 4 ? 1 : 0));
    for (int q = 0; q < PDg && q < kmax; ++q) issue();
    float sc[8], sh[8], e1[8], e2[8], tsc = 1.f, tsh = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) { sc[j] = 1.f; sh[j] = 0.f; e1[j] = 0.f; e2[j] = 0.f; }
    const int img_per_event = p.has_ds ? (int)(a.rows_per_event / p.hw) : 1;
    int n = (t0 + pg) / p.tpi, rem = (t0 + pg) - n * p.tpi, cur_n = -1, b = pg % nbuf;
    for (int k = 0; k < kmax; ++k) {
      if (PDg == 0) issue();
      uint8_t* buf = smem + b * p.buf_bytes;
      if (n != cur_n) {  // per-image constants (one image, one event per tile)
        cur_n = n;
        if (d.in_scale) {
          const int64_t si = d.in_bcast ? 0 : (int64_t)n * cin;
#pragma unroll
          for (int j = 0; j < 8; ++j) { sc[j] = __ldg(d.in_scale + si + xc * 8 + j); sh[j] = __ldg(d.in_shift + si + xc * 8 + j); }
          if (pt < cin) { tsc = __ldg(d.in_scale + si + pt); tsh = __ldg(d.in_shift + si + pt); }
        }
        if (p.has_ds) {
          const int64_t ei = (int64_t)(n / img_per_event) * cout + gc * 8;
#pragma unroll
          for (int j = 0; j < 8; ++j) { e1[j] = __ldg(a.ds1 + ei + j); e2[j] = 2.f * __ldg(a.ds2 + ei + j); }
        }
      }
      if (d.in_scale && pt < cin) {  // the epilogue walks all channels of a row: it gets the table in the buffer
        float* tab = reinterpret_cast<float*>(buf + p.off_tab);
        tab[pt] = tsc;
        tab[cin + pt] = tsh;
      }
      {  // the copies of this tile have landed; the younger requests stay in flight
        const int pend = PDg > 0 ? PDg - 1 : 0;
        const int younger = kmax - 1 - k < pend ? kmax - 1 - k : pend;
        if (younger <= 0) cp_async_wait<0>();
        else if (younger == 1) cp_async_wait<1>();
        else cp_async_wait<2>();
      }
      // every copy of the group and the table are visible to the group
      if (pg == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
      else asm volatile("bar.sync 2, 128;" ::: "memory");
      if (p.has_ds) {  // geff = g + ds1 + 2 y ds2, in place
        uint8_t* q0 = buf + g_so;
#pragma unroll 2
        for (int kk = 0; kk < p.g_planes; ++kk, q0 += grs * 16) {
          float gv[8], yv[8];
          unpack8(*reinterpret_cast<const uint4*>(q0), gv);
          unpack8(*reinterpret_cast<const uint4*>(q0 + p.off_y), yv);
#pragma unroll
          for (int j = 0; j < 8; ++j) gv[j] += fmaf(yv[j], e2[j], e1[j]);
          *reinterpret_cast<uint4*>(q0) = pack8(gv);
        }
      }
      if (p.want_w) {  // xt = relu(x * scale + shift): the second operand of the weight gradient
        uint8_t* q0 = buf + p.off_x + x_so;
        const uint32_t to_xt = p.off_xt - p.off_x;  // 0: in place (no scale: the epilogue's mask x <= 0 survives the ReLU)
        if (d.in_scale || d.in_relu) {
          const float lo = d.in_relu ? 0.f : -INFINITY;
#pragma unroll 2
          for (int kk = 0; kk < p.x_planes; ++kk, q0 += xrs * 16) {
            float xv[8];
            unpack8(*reinterpret_cast<const uint4*>(q0), xv);
#pragma unroll
            for (int j = 0; j < 8; ++j) xv[j] = fmaxf(fmaf(xv[j], sc[j], sh[j]), lo);
            *reinterpret_cast<uint4*>(q0 + to_xt) = pack8(xv);
          }
        } else if (to_xt != 0) {
#pragma unroll 2
          for (int kk = 0; kk < p.x_planes; ++kk, q0 += xrs * 16)
            *reinterpret_cast<uint4*>(q0 + to_xt) = *reinterpret_cast<const uint4*>(q0);
        }
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(full(b));
      if (PDg > 0 && k + PDg < kmax) issue();  // only now, after the hand-over of this tile
      b += 2;
      while (b >= nbuf) b -= nbuf;
      rem += 2;
      while (rem >= p.tpi) { rem -= p.tpi; ++n; }
    }
  } else {
    // ===================== epilogue (two groups, alternate tiles): da -> dx, dscale / dshift; at the end D2 -> dW, db ====
    const int et = tid - 256;            // 0..255
    const int eg = et >> 7;              // group: tiles with (i & 1) == eg, accumulator D1[eg]
    const int el = et & 127;             // thread within the group
    const int q4 = warp & 3;             // this warp may touch TMEM lanes 32*q4 .. +31
    const int row = q4 * 32 + lane;      // TMEM lane == pixel row of the tile
    const uint32_t lane_off = (uint32_t)(q4 * 32) << 16;
    uint8_t* stage = smem + p.off_stage + eg * (BM * p.stage_ld);
    const float isg = a.inv_sigma ? a.inv_sigma[0] : 1.f;
    // column sums: thread -> (8-channel chunk, row group); 16-byte shared-memory reads, registers across tiles
    const int NCH = cin / 8, Q = 128 / NCH, sc_c = el % NCH, sc_q = el / NCH, rows_q = 128 / Q;
    float acc_s[8], acc_h[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { acc_s[j] = 0.f; acc_h[j] = 0.f; }
    int64_t cur_n = -1;
    auto flush = [&]() {
      if (p.want_ss && cur_n >= 0) {
        const int first = (int)((cur_n * p.tpi) / p.tpc);
        const int sl = blockIdx.x - first;
        float* o = a.scratch + ((((cur_n * p.sl_img + sl) * 2 + eg) * Q + sc_q) * cin + sc_c * 8) * 2;
#pragma unroll
        for (int j = 0; j < 8; ++j) { o[2 * j] = acc_s[j]; o[2 * j + 1] = acc_h[j]; }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) { acc_s[j] = 0.f; acc_h[j] = 0.f; }
    };
    auto grp_sync = [&]() {
      if (eg == 0) asm volatile("bar.sync 3, 128;" ::: "memory");
      else asm volatile("bar.sync 4, 128;" ::: "memory");
    };
    int b = eg % nbuf, u = eg / nbuf;  // ring slot of tile i and how often it was filled before
    int n = (t0 + eg) / p.tpi, rem = (t0 + eg) - n * p.tpi;
    for (int i = eg; i < ntile; i += 2) {
      const int k = i >> 1;  // this group's k-th tile
      // producers' images (x planes, tables) of this tile.  A group sees only every other tile: with ONE buffer it
      // would skip a phase of the barrier, and a parity wait cannot tell phase i-2 from phase i -- pass phase i-1 first.
      // (With an even number of slots a slot is always filled by the same producer group, in order.)
      if (nbuf == 1 && i > 0) mbar_wait(full(0), (i - 1) & 1);
      mbar_wait(full(b), u & 1);
      const int bcur = b;
      const int64_t ncur = n;
      b += 2;
      while (b >= nbuf) { b -= nbuf; ++u; }
      rem += 2;
      while (rem >= p.tpi) { rem -= p.tpi; ++n; }
      if (!p.want_x) {                          // (no data gradient wanted: only the buffer release is owed)
        __syncwarp();
        if (lane == 0) mbar_arrive(empty(bcur));
        continue;
      }
      const int64_t m0 = (int64_t)(t0 + i) * BM;
      if (ncur != cur_n) {
        if (cur_n >= 0) flush();
        cur_n = ncur;
      }
      const uint8_t* buf = smem + bcur * p.buf_bytes;
      const float* tab = reinterpret_cast<const float*>(buf + p.off_tab);
      mbar_wait(d1_full(eg), k & 1);            // da of this tile
      tc_fence_after();
      bf16* dxrow = a.dx ? (bf16*)a.dx + (m0 + row) * a.dx_ld : nullptr;
      for (int c16 = 0; c16 < cin; c16 += 16) {  // accumulator columns in batches of 16 (register budget: 96 / thread)
        uint32_t raw[16];
        tmem_ld16_issue(tmem + lane_off + eg * cin + c16, raw);
        uint4 xq[2], oq[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) xq[u] = *reinterpret_cast<const uint4*>(buf + p.off_x + (c16 / 8 + u) * PL + row * 16);
        if (dxrow && a.beta != 0.f) {
#pragma unroll
          for (int u = 0; u < 2; ++u) oq[u] = *reinterpret_cast<const uint4*>(dxrow + c16 + u * 8);
        }
        tmem_ld_wait();
#pragma unroll
        for (int q8 = 0; q8 < 2; ++q8) {  // 8 channels at a time
          const int c0 = c16 + q8 * 8;
          float xv[8], o[8], gm[8], ts[8], th[8];
          unpack8(xq[q8], xv);
          if (d.in_scale) {  // 16-byte broadcast reads of the per-channel table
            const float4* t4 = reinterpret_cast<const float4*>(tab + c0);
            const float4* h4 = reinterpret_cast<const float4*>(tab + cin + c0);
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const float4 a4 = t4[u], b4 = h4[u];
              ts[4 * u] = a4.x; ts[4 * u + 1] = a4.y; ts[4 * u + 2] = a4.z; ts[4 * u + 3] = a4.w;
              th[4 * u] = b4.x; th[4 * u + 1] = b4.y; th[4 * u + 2] = b4.z; th[4 * u + 3] = b4.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) { ts[j] = 1.f; th[j] = 0.f; }
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float g_ = __uint_as_float(raw[q8 * 8 + j]) * isg;
            if (d.in_relu && fmaf(xv[j], ts[j], th[j]) <= 0.f) g_ = 0.f;
            gm[j] = g_;
            o[j] = g_ * ts[j];
          }
          if (dxrow) {
            if (a.beta != 0.f) {
              float old[8];
              unpack8(oq[q8], old);
#pragma unroll
              for (int j = 0; j < 8; ++j) o[j] = fmaf(a.beta, old[j], o[j]);
            }
            *reinterpret_cast<uint4*>(dxrow + c0) = pack8(o);
          }
          if (p.want_ss) *reinterpret_cast<uint4*>(stage + row * p.stage_ld + c0 * 2) = pack8(gm);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(d1_empty(eg));
      if (p.want_ss) {
        grp_sync();  // the staged gm tile is complete
        const int r0 = sc_q * rows_q;
        const uint8_t* xpl = buf + p.off_x + sc_c * PL;
        for (int r = r0; r < r0 + rows_q; ++r) {
          float gv[8], xr[8];
          unpack8(*reinterpret_cast<const uint4*>(stage + r * p.stage_ld + sc_c * 16), gv);
          unpack8(*reinterpret_cast<const uint4*>(xpl + r * 16), xr);
#pragma unroll
          for (int j = 0; j < 8; ++j) { acc_h[j] += gv[j]; acc_s[j] = fmaf(gv[j], xr[j], acc_s[j]); }
        }
        grp_sync();  // the stage may be overwritten by this group's next tile
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty(bcur));  // this warp no longer reads the slot
    }
    if (cur_n >= 0) flush();
    if (p.want_w && eg == 0) {
      mbar_wait(d2_full, 0);
      tc_fence_after();
      const int co = row;
      float* wp = a.wpart + (int64_t)(1 + blockIdx.x) * cout * cin;
      for (int c16 = 0; c16 < cin / 16 + 1; ++c16) {
        float v[16];
        if (ntile > 0) tmem_ld16(tmem + lane_off + 2 * cin + c16 * 16, v);
        else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = 0.f;
        }
        if (co < cout) {
          if (c16 < cin / 16) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              *reinterpret_cast<float4*>(wp + (int64_t)co * cin + c16 * 16 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          } else if (a.dbias) {
            a.wpart[(int64_t)(1 + gridDim.x) * cout * cin + (int64_t)blockIdx.x * cout + co] = v[0];  // column `cin`: sum_px geff
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 16) tmem_free(tmem, p.tmem_cols);
}

// dscale / dshift [n][cin]: fixed-order sum of the partials of the CTAs that touched image n
__global__ void bwd1x1_reduce_ss(const float* part, int64_t n_img, int cin, int tpi, int tpc, int sl_img, int Q, int grid,
                                 float* dscale, float* dshift) {  // Q: row groups per epilogue group (x 2 groups)
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_img * cin) return;
  const int64_t n = i / cin;
  const int c = (int)(i - n * cin);
  const int first = (int)((n * tpi) / tpc);
  int last = (int)(((n + 1) * tpi - 1) / tpc);
  if (last > grid - 1) last = grid - 1;
  float s = 0.f, h = 0.f;
  for (int sl = 0; sl <= last - first; ++sl) {
    // which of the CTA's two epilogue groups saw this image: group eg handled the CTA's tiles t0 + eg, t0 + eg + 2, ...
    const int cta = first + sl;
    const int64_t ta = (int64_t)cta * tpc > n * tpi ? (int64_t)cta * tpc : n * tpi;             // first tile of n in this CTA
    int64_t tb = (int64_t)(cta + 1) * tpc < (n + 1) * tpi ? (int64_t)(cta + 1) * tpc : (n + 1) * tpi;  // one past the last
    for (int eg = 0; eg < 2; ++eg) {
      // tiles of this CTA with (tile - t0) & 1 == eg inside [ta, tb)
      const int64_t t0c = (int64_t)cta * tpc;
      int64_t f = ta + (((ta - t0c) & 1) == eg ? 0 : 1);
      if (f >= tb) continue;
      for (int q = 0; q < Q; ++q) {
        const float* o = part + ((((n * sl_img + sl) * 2 + eg) * Q + q) * cin + c) * 2;
        s += o[0]; h += o[1];
      }
    }
  }
  dscale[i] = s; dshift[i] = h;
}

static bool plan(const iea_conv_desc* d, const iea_bwd1x1_args* a, Params* p) {
  const int cin = d->cin, cout = d->cout;
  if (d->ksize != 1 || d->in_mode != IEA_IN_DIRECT || d->x_dtype != IEA_BF16) return false;
  if (!(cin == 16 || cin == 32 || cin == 64 || cin == 128)) return false;
  if (!(cout == 16 || cout == 32 || cout == 64 || cout == 128)) return false;
  const int hw = d->h * d->w;
  if (hw % BM) return false;
  const int64_t M = d->n * (int64_t)hw;
  if (M / BM >= (1 << 30) || M < 148 * BM) return false;  // small layers: the latency-oriented kernels
  if (d->x_ld % 8 || !aligned16(d->x)) return false;
  p->d = *d;
  p->M = M;
  p->hw = hw;
  p->tpi = hw / BM;
  p->tiles = (int)(M / BM);
  p->g_planes = cout / 8;
  p->x_planes = cin / 8;
  p->want_w = p->want_x = p->want_ss = p->has_ds = 0;
  if (a) {
    if (a->g_ld % 8 || !aligned16(a->g) || !aligned16(a->wd_tc)) return false;
    if (a->ds1 && (a->y_ld % 8 || !aligned16(a->y))) return false;
    if (a->dx && (a->dx_ld % 8 || !aligned16(a->dx))) return false;
    p->a = *a;
    p->want_w = a->wpart != nullptr;
    p->want_x = a->dx != nullptr || a->dscale != nullptr;
    p->want_ss = a->dscale != nullptr;
    p->has_ds = a->ds1 != nullptr;
  }
  return true;
}
static int grid_of(const Params& p) {
  const int sms = sm_count();
  return p.tiles < sms ? p.tiles : sms;
}
static void layout(Params* p, int grid) {
  const int cin = p->d.cin, cout = p->d.cout;
  p->tpc = (p->tiles + grid - 1) / grid;
  p->sl_img = (p->tpi + p->tpc - 1) / p->tpc + 1;
  // a slot: [g planes][y planes, with ds][x planes][xt planes, unless in place][ones plane][tables]
  p->inplace = p->d.in_scale == nullptr;  // no affine: the epilogue needs no raw x (relu mask: max(x, 0) <= 0 <=> x <= 0)
  p->off_y = p->g_planes * PL;
  p->off_x = p->off_y + (p->has_ds ? p->g_planes * PL : 0);
  p->off_xt = p->inplace ? p->off_x : p->off_x + p->x_planes * PL;
  p->off_tab = p->off_xt + (p->x_planes + 1) * PL;
  p->buf_bytes = (p->off_tab + 2 * cin * 4 + 127) / 128 * 128;
  p->stage_ld = cin * 2 + 16;
  const uint32_t stage = p->want_ss ? 2 * BM * p->stage_ld : 0;
  const uint32_t common = cout * cin * 2 + stage + 512 + PL;  // + PL: the B-operand overrun behind the last slot
  // the A operand of MMA2 spans 16 planes from the base of a slot: the last slot's overrun must stay inside the CTA's window
  auto fits = [&](int nb) {
    return nb * p->buf_bytes + common <= 227 * 1024 && (nb - 1) * p->buf_bytes + 16 * PL + 512 <= 227 * 1024;
  };
  p->nbuf = 1;
  for (int nb = 2; nb <= 8; nb += 2)  // even counts: a slot is then always filled by the same producer group
    if (fits(nb)) p->nbuf = nb;
  p->off_w = p->nbuf * p->buf_bytes;
  p->off_stage = p->off_w + cout * cin * 2;
  uint32_t end = p->off_stage + stage + PL;
  if (end < (p->nbuf - 1) * p->buf_bytes + 16 * PL) end = (p->nbuf - 1) * p->buf_bytes + 16 * PL;
  p->off_bar = (end + 127) / 128 * 128;
  p->tmem_cols = 512;
}

}  // namespace b1

extern "C" {
// > 0: the layer is handled by the fused kernel and this is its CTA count (sizes of the partial buffers below)
int iea_conv_bwd1x1_grid(const iea_conv_desc* fwd) {
  b1::Params p;
  if (!b1::plan(fwd, nullptr, &p)) return 0;
  return b1::grid_of(p);
}
// floats of args.scratch (partial dscale / dshift sums) for this layer
int64_t iea_conv_bwd1x1_scratch_floats(const iea_conv_desc* fwd) {
  b1::Params p;
  if (!b1::plan(fwd, nullptr, &p)) return 0;
  const int grid = b1::grid_of(p);
  b1::layout(&p, grid);
  return (int64_t)fwd->n * p.sl_img * 2 * (128 / (fwd->cin / 8)) * fwd->cin * 2;
}
int iea_conv_bwd1x1(const iea_conv_desc* fwd, const iea_bwd1x1_args* args, iea_stream_t stream) {
  b1::Params p;
  IEA_CHECK_ARG(b1::plan(fwd, args, &p), "iea_conv_bwd1x1: layer not handled (cin=%d cout=%d k=%d hw=%d)", fwd->cin, fwd->cout,
                fwd->ksize, fwd->h * fwd->w);
  IEA_CHECK_ARG(!p.want_ss || args->scratch, "iea_conv_bwd1x1: dscale / dshift need the scratch buffer");
  IEA_CHECK_ARG(!args->dbias || args->wpart, "iea_conv_bwd1x1: the bias gradient comes with the weight gradient");
  const int grid = b1::grid_of(p);
  b1::layout(&p, grid);
  cudaStream_t s = (cudaStream_t)stream;
  const uint32_t smem = p.off_bar + 256;
  IEA_CHECK_ARG(smem <= 227 * 1024, "iea_conv_bwd1x1: tile does not fit shared memory (%u bytes)", smem);
  IEA_CUDA(cudaFuncSetAttribute(b1::bwd1x1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  b1::bwd1x1_kernel<<<grid, b1::THREADS, smem, s>>>(p);
  const int cin = fwd->cin, cout = fwd->cout;
  if (p.want_w) {
    const int64_t total = (int64_t)cout * cin;
    int rb = (int)((total + 255) / 256);
    wg::wgrad_reduce_kernel<<<rb, 256, 0, s>>>(args->wpart + total, grid, total, args->wpart);
    if (args->dbias)
      wg::wgrad_reduce_kernel<<<(cout + 255) / 256, 256, 0, s>>>(args->wpart + (int64_t)(1 + grid) * total, grid, cout, args->dbias);
  }
  if (p.want_ss)
    b1::bwd1x1_reduce_ss<<<cdiv(fwd->n * cin, 256), 256, 0, s>>>(args->scratch, fwd->n, cin, p.tpi, p.tpc, p.sl_img,
                                                                   128 / (cin / 8), grid, args->dscale, args->dshift);
  return check_launch("iea_conv_bwd1x1");
}
}
