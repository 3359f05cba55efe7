// conv_generic.cu -- shape-generic fused convolution kernels on the CUDA cores.
//
// These cover every shape the nets contain (Cin = 1 input conv, Cout = 1 output conv,
// odd K of linear_f, tiny spatial sizes) and serve as the in-library cross-check of the
// tcgen05 path (conv_tc.cu), which takes the tensor-core-eligible layers.  Same fused
// semantics as iea_conv_desc documents: prologue T(x) = [pool|up](relu(x*scale+shift)),
// epilogue act(acc*out_scale + bias + residual) and per-tile batch-norm partial sums.
#include "common.cuh"
using namespace iea;

namespace {

struct Geo {
  int64_t M;       // output rows = n*h*w
  int K;           // cin*taps
  int hs, ws;      // stored spatial dims of x
};

__host__ __device__ inline Geo make_geo(const iea_conv_desc& d) {
  Geo g;
  g.M = d.n * (int64_t)d.h * d.w;
  g.K = d.cin * d.ksize * d.ksize;
  g.hs = stored_res(d, d.h);
  g.ws = stored_res(d, d.w);
  return g;
}

// transformed input element T(x)[n, ih, iw, ci] at conv resolution (ih, iw may be out of range -> 0)
__device__ __forceinline__ float load_t(const iea_conv_desc& d, const Geo& g, int64_t n, int ih, int iw, int ci) {
  if ((unsigned)ih >= (unsigned)d.h || (unsigned)iw >= (unsigned)d.w) return 0.f;
  float sc = 1.f, sh = 0.f;
  if (d.in_scale) { int64_t si = (d.in_bcast ? 0 : n * d.cin) + ci; sc = d.in_scale[si]; sh = d.in_shift[si]; }
  if (d.in_mode == IEA_IN_POOL2) {
    float acc = 0.f;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        float v = ld_act(d.x, d.x_dtype, ((n * g.hs + 2 * ih + a) * (int64_t)g.ws + 2 * iw + b) * d.x_ld + ci);
        v = fmaf(v, sc, sh);
        if (d.in_relu) v = fmaxf(v, 0.f);
        acc += v;
      }
    return 0.25f * acc;
  }
  int sh_ = d.in_mode == IEA_IN_UP2 ? 1 : 0;
  float v = ld_act(d.x, d.x_dtype, ((n * g.hs + (ih >> sh_)) * (int64_t)g.ws + (iw >> sh_)) * d.x_ld + ci);
  v = fmaf(v, sc, sh);
  if (d.in_relu) v = fmaxf(v, 0.f);
  return v;
}

__device__ __forceinline__ float load_res(const iea_conv_desc& d, int64_t n, int oh, int ow, int c) {
  if (d.res_mode == IEA_IN_UP2) {
    int hs = d.h / 2, ws = d.w / 2;
    return ld_act(d.res, d.res_dtype, ((n * hs + (oh >> 1)) * (int64_t)ws + (ow >> 1)) * d.res_ld + c);
  }
  if (d.res_mode == IEA_IN_POOL2) {
    int hs = d.h * 2, ws = d.w * 2;
    float acc = 0.f;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b)
        acc += ld_act(d.res, d.res_dtype, ((n * hs + 2 * oh + a) * (int64_t)ws + 2 * ow + b) * d.res_ld + c);
    return 0.25f * acc;
  }
  return ld_act(d.res, d.res_dtype, ((n * d.h + oh) * (int64_t)d.w + ow) * d.res_ld + c);
}

constexpr int BM = 128, BN = 32, BK = 16;

__global__ void __launch_bounds__(256) conv_fprop_generic(const iea_conv_desc d, const Geo g) {
  __shared__ __align__(16) float As[BK][BM];
  __shared__ __align__(16) float Bs[BK][BN];
  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.x * BM;
  const int c0 = blockIdx.y * BN;
  // A loader: fixed row per thread
  const int lrow = tid & (BM - 1), lk0 = (tid >> 7) * 8;
  const int64_t lm = m0 + lrow;
  const bool lvalid = lm < g.M;
  int l_ow = 0, l_oh = 0;
  int64_t l_n = 0;
  if (lvalid) { l_ow = lm % d.w; int64_t t = lm / d.w; l_oh = t % d.h; l_n = t / d.h; }
  const int tx = tid & 7, ty = tid >> 3;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < g.K; k0 += BK) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int k = k0 + lk0 + j;
      float v = 0.f;
      if (lvalid && k < g.K) {
        int tap = k / d.cin, ci = k - tap * d.cin;
        int ih = l_oh, iw = l_ow;
        if (d.ksize == 3) { ih += tap / 3 - 1; iw += tap % 3 - 1; }
        v = load_t(d, g, l_n, ih, iw, ci);
      }
      As[lk0 + j][lrow] = v;
    }
    for (int e = tid; e < BK * BN; e += 256) {
      int kk = e & (BK - 1), cc = e >> 4;
      int k = k0 + kk, co = c0 + cc;
      float v = 0.f;
      if (k < g.K && co < d.cout) v = ld_act(d.wpack, d.w_dtype, (int64_t)co * g.K + k);
      Bs[kk][cc] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  // epilogue
  float s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int64_t m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
    int ow = m % d.w; int64_t t = m / d.w; int oh = t % d.h; int64_t n = t / d.h;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int c = c0 + tx * 4 + j;
      if (c >= d.cout) continue;
      float v = acc[i][j];
      if (d.out_scale) v *= d.out_scale[d.out_scale_stride ? c : 0];
      if (d.bias) v += d.bias[c];
      if (d.res && c < d.res_c) v += load_res(d, n, oh, ow, c);
      if (d.acc_c0 >= 0 && c >= d.acc_c0) v += ld_act(d.y, d.y_dtype, m * d.y_ld + c);
      if (d.act == IEA_ACT_RELU) v = fmaxf(v, 0.f);
      else if (d.act == IEA_ACT_TANH) v = tanhf(v);
      st_act(d.y, d.y_dtype, m * d.y_ld + c, v);
      v = round_act(d.y_dtype, v);
      s1[j] += v;
      s2[j] = fmaf(v, v, s2[j]);
    }
  }
  if (d.stats) {  // deterministic per-tile column sums (re-using As as scratch)
    float* r1 = &As[0][0];          // [32 ty][32 cols]
    float* r2 = r1 + 32 * 32;
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) { r1[ty * 32 + tx * 4 + j] = s1[j]; r2[ty * 32 + tx * 4 + j] = s2[j]; }
    __syncthreads();
    if (tid < 64) {
      int col = tid & 31, which = tid >> 5;
      const float* r = which ? r2 : r1;
      float a = 0.f;
      for (int y = 0; y < 32; ++y) a += r[y * 32 + col];
      int c = c0 + col;
      if (c < d.cout) d.stats[((int64_t)blockIdx.x * d.cout + c) * 2 + which] = a;
    }
  }
}

// ---------------- weight gradient ----------------
constexpr int WM = 32;  // rows per step
__global__ void __launch_bounds__(256) conv_wgrad_generic(const iea_conv_desc d, const Geo g, const void* gr,
                                                          int g_dtype, int g_ld, float* gpart, int64_t rows_per_split) {
  __shared__ float Gs[WM][33];
  __shared__ float As[WM][33];
  const int tid = threadIdx.x;
  const int k0 = blockIdx.x * 32, c0 = blockIdx.y * 32, split = blockIdx.z;
  const int64_t mb = (int64_t)split * rows_per_split;
  int64_t me = mb + rows_per_split;
  if (me > g.M) me = g.M;
  const int tk = tid & 15, tc = tid >> 4;
  float acc[2][2] = {{0, 0}, {0, 0}};
  const int lrow = tid >> 3, lq = (tid & 7) * 4;
  for (int64_t ms = mb; ms < me; ms += WM) {
    int64_t m = ms + lrow;
    bool valid = m < me;
    int ow = 0, oh = 0; int64_t n = 0;
    if (valid) { ow = m % d.w; int64_t t = m / d.w; oh = t % d.h; n = t / d.h; }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int k = k0 + lq + j;
      float v = 0.f;
      if (valid && k < g.K) {
        int tap = k / d.cin, ci = k - tap * d.cin;
        int ih = oh, iw = ow;
        if (d.ksize == 3) { ih += tap / 3 - 1; iw += tap % 3 - 1; }
        v = load_t(d, g, n, ih, iw, ci);
      }
      As[lrow][lq + j] = v;
      int c = c0 + lq + j;
      Gs[lrow][lq + j] = (valid && c < d.cout) ? ld_act(gr, g_dtype, m * g_ld + c) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int r = 0; r < WM; ++r) {
      float g0 = Gs[r][tc * 2], g1 = Gs[r][tc * 2 + 1], a0 = As[r][tk * 2], a1 = As[r][tk * 2 + 1];
      acc[0][0] = fmaf(g0, a0, acc[0][0]); acc[0][1] = fmaf(g0, a1, acc[0][1]);
      acc[1][0] = fmaf(g1, a0, acc[1][0]); acc[1][1] = fmaf(g1, a1, acc[1][1]);
    }
    __syncthreads();
  }
  float* out = gpart + (int64_t)split * d.cout * g.K;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      int c = c0 + tc * 2 + i, k = k0 + tk * 2 + j;
      if (c < d.cout && k < g.K) out[(int64_t)c * g.K + k] = acc[i][j];
    }
}

// ---------------- backward of the prologue T ----------------
// grid (n, channel chunks); block = CB channels x (256/CB) pixel lanes.
__global__ void __launch_bounds__(256) conv_input_bwd_kernel(const iea_conv_desc d, const Geo g, const void* da,
                                                            int da_dtype, void* dx, int dx_dtype, int dx_ld,
                                                            float beta, float* dscale, float* dshift, int cb) {
  __shared__ float r1[256], r2[256];
  const int64_t n = blockIdx.x;
  const int lanes = 256 / cb;
  const int cl = threadIdx.x % cb, pl = threadIdx.x / cb;
  const int c = blockIdx.y * cb + cl;
  float a_s = 0.f, a_h = 0.f;
  if (c < d.cin) {
    float sc = 1.f, sh = 0.f;
    if (d.in_scale) { int64_t si = (d.in_bcast ? 0 : n * d.cin) + c; sc = d.in_scale[si]; sh = d.in_shift[si]; }
    const int64_t npx = (int64_t)g.hs * g.ws;
    for (int64_t p = pl; p < npx; p += lanes) {
      int xw = p % g.ws, xh = p / g.ws;
      float xv = ld_act(d.x, d.x_dtype, (n * npx + p) * d.x_ld + c);
      float gsum;
      if (d.in_mode == IEA_IN_UP2) {
        gsum = 0.f;
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int b = 0; b < 2; ++b)
            gsum += ld_act(da, da_dtype, ((n * d.h + 2 * xh + a) * (int64_t)d.w + 2 * xw + b) * d.cin + c);
      } else if (d.in_mode == IEA_IN_POOL2) {
        gsum = 0.25f * ld_act(da, da_dtype, ((n * d.h + (xh >> 1)) * (int64_t)d.w + (xw >> 1)) * d.cin + c);
      } else {
        gsum = ld_act(da, da_dtype, (n * npx + p) * d.cin + c);
      }
      float pre = fmaf(xv, sc, sh);
      if (d.in_relu && pre <= 0.f) gsum = 0.f;
      a_h += gsum;
      a_s = fmaf(gsum, xv, a_s);
      if (dx) {
        float v = gsum * sc;
        int64_t o = (n * npx + p) * dx_ld + c;
        if (beta != 0.f) v = fmaf(beta, ld_act(dx, dx_dtype, o), v);
        st_act(dx, dx_dtype, o, v);
      }
    }
  }
  if (dscale) {
    r1[threadIdx.x] = a_s; r2[threadIdx.x] = a_h;
    __syncthreads();
    if (pl == 0 && c < d.cin) {
      float t1 = 0.f, t2 = 0.f;
      for (int l = 0; l < lanes; ++l) { t1 += r1[l * cb + cl]; t2 += r2[l * cb + cl]; }
      dscale[n * d.cin + c] = t1;
      dshift[n * d.cin + c] = t2;
    }
  }
}

// g = dy*act' + ds1 + 2*y*ds2
__global__ void conv_out_bwd_kernel(const void* dy, int dy_dtype, int dy_ld, const void* y, int y_dtype, int y_ld,
                                    int act, const float* ds1, const float* ds2, int64_t rows, int rows_per_event,
                                    int c, void* gout, int g_dtype) {
  const int64_t total = rows * c;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t m = i / c; int cc = i - m * c;
    float v = ld_act(dy, dy_dtype, m * dy_ld + cc);
    float yv = (act == IEA_ACT_TANH || ds2) ? ld_act(y, y_dtype, m * y_ld + cc) : 0.f;
    if (act == IEA_ACT_TANH) v *= (1.f - yv * yv);
    if (ds1) {
      int64_t e = m / rows_per_event;
      v += ds1[e * c + cc] + 2.f * yv * ds2[e * c + cc];
    }
    st_act(gout, g_dtype, i, v);
  }
}

__global__ void __launch_bounds__(256) colsum_part(const void* g, int g_dtype, int g_ld, int64_t rows, int c,
                                                   float* part, int64_t rows_per_block) {
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block; if (r1 > rows) r1 = rows;
  __shared__ float red[256];
  const int cb = c < 256 ? c : 256;          // channels per pass
  const int lanes = 256 / cb > 0 ? 256 / cb : 1;
  for (int cbase = 0; cbase < c; cbase += cb) {
    int cl = threadIdx.x % cb, pl = threadIdx.x / cb;
    int cc = cbase + cl;
    float a = 0.f;
    if (pl < lanes && cc < c)
      for (int64_t m = r0 + pl; m < r1; m += lanes) a += ld_act(g, g_dtype, m * g_ld + cc);
    red[threadIdx.x] = a;
    __syncthreads();
    if (pl == 0 && cc < c) {
      float t = 0.f;
      for (int l = 0; l < lanes; ++l) t += red[l * cb + cl];
      part[(int64_t)blockIdx.x * c + cc] = t;
    }
    __syncthreads();
  }
}
// few rows, many columns (the head linears' bias gradients: 320 x 8192): one thread per column, rows in the loop --
// the row-split kernel above would put the whole matrix on ONE block (0.7 ms for 10 MB)
__global__ void __launch_bounds__(256) colsum_wide(const void* g, int g_dtype, int g_ld, int rows, int c, float* out,
                                                   float beta) {
  const int cc = blockIdx.x * 256 + threadIdx.x;
  if (cc >= c) return;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int m = 0;
  for (; m + 3 < rows; m += 4) {
    a0 += ld_act(g, g_dtype, (int64_t)m * g_ld + cc);
    a1 += ld_act(g, g_dtype, (int64_t)(m + 1) * g_ld + cc);
    a2 += ld_act(g, g_dtype, (int64_t)(m + 2) * g_ld + cc);
    a3 += ld_act(g, g_dtype, (int64_t)(m + 3) * g_ld + cc);
  }
  for (; m < rows; ++m) a0 += ld_act(g, g_dtype, (int64_t)m * g_ld + cc);
  const float t = (a0 + a1) + (a2 + a3);
  out[cc] = beta != 0.f ? fmaf(beta, out[cc], t) : t;
}
__global__ void colsum_final(const float* part, int blocks, int c, float* out, float beta) {
  int cc = blockIdx.x * blockDim.x + threadIdx.x;
  if (cc >= c) return;
  float t = 0.f;
  for (int b = 0; b < blocks; ++b) t += part[(int64_t)b * c + cc];
  out[cc] = beta != 0.f ? fmaf(beta, out[cc], t) : t;
}

__global__ void residual_bwd_kernel(const void* g, int g_dtype, int g_ld, int64_t n, int h, int w, int res_c,
                                    int res_mode, void* dres, int dres_dtype, int dres_ld, int dres_c, float beta) {
  const int hs = res_mode == IEA_IN_UP2 ? h / 2 : (res_mode == IEA_IN_POOL2 ? h * 2 : h);
  const int ws = res_mode == IEA_IN_UP2 ? w / 2 : (res_mode == IEA_IN_POOL2 ? w * 2 : w);
  const int64_t total = n * hs * (int64_t)ws * dres_c;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = i % dres_c; int64_t p = i / dres_c;
    int xw = p % ws; int64_t t = p / ws; int xh = t % hs; int64_t nn = t / hs;
    float v = 0.f;
    if (c < res_c) {
      if (res_mode == IEA_IN_UP2) {
        for (int a = 0; a < 2; ++a)
          for (int b = 0; b < 2; ++b)
            v += ld_act(g, g_dtype, ((nn * h + 2 * xh + a) * (int64_t)w + 2 * xw + b) * g_ld + c);
      } else if (res_mode == IEA_IN_POOL2) {
        v = 0.25f * ld_act(g, g_dtype, ((nn * h + (xh >> 1)) * (int64_t)w + (xw >> 1)) * g_ld + c);
      } else {
        v = ld_act(g, g_dtype, p * g_ld + c);
      }
    }
    int64_t o = p * dres_ld + c;
    if (beta != 0.f) v = fmaf(beta, ld_act(dres, dres_dtype, o), v);
    st_act(dres, dres_dtype, o, v);
  }
}

inline int ew_blocks(int64_t total) {
  int64_t b = (total + 255) / 256;
  if (b > 148 * 16) b = 148 * 16;
  return b < 1 ? 1 : (int)b;
}

}  // namespace

int iea_conv_fprop_generic(const iea_conv_desc* d, cudaStream_t s) {
  Geo g = make_geo(*d);
  dim3 grid(cdiv(g.M, BM), cdiv(d->cout, BN));
  conv_fprop_generic<<<grid, 256, 0, s>>>(*d, g);
  return check_launch("iea_conv_fprop(generic)");
}

extern "C" int iea_conv_wgrad(const iea_conv_desc* d, const void* g, int g_dtype, int g_ld, float* gpart,
                              int nsplit, iea_stream_t stream) {
  IEA_CHECK_ARG(nsplit >= 1, "iea_conv_wgrad: nsplit must be >= 1");
  Geo geo = make_geo(*d);
  int64_t rps = (geo.M + nsplit - 1) / nsplit;
  rps = (rps + WM - 1) / WM * WM;
  dim3 grid(cdiv(geo.K, 32), cdiv(d->cout, 32), nsplit);
  conv_wgrad_generic<<<grid, 256, 0, (cudaStream_t)stream>>>(*d, geo, g, g_dtype, g_ld, gpart, rps);
  return check_launch("iea_conv_wgrad");
}

// vectorised version for bf16 tensors with cin % 8 == 0: grid (pixel chunks, n), 256 threads =
// (cin/8 sixteen-byte columns) x (pixel lanes); per-CTA partial (dscale, dshift) then a fixed-order reduce.
namespace {
__global__ void __launch_bounds__(256) conv_input_bwd_vec(const iea_conv_desc d, const Geo g, const bf16* __restrict__ da,
                                                          bf16* __restrict__ dx, int dx_ld, float beta, float* part,
                                                          int chunks, int px_per_chunk) {
  extern __shared__ float red[];  // [lanes][cin][2]
  const int64_t n = blockIdx.y;
  const int cgs = d.cin >> 3, lanes = 256 / cgs;
  const int cgi = threadIdx.x % cgs, pl = threadIdx.x / cgs, c0 = cgi * 8;
  const int npx = g.hs * g.ws;
  const int p0 = blockIdx.x * px_per_chunk;
  int p1 = p0 + px_per_chunk; if (p1 > npx) p1 = npx;
  float sc[8], sh[8], a_s[8], a_h[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = 1.f; sh[j] = 0.f; a_s[j] = 0.f; a_h[j] = 0.f; }
  if (d.in_scale && pl < lanes) {
    const int64_t si = (d.in_bcast ? 0 : n * d.cin) + c0;
#pragma unroll
    for (int j = 0; j < 8; ++j) { sc[j] = d.in_scale[si + j]; sh[j] = d.in_shift[si + j]; }
  }
  const bf16* __restrict__ xb = (const bf16*)d.x;
  // (read-only operands through the non-coherent path + restrict: the unrolled iterations issue their loads
  //  back to back, four pixels in flight per thread, instead of one load-use round trip per pixel)
  if (pl < lanes)
#pragma unroll 4
    for (int p = p0 + pl; p < p1; p += lanes) {
      const int xh = p / g.ws, xw = p - xh * g.ws;
      float xv[8], gs[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(xb + (n * npx + p) * d.x_ld + c0)), xv);
      if (d.in_mode == IEA_IN_UP2) {
#pragma unroll
        for (int j = 0; j < 8; ++j) gs[j] = 0.f;
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int b = 0; b < 2; ++b) {
            float t[8];
            unpack8(__ldg(reinterpret_cast<const uint4*>(da + ((n * d.h + 2 * xh + a) * (int64_t)d.w + 2 * xw + b) * d.cin + c0)), t);
#pragma unroll
            for (int j = 0; j < 8; ++j) gs[j] += t[j];
          }
      } else if (d.in_mode == IEA_IN_POOL2) {
        unpack8(__ldg(reinterpret_cast<const uint4*>(da + ((n * d.h + (xh >> 1)) * (int64_t)d.w + (xw >> 1)) * d.cin + c0)), gs);
#pragma unroll
        for (int j = 0; j < 8; ++j) gs[j] *= 0.25f;
      } else {
        unpack8(__ldg(reinterpret_cast<const uint4*>(da + (n * npx + p) * d.cin + c0)), gs);
      }
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float pre = fmaf(xv[j], sc[j], sh[j]);
        if (d.in_relu && pre <= 0.f) gs[j] = 0.f;
        a_h[j] += gs[j];
        a_s[j] = fmaf(gs[j], xv[j], a_s[j]);
        o[j] = gs[j] * sc[j];
      }
      if (dx) {
        bf16* q = dx + (n * npx + p) * dx_ld + c0;
        if (beta != 0.f) {
          float old[8];
          unpack8(*reinterpret_cast<const uint4*>(q), old);
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = fmaf(beta, old[j], o[j]);
        }
        *reinterpret_cast<uint4*>(q) = pack8(o);
      }
    }
  if (part) {
    if (pl < lanes)
#pragma unroll
      for (int j = 0; j < 8; ++j) { red[(pl * d.cin + c0 + j) * 2] = a_s[j]; red[(pl * d.cin + c0 + j) * 2 + 1] = a_h[j]; }
    __syncthreads();
    for (int c = threadIdx.x; c < d.cin * 2; c += 256) {
      float t = 0.f;
      for (int l = 0; l < lanes; ++l) t += red[l * d.cin * 2 + c];
      part[((n * chunks + blockIdx.x) * d.cin) * 2 + c] = t;
    }
  }
}
// ---- the common case without batch-norm constants (every discriminator layer, and the gradient that flows through
// D in the generator step): dx = [0.25 *] da * 1[x > 0], same resolution or 2x2 average-pool adjoint.  The mask and the
// power-of-two scale are exact in packed bf16, so the kernel is 2 loads, ~10 packed instructions and 1 store per
// 16-byte chunk instead of ~90 fp32 instructions (the general kernel above is instruction-, not bandwidth-bound).
template <bool POOL, bool RELU, bool ACC>
__global__ void __launch_bounds__(256) conv_input_bwd_plain(const bf16* __restrict__ x, int x_ld, const bf16* __restrict__ da,
                                                            bf16* __restrict__ dx, int dx_ld, int cin, int hs, int ws,
                                                            int ws_sh, int px_per_chunk) {
  const int64_t n = blockIdx.y;
  const int cgs = cin >> 3, lanes = 256 / cgs;
  const int cgi = threadIdx.x % cgs, pl = threadIdx.x / cgs, c0 = cgi * 8;
  if (pl >= lanes) return;
  const int npx = hs * ws;
  const int p0 = blockIdx.x * px_per_chunk;
  int p1 = p0 + px_per_chunk; if (p1 > npx) p1 = npx;
  const int h = POOL ? hs >> 1 : hs, w = POOL ? ws >> 1 : ws;  // resolution of da
  const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f), quarter2 = __floats2bfloat162_rn(0.25f, 0.25f);
  auto da_ptr = [&](int p) -> const bf16* {
    if (!POOL) return da + (n * npx + p) * cin + c0;
    const int xh = ws_sh >= 0 ? p >> ws_sh : p / ws, xw = p - xh * ws;
    return da + ((n * h + (xh >> 1)) * (int64_t)w + (xw >> 1)) * cin + c0;
  };
  constexpr int U = 4;
  for (int pb = p0 + pl; pb < p1; pb += U * lanes) {
    uint4 xv[U], gv[U], ov[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int p = pb + u * lanes;
      if (p < p1) {
        if (RELU) xv[u] = __ldg(reinterpret_cast<const uint4*>(x + (n * npx + p) * x_ld + c0));
        gv[u] = __ldg(reinterpret_cast<const uint4*>(da_ptr(p)));
        if (ACC) ov[u] = *reinterpret_cast<const uint4*>(dx + (n * npx + p) * dx_ld + c0);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int p = pb + u * lanes;
      if (p >= p1) continue;
      __nv_bfloat162* g2 = reinterpret_cast<__nv_bfloat162*>(&gv[u]);
      const __nv_bfloat162* x2 = reinterpret_cast<const __nv_bfloat162*>(&xv[u]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (RELU) g2[j] = __hmul2(g2[j], __hgt2(x2[j], zero2));  // mask: 1.0 / 0.0 per lane
        if (POOL) g2[j] = __hmul2(g2[j], quarter2);
      }
      if (ACC) {  // dx += value, in fp32 and rounded once like the general kernel
        const uint32_t* a = reinterpret_cast<const uint32_t*>(&gv[u]);
        const uint32_t* b = reinterpret_cast<const uint32_t*>(&ov[u]);
        uint32_t* o = reinterpret_cast<uint32_t*>(&gv[u]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float lo = __uint_as_float(a[j] << 16) + __uint_as_float(b[j] << 16);
          const float hi = __uint_as_float(a[j] & 0xFFFF0000u) + __uint_as_float(b[j] & 0xFFFF0000u);
          __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
          o[j] = *reinterpret_cast<uint32_t*>(&t);
        }
      }
      *reinterpret_cast<uint4*>(dx + (n * npx + p) * dx_ld + c0) = gv[u];
    }
  }
}
__global__ void input_bwd_reduce(const float* part, int64_t n, int chunks, int cin, float* dscale, float* dshift) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * cin) return;
  const int64_t nn = i / cin; const int c = i - nn * cin;
  float a = 0.f, b = 0.f;
  for (int k = 0; k < chunks; ++k) {
    const float* q = part + ((nn * chunks + k) * cin + c) * 2;
    a += q[0]; b += q[1];
  }
  dscale[i] = a; dshift[i] = b;
}
}  // namespace

extern "C" int iea_conv_input_bwd(const iea_conv_desc* d, const void* da, int da_dtype, void* dx, int dx_dtype,
                                  int dx_ld, float beta, float* dscale, float* dshift, float* scratch,
                                  iea_stream_t stream) {
  Geo g = make_geo(*d);
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = d->x_dtype == IEA_BF16 && da_dtype == IEA_BF16 && (!dx || dx_dtype == IEA_BF16) && d->cin % 8 == 0 &&
                   d->cin <= 2048 && d->x_ld % 8 == 0 && (!dx || dx_ld % 8 == 0) && scratch != nullptr &&
                   (reinterpret_cast<uintptr_t>(d->x) & 15) == 0 && (reinterpret_cast<uintptr_t>(da) & 15) == 0 &&
                   (!dx || (reinterpret_cast<uintptr_t>(dx) & 15) == 0);
  if (vec && dx && !d->in_scale && !dscale && d->in_mode != IEA_IN_UP2 && (beta == 0.f || beta == 1.f) &&
      256 % (d->cin / 8) == 0) {
    const int npx = g.hs * g.ws;
    int chunks = npx / 2048;
    if (chunks < 1) chunks = 1;
    if (chunks > 64) chunks = 64;
    const int ppc = (npx + chunks - 1) / chunks;
    int ws_sh = -1;
    if ((g.ws & (g.ws - 1)) == 0) { ws_sh = 0; while ((1 << ws_sh) < g.ws) ++ws_sh; }
    const dim3 grid(chunks, (unsigned)d->n);
#define IEA_IBP(P_, R_, A_) conv_input_bwd_plain<P_, R_, A_><<<grid, 256, 0, st>>>((const bf16*)d->x, d->x_ld, (const bf16*)da, \
                                                                              (bf16*)dx, dx_ld, d->cin, g.hs, g.ws, ws_sh, ppc)
    const bool pool = d->in_mode == IEA_IN_POOL2, relu = d->in_relu != 0, acc = beta != 0.f;
    if (pool) { if (relu) { if (acc) IEA_IBP(true, true, true); else IEA_IBP(true, true, false); }
                else      { if (acc) IEA_IBP(true, false, true); else IEA_IBP(true, false, false); } }
    else      { if (relu) { if (acc) IEA_IBP(false, true, true); else IEA_IBP(false, true, false); }
                else      { if (acc) IEA_IBP(false, false, true); else IEA_IBP(false, false, false); } }
#undef IEA_IBP
    return check_launch("iea_conv_input_bwd(plain)");
  }
  if (vec) {
    const int npx = g.hs * g.ws;
    int chunks = npx / 2048;
    if (chunks < 1) chunks = 1;
    if (chunks > 64) chunks = 64;
    const int ppc = (npx + chunks - 1) / chunks;
    const int lanes = 256 / (d->cin / 8);
    const size_t smem = (size_t)lanes * d->cin * 2 * sizeof(float);
    conv_input_bwd_vec<<<dim3(chunks, (unsigned)d->n), 256, smem, st>>>(*d, g, (const bf16*)da, (bf16*)dx, dx_ld, beta,
                                                                         dscale ? scratch : nullptr, chunks, ppc);
    if (dscale)
      input_bwd_reduce<<<cdiv(d->n * d->cin, 256), 256, 0, st>>>(scratch, d->n, chunks, d->cin, dscale, dshift);
    return check_launch("iea_conv_input_bwd(vec)");
  }
  int cb = 1;
  while (cb < d->cin && cb < 32) cb <<= 1;
  dim3 grid((unsigned)d->n, cdiv(d->cin, cb));
  conv_input_bwd_kernel<<<grid, 256, 0, st>>>(*d, g, da, da_dtype, dx, dx_dtype, dx_ld, beta, dscale, dshift, cb);
  return check_launch("iea_conv_input_bwd");
}

// ---- vectorised (bf16, 8 channels per 16-byte load) versions of the two bandwidth-bound adjoints ----
namespace {
__device__ __forceinline__ uint4 ld_nc16(const bf16* p) {  // streaming 16-byte load (read once: keep it out of L1)
  uint4 q;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w) : "l"(p));
  return q;
}
// g = dy*act' + ds1 + 2*y*ds2 on bf16 rows, one thread per (row, 8 channels), two rows in flight
__global__ void __launch_bounds__(256) conv_out_bwd_vec(const bf16* dy, int dy_ld, const bf16* y, int y_ld, int act,
                                                        const float* ds1, const float* ds2, int64_t rows,
                                                        int rows_per_event, int c, bf16* gout) {
  const int cgs = c >> 3;
  const int cgi = (int)(threadIdx.x % cgs), rl = (int)(threadIdx.x / cgs), rpb = 256 / cgs;  // 256 % cgs == 0
  const bool need_y = act == IEA_ACT_TANH || ds2 != nullptr;
  const int64_t stride = (int64_t)gridDim.x * rpb;
  for (int64_t m0 = (int64_t)blockIdx.x * rpb + rl; m0 < rows; m0 += 2 * stride) {
    uint4 qd[2], qy[2];
    bool ok[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int64_t m = m0 + u * stride;
      ok[u] = m < rows;
      if (ok[u]) {
        qd[u] = ld_nc16(dy + m * dy_ld + cgi * 8);
        if (need_y) qy[u] = ld_nc16(y + m * y_ld + cgi * 8);
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (!ok[u]) continue;
      const int64_t m = m0 + u * stride;
      float v[8], yv[8];
      unpack8(qd[u], v);
      if (need_y) unpack8(qy[u], yv);
      if (act == IEA_ACT_TANH) {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] *= (1.f - yv[j] * yv[j]);
      }
      if (ds1) {
        const int64_t e = m / rows_per_event;
        const float4* a1 = reinterpret_cast<const float4*>(ds1 + e * c + cgi * 8);
        const float4* a2 = reinterpret_cast<const float4*>(ds2 + e * c + cgi * 8);
        const float4 s0 = a1[0], s1 = a1[1], t0 = a2[0], t1 = a2[1];
        const float s[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
        const float t[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] += fmaf(2.f * yv[j], t[j], s[j]);
      }
      uint32_t o[4];  // (pack2 in a loop, not pack8: with pack8 the compiler unswitches the row loop into three copies)
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = pack2(v[2 * j], v[2 * j + 1]);
      *reinterpret_cast<uint4*>(gout + m * c + cgi * 8) = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
}
__global__ void __launch_bounds__(256) colsum_part_vec(const bf16* g, int g_ld, int64_t rows, int c, float* part,
                                                       int64_t rows_per_block) {
  extern __shared__ float red[];  // [lanes][c]
  const int cgs = c >> 3, lanes = 256 / cgs;
  const int cgi = threadIdx.x % cgs, pl = threadIdx.x / cgs;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block; if (r1 > rows) r1 = rows;
  float a[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = 0.f;
  if (pl < lanes) {
    int64_t m = r0 + pl;
    for (; m + 3 * lanes < r1; m += 4 * lanes) {  // four independent 16-byte loads in flight per thread
      uint4 q[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) q[u] = ld_nc16(g + (m + u * lanes) * g_ld + cgi * 8);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float f[8];
        unpack8(q[u], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) a[j] += f[j];
      }
    }
    for (; m < r1; m += lanes) {
      float f[8];
      unpack8(ld_nc16(g + m * g_ld + cgi * 8), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] += f[j];
    }
  }
  if (pl < lanes)
#pragma unroll
    for (int j = 0; j < 8; ++j) red[pl * c + cgi * 8 + j] = a[j];
  __syncthreads();
  for (int cc = threadIdx.x; cc < c; cc += 256) {
    float t = 0.f;
    for (int l = 0; l < lanes; ++l) t += red[l * c + cc];
    part[(int64_t)blockIdx.x * c + cc] = t;
  }
}
// dres (at the residual's resolution) from g (at the conv resolution); one thread per (pixel, 8 channels)
__global__ void residual_bwd_vec(const bf16* g, int g_ld, int64_t n, int h, int w, int res_c, int res_mode, bf16* dres,
                                 int dres_ld, int dres_c, float beta) {
  const int hs = res_mode == IEA_IN_UP2 ? h / 2 : (res_mode == IEA_IN_POOL2 ? h * 2 : h);
  const int ws = res_mode == IEA_IN_UP2 ? w / 2 : (res_mode == IEA_IN_POOL2 ? w * 2 : w);
  const int cgs = dres_c >> 3;
  const int64_t total = n * hs * (int64_t)ws * cgs;
  // (index arithmetic in 32 bits with shifts for the power-of-two extents every layer has: the six 64-bit
  //  divisions per chunk of the first version cost more than the memory traffic)
  const bool small = total < (1ll << 31);
  const int cg_sh = (cgs & (cgs - 1)) == 0 ? 31 - __clz(cgs) : -1;
  const int ws_sh = (ws & (ws - 1)) == 0 ? 31 - __clz(ws) : -1;
  const int hs_sh = (hs & (hs - 1)) == 0 ? 31 - __clz(hs) : -1;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int cgi; int64_t p;
    if (small) {
      const unsigned iu = (unsigned)i;
      const unsigned pu = cg_sh >= 0 ? iu >> cg_sh : iu / (unsigned)cgs;
      cgi = (int)(iu - pu * (unsigned)cgs); p = pu;
    } else {
      cgi = (int)(i % cgs); p = i / cgs;
    }
    const int c0 = cgi * 8;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = 0.f;
    if (c0 < res_c) {
      if (res_mode == IEA_IN_DIRECT) {
        unpack8(*reinterpret_cast<const uint4*>(g + p * g_ld + c0), v);
      } else {
        int xw, xh; int64_t nn;
        if (small) {
          const unsigned pu = (unsigned)p;
          const unsigned t = ws_sh >= 0 ? pu >> ws_sh : pu / (unsigned)ws;
          xw = (int)(pu - t * (unsigned)ws);
          const unsigned nu = hs_sh >= 0 ? t >> hs_sh : t / (unsigned)hs;
          xh = (int)(t - nu * (unsigned)hs); nn = nu;
        } else {
          xw = (int)(p % ws); const int64_t t = p / ws; xh = (int)(t % hs); nn = t / hs;
        }
        if (res_mode == IEA_IN_UP2) {
#pragma unroll
          for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) {
              float f[8];
              unpack8(*reinterpret_cast<const uint4*>(g + ((nn * h + 2 * xh + a) * (int64_t)w + 2 * xw + b) * g_ld + c0), f);
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] += f[j];
            }
        } else {
          unpack8(*reinterpret_cast<const uint4*>(g + ((nn * h + (xh >> 1)) * (int64_t)w + (xw >> 1)) * g_ld + c0), v);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] *= 0.25f;
        }
      }
    }
    bf16* q = dres + p * dres_ld + c0;
    if (beta != 0.f) {
      float old[8];
      unpack8(*reinterpret_cast<const uint4*>(q), old);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaf(beta, old[j], v[j]);
    }
    *reinterpret_cast<uint4*>(q) = pack8(v);
  }
}
inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
}  // namespace

extern "C" int iea_colsum(const void* g, int g_dtype, int g_ld, int64_t rows, int c, float* out, float beta,
                          float* scratch, iea_stream_t stream) {
  if (rows <= 4096 && c >= 256) {
    colsum_wide<<<cdiv(c, 256), 256, 0, (cudaStream_t)stream>>>(g, g_dtype, g_ld, (int)rows, c, out, beta);
    return check_launch("iea_colsum(wide)");
  }
  int blocks = (int)((rows + 127) / 128);  // (512 rows per block left 5 blocks for a 2560 x 512 gradient: 90 us)
  if (blocks > 296) blocks = 296;
  if (blocks < 1) blocks = 1;
  int64_t rpb = (rows + blocks - 1) / blocks;
  if (g_dtype == IEA_BF16 && c % 8 == 0 && c <= 2048 && g_ld % 8 == 0 && al16(g)) {
    const int lanes = 256 / (c / 8);
    colsum_part_vec<<<blocks, 256, (size_t)lanes * c * sizeof(float), (cudaStream_t)stream>>>((const bf16*)g, g_ld, rows,
                                                                                                 c, scratch, rpb);
  } else {
    colsum_part<<<blocks, 256, 0, (cudaStream_t)stream>>>(g, g_dtype, g_ld, rows, c, scratch, rpb);
  }
  colsum_final<<<cdiv(c, 128), 128, 0, (cudaStream_t)stream>>>(scratch, blocks, c, out, beta);
  return check_launch("iea_colsum");
}

extern "C" int iea_residual_bwd(const void* g, int g_dtype, int g_ld, int64_t n, int h, int w, int res_c,
                                int res_mode, void* dres, int dres_dtype, int dres_ld, int dres_c, float beta,
                                iea_stream_t stream) {
  int hs = res_mode == IEA_IN_UP2 ? h / 2 : (res_mode == IEA_IN_POOL2 ? h * 2 : h);
  int ws = res_mode == IEA_IN_UP2 ? w / 2 : (res_mode == IEA_IN_POOL2 ? w * 2 : w);
  if (g_dtype == IEA_BF16 && dres_dtype == IEA_BF16 && dres_c % 8 == 0 && res_c % 8 == 0 && g_ld % 8 == 0 &&
      dres_ld % 8 == 0 && al16(g) && al16(dres)) {
    residual_bwd_vec<<<ew_blocks(n * hs * (int64_t)ws * (dres_c / 8)), 256, 0, (cudaStream_t)stream>>>(
        (const bf16*)g, g_ld, n, h, w, res_c, res_mode, (bf16*)dres, dres_ld, dres_c, beta);
    return check_launch("iea_residual_bwd(vec)");
  }
  residual_bwd_kernel<<<ew_blocks(n * hs * (int64_t)ws * dres_c), 256, 0, (cudaStream_t)stream>>>(
      g, g_dtype, g_ld, n, h, w, res_c, res_mode, dres, dres_dtype, dres_ld, dres_c, beta);
  return check_launch("iea_residual_bwd");
}

extern "C" int iea_conv_out_bwd(const void* dy, int dy_dtype, int dy_ld, const void* y, int y_dtype, int y_ld,
                                int act, const float* ds1, const float* ds2, int64_t rows, int rows_per_event,
                                int c, void* g, int g_dtype, iea_stream_t stream) {
  if (dy_dtype == IEA_BF16 && y_dtype == IEA_BF16 && g_dtype == IEA_BF16 && c % 8 == 0 && 256 % (c / 8) == 0 &&
      dy_ld % 8 == 0 && y_ld % 8 == 0 && al16(dy) && al16(y) && al16(g)) {
    const int rpb = 256 / (c / 8);
    int64_t blocks = (rows + 2 * rpb - 1) / (2 * rpb);
    if (blocks > 148 * 16) blocks = 148 * 16;
    conv_out_bwd_vec<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const bf16*)dy, dy_ld, (const bf16*)y, y_ld, act, ds1,
                                                                   ds2, rows, rows_per_event, c, (bf16*)g);
    return check_launch("iea_conv_out_bwd(vec)");
  }
  conv_out_bwd_kernel<<<ew_blocks(rows * c), 256, 0, (cudaStream_t)stream>>>(dy, dy_dtype, dy_ld, y, y_dtype, y_ld,
                                                                             act, ds1, ds2, rows, rows_per_event, c,
                                                                             g, g_dtype);
  return check_launch("iea_conv_out_bwd");
}

