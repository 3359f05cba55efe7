// conv_c1.cu -- the two 3x3 convolutions with a single-channel side: the discriminator stem
// (1 -> 32, model.py:717 input_conv) and the generator output layer (32 -> 1, model.py:379-387), whose
// data gradient is again a 1 -> 32 convolution.
//
// Zero-extending the single channel to a 16-wide tensor-core operand makes these layers cost as much as a
// 16-channel layer (shared-memory operand traffic, 9 UMMAs per tile) for 1/16 of the useful work; they
// are 288 FMA per pixel and purely bandwidth-bound, so they run on the CUDA cores with packed fp32x2 FMAs:
//   c1_fwd_kernel    y[px][C]  = (sum_tap W[c][tap] x[px+tap]) * out_scale + bias          (C = 8*CG)
//   c1_wgrad_kernel  R[c][tap] = sum_q  a[q][c] * b[q + sgn*tap]
//        stem:        a = g (C channels),  b = x,  sgn = +1   ->  dW[co][tap]
//        output conv: a = T(x) (C channels, fused BN-affine + ReLU),  b = g,  sgn = -1   ->  dW[0][tap][ci]
// Thread = 4 consecutive pixels x 8 channels: the 8x9 weights (forward) / 9x8 accumulators (gradient)
// live in registers, each wide tensor element is touched once with a 16-byte access.
#include "common.cuh"
using namespace iea;

namespace c1 {

struct Geo { int64_t n; int h, w; int64_t groups; };  // groups = n*h*(w/4) pixel quads

// 3 x 6 window of the single-channel tensor around pixel quad (nn, hh, w0..w0+3); zero outside the image
__device__ __forceinline__ void load_window(const void* b, int dtype, int ld, const Geo& g, int64_t nn, int hh, int w0,
                                            float (&win)[3][6]) {
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const int ih = hh - 1 + r;
    const bool rok = (unsigned)ih < (unsigned)g.h;
    const int64_t base = ((nn * g.h + ih) * (int64_t)g.w + w0) * ld;
    if (rok && dtype == IEA_F32 && ld == 1) {
      const float4 q = __ldg(reinterpret_cast<const float4*>((const float*)b + base));  // w0 % 4 == 0, w % 4 == 0: 16-byte aligned
      win[r][1] = q.x; win[r][2] = q.y; win[r][3] = q.z; win[r][4] = q.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) win[r][1 + i] = rok ? ld_act(b, dtype, base + (int64_t)i * ld) : 0.f;
    }
    win[r][0] = (rok && w0 > 0) ? ld_act(b, dtype, base - ld) : 0.f;
    win[r][5] = (rok && w0 + 4 < g.w) ? ld_act(b, dtype, base + 4ll * ld) : 0.f;
  }
}

// ---------------------------------------------------------------- forward / data gradient: 1 -> C
template <int CG>
__global__ void __launch_bounds__(256, 2) c1_fwd_kernel(const iea_conv_desc d, const Geo g) {
  const int cg = threadIdx.x % CG;
  float2 w2[9][4], b2[4];
  {
    const float os = d.out_scale ? d.out_scale[0] : 1.f;
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = cg * 8 + 2 * j;
        w2[t][j] = make_float2(ld_act(d.wpack, d.w_dtype, (int64_t)c * 9 + t) * os, ld_act(d.wpack, d.w_dtype, (int64_t)(c + 1) * 9 + t) * os);
      }
#pragma unroll
    for (int j = 0; j < 4; ++j) b2[j] = d.bias ? make_float2(d.bias[cg * 8 + 2 * j], d.bias[cg * 8 + 2 * j + 1]) : make_float2(0.f, 0.f);
  }
  const int wq = g.w >> 2;
  const int64_t stride = (int64_t)gridDim.x * (256 / CG);
  for (int64_t q = (int64_t)blockIdx.x * (256 / CG) + threadIdx.x / CG; q < g.groups; q += stride) {
    const int w0 = (int)(q % wq) * 4;
    const int64_t t = q / wq;
    const int hh = (int)(t % g.h);
    const int64_t nn = t / g.h;
    float win[3][6];
    load_window(d.x, d.x_dtype, d.x_ld, g, nn, hh, w0, win);
    float2 acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = b2[j];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int s = 0; s < 3; ++s)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 xv = make_float2(win[r][i + s], win[r][i + s]);
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = ffma2(w2[r * 3 + s][j], xv, acc[i][j]);
        }
    bf16* yp = (bf16*)d.y + ((nn * g.h + hh) * (int64_t)g.w + w0) * d.y_ld + cg * 8;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      *reinterpret_cast<uint4*>(yp + (int64_t)i * d.y_ld) =
          make_uint4(pack2(acc[i][0].x, acc[i][0].y), pack2(acc[i][1].x, acc[i][1].y), pack2(acc[i][2].x, acc[i][2].y),
                     pack2(acc[i][3].x, acc[i][3].y));
  }
}

// ---------------------------------------------------------------- weight gradient
struct WgP {
  const bf16* a; int a_ld;                  // wide tensor [n][h][w][C]
  const float* sc; const float* sh; int bcast, relu;  // fused T() on a (output conv) or NULL
  const void* b; int b_dtype, b_ld;         // single-channel tensor
  int sgn;                                  // +1: b[q + tap], -1: b[q - tap]
  int out_c_stride, out_t_stride;           // partial layout: R[c][tap] at c*out_c_stride + tap*out_t_stride
  int C;
  float* parts;                             // [gridDim.x][9*C]
};

template <int CG>
__global__ void __launch_bounds__(256) c1_wgrad_kernel(const WgP p, const Geo g) {
  __shared__ float red[8][CG * 72];
  const int cg = threadIdx.x % CG;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float2 acc[9][4];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[t][j] = make_float2(0.f, 0.f);
  const int wq = g.w >> 2;
  const int64_t stride = (int64_t)gridDim.x * (256 / CG);
  float2 s2[4], h2[4];
  int64_t ss_n = -1;
  for (int64_t q = (int64_t)blockIdx.x * (256 / CG) + threadIdx.x / CG; q < g.groups; q += stride) {
    const int w0 = (int)(q % wq) * 4;
    const int64_t t = q / wq;
    const int hh = (int)(t % g.h);
    const int64_t nn = t / g.h;
    const bf16* ap = p.a + ((nn * g.h + hh) * (int64_t)g.w + w0) * p.a_ld + cg * 8;
    uint4 raw[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) raw[i] = __ldg(reinterpret_cast<const uint4*>(ap + (int64_t)i * p.a_ld));
    float win[3][6];
    load_window(p.b, p.b_dtype, p.b_ld, g, nn, hh, w0, win);
    if (p.sc && nn != ss_n) {
      ss_n = nn;
      const int64_t si = (p.bcast ? 0 : nn * p.C) + cg * 8;
#pragma unroll
      for (int j = 0; j < 4; ++j) { s2[j] = make_float2(p.sc[si + 2 * j], p.sc[si + 2 * j + 1]); h2[j] = make_float2(p.sh[si + 2 * j], p.sh[si + 2 * j + 1]); }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t wds[4] = {raw[i].x, raw[i].y, raw[i].z, raw[i].w};
      float2 a2[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        a2[j] = bf2_to_f2(wds[j]);
        if (p.sc) a2[j] = ffma2(a2[j], s2[j], h2[j]);
        if (p.relu) { a2[j].x = fmaxf(a2[j].x, 0.f); a2[j].y = fmaxf(a2[j].y, 0.f); }
      }
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          // tap (r, s) has offset (r-1, s-1); b is read at q + sgn*offset
          const float bv = p.sgn > 0 ? win[r][i + s] : win[2 - r][i + 2 - s];
          const float2 b2 = make_float2(bv, bv);
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[r * 3 + s][j] = ffma2(a2[j], b2, acc[r * 3 + s][j]);
        }
    }
  }
  // fold the pixel-quad lanes of each warp (lanes with equal cg), then the 8 warps, in a fixed order
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
      for (int o = CG; o < 32; o <<= 1) {
        acc[t][j].x += __shfl_xor_sync(0xffffffffu, acc[t][j].x, o);
        acc[t][j].y += __shfl_xor_sync(0xffffffffu, acc[t][j].y, o);
      }
    }
  if (lane < CG)
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        red[warp][(lane * 9 + t) * 8 + 2 * j] = acc[t][j].x;
        red[warp][(lane * 9 + t) * 8 + 2 * j + 1] = acc[t][j].y;
      }
  __syncthreads();
  for (int e = threadIdx.x; e < CG * 72; e += 256) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += red[w][e];
    const int c = (e / 72) * 8 + (e & 7), t = (e / 8) % 9;
    p.parts[(int64_t)blockIdx.x * 9 * p.C + (int64_t)c * p.out_c_stride + t * p.out_t_stride] = v;
  }
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
inline int grid_for(int64_t groups, int cgn) {
  const int sms = sm_count();
  const int64_t per_block = 256 / cgn;
  int64_t blocks = (groups + per_block - 1) / per_block;
  if (blocks > sms * 4) blocks = sms * 4;
  return (int)blocks;
}

}  // namespace c1

// forward / data-gradient 1 -> C 3x3 (plain: no prologue, residual, statistics or activation)
int iea_conv_c1_fwd_ok(const iea_conv_desc* d) {
  return d->cin == 1 && d->ksize == 3 && (d->cout == 32 || d->cout == 16 || d->cout == 64) && d->in_mode == IEA_IN_DIRECT &&
         !d->in_scale && !d->in_relu && !d->res && !d->stats && d->acc_c0 < 0 && d->act == IEA_ACT_NONE &&
         d->y_dtype == IEA_BF16 && d->y_ld % 8 == 0 && c1::al16(d->y) && d->w % 4 == 0 && d->out_scale_stride == 0 &&
         (d->x_dtype != IEA_F32 || d->x_ld != 1 || c1::al16(d->x));
}
int iea_conv_c1_fwd(const iea_conv_desc* d, cudaStream_t s) {
  c1::Geo g{d->n, d->h, d->w, d->n * (int64_t)d->h * (d->w / 4)};
  const int cgn = d->cout / 8;
  const int grid = c1::grid_for(g.groups, cgn);
  if (cgn == 4) c1::c1_fwd_kernel<4><<<grid, 256, 0, s>>>(*d, g);
  else if (cgn == 2) c1::c1_fwd_kernel<2><<<grid, 256, 0, s>>>(*d, g);
  else c1::c1_fwd_kernel<8><<<grid, 256, 0, s>>>(*d, g);
  return check_launch("iea_conv_fprop(1-channel)");
}

// weight gradient of the stem (cin 1) and of the output conv (cout 1): 0 = not this kernel's shape
int iea_conv_c1_wgrad_grid(const iea_conv_desc* d, int g_dtype, int g_ld) {
  if (d->ksize != 3 || d->w % 4 || d->in_mode != IEA_IN_DIRECT) return 0;
  int C;
  if (d->cin == 1 && d->cout > 1) {        // stem: a = g
    if (d->in_scale || d->in_relu || g_dtype != IEA_BF16 || g_ld % 8) return 0;
    if (d->x_dtype == IEA_F32 && d->x_ld == 1 && !c1::al16(d->x)) return 0;
    C = d->cout;
  } else if (d->cout == 1 && d->cin > 1) {  // output conv: a = T(x)
    if (d->x_dtype != IEA_BF16 || d->x_ld % 8 || !c1::al16(d->x)) return 0;
    C = d->cin;
  } else {
    return 0;
  }
  if (C != 16 && C != 32 && C != 64) return 0;
  return c1::grid_for(d->n * (int64_t)d->h * (d->w / 4), C / 8);
}
int iea_conv_c1_wgrad(const iea_conv_desc* d, const void* g, int g_dtype, int g_ld, float* parts, cudaStream_t s) {
  const int grid = iea_conv_c1_wgrad_grid(d, g_dtype, g_ld);
  IEA_CHECK_ARG(grid > 0, "iea_conv_wgrad(1-channel): shape not handled");
  c1::Geo geo{d->n, d->h, d->w, d->n * (int64_t)d->h * (d->w / 4)};
  c1::WgP p;
  if (d->cin == 1) {
    IEA_CHECK_ARG(c1::al16(g), "iea_conv_wgrad(1-channel): gradient not 16-byte aligned");
    p = c1::WgP{(const bf16*)g, g_ld, nullptr, nullptr, 0, 0, d->x, d->x_dtype, d->x_ld, +1, 9, 1, d->cout, parts};
  } else {
    const bool g_al = g_dtype != IEA_F32 || g_ld != 1 || c1::al16(g);
    IEA_CHECK_ARG(g_al, "iea_conv_wgrad(1-channel): gradient not 16-byte aligned");
    p = c1::WgP{(const bf16*)d->x, d->x_ld, d->in_scale, d->in_shift, d->in_bcast, d->in_relu, g, g_dtype, g_ld, -1, 1, d->cin,
                d->cin, parts};
  }
  const int cgn = p.C / 8;
  if (cgn == 4) c1::c1_wgrad_kernel<4><<<grid, 256, 0, s>>>(p, geo);
  else if (cgn == 2) c1::c1_wgrad_kernel<2><<<grid, 256, 0, s>>>(p, geo);
  else c1::c1_wgrad_kernel<8><<<grid, 256, 0, s>>>(p, geo);
  return check_launch("iea_conv_wgrad(1-channel)");
}
