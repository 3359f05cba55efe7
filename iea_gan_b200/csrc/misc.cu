// misc.cu -- small bandwidth-bound kernels around the conv path: layout conversion,
// elementwise combine, embedding, pooling, LayerNorm, L2-normalise, the RRM's 40x40
// per-head attention, and the sampling post-process.  All coalesced along the channel /
// feature dimension; reductions are fixed-order (deterministic).
#include "common.cuh"
using namespace iea;

namespace {
inline int ew_blocks(int64_t total, int per = 256) {
  int64_t b = (total + per - 1) / per;
  if (b > 148 * 16) b = 148 * 16;
  return b < 1 ? 1 : (int)b;
}

// ---- layout ----
__global__ void nchw_to_nhwc_kernel(const void* src, int sdt, void* dst, int ddt, int64_t n, int c, int64_t hw) {
  __shared__ float tile[32][33];
  // grid: (hw tiles, c tiles, n)
  const int64_t p0 = (int64_t)blockIdx.x * 32; const int c0 = blockIdx.y * 32; const int64_t nn = blockIdx.z;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int cc = c0 + j; int64_t p = p0 + threadIdx.x;
    tile[j][threadIdx.x] = (cc < c && p < hw) ? ld_act(src, sdt, (nn * c + cc) * hw + p) : 0.f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int64_t p = p0 + j; int cc = c0 + threadIdx.x;
    if (cc < c && p < hw) st_act(dst, ddt, (nn * hw + p) * c + cc, tile[threadIdx.x][j]);
  }
}
__global__ void nhwc_to_nchw_kernel(const void* src, int sdt, void* dst, int ddt, int64_t n, int c, int64_t hw) {
  __shared__ float tile[32][33];
  const int64_t p0 = (int64_t)blockIdx.x * 32; const int c0 = blockIdx.y * 32; const int64_t nn = blockIdx.z;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int64_t p = p0 + j; int cc = c0 + threadIdx.x;
    tile[j][threadIdx.x] = (cc < c && p < hw) ? ld_act(src, sdt, (nn * hw + p) * c + cc) : 0.f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int cc = c0 + j; int64_t p = p0 + threadIdx.x;
    if (cc < c && p < hw) st_act(dst, ddt, (nn * c + cc) * hw + p, tile[threadIdx.x][j]);
  }
}

__global__ void axpby_kernel(const void* a, int adt, float alpha, const void* b, int bdt, float beta, void* y,
                             int ydt, int64_t count) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
    float v = alpha * ld_act(a, adt, i);
    if (b) v = fmaf(beta, ld_act(b, bdt, i), v);
    st_act(y, ydt, i, v);
  }
}

// 8 bf16 per thread and access (16 bytes): the scalar forms below move 2 bytes per load and ran at 1.4 TB/s
__global__ void __launch_bounds__(256) gamma_res_vec_kernel(const uint4* o, const uint4* x, const float* gamma, uint4* y,
                                                            int64_t n8) {
  const float g = gamma[0];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    float a[8], b[8];
    unpack8(o[i], a); unpack8(x[i], b);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = fmaf(g, a[j], b[j]);
    y[i] = pack8(a);
  }
}
__global__ void __launch_bounds__(256) gamma_res_bwd_vec_kernel(const uint4* dy, const uint4* o, const float* gamma,
                                                                uint4* d_o, float* part, int64_t n8) {
  __shared__ float red[33];
  const float g = gamma[0];
  float acc = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    float d[8], v[8];
    unpack8(dy[i], d); unpack8(o[i], v);
#pragma unroll
    for (int j = 0; j < 8; ++j) { acc = fmaf(d[j], v[j], acc); d[j] *= g; }
    d_o[i] = pack8(d);
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) part[blockIdx.x] = acc;
}
__global__ void __launch_bounds__(256) axpby_bf16_vec_kernel(const uint4* a, float alpha, const uint4* b, float beta,
                                                             uint4* y, int64_t n8) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    float u[8], v[8];
    unpack8(a[i], u);
    if (b) {
      unpack8(b[i], v);
#pragma unroll
      for (int j = 0; j < 8; ++j) u[j] = fmaf(beta, v[j], alpha * u[j]);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) u[j] *= alpha;
    }
    y[i] = pack8(u);
  }
}
__device__ __host__ inline bool al16_3(const void* a, const void* b, const void* c) {
  return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c)) & 15) == 0;
}
__global__ void gamma_res_kernel(const void* o, const void* x, int dt, const float* gamma, void* y, int64_t count) {
  const float g = gamma[0];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
    st_act(y, dt, i, fmaf(g, ld_act(o, dt, i), ld_act(x, dt, i)));
}
__global__ void __launch_bounds__(256) gamma_res_bwd_kernel(const void* dy, const void* o, int dt, const float* gamma,
                                                            void* d_o, float* part, int64_t count) {
  __shared__ float red[33];
  const float g = gamma[0];
  float acc = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
    float d = ld_act(dy, dt, i);
    acc = fmaf(d, ld_act(o, dt, i), acc);
    st_act(d_o, dt, i, g * d);
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) part[blockIdx.x] = acc;
}
__global__ void sum_parts_kernel(const float* part, int n, float* out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < n; ++i) t += part[i];
    out[0] = t;
  }
}

// ---- embedding ----
__global__ void embedding_fwd_kernel(const int64_t* idx, const float* w, const float* scale, int64_t n, int dim,
                                     float* out) {
  const float s = scale ? scale[0] : 1.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * dim; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = i / dim; int j = i - r * dim;
    out[i] = w[idx[r] * dim + j] * s;
  }
}
__global__ void embedding_bwd_kernel(const int64_t* idx, const float* dout, const float* scale, int64_t n, int dim,
                                     float* dw) {
  const int r = blockIdx.x;
  const float s = scale ? scale[0] : 1.f;
  for (int j = threadIdx.x; j < dim; j += blockDim.x) {
    float acc = 0.f;
    for (int64_t i = 0; i < n; ++i)
      if (idx[i] == r) acc += dout[i * dim + j];
    dw[(int64_t)r * dim + j] = acc * s;
  }
}

// ---- relu + spatial sum ----
__global__ void __launch_bounds__(256) relu_sumpool_kernel(const void* x, int dt, int64_t hw, int c, float* out, int cb) {
  __shared__ float red[256];
  const int64_t n = blockIdx.x;
  const int lanes = 256 / cb, cl = threadIdx.x % cb, pl = threadIdx.x / cb, cc = blockIdx.y * cb + cl;
  float a = 0.f;
  if (cc < c)
    for (int64_t p = pl; p < hw; p += lanes) a += fmaxf(ld_act(x, dt, (n * hw + p) * c + cc), 0.f);
  red[threadIdx.x] = a;
  __syncthreads();
  if (pl == 0 && cc < c) {
    float t = 0.f;
    for (int l = 0; l < lanes; ++l) t += red[l * cb + cl];
    out[n * c + cc] = t;
  }
}
__global__ void relu_sumpool_bwd_kernel(const void* x, int dt, const float* dout, int64_t n, int64_t hw, int c,
                                        void* dx, int ddt) {
  const int64_t total = n * hw * c;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int cc = i % c; int64_t nn = i / (hw * c);
    st_act(dx, ddt, i, ld_act(x, dt, i) > 0.f ? dout[nn * c + cc] : 0.f);
  }
}

// ---- 2x2 average pool (the DBlock shortcut: model.py:541-557 pools x once for both conv_sc and the identity half) ----
// one thread per (output pixel, 16-byte chunk): vector loads of the four source pixels, fp32 average
template <typename T, int V>
__global__ void __launch_bounds__(256) avgpool2_fwd_kernel(const T* x, int64_t n, int h, int w, int c, int x_ld, T* y, int y_ld) {
  const int ho = h / 2, wo = w / 2, cv = c / V;
  const int64_t total = n * ho * (int64_t)wo * cv;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int cc = (int)(i % cv) * V;
    const int64_t pix = i / cv;
    const int xo = (int)(pix % wo);
    const int64_t t = pix / wo;
    const int yo = (int)(t % ho);
    const int64_t nn = t / ho;
    const T* s0 = x + ((nn * h + 2 * yo) * (int64_t)w + 2 * xo) * x_ld + cc;
    float acc[V];
#pragma unroll
    for (int j = 0; j < V; ++j) acc[j] = 0.f;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        const uint4 q = *reinterpret_cast<const uint4*>(s0 + ((int64_t)a * w + b) * x_ld);
        const T* e = reinterpret_cast<const T*>(&q);
#pragma unroll
        for (int j = 0; j < V; ++j) acc[j] += (float)e[j];
      }
    uint4 o;
    T* eo = reinterpret_cast<T*>(&o);
#pragma unroll
    for (int j = 0; j < V; ++j) eo[j] = (T)(0.25f * acc[j]);
    *reinterpret_cast<uint4*>(y + pix * y_ld + cc) = o;
  }
}

// ---- 2x2 max pool ----
__global__ void maxpool2_fwd_kernel(const void* x, int dt, int64_t n, int h, int w, int c, void* y, uint8_t* idx) {
  const int ho = h / 2, wo = w / 2;
  const int64_t total = n * ho * (int64_t)wo * c;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int cc = i % c; int64_t p = i / c; int xo = p % wo; int64_t t = p / wo; int yo = t % ho; int64_t nn = t / ho;
    float best = -3.4e38f; int bi = 0;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        float v = ld_act(x, dt, ((nn * h + 2 * yo + a) * (int64_t)w + 2 * xo + b) * c + cc);
        if (v > best) { best = v; bi = a * 2 + b; }
      }
    st_act(y, dt, i, best);
    idx[i] = (uint8_t)bi;
  }
}
__global__ void maxpool2_bwd_kernel(const void* dy, int dt, const uint8_t* idx, int64_t n, int h, int w, int c, void* dx) {
  const int ho = h / 2, wo = w / 2;
  const int64_t total = n * h * (int64_t)w * c;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int cc = i % c; int64_t p = i / c; int xx = p % w; int64_t t = p / w; int yy = t % h; int64_t nn = t / h;
    int64_t o = ((nn * ho + (yy >> 1)) * (int64_t)wo + (xx >> 1)) * c + cc;
    int sel = (yy & 1) * 2 + (xx & 1);
    st_act(dx, dt, i, idx[o] == sel ? ld_act(dy, dt, o) : 0.f);
  }
}

// ---- LayerNorm ----
__global__ void __launch_bounds__(128) layernorm_fwd_kernel(const float* x, const float* g, const float* b, int dim,
                                                            float eps, float* y, float* mean, float* rstd) {
  __shared__ float red[33];
  const int64_t r = blockIdx.x;
  const float* xr = x + r * dim;
  float s = 0.f;
  for (int j = threadIdx.x; j < dim; j += blockDim.x) s += xr[j];
  const float mu = block_sum(s, red) / dim;
  float v = 0.f;
  for (int j = threadIdx.x; j < dim; j += blockDim.x) { float d = xr[j] - mu; v = fmaf(d, d, v); }
  const float rs = rsqrtf(block_sum(v, red) / dim + eps);
  for (int j = threadIdx.x; j < dim; j += blockDim.x) y[r * dim + j] = (xr[j] - mu) * rs * g[j] + b[j];
  if (threadIdx.x == 0 && mean) { mean[r] = mu; rstd[r] = rs; }
}
__global__ void __launch_bounds__(128) layernorm_bwd_dx_kernel(const float* dy, const float* x, const float* g,
                                                               const float* mean, const float* rstd, int dim,
                                                               float* dx) {
  __shared__ float red[33];
  const int64_t r = blockIdx.x;
  const float mu = mean[r], rs = rstd[r];
  float a = 0.f, b = 0.f;
  for (int j = threadIdx.x; j < dim; j += blockDim.x) {
    float d = dy[r * dim + j] * g[j], xh = (x[r * dim + j] - mu) * rs;
    a += d; b = fmaf(d, xh, b);
  }
  a = block_sum(a, red) / dim;
  b = block_sum(b, red) / dim;
  for (int j = threadIdx.x; j < dim; j += blockDim.x) {
    float d = dy[r * dim + j] * g[j], xh = (x[r * dim + j] - mu) * rs;
    dx[r * dim + j] = rs * (d - a - xh * b);
  }
}
__global__ void layernorm_bwd_gb_kernel(const float* dy, const float* x, const float* mean, const float* rstd,
                                        int64_t rows, int dim, float* dg, float* db) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= dim) return;
  float a = 0.f, b = 0.f;
  for (int64_t r = 0; r < rows; ++r) {
    float d = dy[r * dim + j];
    a = fmaf(d, (x[r * dim + j] - mean[r]) * rstd[r], a);
    b += d;
  }
  dg[j] = a; db[j] = b;
}

// ---- L2 normalise ----
__global__ void __launch_bounds__(128) l2norm_fwd_kernel(const float* x, int dim, float eps, float* y, float* norm) {
  __shared__ float red[33];
  const int64_t r = blockIdx.x;
  float s = 0.f;
  for (int j = threadIdx.x; j < dim; j += blockDim.x) s = fmaf(x[r * dim + j], x[r * dim + j], s);
  const float nr = sqrtf(block_sum(s, red));
  const float inv = 1.f / fmaxf(nr, eps);
  for (int j = threadIdx.x; j < dim; j += blockDim.x) y[r * dim + j] = x[r * dim + j] * inv;
  if (threadIdx.x == 0 && norm) norm[r] = nr;
}
__global__ void __launch_bounds__(128) l2norm_bwd_kernel(const float* dy, const float* y, const float* norm, int dim,
                                                         float eps, float* dx) {
  __shared__ float red[33];
  const int64_t r = blockIdx.x;
  float s = 0.f;
  for (int j = threadIdx.x; j < dim; j += blockDim.x) s = fmaf(dy[r * dim + j], y[r * dim + j], s);
  const float dot = block_sum(s, red);
  const float nr = norm[r];
  const float inv = 1.f / fmaxf(nr, eps);
  const float k = nr > eps ? dot : 0.f;  // below eps the denominator is the constant eps
  for (int j = threadIdx.x; j < dim; j += blockDim.x) dx[r * dim + j] = (dy[r * dim + j] - y[r * dim + j] * k) * inv;
}

// ---- RRM per-head attention over the `seq` (=40) sensors of an event ----
// block per (event, head); dynamic smem: q,k,v [seq][d] + att [seq][seq]
__global__ void __launch_bounds__(256) mha_fwd_kernel(const float* qkv, int seq, int heads, int d, float* val,
                                                      float* att_out) {
  extern __shared__ float sm[];
  float* q = sm; float* k = q + seq * d; float* v = k + seq * d; float* att = v + seq * d;
  const int e = blockIdx.x / heads, hd = blockIdx.x % heads;
  const float* base = qkv + ((int64_t)e * seq * heads + hd) * 3 * d;
  const int rs = heads * 3 * d;
  for (int i = threadIdx.x; i < seq * d; i += blockDim.x) {
    int s = i / d, j = i - s * d;
    q[i] = base[(int64_t)s * rs + j];
    k[i] = base[(int64_t)s * rs + d + j];
    v[i] = base[(int64_t)s * rs + 2 * d + j];
  }
  __syncthreads();
  const float scl = rsqrtf((float)d);
  for (int i = threadIdx.x; i < seq * seq; i += blockDim.x) {
    int a = i / seq, b = i - a * seq;
    float acc = 0.f;
    for (int j = 0; j < d; ++j) acc = fmaf(q[a * d + j], k[b * d + j], acc);
    att[i] = acc * scl;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int a = wid; a < seq; a += 8) {  // one warp per row
    float m = -3.4e38f;
    for (int b = lane; b < seq; b += 32) m = fmaxf(m, att[a * seq + b]);
    m = warp_max(m);
    float s = 0.f;
    for (int b = lane; b < seq; b += 32) { float ex = __expf(att[a * seq + b] - m); att[a * seq + b] = ex; s += ex; }
    s = warp_sum(s);
    float inv = 1.f / s;
    for (int b = lane; b < seq; b += 32) att[a * seq + b] *= inv;
  }
  __syncthreads();
  float* ao = att_out + (int64_t)blockIdx.x * seq * seq;
  for (int i = threadIdx.x; i < seq * seq; i += blockDim.x) ao[i] = att[i];
  for (int i = threadIdx.x; i < seq * d; i += blockDim.x) {
    int a = i / d, j = i - a * d;
    float acc = 0.f;
    for (int b = 0; b < seq; ++b) acc = fmaf(att[a * seq + b], v[b * d + j], acc);
    val[((int64_t)e * seq + a) * heads * d + hd * d + j] = acc;
  }
}

__global__ void __launch_bounds__(256) mha_bwd_kernel(const float* dval, const float* qkv, const float* att_in,
                                                      int seq, int heads, int d, float* dqkv) {
  extern __shared__ float sm[];
  float* q = sm; float* k = q + seq * d; float* v = k + seq * d; float* dO = v + seq * d;
  float* att = dO + seq * d; float* dS = att + seq * seq;
  const int e = blockIdx.x / heads, hd = blockIdx.x % heads;
  const int rs = heads * 3 * d;
  const float* base = qkv + ((int64_t)e * seq * heads + hd) * 3 * d;
  float* dbase = dqkv + ((int64_t)e * seq * heads + hd) * 3 * d;
  for (int i = threadIdx.x; i < seq * d; i += blockDim.x) {
    int s = i / d, j = i - s * d;
    q[i] = base[(int64_t)s * rs + j];
    k[i] = base[(int64_t)s * rs + d + j];
    v[i] = base[(int64_t)s * rs + 2 * d + j];
    dO[i] = dval[((int64_t)e * seq + s) * heads * d + hd * d + j];
  }
  const float* ai = att_in + (int64_t)blockIdx.x * seq * seq;
  for (int i = threadIdx.x; i < seq * seq; i += blockDim.x) att[i] = ai[i];
  __syncthreads();
  // dAtt = dO V^T
  for (int i = threadIdx.x; i < seq * seq; i += blockDim.x) {
    int a = i / seq, b = i - a * seq;
    float acc = 0.f;
    for (int j = 0; j < d; ++j) acc = fmaf(dO[a * d + j], v[b * d + j], acc);
    dS[i] = acc;
  }
  __syncthreads();
  const float scl = rsqrtf((float)d);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int a = wid; a < seq; a += 8) {
    float s = 0.f;
    for (int b = lane; b < seq; b += 32) s = fmaf(dS[a * seq + b], att[a * seq + b], s);
    s = warp_sum(s);
    for (int b = lane; b < seq; b += 32) dS[a * seq + b] = att[a * seq + b] * (dS[a * seq + b] - s) * scl;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < seq * d; i += blockDim.x) {
    int a = i / d, j = i - a * d;
    float dq = 0.f, dk = 0.f, dv = 0.f;
    for (int b = 0; b < seq; ++b) {
      dq = fmaf(dS[a * seq + b], k[b * d + j], dq);
      dk = fmaf(dS[b * seq + a], q[b * d + j], dk);
      dv = fmaf(att[b * seq + a], dO[b * d + j], dv);
    }
    dbase[(int64_t)a * rs + j] = dq;
    dbase[(int64_t)a * rs + d + j] = dk;
    dbase[(int64_t)a * rs + 2 * d + j] = dv;
  }
}

__global__ void adu_kernel(const float* img, int64_t n, int h, int w, float* out) {
  const int ho = h - 6;
  const int64_t total = n * ho * (int64_t)w;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int x = i % w; int64_t t = i / w; int y = t % ho; int64_t nn = t / ho;
    float v = img[(nn * h + y + 3) * (int64_t)w + x];
    v = v > -0.26f ? v : -1.f;
    v = exp2f(8.f * (v * 0.5f + 0.5f)) - 1.f;
    out[i] = fminf(fmaxf(v, 0.f), 255.f);
  }
}
// Input side of the step (SURVEY 8(f) N4): what utils/dataloader.py:69-77 does per decoded PNG on the CPU --
// Pad((0,3,0,3)) with zeros, ToTensor (/255), fn_lognorm255 = log(255 v + 1) / log 256 (utils/norm.py:8-18),
// UniformNoise(scale) = + scale * U[0,1) (utils/noise.py:32-35, padding rows included), Normalize(0.5, 0.5) --
// as one pass over a pre-decoded uint8 event tensor: 1 byte in (+ 4 of noise), 4 bytes out per pixel.
__global__ void event_preprocess_kernel(const uint8_t* img, int64_t n, int h_in, int w, int pad, const float* noise,
                                        float scale, float* out) {
  const int h = h_in + 2 * pad;
  const int64_t total = n * h * (int64_t)w;
  const float inv_log256 = 0.18033688011112042f;  // 1 / ln 256
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int x = i % w; const int64_t t = i / w; const int y = t % h; const int64_t nn = t / h;
    const int ys = y - pad;
    float v = 0.f;
    if (ys >= 0 && ys < h_in) v = logf((float)img[(nn * h_in + ys) * (int64_t)w + x] + 1.f) * inv_log256;
    if (noise) v = fmaf(scale, noise[i], v);
    out[i] = (v - 0.5f) / 0.5f;
  }
}
}  // namespace

extern "C" {
int iea_event_preprocess(const uint8_t* img, int64_t n, int h_in, int w, int pad, const float* noise, float scale,
                         float* out, iea_stream_t st) {
  IEA_CHECK_ARG(n > 0 && h_in > 0 && w > 0 && pad >= 0, "iea_event_preprocess: bad geometry");
  event_preprocess_kernel<<<ew_blocks(n * (h_in + 2 * pad) * (int64_t)w), 256, 0, (cudaStream_t)st>>>(
      img, n, h_in, w, pad, noise, scale, out);
  return check_launch("iea_event_preprocess");
}
int iea_nchw_to_nhwc(const void* src, int sdt, void* dst, int ddt, int64_t n, int c, int64_t hw, iea_stream_t st) {
  dim3 grid(cdiv(hw, 32), cdiv(c, 32), (unsigned)n), block(32, 8);
  nchw_to_nhwc_kernel<<<grid, block, 0, (cudaStream_t)st>>>(src, sdt, dst, ddt, n, c, hw);
  return check_launch("iea_nchw_to_nhwc");
}
int iea_nhwc_to_nchw(const void* src, int sdt, void* dst, int ddt, int64_t n, int c, int64_t hw, iea_stream_t st) {
  dim3 grid(cdiv(hw, 32), cdiv(c, 32), (unsigned)n), block(32, 8);
  nhwc_to_nchw_kernel<<<grid, block, 0, (cudaStream_t)st>>>(src, sdt, dst, ddt, n, c, hw);
  return check_launch("iea_nhwc_to_nchw");
}
int iea_axpby(const void* a, int adt, float alpha, const void* b, int bdt, float beta, void* y, int ydt,
              int64_t count, iea_stream_t st) {
  if (adt == IEA_BF16 && ydt == IEA_BF16 && (!b || bdt == IEA_BF16) && count % 8 == 0 && al16_3(a, b ? b : a, y)) {
    axpby_bf16_vec_kernel<<<ew_blocks(count / 8), 256, 0, (cudaStream_t)st>>>((const uint4*)a, alpha, (const uint4*)b, beta,
                                                                               (uint4*)y, count / 8);
    return check_launch("iea_axpby");
  }
  axpby_kernel<<<ew_blocks(count), 256, 0, (cudaStream_t)st>>>(a, adt, alpha, b, bdt, beta, y, ydt, count);
  return check_launch("iea_axpby");
}
int iea_gamma_residual(const void* o, const void* x, int dt, const float* gamma, void* y, int64_t count,
                       iea_stream_t st) {
  if (dt == IEA_BF16 && count % 8 == 0 && al16_3(o, x, y)) {
    gamma_res_vec_kernel<<<ew_blocks(count / 8), 256, 0, (cudaStream_t)st>>>((const uint4*)o, (const uint4*)x, gamma, (uint4*)y,
                                                                               count / 8);
    return check_launch("iea_gamma_residual");
  }
  gamma_res_kernel<<<ew_blocks(count), 256, 0, (cudaStream_t)st>>>(o, x, dt, gamma, y, count);
  return check_launch("iea_gamma_residual");
}
int iea_gamma_residual_bwd(const void* dy, const void* o, int dt, const float* gamma, void* d_o, float* dgamma,
                           float* scratch, int64_t count, iea_stream_t st) {
  int blocks = ew_blocks(count, 1024);
  if (blocks > 512) blocks = 512;
  if (dt == IEA_BF16 && count % 8 == 0 && al16_3(dy, o, d_o))
    gamma_res_bwd_vec_kernel<<<blocks, 256, 0, (cudaStream_t)st>>>((const uint4*)dy, (const uint4*)o, gamma, (uint4*)d_o,
                                                                     scratch, count / 8);
  else
    gamma_res_bwd_kernel<<<blocks, 256, 0, (cudaStream_t)st>>>(dy, o, dt, gamma, d_o, scratch, count);
  sum_parts_kernel<<<1, 32, 0, (cudaStream_t)st>>>(scratch, blocks, dgamma);
  return check_launch("iea_gamma_residual_bwd");
}
int iea_embedding_fwd(const int64_t* idx, const float* w, const float* scale, int64_t n, int dim, float* out,
                      iea_stream_t st) {
  embedding_fwd_kernel<<<ew_blocks(n * dim), 256, 0, (cudaStream_t)st>>>(idx, w, scale, n, dim, out);
  return check_launch("iea_embedding_fwd");
}
int iea_embedding_bwd(const int64_t* idx, const float* dout, const float* scale, int64_t n, int dim, int rows,
                      float* dw, iea_stream_t st) {
  embedding_bwd_kernel<<<rows, 256, 0, (cudaStream_t)st>>>(idx, dout, scale, n, dim, dw);
  return check_launch("iea_embedding_bwd");
}
int iea_relu_sumpool_fwd(const void* x, int dt, int64_t n, int64_t hw, int c, float* out, iea_stream_t st) {
  int cb = 1;
  while (cb < c && cb < 32) cb <<= 1;
  dim3 grid((unsigned)n, cdiv(c, cb));
  relu_sumpool_kernel<<<grid, 256, 0, (cudaStream_t)st>>>(x, dt, hw, c, out, cb);
  return check_launch("iea_relu_sumpool_fwd");
}
int iea_relu_sumpool_bwd(const void* x, int dt, const float* dout, int64_t n, int64_t hw, int c, void* dx, int ddt,
                         iea_stream_t st) {
  relu_sumpool_bwd_kernel<<<ew_blocks(n * hw * c), 256, 0, (cudaStream_t)st>>>(x, dt, dout, n, hw, c, dx, ddt);
  return check_launch("iea_relu_sumpool_bwd");
}
int iea_avgpool2_fwd(const void* x, int dt, int64_t n, int h, int w, int c, int x_ld, void* y, int y_ld, iea_stream_t st) {
  IEA_CHECK_ARG(h % 2 == 0 && w % 2 == 0, "iea_avgpool2_fwd: odd spatial size %dx%d", h, w);
  const int v = dt == IEA_BF16 ? 8 : 4;
  IEA_CHECK_ARG(c % v == 0 && x_ld % v == 0 && y_ld % v == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)y & 15) == 0,
                "iea_avgpool2_fwd: channel counts / pitches must be multiples of %d elements and 16-byte aligned", v);
  const int64_t total = n * (h / 2) * (int64_t)(w / 2) * (c / v);
  if (dt == IEA_BF16)
    avgpool2_fwd_kernel<bf16, 8><<<ew_blocks(total), 256, 0, (cudaStream_t)st>>>((const bf16*)x, n, h, w, c, x_ld, (bf16*)y, y_ld);
  else
    avgpool2_fwd_kernel<float, 4><<<ew_blocks(total), 256, 0, (cudaStream_t)st>>>((const float*)x, n, h, w, c, x_ld, (float*)y, y_ld);
  return check_launch("iea_avgpool2_fwd");
}
int iea_maxpool2_fwd(const void* x, int dt, int64_t n, int h, int w, int c, void* y, uint8_t* idx, iea_stream_t st) {
  IEA_CHECK_ARG(h % 2 == 0 && w % 2 == 0, "iea_maxpool2_fwd: odd spatial size %dx%d", h, w);
  maxpool2_fwd_kernel<<<ew_blocks(n * (h / 2) * (int64_t)(w / 2) * c), 256, 0, (cudaStream_t)st>>>(x, dt, n, h, w, c, y, idx);
  return check_launch("iea_maxpool2_fwd");
}
int iea_maxpool2_bwd(const void* dy, int dt, const uint8_t* idx, int64_t n, int h, int w, int c, void* dx,
                     iea_stream_t st) {
  maxpool2_bwd_kernel<<<ew_blocks(n * h * (int64_t)w * c), 256, 0, (cudaStream_t)st>>>(dy, dt, idx, n, h, w, c, dx);
  return check_launch("iea_maxpool2_bwd");
}
int iea_layernorm_fwd(const float* x, const float* g, const float* b, int64_t rows, int dim, float eps, float* y,
                      float* mean, float* rstd, iea_stream_t st) {
  layernorm_fwd_kernel<<<(unsigned)rows, 128, 0, (cudaStream_t)st>>>(x, g, b, dim, eps, y, mean, rstd);
  return check_launch("iea_layernorm_fwd");
}
int iea_layernorm_bwd(const float* dy, const float* x, const float* g, const float* mean, const float* rstd,
                      int64_t rows, int dim, float* dx, float* dg_part, float* db_part, int nparts, iea_stream_t st) {
  (void)nparts;
  layernorm_bwd_dx_kernel<<<(unsigned)rows, 128, 0, (cudaStream_t)st>>>(dy, x, g, mean, rstd, dim, dx);
  if (dg_part)
    layernorm_bwd_gb_kernel<<<cdiv(dim, 64), 64, 0, (cudaStream_t)st>>>(dy, x, mean, rstd, rows, dim, dg_part, db_part);
  return check_launch("iea_layernorm_bwd");
}
int iea_l2norm_fwd(const float* x, int64_t rows, int dim, float eps, float* y, float* norm, iea_stream_t st) {
  l2norm_fwd_kernel<<<(unsigned)rows, 128, 0, (cudaStream_t)st>>>(x, dim, eps, y, norm);
  return check_launch("iea_l2norm_fwd");
}
int iea_l2norm_bwd(const float* dy, const float* y, const float* norm, int64_t rows, int dim, float eps, float* dx,
                   iea_stream_t st) {
  l2norm_bwd_kernel<<<(unsigned)rows, 128, 0, (cudaStream_t)st>>>(dy, y, norm, dim, eps, dx);
  return check_launch("iea_l2norm_bwd");
}
int iea_mha_fwd(const float* qkv, int events, int seq, int heads, int d, float* val, float* att, iea_stream_t st) {
  size_t smem = (size_t)(3 * seq * d + seq * seq) * sizeof(float);
  IEA_CHECK_ARG(smem <= 200 * 1024, "iea_mha_fwd: seq=%d d=%d needs %zu B of shared memory", seq, d, smem);
  IEA_CUDA(cudaFuncSetAttribute(mha_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mha_fwd_kernel<<<events * heads, 256, smem, (cudaStream_t)st>>>(qkv, seq, heads, d, val, att);
  return check_launch("iea_mha_fwd");
}
int iea_mha_bwd(const float* dval, const float* qkv, const float* att, int events, int seq, int heads, int d,
                float* dqkv, iea_stream_t st) {
  size_t smem = (size_t)(4 * seq * d + 2 * seq * seq) * sizeof(float);
  IEA_CHECK_ARG(smem <= 200 * 1024, "iea_mha_bwd: seq=%d d=%d needs %zu B of shared memory", seq, d, smem);
  IEA_CUDA(cudaFuncSetAttribute(mha_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mha_bwd_kernel<<<events * heads, 256, smem, (cudaStream_t)st>>>(dval, qkv, att, seq, heads, d, dqkv);
  return check_launch("iea_mha_bwd");
}
int iea_adu_postprocess(const float* img, int64_t n, int h, int w, float* out, iea_stream_t st) {
  IEA_CHECK_ARG(h > 6, "iea_adu_postprocess: image height %d too small for the 3-row crop", h);
  adu_kernel<<<ew_blocks(n * (h - 6) * (int64_t)w), 256, 0, (cudaStream_t)st>>>(img, n, h, w, out);
  return check_launch("iea_adu_postprocess");
}
}
