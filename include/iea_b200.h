/* iea_b200.h -- C ABI of libiea_sm100.so, the sm_100a (B200) implementation of the
 * IEA-GAN Generator/Discriminator hot path.
 *
 * Conventions
 *   - every entry point returns 0 on success and a negative code on failure; the
 *     message is available from iea_last_error() (thread local).
 *   - all pointers are DEVICE pointers unless a comment says host; the library never
 *     allocates, frees or synchronises: the caller owns every buffer (inputs, outputs,
 *     saved tensors and scratch) and passes the CUDA stream to enqueue on.
 *   - activations are NHWC ([n][h][w][c], channel stride 1, pixel stride `ld`), element
 *     type given by an iea_dtype code; parameters stay fp32 in the reference's layout.
 *   - rows of a batch are grouped by event: 40 consecutive images (model.py:466).
 *
 * Each declaration cites the reference interface (file:line in Baran-phys/IEA-GAN) whose
 * arithmetic it replaces.  INTEGRATION.md shows the ctypes binding.
 */
#ifndef IEA_B200_H
#define IEA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* iea_stream_t; /* cudaStream_t */

enum iea_dtype { IEA_F32 = 0, IEA_BF16 = 1 };
enum iea_in_mode { IEA_IN_DIRECT = 0, IEA_IN_UP2 = 1, IEA_IN_POOL2 = 2 };
enum iea_act { IEA_ACT_NONE = 0, IEA_ACT_RELU = 1, IEA_ACT_TANH = 2 };
/* convolution kernel choice (iea_conv_desc.impl): AUTO picks by shape; GENERIC forces the CUDA-core kernel;
 * TCGEN05 forces the tcgen05 kernels (an error where they reject the shape); TC_STREAM is TCGEN05 with the
 * streaming conv_tc kernel wherever it accepts the shape (the reference the other tcgen05 kernels are checked
 * against), else the resident-weight conv_tc2 kernel; TC2 routes as AUTO except that the 1x1 layers conv_wide takes run
 * on conv_tc2 (the reference conv_wide is checked against). */
enum iea_impl { IEA_IMPL_AUTO = 0, IEA_IMPL_GENERIC = 1, IEA_IMPL_TCGEN05 = 2, IEA_IMPL_TC_STREAM = 3, IEA_IMPL_TC2 = 4 };

/* ---- library ------------------------------------------------------------------ */
int iea_version(void);
const char* iea_last_error(void);
/* fails unless the current device is compute capability 10.x (no fallback path) */
int iea_require_sm100(int device);
int iea_sm_count(int device);

/* ---- spectral norm: layers.py:89-111 power_iteration, layers.py:151-165 SN.W_ ----
 * One grouped call runs the power iteration of EVERY listed layer (v = norm(uW),
 * u' = norm(vW^T), sigma = |vW^T|) and repacks the fp32 master weight into the
 * activation dtype in the two layouts the conv kernels consume.  W/sigma is never
 * materialised: 1/sigma is applied in the conv epilogue. */
typedef struct {
  const float* w;        /* [rows][cin][taps] fp32 master weight (taps = k*k, cols = cin*taps) */
  const float* u_in;     /* [rows] stored u0 */
  float* u_out;          /* [rows] u' (u0 itself when training, scratch otherwise) */
  float* v_out;          /* [cols] v, saved for the backward rank-1 correction */
  float* sigma_out;      /* [1] sv0 when training, scratch otherwise; may be NULL */
  float* inv_sigma_out;  /* [1] 1/sigma (1.0 when !spectral) */
  float* colscale_out;   /* optional [colscale_n]: filled with 1/sigma (grouped ccbn GEMM) */
  void* pack_fprop;      /* optional [rows][taps][cin] in pack_dtype */
  void* pack_dgrad;      /* optional [cin][taps, spatially flipped][pack_dgrad_ld >= rows] in pack_dtype */
  int32_t rows, cin, taps, colscale_n;
  int32_t pack_dgrad_ld; /* row stride of pack_dgrad (lets several layers share one dgrad matrix) */
  /* optional bf16 copies in the tcgen05 kernel's smem-image order [tap][k block][16-byte chunk][row][8]:
   * one contiguous slice per (tap, k block) so the weight operand is a plain TMA bulk copy */
  void* pack_tc_fprop;   /* rows = cout, k blocks over cin */
  void* pack_tc_dgrad;   /* rows = cin, k blocks over cout, taps spatially flipped */
  int32_t pack_tc_rows;  /* row count of the pack_tc_fprop layout (cout rounded up to 16; extra rows stay 0) */
  int32_t pack_tc_cin;   /* row count of the pack_tc_dgrad layout (cin rounded up to 16) */
  int32_t pack_dtype;    /* iea_dtype */
  int32_t spectral;      /* 0: plain layer, only repack */
  float eps;
  int32_t chunk0;        /* first entry of this layer in the chunk table */
  int32_t nchunks;
  int64_t scratch_off;   /* float offset of this layer's scratch (partials + t) */
} iea_sn_layer;
/* chunk table: int32 triples (layer, row_begin, row_end); scratch: fp32 */
int iea_sn_power_iter(const iea_sn_layer* layers_dev, int n_layers, const int32_t* chunks_dev,
                      int n_chunks, float* scratch, int max_cols, iea_stream_t stream);

/* backward of W/sigma (SURVEY.md Appendix B.1): dW = G/sigma - (<G,W>/sigma^2) u'^T v, where
 * G = sum over `nsplit` wgrad partials [nsplit][rows][taps][cin] (fp32).  Writes (beta=0) or
 * accumulates (beta=1) dW in the master layout [rows][cin][taps]. */
int iea_sn_weight_bwd(const float* gpart, int nsplit, const float* w, const float* u, const float* v,
                      const float* inv_sigma, int spectral, float* dw, float beta, int rows, int cin,
                      int taps, float* scratch /* >= 2 + 2*gridcap floats */, iea_stream_t stream);

/* the same for many layers in two launches: items live in device memory, sorted by block0; item i owns the
 * blocks [block0, block0 + nblocks) of the grid of total_blocks (nblocks = ceil(rows*cin*taps / 1024), <= 256);
 * scratch >= total_blocks floats. */
typedef struct {
  const float* gpart; const float* w; const float* u; const float* v; const float* inv_sigma; float* dw;
  int32_t nsplit, spectral, rows, cin, taps; float beta;
  int32_t block0, nblocks;
} iea_sn_bwd_item;
int iea_sn_weight_bwd_grouped(const iea_sn_bwd_item* items_dev, int n_items, int total_blocks, float* scratch,
                              iea_stream_t stream);

/* ---- fused convolution / linear: layers.py:197-206 SNConv2d.forward, :223-224 SNLinear ----
 * y = act( conv_k(T(x), Wpack) * out_scale + bias + residual ), with
 *   T(x) = [avgpool2 | nearest-up2]( relu?( x * in_scale[n][c] + in_shift[n][c] ) )
 * (T fuses ccbn/bn apply + ReLU + F.interpolate / AvgPool2d: model.py:56-70, 545-556) and an
 * optional per-128-row-tile (sum, sum of squares) of y for the next batch-norm. A linear
 * layer is the 1x1 case with h = w = 1.  The same kernel is the data-gradient when given
 * pack_dgrad weights. */
typedef struct {
  int64_t n; int32_t h, w;             /* output (= conv input after T) geometry */
  int32_t cin, cout, ksize;            /* ksize 1 or 3, stride 1, padding ksize/2 */
  const void* x; int32_t x_dtype, x_ld, in_mode, in_relu;
  const float* in_scale; const float* in_shift;   /* [n][cin] ([cin] when in_bcast) or NULL */
  int32_t in_bcast;
  const void* wpack; int32_t w_dtype;  /* [cout][taps][cin] */
  const void* wpack_tc;                /* same weights in the tcgen05 order (iea_sn_layer.pack_tc_*) or NULL */
  int32_t cout_tc;                     /* row count of wpack_tc (cout rounded up to 16); 0: = cout */
  const float* out_scale; int32_t out_scale_stride; /* 0: scalar, 1: per out channel; NULL: 1 */
  const float* bias;                   /* [cout] or NULL */
  const void* res; int32_t res_dtype, res_ld, res_mode, res_c; /* residual for channels < res_c */
  int32_t acc_c0;                      /* channels >= acc_c0 add the existing y value; <0: off */
  void* y; int32_t y_dtype, y_ld, act;
  float* stats;                        /* [events][iea_conv_stats_slots()][cout][2] or NULL */
  int32_t impl;                        /* iea_impl */
} iea_conv_desc;
int iea_conv_fprop(const iea_conv_desc* d /* host */, iea_stream_t stream);
/* number of batch-norm partial-sum slots PER EVENT that iea_conv_fprop writes into d->stats for this
 * descriptor (d->stats must be non-NULL when asking): the buffer is [events][slots][cout][2] floats and
 * must be zero-filled by the caller; 0 = the kernel cannot emit statistics for this geometry.  The count
 * comes from the same kernel choice iea_conv_fprop makes, d->impl included. */
int iea_conv_stats_slots(const iea_conv_desc* d /* host */);
/* 1 if the tcgen05 path accepts this descriptor */
int iea_conv_tc_supported(const iea_conv_desc* d /* host */);

/* weight gradient: gpart[s][cout][taps][cin] = sum over the rows of split s of g[m][co]*T(x)[m][k];
 * g is the gradient at the conv accumulator (dtype g_dtype, pixel stride g_ld). */
int iea_conv_wgrad(const iea_conv_desc* d /* host; x/T fields and geometry are used */, const void* g,
                   int g_dtype, int g_ld, float* gpart, int nsplit, iea_stream_t stream);

/* tensor-core (mma.sync m16n8k16) split-K weight gradient for the thin high-resolution layers.
 * iea_conv_wgrad_mma_slices returns the number of partial slices the kernel will write for this shape
 * (0: shape not handled -> use iea_conv_wgrad); gpart must hold slices*cout*taps*cin floats.  On return
 * slice 0 holds the fixed-order sum of the per-CTA partials (pass it to iea_sn_weight_bwd with nsplit 1).
 * dbias != NULL asks for the bias gradient sum_px g[px][co] from the same pass (one extra MMA per k-step
 * on the g fragments already in registers); returns 1 when dbias was written, 0 when the shape's kernel
 * does not produce it (the caller then runs iea_colsum), < 0 on error. */
int iea_conv_wgrad_mma_slices(const iea_conv_desc* d /* host */, int g_dtype, int g_ld);
int iea_conv_wgrad_mma(const iea_conv_desc* d /* host */, const void* g, int g_dtype, int g_ld, float* gpart,
                       float* dbias /* [cout] or NULL */, iea_stream_t stream);

/* backward of T: da [n][h][w][cin] (at conv resolution) -> dx at x's resolution and the
 * per-(n,c) reductions dscale = sum da*relu'*x, dshift = sum da*relu'.  beta=1 accumulates dx. */
int iea_conv_input_bwd(const iea_conv_desc* d /* host */, const void* da, int da_dtype, void* dx,
                       int dx_dtype, int dx_ld, float beta, float* dscale, float* dshift,
                       float* scratch /* >= n*64*cin*2 floats, or NULL (slow path) */, iea_stream_t stream);

/* g = (dy [* (1 - y^2) if act == TANH]) + ds1[e][c] + 2*y*ds2[e][c]   (batch-norm statistics path) */
int iea_conv_out_bwd(const void* dy, int dy_dtype, int dy_ld, const void* y, int y_dtype, int y_ld,
                     int act, const float* ds1, const float* ds2, int64_t rows, int rows_per_event,
                     int c, void* g, int g_dtype, iea_stream_t stream);

/* out[c] = sum_m g[m][c] (bias gradient); scratch >= blocks*c floats */
int iea_colsum(const void* g, int g_dtype, int g_ld, int64_t rows, int c, float* out, float beta,
               float* scratch, iea_stream_t stream);

/* residual gradient: dres[n][h'][w'][c<res_c] (+)= adjoint of the epilogue's residual read */
int iea_residual_bwd(const void* g, int g_dtype, int g_ld, int64_t n, int h, int w, int res_c,
                     int res_mode, void* dres, int dres_dtype, int dres_ld, int dres_c, float beta,
                     iea_stream_t stream);

/* ---- batch norm: layers.py:656-689 ccbn.forward, :728-742 bn.forward --------------- */
/* stand-alone statistics partials: [events][tiles][c][2] */
int iea_bn_stats(const void* x, int x_dtype, int x_ld, int64_t rows, int rows_per_event, int c,
                 int tiles_per_event, float* partials, iea_stream_t stream);
/* partials -> batch mean / rstd per (event, c) (biased variance), running-stat update when
 * training; eval (mode 0) uses the stored statistics.
 * mode bits: 1 = batch statistics + F.batch_norm running update (momentum, UNBIASED variance,
 * layers.py:664-673); 1|2 = myBN running update (momentum, biased variance, layers.py:585-592);
 * 1|4 = myBN standing statistics (stored += batch statistic, layers.py:579-582).
 * scale[n][c] = rstd*(gain_add + gain[n*gain_ld + c]); shift = bias - mean*scale.
 * ticket: caller-owned, ceil(c/8) zero-initialised counters private to this layer (self-resetting);
 * with it the training path is ONE launch, without it (NULL) three. */
int iea_bn_finalize(const float* partials, int events, int tiles_per_event, int64_t count_per_event,
                    int imgs_per_event, int c, const float* gain, int64_t gain_ld, float gain_add,
                    const float* bias, int64_t bias_ld, float* stored_mean, float* stored_var,
                    int mode, float momentum, float eps, float* mean_out, float* rstd_out,
                    float* scale, float* shift, unsigned int* ticket, iea_stream_t stream);
/* backward: (dscale, dshift)[n][c] -> dgain[n][c], dbias[n][c] (pixel-stride ld, beta accumulate)
 * and the statistics gradients ds1, ds2 [events][c] consumed by iea_conv_out_bwd. */
int iea_bn_finalize_bwd(const float* dscale, const float* dshift, const float* scale,
                        const float* mean, const float* rstd, int events, int imgs_per_event,
                        int64_t count_per_event, int c, const float* gain, int64_t gain_ld,
                        float gain_add, float* dgain, int64_t dgain_ld, float* dbias,
                        int64_t dbias_ld, int reduce_over_n, int training, float* ds1, float* ds2,
                        iea_stream_t stream);
/* y = [relu](x*scale[n][c] + shift[n][c]) : stand-alone apply for the module-level API */
int iea_affine_act(const void* x, int x_dtype, const float* scale, const float* shift, int64_t n,
                   int64_t hw, int c, int relu, void* y, int y_dtype, iea_stream_t stream);

/* ---- the whole backward of a 1x1 SNConv2d layer in one kernel (csrc/conv_bwd1x1.cu) ----
 * Replaces, for same-resolution 1x1 layers with Cin, Cout in {16, 32, 64, 128} and whole 128-pixel tiles per image,
 * the sequence iea_conv_out_bwd -> iea_conv_wgrad_mma -> iea_conv_fprop(dgrad pack) -> iea_conv_input_bwd:
 *   geff = g + ds1[e][co] + 2 y ds2[e][co]  (ds1 == NULL: geff = g);   dW += geff^T . T(x),  db += colsum(geff);
 *   da = geff . W / sigma;  gm = da * 1[x*scale+shift > 0];  dx = beta*dx + gm*scale;
 *   dscale[n][c] = sum_px gm * x,  dshift[n][c] = sum_px gm.
 * `fwd` is the FORWARD descriptor of the layer (x, x_ld, cin, cout, in_scale / in_shift / in_relu / in_bcast). */
typedef struct iea_bwd1x1_args {
  const void* g;           /* dL/dy rows, bf16 */
  const void* y;           /* forward output rows, bf16 (read only when ds1 != NULL) */
  const float* ds1;        /* [events][cout] or NULL */
  const float* ds2;
  const void* wd_tc;       /* iea_sn_layer.pack_tc_dgrad of the layer */
  const float* inv_sigma;  /* 1/sigma of the forward call (NULL: 1) */
  void* dx;                /* bf16 rows of the input gradient, or NULL */
  float* wpart;            /* NULL: no weight gradient.  Else (grid+1)*cout*cin + grid*cout floats; slice 0 receives dW */
  float* dbias;            /* [cout] or NULL (needs wpart) */
  float* dscale;           /* [n][cin] or NULL */
  float* dshift;
  float* scratch;          /* iea_conv_bwd1x1_scratch_floats(fwd) floats when dscale != NULL */
  int64_t rows_per_event;
  int32_t g_ld, y_ld, dx_ld;
  float beta;
} iea_bwd1x1_args;
/* > 0: the layer is handled and this is the CTA count `grid` that sizes wpart; 0: use the unfused sequence */
int iea_conv_bwd1x1_grid(const iea_conv_desc* fwd);
int64_t iea_conv_bwd1x1_scratch_floats(const iea_conv_desc* fwd);
int iea_conv_bwd1x1(const iea_conv_desc* fwd, const iea_bwd1x1_args* args, iea_stream_t stream);

/* ---- optimizer step (SURVEY 8(f) N2): clip + Adam + EMA as multi-tensor kernels ----- */
/* One <= 65536-element slice of one tensor.  p: parameter (updated in place); g: its gradient;
 * m, v: Adam's exp_avg / exp_avg_sq; ema: the moving-average copy of p (NULL: none).
 * iea_mt_lerp reads p as the destination and g as the source. */
typedef struct iea_mt_chunk {
  float* p;
  const float* g;
  float* m;
  float* v;
  float* ema;
  int32_t n;
  int32_t tensor;
} iea_mt_chunk;
/* partial[i] = sum of squares of chunk i's gradient (torch.nn.utils.clip_grad_norm_'s norm,
 * train_fns.py:133-136,190-191; reduced in iea_mt_adam in a fixed order). */
int iea_mt_sqnorm(const iea_mt_chunk* chunks, int n_chunks, float* partial, iea_stream_t stream);
/* torch.optim.Adam step (model.py:410-416, 858-864: no weight decay, no amsgrad) on every chunk, with
 * the gradient scaled by min(1, max_norm / (norm + 1e-6)) when partial != NULL and max_norm > 0, and
 * ema = d*ema + (1-d)*p for chunks that carry one (utils/__init__.py:825-837).
 * scalars (device, 5 floats, zero before the first step): [0] step count, incremented here;
 * [1] clip coefficient; [2] 1-beta1^t; [3] sqrt(1-beta2^t); [4] gradient norm before clipping.
 * hyper (device, 2 floats): [0] learning rate, [1] EMA decay d.  Two launches. */
int iea_mt_adam(const iea_mt_chunk* chunks, int n_chunks, const float* partial, float max_norm, float beta1,
                float beta2, float eps, float* scalars, const float* hyper, iea_stream_t stream);
/* p = d*p + (1-d)*g per chunk (d = hyper[1]): the moving average of buffers (u0, sv0, running stats) */
int iea_mt_lerp(const iea_mt_chunk* chunks, int n_chunks, const float* hyper, iea_stream_t stream);

/* ---- modified orthogonal regularisation (SURVEY 8(f) N1) ------------------------------ */
/* One >= 2-D parameter viewed as W (rows x cols), row-major fp32.  gram: scratch of d*d floats with
 * d = tall ? cols : rows; rownorm: rows floats (tall only).  utils.ortho (utils/__init__.py:843-859):
 * grad += strength * 2 * ((W W^T) o (1 - I)) W; tall = evaluate it as W (W^T W) - diag(|w_i|^2) W. */
typedef struct iea_ortho_item {
  const float* w;
  float* grad;
  float* gram;
  float* rownorm;
  float* gram_part; /* tall only: ksplits partial d*d Gram matrices (the rows are split over ksplits CTAs) */
  int32_t rows, cols;
  int32_t tall;
  float strength;
  int32_t ksplits;
  int32_t pad_;
} iea_ortho_item;
/* rownorm_rows: (item, row) pairs of the tall items; gram_tiles: (item, tile row, tile col, k split) and
 * apply_tiles: (item, tile row, tile col, 0) with 64 x 64 tiles of the Gram matrix / of the parameter;
 * reduce_blocks: (item, first element) per 256-element span of a tall item's Gram matrix (fixed-order sum of
 * its k-split partials).  Three launches for the whole net (four when it has tall matrices). */
int iea_ortho_grouped(const iea_ortho_item* items, const int32_t* rownorm_rows, int n_rownorm_rows,
                      const int32_t* gram_tiles, int n_gram_tiles, const int32_t* reduce_blocks,
                      int n_reduce_blocks, const int32_t* apply_tiles, int n_apply_tiles, iea_stream_t stream);

/* ---- layout / elementwise helpers ------------------------------------------------- */
/* NCHW (src_dtype) <-> NHWC (dst_dtype) */
int iea_nchw_to_nhwc(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, int c,
                     int64_t hw, iea_stream_t stream);
int iea_nhwc_to_nchw(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n, int c,
                     int64_t hw, iea_stream_t stream);
/* y = alpha*a + beta*b (b may be NULL); all contiguous with count elements */
int iea_axpby(const void* a, int a_dtype, float alpha, const void* b, int b_dtype, float beta,
              void* y, int y_dtype, int64_t count, iea_stream_t stream);
/* y = gamma[0]*o + x (layers.py:300); backward: dgamma = sum(dy*o), do = gamma*dy */
int iea_gamma_residual(const void* o, const void* x, int dtype, const float* gamma, void* y,
                       int64_t count, iea_stream_t stream);
int iea_gamma_residual_bwd(const void* dy, const void* o, int dtype, const float* gamma, void* d_o,
                           float* dgamma, float* scratch, int64_t count, iea_stream_t stream);
/* F.embedding(idx, W*scale): layers.py:259, model.py:462 */
int iea_embedding_fwd(const int64_t* idx, const float* w, const float* scale, int64_t n, int dim,
                      float* out, iea_stream_t stream);
int iea_embedding_bwd(const int64_t* idx, const float* dout, const float* scale, int64_t n, int dim,
                      int rows, float* dw /* [rows][dim], zeroed inside */, iea_stream_t stream);
/* torch.sum(relu(h), [2,3]): model.py:912 */
int iea_relu_sumpool_fwd(const void* x, int x_dtype, int64_t n, int64_t hw, int c, float* out,
                         iea_stream_t stream);
int iea_relu_sumpool_bwd(const void* x, int x_dtype, const float* dout, int64_t n, int64_t hw, int c,
                         void* dx, int dx_dtype, iea_stream_t stream);
/* nn.AvgPool2d(2) of an NHWC tensor (channel windows: x_ld / y_ld are the row pitches in elements): the DBlock
 * shortcut pools its input once, model.py:541-557 (`downsample(x)` feeds both conv_sc and the identity half).
 * The adjoint is iea_residual_bwd with res_mode = IEA_IN_POOL2. */
int iea_avgpool2_fwd(const void* x, int dtype, int64_t n, int h, int w, int c, int x_ld, void* y, int y_ld,
                     iea_stream_t stream);

/* F.max_pool2d(x, 2): layers.py:286-287 (index saved as uint8 0..3) */
int iea_maxpool2_fwd(const void* x, int dtype, int64_t n, int h, int w, int c, void* y, uint8_t* idx,
                     iea_stream_t stream);
int iea_maxpool2_bwd(const void* dy, int dtype, const uint8_t* idx, int64_t n, int h, int w, int c,
                     void* dx, iea_stream_t stream);
/* nn.LayerNorm over the last dim (RRM.py:94-95,118; model.py:798) fp32 rows */
int iea_layernorm_fwd(const float* x, const float* g, const float* b, int64_t rows, int dim, float eps,
                      float* y, float* mean, float* rstd, iea_stream_t stream);
int iea_layernorm_bwd(const float* dy, const float* x, const float* g, const float* mean,
                      const float* rstd, int64_t rows, int dim, float* dx, float* dg_part,
                      float* db_part, int nparts, iea_stream_t stream);
/* F.normalize(x, dim=1): model.py:934-935 */
int iea_l2norm_fwd(const float* x, int64_t rows, int dim, float eps, float* y, float* norm,
                   iea_stream_t stream);
int iea_l2norm_bwd(const float* dy, const float* y, const float* norm, int64_t rows, int dim, float eps,
                   float* dx, iea_stream_t stream);

/* ---- RRM attention: RRM.py:10-16 scaled_dot_product on the per-head-interleaved qkv ---- */
/* qkv [events][40][heads][3*d] fp32 -> val [events][40][heads*d]; att [events][heads][40][40] saved */
int iea_mha_fwd(const float* qkv, int events, int seq, int heads, int d, float* val, float* att,
                iea_stream_t stream);
int iea_mha_bwd(const float* dval, const float* qkv, const float* att, int events, int seq, int heads,
                int d, float* dqkv, iea_stream_t stream);

/* ---- BigGAN self-attention core: layers.py:289-299 (softmax(theta^T phi), o = g beta^T) ---- */
/* theta [n][hw][ck], phi [n][hw/4][ck], g [n][hw/4][cv] -> o [n][hw][cv]; lse [n][hw] saved */
int iea_attn_fwd(const void* theta, const void* phi, const void* g, int dtype, int64_t n, int hw,
                 int hwk, int ck, int cv, void* o, float* lse, iea_stream_t stream);
int iea_attn_bwd(const void* d_o, const void* theta, const void* phi, const void* g, const void* o,
                 const float* lse, int dtype, int64_t n, int hw, int hwk, int ck, int cv,
                 void* dtheta, void* dphi, void* dg, float* dq_scratch /* [n][hw] */,
                 iea_stream_t stream);

/* ---- DiffAugment: diff_aug.py:23-102, closed form of SURVEY.md Appendix B.9 ---------- */
typedef struct {
  const float* brightness; const float* contrast;     /* [n] raw U(0,1) draws or NULL */
  const int64_t* tx; const int64_t* ty;               /* [n] or NULL */
  const int64_t* ox; const int64_t* oy; int32_t cut_h, cut_w; /* [n] or NULL */
} iea_aug_draws;
int iea_diffaug_fwd(const float* x, const iea_aug_draws* d /* host */, int64_t n, int h, int w, float* y,
                    float* mean_scratch /* [n] */, iea_stream_t stream);
int iea_diffaug_bwd(const float* dy, const iea_aug_draws* d /* host */, int64_t n, int h, int w,
                    float* dx, float* mean_scratch /* [n] */, iea_stream_t stream);

/* ---- losses: loss.py:8-9, 14-27, 30-38, 79-132 (per event of `seq` rows, then averaged) ---- */
/* out[0] = mean relu(1 - real), out[1] = mean relu(1 + fake) */
int iea_loss_hinge_dis(const float* fake, const float* real, int64_t n, float* out, iea_stream_t stream);
int iea_loss_hinge_dis_bwd(const float* fake, const float* real, const float* dout /* [2] */, int64_t n,
                           float* dfake, float* dreal, iea_stream_t stream);
/* out[0] = scale * mean(x) (loss_hinge_gen: scale = -1) and its backward dx[i] = dout*scale/n */
int iea_loss_mean(const float* x, int64_t n, float scale, float* out, iea_stream_t stream);
int iea_loss_mean_bwd(const float* dout, int64_t n, float scale, float* dx, iea_stream_t stream);
/* loss.py:41-44 l2_loss: out[0] = mean((a-b)^2); backward da = 2(a-b) dout/n, db = -da (either may be NULL) */
int iea_loss_l2(const float* a, const float* b, int64_t n, float* out, iea_stream_t stream);
int iea_loss_l2_bwd(const float* a, const float* b, const float* dout, int64_t n, float* da, float* db,
                    iea_stream_t stream);
/* The three Gram-based losses split the (seq x seq x dim) products of an event over ceil(dim/128) CTAs;
 * `scratch` receives the partial Gram matrices: iea_loss_scratch_floats(events, seq, dim) floats. */
int64_t iea_loss_scratch_floats(int events, int seq, int dim);
int iea_loss_contrastive_fwd(const float* embed, const float* proxy, int events, int seq, int dim,
                             float temperature, float margin, float* loss, float* saved /* events*(2*seq*seq+4*seq+1) */,
                             float* scratch, iea_stream_t stream);
int iea_loss_contrastive_bwd(const float* embed, const float* proxy, const float* saved,
                             const float* dloss, int events, int seq, int dim, float temperature,
                             float* dembed, float* dproxy, iea_stream_t stream);
int iea_loss_iea_fwd(const float* kf, const float* kr, int events, int seq, int dim, float* loss,
                     float* saved /* events*(seq*seq+1) */, float* scratch, iea_stream_t stream);
int iea_loss_iea_bwd(const float* kf, const float* saved, const float* dloss, int events, int seq,
                     int dim, float* dkf, iea_stream_t stream);
int iea_loss_unif_fwd(const float* x, int events, int seq, int dim, float t, float* loss,
                      float* saved /* events*(seq*seq+2) */, float* scratch, iea_stream_t stream);
int iea_loss_unif_bwd(const float* x, const float* saved, const float* dloss, int events, int seq,
                      int dim, float t, float* dx, iea_stream_t stream);

/* ---- input pipeline (SURVEY 8(f) N4): utils/dataloader.py:69-77 on a pre-decoded uint8 event tensor ----
 * out[n][h_in+2*pad][w] = 2*(log(u8 + 1)/log 256 + scale*noise) - 1 with `pad` zero rows above and below
 * (Pad((0,3,0,3)) -> ToTensor -> fn_lognorm255 -> UniformNoise(scale) -> Normalize(0.5, 0.5));
 * noise: U[0,1) draws of the output's shape (torch.rand_like in the reference), or NULL for none. */
int iea_event_preprocess(const uint8_t* img, int64_t n, int h_in, int w, int pad, const float* noise,
                         float scale, float* out, iea_stream_t stream);

/* ---- sampling post-process: model.py:1139-1147 (7-ADU cut, 256^x - 1, clamp, crop 3 rows) ---- */
int iea_adu_postprocess(const float* img, int64_t n, int h, int w, float* out /* [n][h-6][w] */,
                        iea_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* IEA_B200_H */
