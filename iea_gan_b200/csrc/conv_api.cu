// conv_api.cu -- iea_conv_fprop: validates the descriptor and dispatches to the tcgen05
// implicit-GEMM kernel (conv_tc.cu) or to the shape-generic kernel (conv_generic.cu).
#include "common.cuh"
#include <stdlib.h>
using namespace iea;

int iea_conv_fprop_generic(const iea_conv_desc* d, cudaStream_t s);
int iea_conv_fprop_tc(const iea_conv_desc* d, cudaStream_t s);
int iea_conv_tc_ok(const iea_conv_desc* d);
int iea_conv_lowres_ok(const iea_conv_desc* d);
int iea_conv_fprop_lowres(const iea_conv_desc* d, cudaStream_t s);
int iea_conv_tc2_ok(const iea_conv_desc* d);
int iea_conv_fprop_tc2(const iea_conv_desc* d, cudaStream_t s);
int iea_conv_thin_ok(const iea_conv_desc* d);
int iea_conv_fprop_thin(const iea_conv_desc* d, cudaStream_t s);
int iea_conv_thin_stats_slots(const iea_conv_desc* d);
int iea_conv_c1_fwd_ok(const iea_conv_desc* d);
int iea_conv_c1_fwd(const iea_conv_desc* d, cudaStream_t s);
int iea_linear_skinny_ok(const iea_conv_desc* d);
int iea_linear_skinny(const iea_conv_desc* d, cudaStream_t s);

// tcgen05 variant selection: resident-weights/patch kernel when it applies, then the staged-patch kernel with
// streamed weights (wide 3x3 layers at low resolution), else the streaming one.
// IEA_TC_VARIANT=stream forces the streaming kernel (used by the tests to cover both); IEA_LOWRES_TC=0 turns the
// staged-patch kernel off.  Both kernels tile the pixels alike, so the statistics slots do not depend on the choice.
static bool lowres_on() {
  const char* v = getenv("IEA_LOWRES_TC");
  return !(v && v[0] == '0');
}
static int run_tc(const iea_conv_desc* d, cudaStream_t s) {
  const char* v = getenv("IEA_TC_VARIANT");
  const bool force_stream = v && v[0] == 's';
  if (!force_stream && iea_conv_thin_ok(d)) return iea_conv_fprop_thin(d, s);
  if ((!force_stream || !iea_conv_tc_ok(d)) && iea_conv_tc2_ok(d)) return iea_conv_fprop_tc2(d, s);
  if (!force_stream && lowres_on() && iea_conv_lowres_ok(d)) return iea_conv_fprop_lowres(d, s);
  return iea_conv_fprop_tc(d, s);
}

static int validate(const iea_conv_desc* d) {
  IEA_CHECK_ARG(d != nullptr, "iea_conv_fprop: null descriptor");
  IEA_CHECK_ARG(d->ksize == 1 || d->ksize == 3, "iea_conv_fprop: ksize %d not built (1 or 3)", d->ksize);
  IEA_CHECK_ARG(d->n > 0 && d->h > 0 && d->w > 0 && d->cin > 0 && d->cout > 0, "iea_conv_fprop: empty geometry");
  IEA_CHECK_ARG(d->x && d->wpack && d->y, "iea_conv_fprop: null tensor pointer");
  IEA_CHECK_ARG(d->in_mode != IEA_IN_UP2 || (d->h % 2 == 0 && d->w % 2 == 0), "iea_conv_fprop: up2 needs even h,w");
  IEA_CHECK_ARG((d->in_scale == nullptr) == (d->in_shift == nullptr), "iea_conv_fprop: in_scale/in_shift mismatch");
  IEA_CHECK_ARG(d->x_ld >= d->cin && d->y_ld >= 1, "iea_conv_fprop: bad pixel strides");
  return 0;
}

int iea_conv_tc2_stats_slots(const iea_conv_desc* d);
// batch-norm partial-sum slots per event that iea_conv_fprop will write for this descriptor
// (0: none -- the caller runs iea_bn_stats instead).  Mirrors the dispatch below.
extern "C" int iea_conv_stats_slots(const iea_conv_desc* d) {
  const int64_t px = 40ll * d->h * d->w;
  const int tiles = (d->n % 40 == 0 && px % 128 == 0) ? (int)(px / 128) : 0;
  if (d->impl == IEA_IMPL_GENERIC) return tiles;
  const char* v = getenv("IEA_TC_VARIANT");
  const bool force_stream = v && v[0] == 's';
  if (!iea_conv_tc_ok(d) && !iea_conv_tc2_ok(d)) return tiles;  // generic kernel
  if (!force_stream && iea_conv_thin_ok(d)) return iea_conv_thin_stats_slots(d);
  if ((!force_stream || !iea_conv_tc_ok(d)) && iea_conv_tc2_ok(d)) return iea_conv_tc2_stats_slots(d);
  return tiles;  // conv_tc_kernel and conv_lr_kernel: one slot per 128-pixel tile
}

extern "C" int iea_conv_tc_supported(const iea_conv_desc* d) { return iea_conv_tc_ok(d) || iea_conv_tc2_ok(d); }

extern "C" int iea_conv_fprop(const iea_conv_desc* d, iea_stream_t stream) {
  int rc = validate(d);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  if (d->impl == IEA_IMPL_GENERIC) return iea_conv_fprop_generic(d, s);
  if (d->impl == IEA_IMPL_AUTO && iea_conv_c1_fwd_ok(d)) return iea_conv_c1_fwd(d, s);  // 1-channel input: CUDA cores
  if (d->impl == IEA_IMPL_AUTO && iea_linear_skinny_ok(d)) return iea_linear_skinny(d, s);  // few rows, long K: cluster split-K
  if (d->impl == IEA_IMPL_TCGEN05) {
    IEA_CHECK_ARG(iea_conv_tc_ok(d) || iea_conv_tc2_ok(d), "iea_conv_fprop: tcgen05 path requested for an unsupported shape "
                  "(cin=%d cout=%d k=%d)", d->cin, d->cout, d->ksize);
    return run_tc(d, s);
  }
  return (iea_conv_tc_ok(d) || iea_conv_tc2_ok(d)) ? run_tc(d, s) : iea_conv_fprop_generic(d, s);
}
