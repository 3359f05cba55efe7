// conv_api.cu -- iea_conv_fprop: validates the descriptor and routes it to one of the forward kernels.
// conv_route() is the one place that picks the kernel; iea_conv_stats_slots sizes the batch-norm partial buffer
// from the same choice, so the buffer always matches the kernel that writes it.
#include "common.cuh"
using namespace iea;

int iea_conv_fprop_generic(const iea_conv_desc* d, cudaStream_t s);
int iea_conv_fprop_tc(const iea_conv_desc* d, cudaStream_t s);
int iea_conv_tc_ok(const iea_conv_desc* d);
int iea_conv_lowres_ok(const iea_conv_desc* d);
int iea_conv_fprop_lowres(const iea_conv_desc* d, cudaStream_t s);
int iea_conv_tc2_ok(const iea_conv_desc* d);
int iea_conv_fprop_tc2(const iea_conv_desc* d, cudaStream_t s);
int iea_conv_tc2_stats_slots(const iea_conv_desc* d);
int iea_conv_thin_ok(const iea_conv_desc* d);
int iea_conv_fprop_thin(const iea_conv_desc* d, cudaStream_t s);
int iea_conv_thin_stats_slots(const iea_conv_desc* d);
int iea_conv_c1_fwd_ok(const iea_conv_desc* d);
int iea_conv_c1_fwd(const iea_conv_desc* d, cudaStream_t s);
int iea_linear_skinny_ok(const iea_conv_desc* d);
int iea_linear_skinny(const iea_conv_desc* d, cudaStream_t s);

enum class ConvKernel { generic, c1, skinny, thin, tc2, lowres, stream };

// auto: c1, then skinny, then the tcgen05 chain (thin -> tc2 -> lowres -> stream), else generic.  tcgen05 and
// tc_stream run the tcgen05 chain only; tc_stream skips thin and lowres and takes the streaming kernel wherever
// iea_conv_tc_ok accepts the shape.  Returns generic when tcgen05 does not accept the shape.
static ConvKernel conv_route(const iea_conv_desc* d) {
  if (d->impl == IEA_IMPL_GENERIC) return ConvKernel::generic;
  if (d->impl == IEA_IMPL_AUTO && iea_conv_c1_fwd_ok(d)) return ConvKernel::c1;
  if (d->impl == IEA_IMPL_AUTO && iea_linear_skinny_ok(d)) return ConvKernel::skinny;
  const bool tc_ok = iea_conv_tc_ok(d), tc2_ok = iea_conv_tc2_ok(d);
  if (!tc_ok && !tc2_ok) return ConvKernel::generic;
  const bool force_stream = d->impl == IEA_IMPL_TC_STREAM;
  if (!force_stream && iea_conv_thin_ok(d)) return ConvKernel::thin;
  if ((!force_stream || !tc_ok) && tc2_ok) return ConvKernel::tc2;
  if (!force_stream && iea_conv_lowres_ok(d)) return ConvKernel::lowres;
  return ConvKernel::stream;
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

// batch-norm partial-sum slots per event that iea_conv_fprop will write for this descriptor
// (0: none -- the caller runs iea_bn_stats instead)
extern "C" int iea_conv_stats_slots(const iea_conv_desc* d) {
  switch (conv_route(d)) {
    case ConvKernel::thin: return iea_conv_thin_stats_slots(d);
    case ConvKernel::tc2: return iea_conv_tc2_stats_slots(d);
    default: {  // one slot per 128-pixel tile
      const int64_t px = 40ll * d->h * d->w;
      return (d->n % 40 == 0 && px % 128 == 0) ? (int)(px / 128) : 0;
    }
  }
}

extern "C" int iea_conv_tc_supported(const iea_conv_desc* d) { return iea_conv_tc_ok(d) || iea_conv_tc2_ok(d); }

extern "C" int iea_conv_fprop(const iea_conv_desc* d, iea_stream_t stream) {
  int rc = validate(d);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const ConvKernel k = conv_route(d);
  IEA_CHECK_ARG(k != ConvKernel::generic || (d->impl != IEA_IMPL_TCGEN05 && d->impl != IEA_IMPL_TC_STREAM),
                "iea_conv_fprop: tcgen05 path requested for an unsupported shape (cin=%d cout=%d k=%d)", d->cin, d->cout,
                d->ksize);
  switch (k) {
    case ConvKernel::c1: return iea_conv_c1_fwd(d, s);
    case ConvKernel::skinny: return iea_linear_skinny(d, s);
    case ConvKernel::thin: return iea_conv_fprop_thin(d, s);
    case ConvKernel::tc2: return iea_conv_fprop_tc2(d, s);
    case ConvKernel::lowres: return iea_conv_fprop_lowres(d, s);
    case ConvKernel::stream: return iea_conv_fprop_tc(d, s);
    case ConvKernel::generic: break;
  }
  return iea_conv_fprop_generic(d, s);
}
