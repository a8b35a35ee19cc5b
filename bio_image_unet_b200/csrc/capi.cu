// extern "C" boundary (include/biu_b200.h). Plain pointers and sizes only.
#include "../../include/biu_b200.h"
#include "common.cuh"
#include "conv_tc.cuh"
#include "net.h"

#include <cstdarg>
#include <cstring>

namespace biu {
static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }
unsigned long long g_launch_count = 0;
}  // namespace biu

using namespace biu;

// `esz` of the layer entry points: 2 = bf16, BIU_ESZ_FP16 = fp16, 4 = fp32 -> ElemFmt. The tensor-core entry points take
// fp32 storage as tf32 operands (fp32_fmt = FMT_TF32); the CUDA-core ones store it unrounded (FMT_F32).
static int layer_format(int esz, int fp32_fmt, int* fmt) {
  BIU_REQUIRE(esz == 2 || esz == 4 || esz == BIU_ESZ_FP16, "unknown element code esz=%d (2 = bf16, %d = fp16, 4 = fp32)",
              esz, BIU_ESZ_FP16);
  *fmt = esz == 4 ? fp32_fmt : (esz == BIU_ESZ_FP16 ? FMT_F16 : FMT_BF16);
  return 0;
}

struct biu_net {
  Net* n;
};

extern "C" {

const char* biu_last_error(void) { return get_error(); }
int biu_version(void) { return 100; }

biu_net* biu_net_create(int kind, int n_filter, int in_channels, int n_heads, const int* head_channels,
                        const int* head_acts, const char* const* head_names, int siam_mode, int use_interpolation,
                        int precision) {
  if (kind < 0 || kind > 8) { set_error("unknown network kind %d", kind); return nullptr; }
  static_assert(BIU_PREC_BF16 == 0 && BIU_PREC_TF32 == 1 && BIU_PREC_FP32 == 2 && BIU_PREC_FP16 == 3, "prec_fmt order");
  static const int prec_fmt[4] = {FMT_BF16, FMT_TF32, FMT_F32, FMT_F16};
  if (precision < 0 || precision > 3) { set_error("unknown precision %d", precision); return nullptr; }
  if (n_heads < 1 || !head_channels || !head_acts) { set_error("at least one output head is required"); return nullptr; }
  Net* n = new Net();
  n->kind = kind; n->nf = n_filter; n->in_ch = in_channels; n->fmt = prec_fmt[precision];
  n->siam_mode = siam_mode; n->use_interp = use_interpolation;
  for (int i = 0; i < n_heads; ++i) {
    n->head_channels.push_back(head_channels[i]);
    n->head_acts.push_back(head_acts[i]);
    n->head_names.push_back(head_names && head_names[i] ? head_names[i] : "");
  }
  if (net_build(n) != 0) { delete n; return nullptr; }
  biu_net* h = new biu_net();
  h->n = n;
  return h;
}

int biu_net_set_param(biu_net* net, const char* name, const float* data_host, int ndim, const long long* shape) {
  BIU_REQUIRE(net && net->n && name && data_host, "biu_net_set_param: null argument");
  BIU_REQUIRE(!net->n->finalized, "biu_net_set_param after biu_net_finalize");
  HostTensor t;
  long long cnt = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); cnt *= shape[i]; }
  t.data.assign(data_host, data_host + cnt);
  net->n->params[name] = std::move(t);
  return 0;
}
int biu_net_finalize(biu_net* net) {
  BIU_REQUIRE(net && net->n, "null handle");
  return net_finalize(net->n);
}
long long biu_net_plan(biu_net* net, int batch, int d, int h, int w) {
  if (!net || !net->n) { set_error("null handle"); return -1; }
  return net_plan(net->n, batch, d, h, w);
}
int biu_net_forward(biu_net* net, const void* in, int in_kind, const void* in2, float* out_val, uint8_t* out_u8,
                    void* workspace, void* stream) {
  BIU_REQUIRE(net && net->n, "null handle");
  return net_forward(net->n, in, in_kind, in2, out_val, out_u8, workspace, (cudaStream_t)stream);
}
int biu_net_debug_copy(biu_net* net, const char* name, void* workspace, void* dst_host, long long max_bytes) {
  BIU_REQUIRE(net && net->n, "null handle");
  return net_debug_copy(net->n, name, workspace, dst_host, max_bytes);
}
int biu_net_set_force_direct(biu_net* net, int on) {
  BIU_REQUIRE(net && net->n, "null handle");
  net->n->force_direct = on;
  return 0;
}

int biu_net_set_siam_shared(biu_net* net, int tiles_per_frame) {
  BIU_REQUIRE(net && net->n, "null handle");
  BIU_REQUIRE(tiles_per_frame >= 0, "tiles_per_frame must not be negative");
  BIU_REQUIRE(tiles_per_frame == 0 || net->n->kind == NET_SIAM2D, "the shared twin encoder is a Siam_UNet mode");
  net->n->siam_shared = tiles_per_frame;
  net->n->B = 0;                            // buffer sizes change: biu_net_plan has to be called again
  return 0;
}
int biu_net_fallback_ops(biu_net* net) {
  BIU_REQUIRE(net && net->n, "null handle");
  int cnt = 0;
  for (int k : net->n->op_kinds) cnt += (k & 16) ? 1 : 0;
  return cnt;
}

int biu_set_halo_cta2(int on) {
  conv_halo_set_cta2(on);
  return 0;
}

int biu_set_rows_kernel(int on) {
  conv_rows_set_enabled(on);
  return 0;
}

int biu_net_set_fuse_pool(biu_net* net, int on) {
  BIU_REQUIRE(net && net->n, "null handle");
  net->n->no_fuse = on ? 0 : 1;
  return 0;
}
int biu_net_set_debug_stop(biu_net* net, int last_op) {
  BIU_REQUIRE(net && net->n, "null handle");
  BIU_REQUIRE(last_op >= -1, "last_op must be -1 (off) or an op index (got %d)", last_op);
  net->n->debug_stop = last_op;
  return 0;
}
void biu_net_destroy(biu_net* net) {
  if (!net) return;
  if (net->n) net_destroy(net->n);
  delete net;
}

int biu_histogram(const void* img, int dtype_bytes, long long n_per_frame, int frames, uint32_t* hist, void* stream) {
  return launch_histogram(img, dtype_bytes, n_per_frame, frames, hist, (cudaStream_t)stream);
}
int biu_hist_sum(const uint32_t* hist, int frames, uint32_t* out, void* stream) {
  return launch_hist_sum(hist, frames, out, (cudaStream_t)stream);
}
int biu_norm_lut(const uint32_t* hist_bounds, const uint32_t* hist_range, long long bounds_stride,
                 long long range_stride, int frames, double q_lo, double q_hi, int invert, uint8_t* lut,
                 double* params, void* stream) {
  return launch_norm_lut(hist_bounds, hist_range, bounds_stride, range_stride, frames, q_lo, q_hi, invert, lut,
                         params, (cudaStream_t)stream);
}
int biu_apply_lut(const void* img, int dtype_bytes, long long n_per_frame, int frames, const uint8_t* lut,
                  long long lut_stride, uint8_t* out, void* stream) {
  return launch_apply_lut(img, dtype_bytes, n_per_frame, frames, lut, lut_stride, out, (cudaStream_t)stream);
}
int biu_norm_lut_f32(const uint32_t* hist_bounds, const uint32_t* hist_range, long long bounds_stride,
                     long long range_stride, int frames, double q_lo, double q_hi, int mode, float* lut,
                     double* params, void* stream) {
  return launch_norm_lut_f32(hist_bounds, hist_range, bounds_stride, range_stride, frames, q_lo, q_hi, mode, lut,
                             params, (cudaStream_t)stream);
}
int biu_apply_lut_f32(const void* img, int dtype_bytes, long long n_per_frame, int frames, const float* lut,
                      long long lut_stride, float* out, void* stream) {
  return launch_apply_lut_f32(img, dtype_bytes, n_per_frame, frames, lut, lut_stride, out, (cudaStream_t)stream);
}
int biu_gather_tiles_f32(const float* src, int F, int Z, int H, int W, const int* zs, const int* ys, const int* xs,
                         int nz, int ny, int nx, int pd, int ph, int pw, float* dst, void* stream) {
  return launch_gather_tiles_f32(src, F, Z, H, W, zs, ys, xs, nz, ny, nx, pd, ph, pw, dst, (cudaStream_t)stream);
}
int biu_gather_tiles(const uint8_t* src, int F, int Z, int H, int W, int pad_mode, const int* zs, const int* ys,
                     const int* xs, int nz, int ny, int nx, int pd, int ph, int pw, uint8_t* dst, void* stream) {
  GatherArgs a{src, 1, nullptr, 0, F, Z, H, W, pad_mode, zs, ys, xs, nz, ny, nx, pd, ph, pw, dst};
  return launch_gather_tiles(a, (cudaStream_t)stream);
}
int biu_gather_tiles_lut(const void* src, int dtype_bytes, const uint8_t* lut, long long lut_stride, int F, int Z, int H,
                         int W, int pad_mode, const int* zs, const int* ys, const int* xs, int nz, int ny, int nx, int pd,
                         int ph, int pw, uint8_t* dst, void* stream) {
  BIU_REQUIRE(lut != nullptr && (dtype_bytes == 1 || dtype_bytes == 2), "gather_tiles_lut: uint8 / uint16 source and a table");
  GatherArgs a{src, dtype_bytes, lut, lut_stride, F, Z, H, W, pad_mode, zs, ys, xs, nz, ny, nx, pd, ph, pw, dst};
  return launch_gather_tiles(a, (cudaStream_t)stream);
}
static int tta_code(int dims, int t, int* xform) {
  BIU_REQUIRE(dims == 2 || dims == 3, "test-time augmentation: dims must be 2 or 3 (got %d)", dims);
  BIU_REQUIRE(t >= 0 && t < 8, "test-time augmentation: transform code must be 0..7 (got %d)", t);
  *xform = tta_xform(dims, t);
  return 0;
}
int biu_gather_tiles_tta(const void* src, int dtype_bytes, const uint8_t* lut, long long lut_stride, int F, int Z, int H,
                         int W, int pad_mode, const int* zs, const int* ys, const int* xs, int nz, int ny, int nx, int pd,
                         int ph, int pw, int dims, int t, uint8_t* dst, void* stream) {
  BIU_REQUIRE(dtype_bytes == 1 || (dtype_bytes == 2 && lut != nullptr),
              "gather_tiles_tta: a uint8 source, or a uint8 / uint16 source and a table");
  GatherArgs a{src, dtype_bytes, lut, lut_stride, F, Z, H, W, pad_mode, zs, ys, xs, nz, ny, nx, pd, ph, pw, dst, 0};
  if (int rc = tta_code(dims, t, &a.xform)) return rc;
  return launch_gather_tiles(a, (cudaStream_t)stream);
}
int biu_gather_tiles_f32_tta(const float* src, int F, int Z, int H, int W, const int* zs, const int* ys, const int* xs,
                             int nz, int ny, int nx, int pd, int ph, int pw, int dims, int t, float* dst, void* stream) {
  int xform = 0;
  if (int rc = tta_code(dims, t, &xform)) return rc;
  return launch_gather_tiles_f32(src, F, Z, H, W, zs, ys, xs, nz, ny, nx, pd, ph, pw, dst, (cudaStream_t)stream, xform);
}
int biu_tta_accumulate(const float* val, long long planes, int pd, int ph, int pw, int dims, int t, int pass, int passes,
                       float* acc, uint8_t* out_u8, float* out_f32, void* stream) {
  TtaAccArgs a{val, planes, pd, ph, pw, 0, pass, passes, acc, out_u8, out_f32};
  if (int rc = tta_code(dims, t, &a.xform)) return rc;
  return launch_tta_accumulate(a, (cudaStream_t)stream);
}
int biu_stitch_mean_u8(const uint8_t* tiles, int F, int C, int H, int W, const int* ys, const int* xs, int ny, int nx,
                       int ph, int pw, uint8_t* out, void* stream) {
  StitchMeanArgs a{tiles, F, C, H, W, ys, xs, ny, nx, ph, pw, out};
  return launch_stitch_mean(a, (cudaStream_t)stream);
}
int biu_stitch_mod3_u8(const uint8_t* tiles, int Z, int H, int W, const int* zs, const int* ys, const int* xs, int nz,
                       int ny, int nx, int pd, int ph, int pw, uint8_t* out, void* stream) {
  StitchMod3Args a{tiles, Z, H, W, zs, ys, xs, nz, ny, nx, pd, ph, pw, out};
  return launch_stitch_mod3(a, (cudaStream_t)stream);
}
int biu_stitch_weighted_u8(const uint8_t* tiles, int F, int C, int Z, int H, int W, const int* zs, const int* ys,
                           const int* xs, int nz, int ny, int nx, int pd, int ph, int pw, const int* w_d, const int* w_h,
                           const int* w_w, uint8_t* out, void* stream) {
  StitchWeightedArgs a{tiles, F, C, Z, H, W, zs, ys, xs, nz, ny, nx, pd, ph, pw, w_d, w_h, w_w, out};
  return launch_stitch_weighted(a, (cudaStream_t)stream);
}
int biu_stitch_ramp_f32(const float* tiles, int V, int C, int Z, int H, int W, const int* zs, const int* ys,
                        const int* xs, int nz, int ny, int nx, int pd, int ph, int pw, int margin, float* out,
                        void* stream) {
  StitchRampArgs a{tiles, V, C, Z, H, W, zs, ys, xs, nz, ny, nx, pd, ph, pw, margin, out};
  return launch_stitch_ramp(a, (cudaStream_t)stream);
}

int biu_conv_tc(int esz, const void* in, int in_ctot, int in_coff, int cin, int B, int D, int H, int W, int kd,
                int kh, int kw, const void* wgt, int cout, const float* scale, const float* shift, float slope,
                void* out, int out_ctot, int out_coff, void* stream) {
  ConvTcArgs a;
  memset(&a, 0, sizeof(a));
  if (int rc = layer_format(esz, FMT_TF32, &a.fmt)) return rc;
  a.in = in; a.in_ctot = in_ctot; a.in_coff = in_coff; a.cin = cin;
  a.W = W; a.H = H; a.D = D; a.B = B; a.kw = kw; a.kh = kh; a.kd = kd;
  a.wgt = wgt; a.n_total = cout; a.mode = EPI_CONV; a.slope = slope; a.scale = scale; a.shift = shift;
  a.out = out; a.out_ctot = out_ctot; a.out_coff = out_coff;
  return launch_conv_tc(a, (cudaStream_t)stream);
}
int biu_up_tc(int esz, const void* in, int in_ctot, int in_coff, int cin, int B, int D, int H, int W, int dims,
              const void* wgt, int cout, const float* bias_rep, void* out, int out_ctot, int out_coff, void* stream) {
  ConvTcArgs a;
  memset(&a, 0, sizeof(a));
  if (int rc = layer_format(esz, FMT_TF32, &a.fmt)) return rc;
  a.in = in; a.in_ctot = in_ctot; a.in_coff = in_coff; a.cin = cin;
  a.W = W; a.H = H; a.D = D; a.B = B; a.kw = a.kh = a.kd = 1;
  a.wgt = wgt; a.n_total = (dims == 3 ? 8 : 4) * cout; a.mode = EPI_UP; a.slope = 1.f; a.scale = bias_rep;
  a.shift = bias_rep; a.out = out; a.out_ctot = out_ctot; a.out_coff = out_coff; a.up_cout = cout; a.up_dims = dims;
  return launch_conv_tc(a, (cudaStream_t)stream);
}
int biu_conv_direct(int esz, const void* in, int in_ctot, int in_coff, int cin, int B, int D, int H, int W, int kd,
                    int kh, int kw, const float* wgt, int cout, const float* scale, const float* shift, float slope,
                    void* out, int out_ctot, int out_coff, void* stream) {
  DirectConvArgs a;
  memset(&a, 0, sizeof(a));
  if (int rc = layer_format(esz, FMT_F32, &a.fmt)) return rc;
  a.in = in; a.in_ctot = in_ctot; a.in_coff = in_coff; a.cin = cin;
  a.W = W; a.H = H; a.D = D; a.B = B; a.kw = kw; a.kh = kh; a.kd = kd;
  a.wgt = wgt; a.cout = cout; a.slope = slope; a.scale = scale; a.shift = shift;
  a.out = out; a.out_ctot = out_ctot; a.out_coff = out_coff;
  return launch_direct_conv(a, (cudaStream_t)stream);
}
int biu_pool2(int esz, const void* in, int in_ctot, int in_coff, int c, int B, int D, int H, int W, int dims,
              int mode, void* out, int out_ctot, int out_coff, void* stream) {
  PoolArgs a;
  memset(&a, 0, sizeof(a));
  if (int rc = layer_format(esz, FMT_F32, &a.fmt)) return rc;
  a.in = in; a.in_ctot = in_ctot; a.in_coff = in_coff; a.c = c; a.W = W; a.H = H; a.D = D; a.B = B;
  a.dims = dims; a.mode = mode; a.out = out; a.out_ctot = out_ctot; a.out_coff = out_coff;
  return launch_pool2(a, (cudaStream_t)stream);
}
int biu_device_fault(unsigned int* code_host) { return read_device_fault(code_host); }
int biu_stitch_margin_f32(const float* tiles, const int* src_index, int T, int C, int H, int W, const int* ys,
                          const int* xs, int ny, int nx, int ph, int pw, int margin, const float* fill, float* out,
                          void* stream) {
  StitchMarginArgs a;
  memset(&a, 0, sizeof(a));
  a.tiles = tiles; a.src_index = src_index; a.T = T; a.C = C; a.H = H; a.W = W; a.ys = ys; a.xs = xs;
  a.ny = ny; a.nx = nx; a.ph = ph; a.pw = pw; a.margin = margin; a.fill = fill; a.out = out;
  return launch_stitch_margin(a, (cudaStream_t)stream);
}

long long biu_normalize_f32_scratch_bytes(long long n_per_frame, int frames) {
  return normalize_f32_scratch_bytes(n_per_frame, frames);
}
int biu_normalize_f32(const float* img, long long n_per_frame, int frames, int mode, double q_lo, double q_hi, int invert,
                      void* scratch, float* params, uint8_t* out_u8, float* out_f32, void* stream) {
  NormF32Args a;
  memset(&a, 0, sizeof(a));
  a.img = img; a.n_per_frame = n_per_frame; a.frames = frames; a.mode = mode; a.q_lo = q_lo; a.q_hi = q_hi;
  a.invert = invert; a.scratch = reinterpret_cast<char*>(scratch); a.params = params; a.out_u8 = out_u8; a.out_f32 = out_f32;
  return launch_normalize_f32(a, (cudaStream_t)stream);
}

unsigned long long biu_launch_count(void) { return g_launch_count; }
int biu_net_set_profile(biu_net* net, int on) {
  BIU_REQUIRE(net && net->n, "null handle");
  net->n->profile = on;
  return 0;
}
int biu_net_profile_read(biu_net* net, int max_ops, int* kinds, float* ms, int* n_ops) {
  BIU_REQUIRE(net && net->n, "null handle");
  return net_profile_read(net->n, max_ops, kinds, ms, n_ops);
}

}  // extern "C"
