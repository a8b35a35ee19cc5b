// Internal launcher interface shared by the C-ABI (capi.cu) and the network planner (net.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace biu {

// number of kernel launches issued by this library since load (bench.py reports it as gpu_launches)
extern unsigned long long g_launch_count;
inline void count_launch(int n = 1) { g_launch_count += n; }

// ---- tcgen05 implicit-GEMM convolution (conv_tc.cu) -------------------------------------------------------------
// Every argument block below gives the activation storage as `fmt`, the ElemFmt code (common.cuh) that the kernels also
// take as their template argument: FMT_BF16 / FMT_F16 (2-byte elements, tensor-core operands of the same format),
// FMT_TF32 (fp32 storage rounded to tf32) or FMT_F32 (fp32 storage, never rounded: CUDA-core kernels only).
// Byte sizes follow from fmt_esz(fmt).
struct ConvTcArgs {
  int fmt;                      // FMT_BF16 / FMT_F16 / FMT_TF32
  const void* in;               // NHWC / NDHWC activations
  int in_ctot, in_coff;         // channel stride / offset of the source buffer
  int cin;                      // logical input channels (multiple of 16 bf16 / fp16, 8 fp32)
  int W, H, D, B;
  int kw, kh, kd;               // 3 or 1
  const void* wgt;              // packed [tap][n_total][cin]
  int n_total;                  // Cout, or 2^dims * Cout for the transposed convolution
  int mode;                     // EpiMode
  float slope;
  const float* scale;
  const float* shift;
  void* out;
  int out_ctot, out_coff;
  int up_cout, up_dims;
  int head_n;
  const float* head_w;
  const float* head_b;
  int head_act[8];
  float* out_val;
  uint8_t* out_u8;
  int smem_budget;              // 0 = default
  const void* wgt_fold;         // optional: weights packed [kd*3 (dz,dx)][3*cout ((2-dy),co)][cin] for the row-streaming kernel
  const void* wgt_fold_z;       // optional (3D): [9 (dy,dx)][3*cout ((2-dz),co)][cin] for the row kernel's plane mode
  void* acc_scratch;            // optional: fp32 scratch of B*D*H*W*n_total floats for blocks whose K is split over several
  long long acc_scratch_bytes;  // launches (conv_rows.cuh acc_mode): an activation buffer that is dead while the block runs
  void* pool_out;               // optional fused MaxPool2d(2) output (EPI_CONV, 2D, halo-tile / row kernels only)
  int pool_ctot, pool_coff;
  int pool_3d;                  // 3D blocks: pool_out is the MaxPool3d(2) result [B][D/2][H/2][W/2] (plane mode of the row
                                // kernel, conv_tc_can_fuse_pool3d); 0: every plane pooled in (y, x) only
};
bool conv_tc_supported(const ConvTcArgs& a);
bool conv_tc_can_fuse_pool(const ConvTcArgs& a);
bool conv_tc_can_fuse_pool_xy(const ConvTcArgs& a);   // 3D: the row kernel pools every plane in (y, x) only
bool conv_tc_can_fuse_pool3d(const ConvTcArgs& a);    // 3D: the row kernel's plane mode pools in (z, y, x)
void conv_halo_set_cta2(int on);      // test hook: CTA pairs (tcgen05.mma.cta_group::2) in the halo-tile kernel (default on)
void conv_rows_set_enabled(int on);   // test hook: route narrow 3x3 blocks through the row-streaming kernel (default on)
int launch_conv_tc(const ConvTcArgs& a, cudaStream_t stream);
int read_device_fault(unsigned int* out);
int pick_ck(int cin, int fmt);

// ---- CUDA-core kernels (direct.cu): exact-fp32 path and shapes the tensor path cannot take ------------------------
struct DirectConvArgs {
  int fmt;                      // FMT_TF32 rounds the stored fp32 activations to tf32 (so the tensor path can consume them)
  const void* in;
  int in_ctot, in_coff, cin;
  int W, H, D, B;
  int kw, kh, kd;
  const float* wgt;             // fp32 [tap][cin][cout]
  int cout;
  float slope;                  // LeakyReLU slope; 1.0 => identity
  const float* scale;           // [cout] (nullptr => 1)
  const float* shift;           // [cout]
  void* out;
  int out_ctot, out_coff;
};
int launch_direct_conv(const DirectConvArgs& a, cudaStream_t stream);

struct DirectUpArgs {           // ConvTranspose(k=2,s=2): fp32 weights [q][cin][cout], q = (az,ay,ax) bits
  int fmt;
  const void* in;
  int in_ctot, in_coff, cin;
  int W, H, D, B;
  int dims;
  const float* wgt;
  const float* bias;
  int cout;
  void* out;
  int out_ctot, out_coff;
};
int launch_direct_up(const DirectUpArgs& a, cudaStream_t stream);

struct FirstConvArgs {          // planar u8 / f32 input with few channels -> NHWC features
  int in_kind;                  // 0 = u8 (value/255), 1 = f32
  const void* in;               // [B][cin][D][H][W]
  int cin;
  int W, H, D, B;
  int kd;                       // 1 (2D) or 3
  const float* wgt;             // fp32 [tap][cin][cout]
  int cout;                     // channels of the weight / scale / shift arrays (their stride)
  int cout_real;                // 0, or the block's real width when `cout` is a padded count: 8-channel groups at or above it
                                // are pure padding and are written as zeros without arithmetic (3D kernel)
  float slope;
  const float* scale;
  const float* shift;
  int fmt;
  void* out;                    // NHWC, channels [coff, coff+cout_pad) written (pad = zeros)
  int out_ctot, out_coff, cout_pad;
};
int launch_first_conv(const FirstConvArgs& a, cudaStream_t stream);

// First block of the 2D nets on the row kernel (conv_rows.cuh, first mode): uint8 tile in, NHWC features out; the three dx
// taps are the GEMM's K, the dy taps are folded into N. Tensor-core modes only (weights rounded like every other block's).
struct FirstRowsArgs {
  int fmt;                      // FMT_BF16 / FMT_F16 / FMT_TF32
  const uint8_t* in;            // [B][H][W] uint8 (one channel)
  int W, H, B;
  const void* wgt;              // [3 * n_total ((2 - dy), co)][16 bf16 / fp16 | 8 tf32: (dx = 0..2, zeros)]
  int n_total;                  // padded output channels: 16 or 32
  float slope;
  const float* scale;           // BatchNorm scale / 255 (the input rows hold the raw integers)
  const float* shift;
  void* out;
  int out_ctot, out_coff;
};
bool conv_first_rows_supported(const FirstRowsArgs& a);
int launch_conv_first_rows(const FirstRowsArgs& a, cudaStream_t stream);

struct PoolArgs {
  int fmt;
  const void* in;
  int in_ctot, in_coff, c;
  int W, H, D, B;               // input extents
  int dims;                     // 2: pool (h,w); 3: pool (d,h,w)
  int mode;                     // 0 = max, 1 = nearest (take the even-index sample), 2 = max over z pairs only (the
                                // input is already pooled in y and x: extents W, H are those of the output)
  void* out;                    // [B][D'][H/2][W/2][out_ctot]
  int out_ctot, out_coff;
};
int launch_pool2(const PoolArgs& a, cudaStream_t stream);

struct UpNearestArgs {          // nearest-neighbour x2 upsampling (multi_output_unet3d, use_interpolation=True)
  int fmt;
  const void* in;
  int in_ctot, in_coff, c;
  int W, H, D, B;               // input extents
  int dims;
  void* out;
  int out_ctot, out_coff;
};
int launch_up_nearest(const UpNearestArgs& a, cudaStream_t stream);

struct HeadArgs {               // 1x1 head + activation on NHWC features -> planar
  int fmt;
  const void* in;
  int in_ctot, in_coff, cin;
  long long npix_per_img;       // D*H*W
  int B;
  int head_n;
  const float* w;               // [head_n][cin]
  const float* b;
  int act[8];
  float* out_val;
  uint8_t* out_u8;
};
int launch_head(const HeadArgs& a, cudaStream_t stream);

// ---- HBM-bound pipeline kernels (pipeline.cu) -------------------------------------------------------------------
int launch_histogram(const void* img, int dtype_bytes, long long n_per_frame, int frames, unsigned int* hist,
                     cudaStream_t stream);
int launch_hist_sum(const unsigned int* hist, int frames, unsigned int* out, cudaStream_t stream);
int launch_norm_lut(const unsigned int* hist_bounds, const unsigned int* hist_range, long long bounds_stride,
                    long long range_stride, int frames, double q_lo, double q_hi, int invert, uint8_t* lut,
                    double* params, cudaStream_t stream);
int launch_apply_lut(const void* img, int dtype_bytes, long long n_per_frame, int frames, const uint8_t* lut,
                     long long lut_stride, uint8_t* out, cudaStream_t stream);
struct GatherArgs {
  const void* src;              // [F][Z][H][W] uint8, or the raw uint8 / uint16 stack when `lut` is set
  int src_bytes;                // 1 or 2
  const uint8_t* lut;           // optional: fused normalisation, dst = lut[f * lut_stride + src] (unet/predict.py:122-131)
  long long lut_stride;         // 65536 (one table per frame) or 0 (one table for the stack)
  int F, Z, H, W;
  int pad_mode;                 // 0 = reflect, 1 = constant zero
  const int* zs; const int* ys; const int* xs;   // device arrays of tile starts
  int nz, ny, nx;
  int pd, ph, pw;               // tile extents
  uint8_t* dst;                 // [F*nz*ny*nx][pd][ph][pw]
  int xform;                    // test-time augmentation: XF_* bits, 0 = the tile as it is
};
// Transform of a tile's coordinates (test-time augmentation). The flips act first, the transpose (2D square tiles only)
// last; the inverse transposes first. tta_xform maps the public code t (2D: bit 0 x, 1 y, 2 transpose; 3D: bit 0 x,
// 1 y, 2 z) onto these bits.
enum { XF_FLIP_X = 1, XF_FLIP_Y = 2, XF_FLIP_Z = 4, XF_TRANSPOSE = 8 };
inline int tta_xform(int dims, int t) { return dims == 2 ? ((t & 3) | ((t & 4) ? XF_TRANSPOSE : 0)) : (t & 7); }
int launch_gather_tiles(const GatherArgs& a, cudaStream_t stream);
struct TtaAccArgs {             // one pass of the test-time augmentation merge
  const float* val;             // [planes][pd][ph][pw]: the net's output on the transformed tiles
  long long planes;             // tiles * channels
  int pd, ph, pw;
  int xform;                    // XF_* bits of the pass's transform; its inverse is applied on the read
  int pass, passes;             // pass 0 writes acc, the last pass writes the mean to out_u8 / out_f32
  float* acc;                   // [planes][pd][ph][pw] fp32 running sum in pass order
  uint8_t* out_u8;              // trunc(mean * 255), the head epilogue's rule (may be null)
  float* out_f32;               // mean (may be null)
};
int launch_tta_accumulate(const TtaAccArgs& a, cudaStream_t stream);
struct StitchMeanArgs {         // unet/predict.py:204-229 == integer sum // count
  const uint8_t* tiles;         // [F][ny*nx][C][ph][pw]
  int F, C, H, W;               // output extents (already cropped to the image)
  const int* ys; const int* xs;
  int ny, nx, ph, pw;
  uint8_t* out;                 // [F][C][H][W]
};
int launch_stitch_mean(const StitchMeanArgs& a, cudaStream_t stream);
struct StitchMod3Args {         // unet3d/predict.py:173-195
  const uint8_t* tiles;         // [nz*ny*nx][pd][ph][pw]
  int Z, H, W;
  const int* zs; const int* ys; const int* xs;
  int nz, ny, nx, pd, ph, pw;
  uint8_t* out;                 // [Z][H][W]
};
int launch_stitch_mod3(const StitchMod3Args& a, cudaStream_t stream);
struct StitchWeightedArgs {     // engine-only: (sum w * v) // (sum w), w = w_d[tz] * w_h[ty] * w_w[tx]
  const uint8_t* tiles;         // [F][nz*ny*nx][C][pd][ph][pw]
  int F, C, Z, H, W;            // output extents; starts may be negative and tiles may reach past the output
  const int* zs; const int* ys; const int* xs;
  int nz, ny, nx, pd, ph, pw;
  const int* w_d; const int* w_h; const int* w_w;   // device int32 tables of pd / ph / pw entries in [0, 1024]
  uint8_t* out;                 // [F][C][Z][H][W]
};
int launch_stitch_weighted(const StitchWeightedArgs& a, cudaStream_t stream);
struct StitchRampArgs {         // multi_output_unet3d/predict.py:203-307
  const float* tiles;           // [V][nz*ny*nx][C][pd][ph][pw]
  int V, C, Z, H, W;
  const int* zs; const int* ys; const int* xs;
  int nz, ny, nx, pd, ph, pw;
  int margin;
  float* out;                   // [V][C][Z][H][W]
};
int launch_stitch_ramp(const StitchRampArgs& a, cudaStream_t stream);
struct NormF32Args {            // percentile normalisation of a float32 stack to uint8 (unet/predict.py:122-150)
  const float* img;             // [frames][n_per_frame]
  long long n_per_frame;
  int frames;
  int mode;                     // 0 'single' (per frame), 1 'first' (bounds of frame 0), 2 'all'
  double q_lo, q_hi;
  int invert;
  char* scratch;                // normalize_f32_scratch_bytes() bytes
  float* params;                // [frames or 1][4] {lo, hi, mn, mx}
  uint8_t* out_u8;              // [frames][n_per_frame]
  float* out_f32;               // optional: the float32 values the reference stores back into the stack
};
int launch_normalize_f32(const NormF32Args& a, cudaStream_t stream);
long long normalize_f32_scratch_bytes(long long n_per_frame, int frames);
struct StitchMarginArgs {       // multi_output_unet/predict.py:230-285 (ys/ny index image rows, xs/nx columns)
  const float* tiles;           // [P][C][ph][pw] float32 (rounded to float16 on read, as the reference stores them)
  const int* src_index;         // [T][ny][nx] flat patch index of tile (image, j, k)
  int T, C, H, W;
  const int* ys; const int* xs;
  int ny, nx, ph, pw, margin;
  const float* fill;            // device scalar: value of pixels without any weight
  float* out;                   // [T][C][H][W]
};
int launch_stitch_margin(const StitchMarginArgs& a, cudaStream_t stream);
int launch_norm_lut_f32(const unsigned int* hist_bounds, const unsigned int* hist_range, long long bounds_stride,
                        long long range_stride, int frames, double q_lo, double q_hi, int mode, float* lut,
                        double* params, cudaStream_t stream);
int launch_apply_lut_f32(const void* img, int dtype_bytes, long long n_per_frame, int frames, const float* lut,
                         long long lut_stride, float* out, cudaStream_t stream);
int launch_gather_tiles_f32(const float* src, int F, int Z, int H, int W, const int* zs, const int* ys, const int* xs,
                            int nz, int ny, int nx, int pd, int ph, int pw, float* dst, cudaStream_t stream,
                            int xform = 0);



}  // namespace biu
