/* biu_b200 — C-ABI of the B200-native tiled U-Net prediction engine.
 *
 * Drop-in boundary for the prediction path of danihae/bio-image-unet. The reference has no FFI: its seam is
 * the Python call `self.model(patch)` plus the numpy pre/post-processing around it. Each entry point below
 * names the reference code it replaces (paths relative to bio_image_unet/ in the reference, v1.1.1).
 *
 * Conventions
 *   - every function returns 0 on success (biu_net_create returns NULL, biu_net_plan a negative value, on error);
 *     biu_last_error() returns the message of the last failure on the calling thread;
 *   - all data pointers are DEVICE pointers unless the parameter name ends in `_host`; nothing returned by the
 *     library has to be freed by the caller except the handle (biu_net_destroy);
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous and stream-ordered on it;
 *   - a handle is not thread-safe.
 */
#ifndef BIU_B200_H
#define BIU_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- enums ---------------------------------------------------------------------------------------------- */
enum { BIU_NET_UNET2D = 0,   /* unet/unet.py:5 Unet */
       BIU_NET_SIAM2D = 1,   /* siam_unet/siam_unet.py:7 Siam_UNet */
       BIU_NET_UNET3D = 2,   /* unet3d/unet3d.py:6 UNet3D */
       BIU_NET_MO3D   = 3,   /* multi_output_unet3d/multi_output_unet3d.py:7 MultiOutputUnet3D */
       BIU_NET_UNET2D_V0 = 4, /* unet/unet_v0.py:5 Unet_v0 (ReLU blocks, early skips, decode9) */
       BIU_NET_ATTUNET2D = 5, /* unet/attention_unet.py:5 AttentionUnet (gated skip connections) */
       BIU_NET_MO2D = 6,     /* multi_output_unet/multi_output_unet.py:6 MultiOutputUnet (Unet body, named heads) */
       BIU_NET_NESTED2D = 7, /* multi_output_unet/multi_output_nested_unet.py:58 MultiOutputNestedUNet (U-Net++, 4 pools) */
       BIU_NET_NESTED2D_3L = 8 }; /* multi_output_nested_unet.py:151 MultiOutputNestedUNet_3Levels (3 pools) */
enum { BIU_PREC_BF16 = 0,    /* bf16 operands on tcgen05, fp32 accumulate */
       BIU_PREC_TF32 = 1,    /* tf32 operands on tcgen05, fp32 storage */
       BIU_PREC_FP32 = 2,    /* fp32 CUDA-core kernels */
       BIU_PREC_FP16 = 3 };  /* fp16 operands on tcgen05, fp32 accumulate, fp16 storage (beyond +-65504: +-inf) */
enum { BIU_SIAM_CONCAT = 0, BIU_SIAM_MAX = 1, BIU_SIAM_CONTROL = 2, BIU_SIAM_CORR = 3 }; /* siam_unet.py:114-124 */
enum { BIU_ACT_NONE = 0, BIU_ACT_SIGMOID = 1, BIU_ACT_TANH = 2, BIU_ACT_RELU = 3 };      /* multi_output_unet3d.py:97-104 */
enum { BIU_PAD_REFLECT = 0,  /* unet/predict.py:163-168, unet3d/predict.py:134-137 */
       BIU_PAD_ZERO = 1 };   /* siam_unet/predict.py:169-180 */
enum { BIU_IN_U8 = 0,        /* uint8 tiles, converted as float32(u8)/255 (unet/predict.py:192) */
       BIU_IN_F32 = 1 };     /* float32 patches (multi_output_unet3d/predict.py:185) */

const char* biu_last_error(void);
int biu_version(void);

/* ---- network handle: replaces network(...).to(device); load_state_dict; eval; self.model(patch) -----------
 * unet/predict.py:98-101,197  siam_unet/predict.py:73-76,211  unet3d/predict.py:84-88,166
 * multi_output_unet3d/predict.py:55-62,192 */
typedef struct biu_net biu_net;

/* n_heads/head_channels/head_acts/head_names describe the output layer(s): one sigmoid head of `out_channels`
 * channels for Unet/Siam_UNet/UNet3D, the output_heads dict for MultiOutputUnet3D.
 * siam_mode: BIU_SIAM_*; use_interpolation: constructor flag of UNet3D / MultiOutputUnet3D. */
biu_net* biu_net_create(int kind, int n_filter, int in_channels, int n_heads, const int* head_channels,
                        const int* head_acts, const char* const* head_names, int siam_mode, int use_interpolation,
                        int precision);
/* One call per state_dict entry (same key, fp32, C-contiguous, HOST memory; copied). Unknown keys are kept and
 * ignored; missing ones are reported by biu_net_finalize. */
int biu_net_set_param(biu_net* net, const char* name, const float* data_host, int ndim, const long long* shape);
/* Fold BatchNorm (eps 1e-5) into per-channel scale/shift, repack weights, upload. */
int biu_net_finalize(biu_net* net);
/* Fix the batch and tile extents (d = 1 for 2D). Returns the workspace size in bytes. Tile extents must be
 * divisible by 16 (2D) / 8 (3D): the reference raises 'concatenation failed: wrong dimensions' (unet/unet.py:67). */
long long biu_net_plan(biu_net* net, int batch, int d, int h, int w);
/* Forward of `batch` tiles. in: planar [batch][in_channels][d][h][w] (uint8 or float32 per in_kind);
 * in2: previous-frame tiles for Siam_UNet (else NULL). Outputs are planar [batch][sum(head_channels)][d][h][w]:
 * out_val = activated head output (float32, may be NULL), out_u8 = trunc(out_val*255) (may be NULL;
 * unet/predict.py:200). workspace: biu_net_plan bytes, zero-initialised once by the caller. */
int biu_net_forward(biu_net* net, const void* in, int in_kind, const void* in2, float* out_val, uint8_t* out_u8,
                    void* workspace, void* stream);
/* Test hook: copy a named intermediate activation (e.g. "e1", "cat4", "mid2") to host memory. */
int biu_net_debug_copy(biu_net* net, const char* name, void* workspace, void* dst_host, long long max_bytes);
/* Test hook: 1 = run every convolution on the CUDA-core kernels. */
int biu_net_set_force_direct(biu_net* net, int on);
/* Test hook: 0 = run MaxPool2d as its own kernel instead of fusing it into the preceding block's epilogue
 * (default 1; both give bit-identical activations). */
int biu_net_set_fuse_pool(biu_net* net, int on);
/* Test hook: last_op >= 0 makes the following biu_net_forward calls return after op `last_op` of the layer program
 * (a pool fused into that op's epilogue is written, as in a full forward); later ops, out_val and out_u8 are not
 * written, and biu_net_profile_read refuses such a forward. -1 (the default) runs the whole program. */
int biu_net_set_debug_stop(biu_net* net, int last_op);
/* Siam_UNet with per-frame ('single') normalisation (siam_unet/predict.py:102-136, siam_unet/siam_unet.py:85-112): frame t
 * is the current frame of pair t and the previous frame of pair t + 1 and its normalised tiles - hence its encoder
 * output - are the same in both. tiles_per_frame > 0 makes the following biu_net_plan(batch B, ...) / biu_net_forward
 * run the shared-weight encoder ONCE over the B + tiles_per_frame unique tiles of B consecutive tile pairs: `in` then
 * holds [tiles of the previous frame of the first pair | tiles of the current frames] (B + tiles_per_frame tiles, `in2`
 * null); pair j uses tile j as its previous and tile j + tiles_per_frame as its current frame. 0 restores the two-input
 * form. Results are bit-identical; 21 % of the reference's FLOPs are not executed. */
int biu_net_set_siam_shared(biu_net* net, int tiles_per_frame);
/* Number of convolution / transposed-convolution / gate ops of the most recent biu_net_forward that a tensor-core
 * mode (bf16 / fp16 / tf32) had to run on the CUDA-core kernels because the tile shape is outside what the tcgen05 kernels
 * take (planes narrower than 8 px, ...). 0 in the exact-fp32 mode's sense of "as requested"; the Python Predict
 * classes turn a non-zero count into a RuntimeWarning (the result is the same, the speed is not). */
int biu_net_fallback_ops(biu_net* net);
/* Test hook (process-wide): 0 = run every halo-tile convolution on single CTAs instead of CTA pairs (default 1: layers
 * with at least 64 output channels per block run tcgen05.mma.cta_group::2, M = 256 over the two SMs of a TPC, each CTA
 * staging half of every weight tile; the MMAs and their order per output tile are the same, so results are
 * bit-identical). */
int biu_set_halo_cta2(int on);
/* Test hook (process-wide): 0 = run the narrow (Cout <= 32) 3x3 blocks on the halo-tile kernel instead of the
 * row-streaming folded-tap kernel (default 1; results agree to fp32 summation order); 2 = row kernel with its two
 * pipelines per CTA forced on even for workloads with few work items (they are only chosen for large batches). */
int biu_set_rows_kernel(int on);
void biu_net_destroy(biu_net* net);

/* ---- intensity normalisation: replaces Predict.__preprocess ------------------------------------------------
 * unet/predict.py:122-150  siam_unet/predict.py:125-162  unet3d/predict.py:109-117 */
/* hist[frames][65536] (uint32): per-frame histogram of a uint8 (dtype_bytes 1) or uint16 (2) stack. */
int biu_histogram(const void* img, int dtype_bytes, long long n_per_frame, int frames, uint32_t* hist, void* stream);
/* out[65536] = sum over frames ('all' mode, 3D global percentiles). */
int biu_hist_sum(const uint32_t* hist, int frames, uint32_t* out, void* stream);
/* Per frame f: percentile bounds (np.nanpercentile/np.percentile, linear) from hist_bounds + f*bounds_stride,
 * value range from hist_range + f*range_stride, then lut[f][v] = uint8(trunc(((clip(v,lo,hi)-mn)/mx)*255))
 * [255 - . when invert], all in float64 in numpy's operation order. params (may be NULL): [frames][4] doubles
 * {lo, hi, mn, mx}. Strides are in uint32 elements (0 = share one histogram). */
int biu_norm_lut(const uint32_t* hist_bounds, const uint32_t* hist_range, long long bounds_stride,
                 long long range_stride, int frames, double q_lo, double q_hi, int invert, uint8_t* lut,
                 double* params, void* stream);
/* out[f][i] = lut[f*lut_stride + img[f][i]] */
int biu_apply_lut(const void* img, int dtype_bytes, long long n_per_frame, int frames, const uint8_t* lut,
                  long long lut_stride, uint8_t* out, void* stream);

/* Percentile normalisation of a FLOAT32 stack to uint8, unet/predict.py:122-150 as numpy evaluates it on a float32
 * image (float32 percentiles with linear interpolation, clip, - min, / max * 255, optional 255 - x, truncating cast).
 * Exact order statistics by a two-level radix select on the floats' order-preserving keys. mode 0 'single' (per
 * frame), 1 'first' (percentiles of frame 0, range of the stack), 2 'all'. scratch: biu_normalize_f32_scratch_bytes().
 * params [frames or 1][4] = {lo, hi, min, max}; out_f32 (optional) = the float values the reference stores back. */
long long biu_normalize_f32_scratch_bytes(long long n_per_frame, int frames);
int biu_normalize_f32(const float* img, long long n_per_frame, int frames, int mode, double q_lo, double q_hi, int invert,
                      void* scratch, float* params, uint8_t* out_u8, float* out_f32, void* stream);

/* multi_output_unet3d/predict.py:104-125 on an integer-valued stack: float32 LUT of the float64 expression
 * (clip(v,lo,hi) - min) / (ptp + 1e-8) [mode 0, 'single'] or (clip(v,lo,hi) - lo) / (hi - lo + 1e-8) [mode 1];
 * mode 2 = multi_output_unet/predict.py:128-151: (clip(v,lo,hi) - min) / max in float32. */
int biu_norm_lut_f32(const uint32_t* hist_bounds, const uint32_t* hist_range, long long bounds_stride,
                     long long range_stride, int frames, double q_lo, double q_hi, int mode, float* lut,
                     double* params, void* stream);
int biu_apply_lut_f32(const void* img, int dtype_bytes, long long n_per_frame, int frames, const float* lut,
                      long long lut_stride, float* out, void* stream);
/* multi_output_unet3d/predict.py:127-174: float32 patches, src [F][Z][H][W] -> dst [F*nz*ny*nx][pd][ph][pw]. */
int biu_gather_tiles_f32(const float* src, int F, int Z, int H, int W, const int* zs, const int* ys, const int* xs,
                         int nz, int ny, int nx, int pd, int ph, int pw, float* dst, void* stream);

/* ---- tiling: replaces Predict.__split -----------------------------------------------------------------------
 * unet/predict.py:152-182  siam_unet/predict.py:164-197  unet3d/predict.py:119-153
 * src [F][Z][H][W] uint8 -> dst [F*nz*ny*nx][pd][ph][pw]; starts are device int32 arrays. */
int biu_gather_tiles(const uint8_t* src, int F, int Z, int H, int W, int pad_mode, const int* zs, const int* ys,
                     const int* xs, int nz, int ny, int nx, int pd, int ph, int pw, uint8_t* dst, void* stream);
/* Same with the intensity normalisation fused in (unet/predict.py:122-131 + :152-182 in one pass): src is the RAW
 * uint8 / uint16 stack and every value goes through lut[f * lut_stride + value] (tables of biu_norm_lut; lut_stride
 * 65536 = one table per frame, 0 = one for the stack) on its way into the tile - the normalised stack is never written.
 * Padding of undersized sources applies to the normalised values (zeros stay zeros, reflection commutes with the table). */
int biu_gather_tiles_lut(const void* src, int dtype_bytes, const uint8_t* lut, long long lut_stride, int F, int Z, int H,
                         int W, int pad_mode, const int* zs, const int* ys, const int* xs, int nz, int ny, int nx, int pd,
                         int ph, int pw, uint8_t* dst, void* stream);

/* ---- test-time augmentation (engine-only, replaces nothing in the reference) ---------------------------------
 * Transform code t of a tile: 2D (dims 2): bit 0 flips x, bit 1 flips y, bit 2 transposes after the flips (square tiles
 * only); 3D (dims 3): bits 0, 1, 2 flip x, y, z. The transform acts on the tile after the far-end padding, and t = 0 is
 * the plain tile. */
/* biu_gather_tiles / biu_gather_tiles_lut producing T_t(tile): a uint8 source (lut NULL) or a uint8 / uint16 source
 * with its normalisation tables. */
int biu_gather_tiles_tta(const void* src, int dtype_bytes, const uint8_t* lut, long long lut_stride, int F, int Z, int H,
                         int W, int pad_mode, const int* zs, const int* ys, const int* xs, int nz, int ny, int nx, int pd,
                         int ph, int pw, int dims, int t, uint8_t* dst, void* stream);
/* biu_gather_tiles_f32 producing T_t(patch). */
int biu_gather_tiles_f32_tta(const float* src, int F, int Z, int H, int W, const int* zs, const int* ys, const int* xs,
                             int nz, int ny, int nx, int pd, int ph, int pw, int dims, int t, float* dst, void* stream);
/* Pass `pass` of `passes` (a power of two) of the merge: val [planes][pd][ph][pw] is the net's float output on the tiles
 * of transform t; acc (same shape, fp32) = sum in pass order of T_t^-1(val). Pass 0 writes acc, the last pass writes
 * mean = acc * (1 / passes) to out_f32 and / or out_u8 = trunc(mean * 255) (the rule of biu_net_forward's out_u8) and
 * leaves acc as it was. Deterministic (no atomics). */
int biu_tta_accumulate(const float* val, long long planes, int pd, int ph, int pw, int dims, int t, int pass, int passes,
                       float* acc, uint8_t* out_u8, float* out_f32, void* stream);

/* ---- stitching: replaces Predict.__stitch -------------------------------------------------------------------*/
/* unet/predict.py:204-229, siam_unet/predict.py:217-240: uint8(nanmean) == sum // count.
 * tiles [F][ny*nx][C][ph][pw] -> out [F][C][H][W] */
int biu_stitch_mean_u8(const uint8_t* tiles, int F, int C, int H, int W, const int* ys, const int* xs, int ny, int nx,
                       int ph, int pw, uint8_t* out, void* stream);
/* unet3d/predict.py:173-195: three slots, patch n -> slot n % 3, last writer wins, nanmean, uint8. */
int biu_stitch_mod3_u8(const uint8_t* tiles, int Z, int H, int W, const int* zs, const int* ys, const int* xs, int nz,
                       int ny, int nx, int pd, int ph, int pw, uint8_t* out, void* stream);
/* Engine-only (replaces nothing in the reference): weighted overlap stitch of uint8 result tiles,
 *   out[f][c][z][y][x] = (sum w * v) // (sum w)   (0 where no tile covers the element or sum w = 0)
 * over every tile n covering the element, v = its value there, w = w_d[tz] * w_h[ty] * w_w[tx] at the in-tile position
 * (tz, ty, tx). Exact unsigned 64-bit integer sums and floor division: the result does not depend on the order of the
 * tiles. w_d / w_h / w_w: device int32 tables of pd / ph / pw entries, each in [0, 1024]. tiles
 * [F][nz*ny*nx][C][pd][ph][pw] -> out [F][C][Z][H][W]; starts may be negative and tiles may reach past the output.
 * 2D: nz = pd = Z = 1, zs = {0}, w_d = {1}. */
int biu_stitch_weighted_u8(const uint8_t* tiles, int F, int C, int Z, int H, int W, const int* zs, const int* ys,
                           const int* xs, int nz, int ny, int nx, int pd, int ph, int pw, const int* w_d, const int* w_h,
                           const int* w_w, uint8_t* out, void* stream);
/* multi_output_unet3d/predict.py:203-307: ramp-weighted blend, tiles [V][nz*ny*nx][C][pd][ph][pw] float32. */
int biu_stitch_ramp_f32(const float* tiles, int V, int C, int Z, int H, int W, const int* zs, const int* ys,
                        const int* xs, int nz, int ny, int nx, int pd, int ph, int pw, int margin, float* out,
                        void* stream);

/* multi_output_unet/predict.py:230-285: margin-weighted mean (weight 0 on the `margin` border rows / columns that face
 * a neighbouring patch), tiles [P][C][ph][pw] float32 read through float16 rounding like the reference's float16 patch
 * store; src_index [T][ny][nx] = flat patch index of tile (image, j, k); ys/ny along rows, xs/nx along columns;
 * pixels without weight get *fill (device scalar). out [T][C][H][W]. */
int biu_stitch_margin_f32(const float* tiles, const int* src_index, int T, int C, int H, int W, const int* ys,
                          const int* xs, int ny, int nx, int ph, int pw, int margin, const float* fill, float* out,
                          void* stream);

/* ---- single layers (used by the parity tests; same kernels the network handle launches) ------------------- */
/* Element code `esz` of the layer entry points: 2 = bf16 activations (and tcgen05 weights), 4 = fp32 storage / tf32
 * math, BIU_ESZ_FP16 = fp16 activations / weights (2-byte elements). */
enum { BIU_ESZ_FP16 = 3 };
/* Conv(k in {1,3}, pad k/2) + per-channel scale/shift + LeakyReLU(slope) on tcgen05.
 * in: NDHWC with channel stride in_ctot, offset in_coff; wgt: [kd*kh*kw][cout][cin]; out: NDHWC (out_ctot/out_coff). */
int biu_conv_tc(int esz, const void* in, int in_ctot, int in_coff, int cin, int B, int D, int H, int W, int kd,
                int kh, int kw, const void* wgt, int cout, const float* scale, const float* shift, float slope,
                void* out, int out_ctot, int out_coff, void* stream);
/* ConvTranspose(k=2,s=2) + bias on tcgen05; wgt: [2^dims * cout][cin], row q*cout+co with q = (az,ay,ax) bits. */
int biu_up_tc(int esz, const void* in, int in_ctot, int in_coff, int cin, int B, int D, int H, int W, int dims,
              const void* wgt, int cout, const float* bias_rep, void* out, int out_ctot, int out_coff, void* stream);
/* fp32 CUDA-core convolution, wgt fp32 [taps][cin][cout]. */
int biu_conv_direct(int esz, const void* in, int in_ctot, int in_coff, int cin, int B, int D, int H, int W, int kd,
                    int kh, int kw, const float* wgt, int cout, const float* scale, const float* shift, float slope,
                    void* out, int out_ctot, int out_coff, void* stream);
int biu_pool2(int esz, const void* in, int in_ctot, int in_coff, int c, int B, int D, int H, int W, int dims,
              int mode, void* out, int out_ctot, int out_coff, void* stream);
/* Device fault word written by a kernel whose pipeline wait timed out (0 = none). */
int biu_device_fault(unsigned int* code_host);
/* Kernel launches issued by the library since it was loaded. */
unsigned long long biu_launch_count(void);
/* Measurement hooks: with profiling on, biu_net_forward brackets every layer with CUDA events on the caller's
 * stream; biu_net_profile_read synchronises those events and returns, for the most recent forward, the op kind
 * (0 first conv, 1 conv block [tcgen05], 2 conv block + head [tcgen05], 3 transposed conv [tcgen05], 4 pool,
 * 5 nearest upsample, 6 max join; +16 when the op ran on the CUDA-core fallback, +32 when it was fused into the
 * previous op and launched nothing) and its duration in ms. */
int biu_net_set_profile(biu_net* net, int on);
int biu_net_profile_read(biu_net* net, int max_ops, int* kinds, float* ms, int* n_ops);

#ifdef __cplusplus
}
#endif
#endif /* BIU_B200_H */
