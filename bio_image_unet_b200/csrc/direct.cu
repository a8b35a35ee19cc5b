// CUDA-core kernels of the network: first layer (1..4 input channels), 2x pooling / nearest resampling,
// standalone 1x1 head, and a shared-memory-tiled fp32 direct convolution / transposed convolution used for the
// exact-fp32 mode and for channel counts the tensor-core kernel cannot take. All NHWC / NDHWC.
#include "common.cuh"
#include "launch.h"

namespace biu {

template <typename T> __device__ __forceinline__ float ld_act(const T* p);
template <> __device__ __forceinline__ float ld_act<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float ld_act<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}
template <> __device__ __forceinline__ float ld_act<__half>(const __half* p) { return __half2float(*p); }
__device__ __forceinline__ float to_tf32(float v) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
  return __uint_as_float(u);
}
template <typename T> __device__ __forceinline__ void st_act(T* p, float v, int round_tf32);
template <> __device__ __forceinline__ void st_act<float>(float* p, float v, int round_tf32) {
  *p = round_tf32 ? to_tf32(v) : v;
}
template <> __device__ __forceinline__ void st_act<__nv_bfloat16>(__nv_bfloat16* p, float v, int) {
  *p = __float2bfloat16_rn(v);
}
template <> __device__ __forceinline__ void st_act<__half>(__half* p, float v, int) { *p = __float2half_rn(v); }

// ------------------------------------------------------------------------------------------------
// First block: Conv(k=3,pad=1) on a planar few-channel input + folded BN + LeakyReLU (unet/unet.py:20,54-60;
// unet3d/unet3d.py:24). u8 tiles are converted as float32(u8)/255 (unet/predict.py:192). One thread per
// (pixel, 8 output channels): 16-byte bf16 / fp16 stores; weights staged in shared memory.
// ------------------------------------------------------------------------------------------------
template <typename TIN, typename TOUT>
__global__ void __launch_bounds__(256) first_conv_kernel(FirstConvArgs a) {
  extern __shared__ float sw[];  // [taps*cin][cout_pad] then scale[cout_pad], shift[cout_pad]
  const int taps = 9 * a.kd;
  const int kk = taps * a.cin;
  float* s_scale = sw + kk * a.cout_pad;
  float* s_shift = s_scale + a.cout_pad;
  for (int i = threadIdx.x; i < kk * a.cout_pad; i += blockDim.x) {
    const int co = i % a.cout_pad, k = i / a.cout_pad;
    sw[i] = co < a.cout ? a.wgt[k * a.cout + co] : 0.f;
  }
  for (int i = threadIdx.x; i < a.cout_pad; i += blockDim.x) {
    s_scale[i] = i < a.cout ? a.scale[i] : 0.f;
    s_shift[i] = i < a.cout ? a.shift[i] : 0.f;
  }
  __syncthreads();
  const int groups = a.cout_pad / 8;
  const long long npix = (long long)a.B * a.D * a.H * a.W;
  const long long plane = (long long)a.D * a.H * a.W;
  const TIN* in = reinterpret_cast<const TIN*>(a.in);
  TOUT* out = reinterpret_cast<TOUT*>(a.out);
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < npix * groups;
       idx += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(idx % groups);
    const long long pix = idx / groups;
    long long r = pix;
    const int x = (int)(r % a.W); r /= a.W;
    const int y = (int)(r % a.H); r /= a.H;
    const int z = (int)(r % a.D); r /= a.D;
    const int b = (int)r;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    int tap = 0;
    for (int dz = 0; dz < a.kd; ++dz) {
      const int zz = z + dz - (a.kd >> 1);
      for (int dy = 0; dy < 3; ++dy) {
        const int yy = y + dy - 1;
        for (int dx = 0; dx < 3; ++dx, ++tap) {
          const int xx = x + dx - 1;
          if (zz < 0 || zz >= a.D || yy < 0 || yy >= a.H || xx < 0 || xx >= a.W) continue;
          for (int ci = 0; ci < a.cin; ++ci) {
            const long long off = ((long long)b * a.cin + ci) * plane + ((long long)zz * a.H + yy) * a.W + xx;
            float v;
            if (sizeof(TIN) == 1) v = __fdiv_rn((float)in[off], 255.0f); else v = (float)in[off];
            const float* w = sw + (tap * a.cin + ci) * a.cout_pad + g * 8;
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = fmaf(v, w[j], acc[j]);
          }
        }
      }
    }
    TOUT* o = out + pix * a.out_ctot + a.out_coff + g * 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float t = fmaf(acc[j], s_scale[g * 8 + j], s_shift[g * 8 + j]);
      t = t > 0.f ? t : t * a.slope;
      st_act<TOUT>(o + j, t, a.fmt == FMT_TF32);
    }
  }
}

// Fast path for a single input channel (every reference model): one thread per pixel gathers the 9 / 27 taps once
// into registers, then produces all output channels 8 at a time (broadcast weight reads from shared memory,
// 16-byte stores; a warp writes 32 consecutive pixels = one contiguous run of the NHWC buffer).
template <typename TIN, typename TOUT, int TAPS>
__global__ void __launch_bounds__(256) first_conv1_kernel(FirstConvArgs a) {
  extern __shared__ float sw[];  // [TAPS][cout_pad], scale[cout_pad], shift[cout_pad]
  float* s_scale = sw + TAPS * a.cout_pad;
  float* s_shift = s_scale + a.cout_pad;
  for (int i = threadIdx.x; i < TAPS * a.cout_pad; i += blockDim.x) {
    const int co = i % a.cout_pad, k = i / a.cout_pad;
    sw[i] = co < a.cout ? a.wgt[k * a.cout + co] : 0.f;
  }
  for (int i = threadIdx.x; i < a.cout_pad; i += blockDim.x) {
    s_scale[i] = i < a.cout ? a.scale[i] : 0.f;
    s_shift[i] = i < a.cout ? a.shift[i] : 0.f;
  }
  __syncthreads();
  const long long npix = (long long)a.B * a.D * a.H * a.W;
  const long long plane = (long long)a.D * a.H * a.W;
  const TIN* in = reinterpret_cast<const TIN*>(a.in);
  TOUT* out = reinterpret_cast<TOUT*>(a.out);
  constexpr int KD = TAPS / 9;
  for (long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x; pix < npix;
       pix += (long long)gridDim.x * blockDim.x) {
    long long r = pix;
    const int x = (int)(r % a.W); r /= a.W;
    const int y = (int)(r % a.H); r /= a.H;
    const int z = (int)(r % a.D); r /= a.D;
    const TIN* img = in + r * plane;
    float v[TAPS];
#pragma unroll
    for (int dz = 0; dz < KD; ++dz)
#pragma unroll
      for (int dy = 0; dy < 3; ++dy)
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          const int zz = z + dz - (KD >> 1), yy = y + dy - 1, xx = x + dx - 1;
          float t = 0.f;
          if (zz >= 0 && zz < a.D && yy >= 0 && yy < a.H && xx >= 0 && xx < a.W) {
            const TIN raw = __ldg(img + ((long long)zz * a.H + yy) * a.W + xx);
            t = sizeof(TIN) == 1 ? __fdiv_rn((float)raw, 255.0f) : (float)raw;
          }
          v[(dz * 3 + dy) * 3 + dx] = t;
        }
    TOUT* o = out + pix * a.out_ctot + a.out_coff;
    for (int g = 0; g < a.cout_pad; g += 8) {
      float acc[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
      for (int t = 0; t < TAPS; ++t) {
        const float4 w0 = *reinterpret_cast<const float4*>(sw + t * a.cout_pad + g);
        const float4 w1 = *reinterpret_cast<const float4*>(sw + t * a.cout_pad + g + 4);
        acc[0] = fmaf(v[t], w0.x, acc[0]); acc[1] = fmaf(v[t], w0.y, acc[1]);
        acc[2] = fmaf(v[t], w0.z, acc[2]); acc[3] = fmaf(v[t], w0.w, acc[3]);
        acc[4] = fmaf(v[t], w1.x, acc[4]); acc[5] = fmaf(v[t], w1.y, acc[5]);
        acc[6] = fmaf(v[t], w1.z, acc[6]); acc[7] = fmaf(v[t], w1.w, acc[7]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float t = fmaf(acc[j], s_scale[g + j], s_shift[g + j]);
        acc[j] = t > 0.f ? t : t * a.slope;
      }
      if (sizeof(TOUT) == 2) {
        uint32_t w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) w[j] = pack_half2<fmt_of<TOUT>>(acc[2 * j], acc[2 * j + 1]);
        *reinterpret_cast<uint4*>(o + g) = make_uint4(w[0], w[1], w[2], w[3]);
      } else {
        float* of = reinterpret_cast<float*>(o + g);
        if (a.fmt == FMT_TF32) {
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = to_tf32(acc[j]);
        }
        *reinterpret_cast<float4*>(of) = make_float4(acc[0], acc[1], acc[2], acc[3]);
        *reinterpret_cast<float4*>(of + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
      }
    }
  }
}

// 3D, single input channel. A block owns a column of ZC planes of an (8 rows x 128 voxels) tile and slides along z:
// four input planes (10 rows x 130 voxels with the halo, already float32(u8)/255 - exact division,
// unet3d/predict.py:161) rotate through shared memory, the plane needed two steps ahead is fetched from global
// memory while the current plane is computed (one __syncthreads per plane, no global latency and no bounds checks in
// the arithmetic). A thread produces a run of 4 consecutive voxels along x as TWO VOXEL PAIRS: the arithmetic runs on
// packed float pairs (FFMA2: {out[x], out[x+1]} += {in[x+dx], in[x+1+dx]} * {w, w}), so the input pairs of all three dx
// taps come straight out of shared memory as aligned 64-bit register pairs - the planes are kept twice, the second
// copy shifted by one voxel, which makes the odd-aligned pairs of the dx = 0 / 2 taps 16- / 8-byte aligned loads - and
// the weights are kept pre-duplicated ({w, w}), one 16-byte broadcast load per two output channels: no register
// shuffling between the loads and the FMAs (the previous form spent two moves per FFMA2 operand on {v, v} pairs).
// The FMA order of every output is unchanged ((dz, dy, dx) ascending): results are bit-identical to the scalar form.
// Channel groups that are pure padding (UNet3D's first block has n_filter / 2 = 8 real channels in a 16-channel
// buffer) are written as zeros without any arithmetic; a thread's stores cover 4 * C_out contiguous elements.
constexpr int kFc3Rows = 8, kFc3Cols = 128, kFc3Pitch = 136, kFc3Planes = 4, kFc3ZC = 16;
constexpr int kFc3PlaneF = (kFc3Rows + 2) * kFc3Pitch;                 // floats of one staged plane
static size_t first_conv1_3d_smem(int cout_pad) {
  return ((size_t)27 * cout_pad * 2 + 4 * cout_pad + 256 + 2 * kFc3Planes * kFc3PlaneF) * sizeof(float);
}
template <typename TIN, typename TOUT>
__global__ void __launch_bounds__(256, 2) first_conv1_3d_kernel(FirstConvArgs a) {
  extern __shared__ __align__(16) float fc3_smem[];
  float* sw2 = fc3_smem;                                   // [27][cout_pad] x {w, w}
  float* s_scale2 = sw2 + 27 * a.cout_pad * 2;             // [cout_pad] x {s, s}
  float* s_shift2 = s_scale2 + 2 * a.cout_pad;
  float* lut = s_shift2 + 2 * a.cout_pad;                  // u8 -> float32(u8)/255
  float* tile_a = lut + 256;                               // voxel xt - 4 + j of a row at index j
  float* tile_b = tile_a + kFc3Planes * kFc3PlaneF;        // the same rows one voxel further right: b[j] = a[j - 1]
  for (int i = threadIdx.x; i < 27 * a.cout_pad; i += blockDim.x) {
    const int co = i % a.cout_pad, k = i / a.cout_pad;
    const float w = co < a.cout ? a.wgt[k * a.cout + co] : 0.f;
    sw2[2 * i] = w; sw2[2 * i + 1] = w;
  }
  for (int i = threadIdx.x; i < a.cout_pad; i += blockDim.x) {
    const float sc = i < a.cout ? a.scale[i] : 0.f, sh = i < a.cout ? a.shift[i] : 0.f;
    s_scale2[2 * i] = sc; s_scale2[2 * i + 1] = sc;
    s_shift2[2 * i] = sh; s_shift2[2 * i + 1] = sh;
  }
  if (sizeof(TIN) == 1) lut[threadIdx.x] = __fdiv_rn((float)threadIdx.x, 255.0f);
  __syncthreads();
  constexpr int PLANE = kFc3PlaneF, NVAL = (kFc3Rows + 2) * (kFc3Cols + 2), NLD = (NVAL + 255) / 256;
  const int tiles_x = (a.W + kFc3Cols - 1) / kFc3Cols, tiles_y = (a.H + kFc3Rows - 1) / kFc3Rows;
  const int zchunks = (a.D + kFc3ZC - 1) / kFc3ZC;
  const int ncols = a.B * zchunks * tiles_y * tiles_x;
  const long long plane = (long long)a.D * a.H * a.W;
  const int real_c = ((a.cout_real > 0 ? min(a.cout_real, a.cout) : a.cout) + 7) & ~7;   // channels [real_c, cout_pad) are padding
  const TIN* in = reinterpret_cast<const TIN*>(a.in);
  TOUT* out = reinterpret_cast<TOUT*>(a.out);
  const unsigned long long slope2 = pack_f32x2(a.slope, a.slope);
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int col = blockIdx.x; col < ncols; col += gridDim.x) {
    int rem = col;
    const int xt = (rem % tiles_x) * kFc3Cols; rem /= tiles_x;
    const int yt = (rem % tiles_y) * kFc3Rows; rem /= tiles_y;
    const int z0 = (rem % zchunks) * kFc3ZC; const int r = rem / zchunks;
    const int z1 = min(z0 + kFc3ZC, a.D);
    const TIN* img = in + r * plane;
    // one input plane zz of the tile (rows yt-1 .. yt+8, voxels xt-1 .. xt+128), zero outside the volume
    TIN stg[NLD];                                                  // raw values: converted only when they are stashed,
    bool stg_ok[NLD];                                              // so the global loads stay in flight during the arithmetic
    int g_off[NLD], s_off[NLD];                                    // z-invariant part of this thread's staging work
    bool in_ok[NLD];
#pragma unroll
    for (int k = 0; k < NLD; ++k) {
      const int i = threadIdx.x + k * 256;
      const int ry = i / (kFc3Cols + 2), rx = i - ry * (kFc3Cols + 2);
      const int yy = yt - 1 + ry, xx = xt - 1 + rx;
      in_ok[k] = i < NVAL && yy >= 0 && yy < a.H && xx >= 0 && xx < a.W;
      g_off[k] = yy * a.W + xx;
      s_off[k] = i < NVAL ? ry * kFc3Pitch + 3 + rx : -1;         // voxel xt - 4 + j lives at index j
    }
    const int hw = a.H * a.W;
    auto fetch = [&](int zz) {
      const bool z_ok = zz >= 0 && zz < a.D;
      const TIN* pz = img + (long long)zz * hw;
#pragma unroll
      for (int k = 0; k < NLD; ++k) {
        stg_ok[k] = z_ok && in_ok[k];
        stg[k] = 0;
        if (stg_ok[k]) stg[k] = __ldg(pz + g_off[k]);
      }
    };
    auto stash = [&](int zz) {
      const int po = ((zz + kFc3Planes) % kFc3Planes) * PLANE;
#pragma unroll
      for (int k = 0; k < NLD; ++k) {
        float t = 0.f;
        if (stg_ok[k]) t = sizeof(TIN) == 1 ? lut[(int)stg[k]] : (float)stg[k];
        if (s_off[k] >= 0) { tile_a[po + s_off[k]] = t; tile_b[po + s_off[k] + 1] = t; }
      }
    };
    __syncthreads();                                               // the previous column's planes are consumed
    for (int zz = z0 - 1; zz <= z0 + 1; ++zz) { fetch(zz); stash(zz); }
    __syncthreads();
    const int y = yt + wid, x0 = xt + 4 * lane;
    const bool active = y < a.H && x0 < a.W;
    const int t_off = wid * kFc3Pitch + 4 * lane;                  // a[t_off + 3 + i] = voxel x0 - 1 + i of row y - 1
    for (int z = z0; z < z1; ++z) {
      const bool more = z + 1 < z1;
      if (more) fetch(z + 2);                                      // in flight while this plane is computed
      if (active) {
        TOUT* o = out + ((r * plane + ((long long)z * a.H + y) * a.W + x0) * a.out_ctot + a.out_coff);
        for (int g = 0; g < a.cout_pad; g += 8) {
          if (g >= real_c) {
#pragma unroll
            for (int xi = 0; xi < 4; ++xi) {
              if (x0 + xi >= a.W) break;
              TOUT* ov = o + (long long)xi * a.out_ctot + g;
              if (sizeof(TOUT) == 2) *reinterpret_cast<uint4*>(ov) = make_uint4(0, 0, 0, 0);
              else { *reinterpret_cast<float4*>(ov) = make_float4(0.f, 0.f, 0.f, 0.f); *reinterpret_cast<float4*>(reinterpret_cast<float*>(ov) + 4) = make_float4(0.f, 0.f, 0.f, 0.f); }
            }
            continue;
          }
          unsigned long long acc2[2][8];                           // [voxel pair (x0, x0+1) / (x0+2, x0+3)][channel]
#pragma unroll
          for (int xp = 0; xp < 2; ++xp)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc2[xp][c] = 0ull;
#pragma unroll
          for (int dz = 0; dz < 3; ++dz) {
            const int po = ((z + dz - 1 + kFc3Planes) % kFc3Planes) * PLANE + t_off;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
              const float* ra = tile_a + po + dy * kFc3Pitch;
              const float* rbp = tile_b + po + dy * kFc3Pitch;
              // voxels x0-1 .. x0+4 = a[3..8]: pairs (a3,a4) (a5,a6) = b[4..7]; (a4,a5) (a6,a7) = a[4..7]; (a7,a8) = b[8..9]
              const ulonglong2 p0 = *reinterpret_cast<const ulonglong2*>(rbp + 4);
              const ulonglong2 p1 = *reinterpret_cast<const ulonglong2*>(ra + 4);
              const unsigned long long p2 = *reinterpret_cast<const unsigned long long*>(rbp + 8);
              const unsigned long long pr[3][2] = {{p0.x, p0.y}, {p1.x, p1.y}, {p0.y, p2}};
#pragma unroll
              for (int dx = 0; dx < 3; ++dx) {
                const float* wt = sw2 + (((dz * 3 + dy) * 3 + dx) * a.cout_pad + g) * 2;
#pragma unroll
                for (int c2 = 0; c2 < 4; ++c2) {
                  const ulonglong2 w = *reinterpret_cast<const ulonglong2*>(wt + 4 * c2);    // {w, w} of channels 2 c2, 2 c2 + 1
                  acc2[0][2 * c2] = fma_f32x2(pr[dx][0], w.x, acc2[0][2 * c2]);
                  acc2[1][2 * c2] = fma_f32x2(pr[dx][1], w.x, acc2[1][2 * c2]);
                  acc2[0][2 * c2 + 1] = fma_f32x2(pr[dx][0], w.y, acc2[0][2 * c2 + 1]);
                  acc2[1][2 * c2 + 1] = fma_f32x2(pr[dx][1], w.y, acc2[1][2 * c2 + 1]);
                }
              }
            }
          }
          // BatchNorm + LeakyReLU (t > 0 ? t : t * slope == max(t, t * slope) for 0 <= slope <= 1), per voxel 8 channels
          float res[4][8];
#pragma unroll
          for (int c2 = 0; c2 < 4; ++c2) {
            const ulonglong2 sc = *reinterpret_cast<const ulonglong2*>(s_scale2 + (g + 2 * c2) * 2);
            const ulonglong2 sh = *reinterpret_cast<const ulonglong2*>(s_shift2 + (g + 2 * c2) * 2);
#pragma unroll
            for (int xp = 0; xp < 2; ++xp) {
              const unsigned long long t0 = fma_f32x2(acc2[xp][2 * c2], sc.x, sh.x);
              const unsigned long long t1 = fma_f32x2(acc2[xp][2 * c2 + 1], sc.y, sh.y);
              const unsigned long long u0 = mul_f32x2(t0, slope2), u1 = mul_f32x2(t1, slope2);
              float ta, tb, ua, ub;
              unpack_f32x2(t0, ta, tb); unpack_f32x2(u0, ua, ub);
              res[2 * xp][2 * c2] = fmaxf(ta, ua); res[2 * xp + 1][2 * c2] = fmaxf(tb, ub);
              unpack_f32x2(t1, ta, tb); unpack_f32x2(u1, ua, ub);
              res[2 * xp][2 * c2 + 1] = fmaxf(ta, ua); res[2 * xp + 1][2 * c2 + 1] = fmaxf(tb, ub);
            }
          }
#pragma unroll
          for (int xi = 0; xi < 4; ++xi) {
            if (x0 + xi >= a.W) break;
            TOUT* ov = o + (long long)xi * a.out_ctot + g;
            if (sizeof(TOUT) == 2) {
              uint32_t w[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) w[j] = pack_half2<fmt_of<TOUT>>(res[xi][2 * j], res[xi][2 * j + 1]);
              *reinterpret_cast<uint4*>(ov) = make_uint4(w[0], w[1], w[2], w[3]);
            } else {
              float* of = reinterpret_cast<float*>(ov);
              float v8[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) v8[j] = a.fmt == FMT_TF32 ? to_tf32(res[xi][j]) : res[xi][j];
              *reinterpret_cast<float4*>(of) = make_float4(v8[0], v8[1], v8[2], v8[3]);
              *reinterpret_cast<float4*>(of + 4) = make_float4(v8[4], v8[5], v8[6], v8[7]);
            }
          }
        }
      }                                                            // active
      if (more) stash(z + 2);
      __syncthreads();
    }
  }
}

// 2D, single input channel, third generation: a block stages its input patch (8 warps x 32/G pixels wide, 64 rows,
// 1-pixel halo) in shared memory as float32(u8)/255 (exact division, unet/predict.py:192), then every warp walks down
// its strip, lane = (pixel x, channel group g of 8). The 72 weights of the group stay in registers for the whole
// kernel, the 3x3 window slides down the strip (3 new values per output row from shared memory - the second
// generation fetched them from global memory one row ahead and stalled on that latency), the arithmetic runs on
// packed float pairs (FFMA2), and for every row the warp's 16-byte stores cover one contiguous run of the NHWC
// buffer (full sectors, not 16 B pieces of 32 pixels).
constexpr int kFcRows = 64;
template <typename TIN, typename TOUT, int G>
__global__ void __launch_bounds__(256, 2) first_conv1_2d_kernel(FirstConvArgs a) {
  constexpr int PXW = 32 / G;                   // pixels per warp row
  constexpr int TX = 8 * PXW;                   // block tile: 8 warps side by side ...
  constexpr int TY = G >= 4 ? kFcRows : kFcRows / 2;   // ... TY rows tall
  constexpr int PITCH = TX + 2;
  __shared__ float tile[(TY + 2) * PITCH];      // input patch with its 1-pixel halo, already float32(u8)/255
  __shared__ __align__(16) float s_sc[64], s_sh[64];
  if (threadIdx.x < 64) {
    s_sc[threadIdx.x] = threadIdx.x < a.cout ? a.scale[threadIdx.x] : 0.f;
    s_sh[threadIdx.x] = threadIdx.x < a.cout ? a.shift[threadIdx.x] : 0.f;
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int g = lane % G, lx = lane / G;
  // weights, accumulators and the BatchNorm affine as float PAIRS: fma.rn.f32x2 (FFMA2 on sm_100) does two IEEE
  // fp32 FMAs per issue slot; results are bit-identical to the scalar form
  unsigned long long w2[9][4];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const float wa = (g * 8 + 2 * m) < a.cout ? __ldg(a.wgt + t * a.cout + g * 8 + 2 * m) : 0.f;
      const float wb = (g * 8 + 2 * m + 1) < a.cout ? __ldg(a.wgt + t * a.cout + g * 8 + 2 * m + 1) : 0.f;
      w2[t][m] = pack_f32x2(wa, wb);
    }
  const int tiles_x = (a.W + TX - 1) / TX, tiles_y = (a.H + TY - 1) / TY;
  const int total = a.B * tiles_y * tiles_x;
  const TIN* in = reinterpret_cast<const TIN*>(a.in);
  TOUT* out = reinterpret_cast<TOUT*>(a.out);
  const int W = a.W, H = a.H;
  const unsigned long long slope2 = pack_f32x2(a.slope, a.slope);
  for (int t = blockIdx.x; t < total; t += gridDim.x) {
    int r = t;
    const int tx = r % tiles_x; r /= tiles_x;
    const int ty = r % tiles_y; r /= tiles_y;
    const int x0 = tx * TX, y0 = ty * TY;
    __syncthreads();                                                // the previous tile has been consumed
    // the block stages its input patch once: coalesced loads, conversion (exact division, unet/predict.py:192) and
    // zero padding happen here, so the row loop below has no global-memory latency on its critical path
    const TIN* img = in + (long long)r * H * W;
    for (int i = threadIdx.x; i < (TY + 2) * PITCH; i += 256) {
      const int yy = i / PITCH, xx = i - yy * PITCH;
      const int gy = y0 + yy - 1, gx = x0 + xx - 1;
      float v = 0.f;
      if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
        const TIN raw = __ldg(img + (long long)gy * W + gx);
        v = sizeof(TIN) == 1 ? __fdiv_rn((float)raw, 255.0f) : (float)raw;
      }
      tile[i] = v;
    }
    __syncthreads();
    const int xl = wid * PXW + lx, x = x0 + xl;                     // this thread's pixel column
    const int y1 = min(TY, H - y0);
    const bool c1 = x < W;
    const float* tp = tile + xl;                                     // tile[yy][xl + dx] = input (y0 + yy - 1, x + dx - 1)
    float v0[3], v1[3], v2[3];
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) { v0[dx] = tp[dx]; v1[dx] = tp[PITCH + dx]; }
    TOUT* o = out + (((long long)r * H + y0) * W + x) * a.out_ctot + a.out_coff + g * 8;
    const long long o_step = (long long)W * a.out_ctot;
    for (int y = 0; y < y1; ++y, o += o_step) {
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) v2[dx] = tp[(y + 2) * PITCH + dx];
      unsigned long long acc2[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const unsigned long long b0 = pack_f32x2(v0[dx], v0[dx]), b1 = pack_f32x2(v1[dx], v1[dx]),
                                 b2 = pack_f32x2(v2[dx], v2[dx]);
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          acc2[m] = fma_f32x2(b0, w2[dx][m], acc2[m]);
          acc2[m] = fma_f32x2(b1, w2[3 + dx][m], acc2[m]);
          acc2[m] = fma_f32x2(b2, w2[6 + dx][m], acc2[m]);
        }
      }
      const ulonglong2 sc01 = *reinterpret_cast<const ulonglong2*>(s_sc + g * 8), sc23 = *reinterpret_cast<const ulonglong2*>(s_sc + g * 8 + 4);
      const ulonglong2 sh01 = *reinterpret_cast<const ulonglong2*>(s_sh + g * 8), sh23 = *reinterpret_cast<const ulonglong2*>(s_sh + g * 8 + 4);
      const unsigned long long sc2[4] = {sc01.x, sc01.y, sc23.x, sc23.y}, sh2[4] = {sh01.x, sh01.y, sh23.x, sh23.y};
      float acc[8];
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const unsigned long long t2 = fma_f32x2(acc2[m], sc2[m], sh2[m]);
        const unsigned long long u2 = mul_f32x2(t2, slope2);
        float ta, tb, ua, ub;
        unpack_f32x2(t2, ta, tb);
        unpack_f32x2(u2, ua, ub);
        acc[2 * m] = ta > 0.f ? ta : ua;             // LeakyReLU / ReLU: t > 0 ? t : t * slope
        acc[2 * m + 1] = tb > 0.f ? tb : ub;
      }
      if (c1) {
        if (sizeof(TOUT) == 2) {
          uint32_t pk[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) pk[j] = pack_half2<fmt_of<TOUT>>(acc[2 * j], acc[2 * j + 1]);
          *reinterpret_cast<uint4*>(o) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        } else {
          float* of = reinterpret_cast<float*>(o);
          if (a.fmt == FMT_TF32) {
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = to_tf32(acc[j]);
          }
          *reinterpret_cast<float4*>(of) = make_float4(acc[0], acc[1], acc[2], acc[3]);
          *reinterpret_cast<float4*>(of + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
        }
      }
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) { v0[dx] = v1[dx]; v1[dx] = v2[dx]; }
    }
  }
}

template <typename TIN, typename TOUT>
static void launch_first_conv1_2d(const FirstConvArgs& a, cudaStream_t stream) {
  const int G = a.cout_pad / 8;
  const int ty = G >= 4 ? kFcRows : kFcRows / 2, tx = 8 * (32 / G);          // block tile (first_conv1_2d_kernel)
  long long blocks = (long long)a.B * ((a.H + ty - 1) / ty) * ((a.W + tx - 1) / tx);
  if (blocks > 148LL * 8) blocks = 148LL * 8;
  if (blocks < 1) blocks = 1;
  if (G == 1) first_conv1_2d_kernel<TIN, TOUT, 1><<<(int)blocks, 256, 0, stream>>>(a);
  else if (G == 2) first_conv1_2d_kernel<TIN, TOUT, 2><<<(int)blocks, 256, 0, stream>>>(a);
  else if (G == 4) first_conv1_2d_kernel<TIN, TOUT, 4><<<(int)blocks, 256, 0, stream>>>(a);
  else first_conv1_2d_kernel<TIN, TOUT, 8><<<(int)blocks, 256, 0, stream>>>(a);
}

int launch_first_conv(const FirstConvArgs& a, cudaStream_t stream) {
  BIU_REQUIRE(a.cout_pad % 8 == 0 && a.cout_pad >= a.cout, "first_conv: cout_pad must be a multiple of 8");
  BIU_REQUIRE(a.cin >= 1 && a.cin <= 16, "first_conv: 1..16 input channels supported (got %d)", a.cin);
  const int taps = 9 * a.kd;
  const size_t smem = ((size_t)taps * a.cin * a.cout_pad + 2 * a.cout_pad) * sizeof(float);
  BIU_REQUIRE(smem <= 200 * 1024, "first_conv: weights do not fit shared memory");
  const long long work = (long long)a.B * a.D * a.H * a.W * (a.cout_pad / 8);
  long long blocks = ceil_div_ll(work, 256);
  if (blocks > 148LL * 8) blocks = 148LL * 8;
  if (blocks < 1) blocks = 1;
  const bool fast = a.cin == 1 && a.out_ctot % 8 == 0 && a.out_coff % 8 == 0 && smem <= 48 * 1024 &&
                    (a.kd == 1 || first_conv1_3d_smem(a.cout_pad) <= 100 * 1024);   // 3D: two blocks of it per SM
  const int groups = a.cout_pad / 8;
  const bool fast2d = fast && a.kd == 1 && a.D == 1 && (groups == 1 || groups == 2 || groups == 4 || groups == 8);
  long long fb = ceil_div_ll((long long)a.B * a.D * a.H * a.W, 256);
  if (fb > 148LL * 16) fb = 148LL * 16;
  if (fb < 1) fb = 1;
  long long rb3 = (long long)a.B * ((a.D + kFc3ZC - 1) / kFc3ZC) * ((a.H + kFc3Rows - 1) / kFc3Rows) *
                  ((a.W + kFc3Cols - 1) / kFc3Cols);                                   // tile columns (3D kernel)
  if (rb3 > 148LL * 2) rb3 = 148LL * 2;
  if (rb3 < 1) rb3 = 1;
  BIU_REQUIRE(a.in_kind == 0 || a.in_kind == 1, "first_conv: bad in_kind %d", a.in_kind);
  const int rc = with_elem_type(a.fmt, [&](auto out_tag) {
    using TOUT = typename decltype(out_tag)::type;
    auto run = [&](auto in_tag) -> int {
      using TIN = typename decltype(in_tag)::type;
      if (fast2d) {
        launch_first_conv1_2d<TIN, TOUT>(a, stream);
      } else if (fast && a.kd == 1) {
        first_conv1_kernel<TIN, TOUT, 9><<<(int)fb, 256, smem, stream>>>(a);
      } else if (fast) {
        static int attr_set = 0;
        const int sm3 = (int)first_conv1_3d_smem(a.cout_pad);
        if (sm3 > attr_set) {
          BIU_CHECK_CUDA(cudaFuncSetAttribute(first_conv1_3d_kernel<TIN, TOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              sm3));
          attr_set = sm3;
        }
        first_conv1_3d_kernel<TIN, TOUT><<<(int)rb3, 256, sm3, stream>>>(a);
      } else {
        if (smem > 48 * 1024)
          BIU_CHECK_CUDA(cudaFuncSetAttribute(first_conv_kernel<TIN, TOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              (int)smem));
        first_conv_kernel<TIN, TOUT><<<(int)blocks, 256, smem, stream>>>(a);
      }
      return 0;
    };
    return a.in_kind == 0 ? run(ElemTag<uint8_t>{}) : run(ElemTag<float>{});
  });
  if (rc) return rc;
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// MaxPool(k=2,s=2) (unet/unet.py:22, unet3d/unet3d.py:26) or nearest x0.5 (multi_output_unet3d.py:112):
// 16-byte vectors along the channel dim.
// ------------------------------------------------------------------------------------------------
template <typename T, int VEC>
__global__ void __launch_bounds__(256) pool2_kernel(PoolArgs a) {
  // output rows flattened over the threads, one 64-bit division per thread and 32-bit arithmetic below it;
  // consecutive threads read consecutive vectors of
  // consecutive input voxels (x = 2 ox, 2 ox + 1 are adjacent), i.e. contiguous runs of the 2 (x 2) input rows
  const bool zonly = a.mode == 2;                   // input already pooled in (y, x): reduce the z pairs
  const int oW = zonly ? a.W : a.W / 2, oH = zonly ? a.H : a.H / 2, oD = a.dims == 3 ? a.D / 2 : a.D;
  const int cv = a.c / VEC;
  const int rows = a.B * oD * oH, per_row = oW * cv;
  const T* in = reinterpret_cast<const T*>(a.in);
  T* out = reinterpret_cast<T*>(a.out);
  const int nz = (a.dims == 3 && a.mode != 1) ? 2 : 1;
  const int nyx = a.mode == 0 ? 2 : 1;
  const int xy = zonly ? 1 : 2;
  const int zs = a.dims == 3 ? 2 : 1;
  const long long i_y = (long long)a.W * a.in_ctot, i_z = (long long)a.H * a.W * a.in_ctot;
  const long long total = (long long)rows * per_row;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    {
      const int row = (int)(idx / per_row), i = (int)(idx - (long long)row * per_row);
      const int y = row % oH, bz = row / oH;
      const int z = bz % oD, b = bz / oD;
      const T* i00 = in + ((((long long)b * a.D + zs * z) * a.H + xy * y) * a.W) * a.in_ctot + a.in_coff;
      T* orow = out + (long long)row * oW * a.out_ctot + a.out_coff;
      const int x = i / cv, c = (i - x * cv) * VEC;
      float m[VEC];
#pragma unroll
      for (int k = 0; k < VEC; ++k) m[k] = -INFINITY;
      const T* ip = i00 + (long long)(xy * x) * a.in_ctot + c;
      for (int dz = 0; dz < nz; ++dz)
        for (int dy = 0; dy < nyx; ++dy)
          for (int dx = 0; dx < nyx; ++dx) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(ip + dz * i_z + dy * i_y + dx * a.in_ctot));
            const T* e = reinterpret_cast<const T*>(&q);
#pragma unroll
            for (int k = 0; k < VEC; ++k) m[k] = fmaxf(m[k], (float)e[k]);
          }
      uint4 q;
      T* e = reinterpret_cast<T*>(&q);
#pragma unroll
      for (int k = 0; k < VEC; ++k) e[k] = (T)m[k];
      *reinterpret_cast<uint4*>(orow + x * a.out_ctot + c) = q;
    }
  }
}

int launch_pool2(const PoolArgs& a, cudaStream_t stream) {
  const int vec = 16 / fmt_esz(a.fmt);
  BIU_REQUIRE(a.c % vec == 0 && a.in_ctot % vec == 0 && a.in_coff % vec == 0 && a.out_ctot % vec == 0 &&
                  a.out_coff % vec == 0,
              "pool2: channel counts must be multiples of %d", vec);
  const int oh = a.mode == 2 ? a.H : a.H / 2, ow = a.mode == 2 ? a.W : a.W / 2;
  long long blocks = ceil_div_ll((long long)a.B * (a.dims == 3 ? a.D / 2 : a.D) * oh * ow * (a.c / vec), 256);
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  if (blocks < 1) blocks = 1;
  if (int rc = with_elem_type(a.fmt, [&](auto tag) {
        using T = typename decltype(tag)::type;
        pool2_kernel<T, 16 / sizeof(T)><<<(int)blocks, 256, 0, stream>>>(a);
        return 0;
      }))
    return rc;
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// nearest x2 upsampling: out[2z+a, 2y+b, 2x+c] = in[z, y, x] (multi_output_unet3d.py:138,147,156)
// One block iteration per INPUT row: a thread reads one 16-byte channel vector and writes its 4 (2D) / 8 (3D) copies;
// consecutive threads cover consecutive vectors of consecutive voxels, so every output row receives one contiguous
// run. 32-bit index arithmetic (the output-indexed first version spent its time in 64-bit divisions: 2.6 TB/s).
template <typename T, int VEC>
__global__ void __launch_bounds__(256) up_nearest_kernel(UpNearestArgs a) {
  const int oW = a.W * 2, oH = a.H * 2;
  const int zc = a.dims == 3 ? 2 : 1, oD = a.D * zc;
  const int cv = a.c / VEC;
  const int rows = a.B * a.D * a.H, per_row = a.W * cv;
  const T* in = reinterpret_cast<const T*>(a.in);
  T* out = reinterpret_cast<T*>(a.out);
  for (int row = blockIdx.x; row < rows; row += gridDim.x) {
    const int y = row % a.H, bz = row / a.H;
    const int z = bz % a.D, b = bz / a.D;
    const T* irow = in + (long long)row * a.W * a.in_ctot + a.in_coff;
    T* o00 = out + ((((long long)b * oD + zc * z) * oH + 2 * y) * oW) * a.out_ctot + a.out_coff;
    const long long o_y = (long long)oW * a.out_ctot, o_z = (long long)oH * oW * a.out_ctot;
    for (int i = threadIdx.x; i < per_row; i += blockDim.x) {
      const int x = i / cv, c = (i - x * cv) * VEC;
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(irow + x * a.in_ctot + c));
      T* o = o00 + (long long)(2 * x) * a.out_ctot + c;
      for (int dz = 0; dz < zc; ++dz)
#pragma unroll
        for (int dy = 0; dy < 2; ++dy) {
          T* orow = o + dz * o_z + dy * o_y;
          *reinterpret_cast<uint4*>(orow) = q;
          *reinterpret_cast<uint4*>(orow + a.out_ctot) = q;
        }
    }
  }
}
int launch_up_nearest(const UpNearestArgs& a, cudaStream_t stream) {
  const int vec = 16 / fmt_esz(a.fmt);
  BIU_REQUIRE(a.c % vec == 0 && a.in_ctot % vec == 0 && a.in_coff % vec == 0 && a.out_ctot % vec == 0 &&
                  a.out_coff % vec == 0,
              "up_nearest: channel counts must be multiples of %d", vec);
  long long blocks = (long long)a.B * a.D * a.H;             // one block iteration per input row
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  if (blocks < 1) blocks = 1;
  if (int rc = with_elem_type(a.fmt, [&](auto tag) {
        using T = typename decltype(tag)::type;
        up_nearest_kernel<T, 16 / sizeof(T)><<<(int)blocks, 256, 0, stream>>>(a);
        return 0;
      }))
    return rc;
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Standalone 1x1 head + activation (unet/unet.py:50-52,104; multi_output_unet3d.py:164-168)
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) head_kernel(HeadArgs a) {
  const long long total = a.npix_per_img * a.B;
  const T* in = reinterpret_cast<const T*>(a.in);
  for (long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x; pix < total;
       pix += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(pix / a.npix_per_img);
    const long long sp = pix - (long long)b * a.npix_per_img;
    const T* src = in + pix * a.in_ctot + a.in_coff;
    for (int h = 0; h < a.head_n; ++h) {
      float s = 0.f;
      for (int c = 0; c < a.cin; ++c) s = fmaf(ld_act<T>(src + c), __ldg(a.w + h * a.cin + c), s);
      s += __ldg(a.b + h);
      float v;
      switch (a.act[h]) {
        case 1: v = 1.0f / (1.0f + expf(-s)); break;
        case 2: v = tanhf(s); break;
        case 3: v = fmaxf(s, 0.f); break;
        default: v = s;
      }
      const long long o = ((long long)b * a.head_n + h) * a.npix_per_img + sp;
      if (a.out_val) a.out_val[o] = v;
      if (a.out_u8) a.out_u8[o] = (uint8_t)(v * 255.0f);
    }
  }
}
int launch_head(const HeadArgs& a, cudaStream_t stream) {
  const long long total = a.npix_per_img * a.B;
  long long blocks = ceil_div_ll(total, 256);
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  if (blocks < 1) blocks = 1;
  if (int rc = with_elem_type(a.fmt, [&](auto tag) {
        head_kernel<typename decltype(tag)::type><<<(int)blocks, 256, 0, stream>>>(a);
        return 0;
      }))
    return rc;
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Direct convolution, fp32 accumulate on CUDA cores. Block = 64 pixels x 64 output channels, 256 threads,
// each thread 4 pixels x 4 channels; K loop over (tap, 16-channel slices) staged through shared memory.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) direct_conv_kernel(DirectConvArgs a) {
  __shared__ float As[16][64 + 4];
  __shared__ float Ws[16][64 + 4];
  const long long npix = (long long)a.B * a.D * a.H * a.W;
  const long long pix0 = (long long)blockIdx.x * 64;
  const int co0 = blockIdx.y * 64;
  const int tp = threadIdx.x & 15;        // pixel group (4 pixels: tp*4..)
  const int tc = threadIdx.x >> 4;        // channel group (4 channels: tc*4..)
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const T* in = reinterpret_cast<const T*>(a.in);

  // staging roles: thread loads A element (pixel lp, channel lc..)
  const int lp = threadIdx.x & 63;        // pixel within tile
  const int lq = threadIdx.x >> 6;        // 0..3 -> channels lq*4..lq*4+3
  const long long my_pix = pix0 + lp;
  int mx = 0, my = 0, mz = 0, mb = 0;
  if (my_pix < npix) {
    long long r = my_pix;
    mx = (int)(r % a.W); r /= a.W;
    my = (int)(r % a.H); r /= a.H;
    mz = (int)(r % a.D); r /= a.D;
    mb = (int)r;
  }
  int tap = 0;
  for (int dz = 0; dz < a.kd; ++dz)
    for (int dy = 0; dy < a.kh; ++dy)
      for (int dx = 0; dx < a.kw; ++dx, ++tap) {
        const int zz = mz + dz - (a.kd >> 1), yy = my + dy - (a.kh >> 1), xx = mx + dx - (a.kw >> 1);
        const bool inb = my_pix < npix && zz >= 0 && zz < a.D && yy >= 0 && yy < a.H && xx >= 0 && xx < a.W;
        const long long spix = (((long long)mb * a.D + zz) * a.H + yy) * a.W + xx;
        for (int c0 = 0; c0 < a.cin; c0 += 16) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int c = c0 + lq * 4 + k;
            As[lq * 4 + k][lp] = (inb && c < a.cin) ? ld_act<T>(in + spix * a.in_ctot + a.in_coff + c) : 0.f;
          }
          // weights: 16 x 64 slice; thread -> (row = tid/16, cols (tid%16)*4..+3)
          {
            const int wr = threadIdx.x >> 4, wc = (threadIdx.x & 15) * 4;
            const int c = c0 + wr;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int co = co0 + wc + k;
              Ws[wr][wc + k] = (c < a.cin && co < a.cout) ? __ldg(a.wgt + ((long long)tap * a.cin + c) * a.cout + co) : 0.f;
            }
          }
          __syncthreads();
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            float av[4], wv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) av[i] = As[k][tp * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) wv[j] = Ws[k][tc * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
          }
          __syncthreads();
        }
      }
  T* out = reinterpret_cast<T*>(a.out);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long pix = pix0 + tp * 4 + i;
    if (pix >= npix) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int co = co0 + tc * 4 + j;
      if (co >= a.cout) continue;
      float t = acc[i][j];
      t = fmaf(t, a.scale ? __ldg(a.scale + co) : 1.f, __ldg(a.shift + co));
      t = t > 0.f ? t : t * a.slope;
      st_act<T>(out + pix * a.out_ctot + a.out_coff + co, t, a.fmt == FMT_TF32);
    }
  }
}

int launch_direct_conv(const DirectConvArgs& a, cudaStream_t stream) {
  const long long npix = (long long)a.B * a.D * a.H * a.W;
  dim3 grid((unsigned)ceil_div_ll(npix, 64), (unsigned)ceil_div(a.cout, 64));
  if (int rc = with_elem_type(a.fmt, [&](auto tag) {
        direct_conv_kernel<typename decltype(tag)::type><<<grid, 256, 0, stream>>>(a);
        return 0;
      }))
    return rc;
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ConvTranspose(k=2,s=2): out[2p+q] = bias + sum_ci in[p,ci] * W[q][ci][co] (unet/unet.py:38, unet3d/unet3d.py:40-42)
template <typename T>
__global__ void __launch_bounds__(256) direct_up_kernel(DirectUpArgs a) {
  const int nq = a.dims == 3 ? 8 : 4;
  const long long npix = (long long)a.B * a.D * a.H * a.W;
  const long long total = npix * nq * a.cout;
  const T* in = reinterpret_cast<const T*>(a.in);
  T* out = reinterpret_cast<T*>(a.out);
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long r = idx;
    const int co = (int)(r % a.cout); r /= a.cout;
    const int q = (int)(r % nq); r /= nq;
    const long long pix = r;
    const int x = (int)(r % a.W); r /= a.W;
    const int y = (int)(r % a.H); r /= a.H;
    const int z = (int)(r % a.D); r /= a.D;
    const int b = (int)r;
    float s = 0.f;
    const T* src = in + pix * a.in_ctot + a.in_coff;
    const float* w = a.wgt + (long long)q * a.cin * a.cout + co;
    for (int c = 0; c < a.cin; ++c) s = fmaf(ld_act<T>(src + c), __ldg(w + (long long)c * a.cout), s);
    s += __ldg(a.bias + co);
    const int ax = q & 1, ay = (q >> 1) & 1, az = (q >> 2) & 1;
    const int oW = 2 * a.W, oH = 2 * a.H, oD = a.dims == 3 ? 2 * a.D : a.D;
    const int oz = a.dims == 3 ? 2 * z + az : z;
    const long long op = (((long long)b * oD + oz) * oH + (2 * y + ay)) * oW + (2 * x + ax);
    st_act<T>(out + op * a.out_ctot + a.out_coff + co, s, a.fmt == FMT_TF32);
  }
}
int launch_direct_up(const DirectUpArgs& a, cudaStream_t stream) {
  const long long total = (long long)a.B * a.D * a.H * a.W * (a.dims == 3 ? 8 : 4) * a.cout;
  long long blocks = ceil_div_ll(total, 256);
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  if (blocks < 1) blocks = 1;
  if (int rc = with_elem_type(a.fmt, [&](auto tag) {
        direct_up_kernel<typename decltype(tag)::type><<<(int)blocks, 256, 0, stream>>>(a);
        return 0;
      }))
    return rc;
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

}  // namespace biu
